"""Restart files across GPUs (needs >= 2 B200 in the box; skipped on a one-GPU box): two ranks, one process per GPU, each save their
slab of one plane into one file on a shared path; after the barrier one rank resumes the whole plane from it, bitwise."""
import os
import socket
import subprocess
import sys

import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_two_ranks_save_one_file_and_one_rank_resumes(dfb, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    env = dict(os.environ, DFB_RESTART_TEST_FILE=str(tmp_path / "slabs.dfbr"))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "restart_slab_worker.py")],
                       capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0 and "RESTART_SLABS_OK 2" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])
