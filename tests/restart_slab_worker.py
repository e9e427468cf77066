"""tests/restart_slab_worker.py -- one rank of the 2-GPU restart test (launched by tests/test_restart_multi_gpu.py through
torch.distributed.run): every rank filters its spanwise slab of one plane on its own GPU for n steps and saves it into ONE restart file
on a shared path; after the barrier rank 0 alone loads the file into a whole-plane handle and checks its next n steps, bit for bit,
against the same plane filtered whole without interruption."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import _dfb_import  # noqa: E402,F401
import digital_filtering_b200 as dfb  # noqa: E402
from digital_filtering_b200 import workloads as W  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    path = os.environ["DFB_RESTART_TEST_FILE"]
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    plane = W.plane_profile(64, 400, 16, 24)
    k0, k1 = plane["Nz"] * rank // world, plane["Nz"] * (rank + 1) // world
    dts = [2e-7, 1e-7, 0.0, 3e-7, 5e-8, 1e-7]
    n = 3
    slab = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, device=local, k_begin=k0, k_end=k1), fetch=False)
    for dt in dts[:n]:
        slab.filter(dt)
    slab.save_restart(path)
    slab.close()
    dist.barrier()                                  # every writer has returned: the file is complete
    ok = True
    if rank == 0:
        which = (dfb.U_FLUC, dfb.V_FLUC, dfb.W_FLUC, dfb.T_FLUC, dfb.RHO_FLUC, dfb.U_FILT, dfb.V_FILT, dfb.W_FILT)
        ref = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, device=local), fetch=False)
        got = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, device=local), fetch=False)
        for dt in dts[:n]:
            ref.filter(dt)
        assert dfb.restart_info(path)["records"] == world
        got.load_restart(path)
        for dt in dts[n:]:
            ref.filter(dt)
            got.filter(dt)
            ok &= all(np.array_equal(ref.get(w), got.get(w)) for w in which)
        ref.close()
        got.close()
    flag = torch.tensor([1.0 if ok else 0.0])
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if rank == 0:
        print("RESTART_SLABS_OK" if flag.item() == 1.0 else "RESTART_SLABS_FAIL", world)
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
