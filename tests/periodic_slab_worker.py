"""tests/periodic_slab_worker.py -- one rank of the 2-GPU periodic slab test (launched by tests/test_periodic_z.py through
torch.distributed.run): parallel.SlabFilter over spanwise-periodic slabs (dfb_config.periodic_z = 1; the edge slabs regenerate their
wrapped neighbour columns locally, no exchange); rank 0 checks every gathered field of every step, bit for bit, against the
periodic plane filtered whole on its own GPU."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import _dfb_import  # noqa: E402,F401
import digital_filtering_b200 as dfb  # noqa: E402
from digital_filtering_b200 import parallel as P, workloads as W  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")
    plane = W.plane_profile(64, 1400, 16, 24)
    mk = lambda k0, k1: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, device=local, k_begin=k0, k_end=k1, periodic_z=1),
                                           fetch=False)
    sf = P.SlabFilter(dist, plane["Nz"], mk)
    dts = [2e-7, 1e-7]
    got = []
    sf.gather()
    got.append([sf.plane(w) for w in range(5)])
    for dt in dts:
        sf.filter(dt)
        sf.gather()
        got.append([sf.plane(w) for w in range(5)])
    ok = True
    if rank == 0:
        whole = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=3, device=local, periodic_z=1))
        for s in range(len(dts) + 1):
            if s:
                whole.filter(dts[s - 1])
            ref = [whole.u.fluc, whole.v.fluc, whole.w.fluc, whole.T_fluc, whole.rho_fluc]
            for w in range(5):
                ok &= bool(np.array_equal(got[s][w], ref[w]))
        whole.close()
    flag = torch.tensor([1.0 if ok else 0.0])
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    sf.filt.close()
    dist.destroy_process_group()
    if rank == 0:
        print("PERIODIC_SLAB_OK" if flag.item() == 1.0 else "PERIODIC_SLAB_FAIL")
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
