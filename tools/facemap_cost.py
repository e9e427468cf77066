"""tools/facemap_cost.py -- what the face maps of the CFD hand-off (dfb_facemap_create, dfb_interp_to_cells, dfb_interp_to_host) cost.

On the 1024x2048 profile plane:
  - apply time of dfb_interp_to_cells (all five fields, mean given, scale 1, a permuted dst_index) from CUDA events on the handle's
    stream, and its share of the 6 453 GB/s HBM roof by the bytes the kernel must move: the taps (POINT 48 B per face; AREA 4 B of CSR
    pointer + 12 B per tap), dst_index, five means read, five values written, and five fields read once per distinct cell the map
    touches.  Maps: POINT one face per cell (centres moved off the cell centres: four taps each), AREA faces of 2x2 cells, POINT 10^4
    random faces.  The working set of the full-plane maps (> 300 MB) does not fit the 126 MB L2;
  - dfb_interp_to_host after a step against dfb_filter_to_host into page-locked arrays, for the same faces (host clock, synchronous);
  - ms/step of a handle with three maps alive against a handle without, alternating windows in one process.
Records the device name and power limit; writes a JSON record (default profiles/facemap_cost.json).

    python tools/facemap_cost.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import _dfb_import  # noqa: E402,F401
import digital_filtering_b200 as dfb  # noqa: E402
from digital_filtering_b200 import workloads as W  # noqa: E402

HBM_GBS = 6453.0      # DESIGN.md section 5
PLANE = "1024x2048_profile_N128"
DT = 1e-7


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip()
    except Exception as e:               # the measurement still stands; the record says what could not be read
        smi = "nvidia-smi unavailable: %s" % e
    return name, smi


def face_sets(df, rng):
    Ny, Nz = df.Ny, df.Nz
    yc, vy, vz = df.table(8), df.table(12, n=Ny + 1), df.table(13, n=Nz + 1)
    zc = 0.5 * (vz[1:] + vz[:-1])
    # POINT, one face per cell, 0.37 of the way to the next centre in y and z: four taps of nonzero weight
    ym = np.r_[yc[:-1] + 0.37 * np.diff(yc), yc[-1]]
    zm = np.r_[zc[:-1] + 0.37 * np.diff(zc), zc[-1]]
    jj, kk = np.meshgrid(np.arange(Ny), np.arange(Nz), indexing="ij")
    point = dict(yf=ym[jj.ravel()], zf=zm[kk.ravel()])
    # AREA, faces of 2x2 cells
    j2, k2 = np.meshgrid(np.arange(0, Ny - 1, 2), np.arange(0, Nz - 1, 2), indexing="ij")
    j2, k2 = j2.ravel(), k2.ravel()
    area = dict(yf=0.5 * (vy[j2] + vy[j2 + 2]), zf=0.5 * (vz[k2] + vz[k2 + 2]), hy=vy[j2 + 2] - vy[j2], hz=vz[k2 + 2] - vz[k2])
    n = 10000
    rand = dict(yf=rng.uniform(yc[0], yc[-1], n), zf=rng.uniform(zc[0], zc[-1], n))
    return {"point_per_cell": (point, 4, Ny * Nz), "area_2x2": (area, 4, Ny * Nz), "point_random_1e4": (rand, 4, 4 * n)}


def bytes_moved(name, n, taps_per_face, cells):
    taps = (48 * n) if name.startswith("point") else (4 * (n + 1) + 12 * taps_per_face * n)
    return taps + 4 * n + 5 * 8 * n * 2 + 5 * 8 * cells


def apply_ms(fm, args, st, reps, n_apply):
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(n_apply):
            fm.to_cells(*args)
        b.record(st)
        b.synchronize()
        out.append(a.elapsed_time(b) / n_apply)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "facemap_cost.json"))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    name, smi = gpu_identity()
    rng = np.random.default_rng(0)
    plane = W.NAMED[PLANE]()
    dev = torch.device("cuda", 0)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=5, device=0), fetch=False)
    for _ in range(5):
        df.filter(DT)
    df.sync()
    st = torch.cuda.ExternalStream(df.stream())
    rec = dict(device=name, nvidia_smi=smi, plane=PLANE, Ny=df.Ny, Nz=df.Nz, hbm_gbs=HBM_GBS, maps={})
    host5 = [torch.zeros((df.Ny, df.Nz), dtype=torch.float64).pin_memory().numpy() for _ in range(5)]   # page-locked, as bench.py's e2e leg
    for key, (f, tpf, cells) in face_sets(df, rng).items():
        t0 = time.perf_counter()
        fm = df.facemap(**f)
        t_create = time.perf_counter() - t0
        n = fm.n
        dst = [torch.zeros(n * 1, dtype=torch.float64, device=dev) for _ in range(5)]
        mean = [torch.rand(n, dtype=torch.float64, device=dev) for _ in range(5)]
        perm = torch.as_tensor(rng.permutation(n).astype(np.int32), device=dev) if key.startswith("point_random") else \
            torch.arange(n, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        args = (dst, perm, mean, None)
        for _ in range(20):
            fm.to_cells(*args)
        n_apply = 200 if n > 100000 else 2000
        ms = apply_ms(fm, args, st, a.reps, n_apply)
        by = bytes_moved(key, n, tpf, cells)
        med = float(np.median(ms))
        # host delivery: one step + the faces to the host, against one step + the five whole fields to pinned host arrays
        out = np.zeros((5, n))
        th, tf = [], []
        for _ in range(a.reps):
            for _ in range(3):
                df.filter(DT); fm.to_host(out=out)
            df.sync()
            t0 = time.perf_counter()
            for _ in range(20):
                df.filter(DT)
                fm.to_host(out=out)
            th.append((time.perf_counter() - t0) / 20 * 1e3)
            t0 = time.perf_counter()
            for _ in range(20):
                dfb._check(dfb.lib().dfb_filter_to_host(df._h, DT, *[h.ctypes.data for h in host5]))
            tf.append((time.perf_counter() - t0) / 20 * 1e3)
        rec["maps"][key] = dict(faces=n, create_s=t_create, apply_ms=ms, apply_ms_median=med, bytes=by, gbs=by / (med * 1e-3) / 1e9,
                                hbm_roof_fraction=by / (med * 1e-3) / 1e9 / HBM_GBS,
                                step_plus_to_host_ms=float(np.median(th)), step_plus_filter_to_host_ms=float(np.median(tf)))
        print("%-18s faces %8d  apply %.4f ms  %.0f GB/s  roof %.2f  | step+to_host %.3f ms  step+filter_to_host %.3f ms" % (
            key, n, med, by / (med * 1e-3) / 1e9, by / (med * 1e-3) / 1e9 / HBM_GBS, np.median(th), np.median(tf)))
        fm.close()
    df.close()

    # step time with maps alive on the handle, against a control handle without, alternating windows
    hs = {k: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=5, device=0), fetch=False) for k in ("maps", "control")}
    alive = [hs["maps"].facemap(**f) for (f, _, _) in face_sets(hs["maps"], rng).values()]
    times = {k: [] for k in hs}
    for d in hs.values():
        for _ in range(20):
            d.filter(DT)
        d.sync()
    for _ in range(a.reps):
        for k, d in hs.items():
            s = torch.cuda.ExternalStream(d.stream())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            for _ in range(200):
                d.filter(DT)
            e1.record(s)
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / 200)
    rec["step_ms"] = {k: dict(windows=v, median=float(np.median(v))) for k, v in times.items()}
    print("step ms/step: maps alive %.4f  control %.4f" % (rec["step_ms"]["maps"]["median"], rec["step_ms"]["control"]["median"]))
    for m in alive:
        m.close()
    for d in hs.values():
        d.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
