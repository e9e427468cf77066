"""tools/profiles_cost.py -- what per-cell profiles (dfb_set_profiles) cost.

Step time: ms/step of six handles of one plane, alternating window by window in one process (best and median of the windows): two
handles that never set profiles (the first is the reference, the second a control that shows the run-to-run spread), a handle that set
profiles and cleared them again, profiles on, profiles with N2 statistics, and profiles with the mass-flux correction (DFB_FLUX_MASS);
on the reference's default plane, a batch of 8 of those, and the 1024x2048 and 4096x8192 profile planes.  The profiles are the plane's
row tables with the Reynolds stresses thickened linearly along the span, up to 1.5x at the last column.
Kernel time: profiles_kernel from torch.profiler (CUDA activities) over the profiles handle's steps in a run of its own; the bytes it must
move (filt_old 24 B/cell and the constants 56 B/cell read, u', v', w', T', rho' 40 B/cell written: 120 B/cell) over the kernel time,
against the 7.7 TB/s of the B200 data sheet.
Prints the device name and power limit, and writes a JSON record (default profiles/profiles_cost.json).

    python tools/profiles_cost.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from time_scales_cost import WORKLOADS, gpu_identity, plane_of, summary  # noqa: E402

HANDLES = ("never", "control", "cleared", "profiles", "profiles_n2", "profiles_flux")
HBM_TBS = 7.7
BYTES_PER_CELL = 120


def cells_for(d):
    rows = d.rows()
    Nz = d.info(5)
    f = 1.0 + 0.5 * np.arange(Nz) / Nz
    cells = np.repeat(rows[:, :, None], Nz, axis=2)
    cells[:4] *= f[None, None, :]
    return cells


def make(dfb, pl, nplanes, which):
    d = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=1), fetch=False, nplanes=nplanes)
    if which in ("never", "control"):
        return d
    d.set_profiles(cells_for(d))
    if which == "cleared":
        d.set_profiles(None)
    if which == "profiles_n2":
        d.stats_enable(True)
    if which == "profiles_flux":
        d.set_flux_correction(dfb.FLUX_MASS)
    return d


def kernel_us(d, dt, n):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(5):
        d.filter(dt)
    d.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            d.filter(dt)
        d.sync()
    for e in prof.key_averages():
        if "profiles_kernel" in e.key:
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            return t / max(e.count, 1)
    return 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "profiles_cost.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    import _dfb_import  # noqa: F401
    import digital_filtering_b200 as dfb
    name, smi = gpu_identity(torch)
    print("device:", name, "|", smi)
    rec = dict(device=name, nvidia_smi=smi, reps=args.reps,
               method="ms/step: CUDA events around n steps per window on each handle's own stream (fetch=False), ended by a "
                      "synchronise; the six handles alternate window by window; best and median of the windows.  kernel_us: "
                      "torch.profiler CUDA activities over the profiles handle's steps, mean per launch.  hbm_fraction: 120 B/cell "
                      "/ kernel time / 7.7 TB/s (data sheet).",
               workloads={})
    for wname, nplanes, dt, n in WORKLOADS:
        pl = plane_of(wname)
        h = {s: make(dfb, pl, nplanes, s) for s in HANDLES}
        st = {s: torch.cuda.ExternalStream(d.stream()) for s, d in h.items()}

        def window(s, k):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st[s])
            for _ in range(k):
                h[s].filter(dt)
            b.record(st[s])
            h[s].sync()
            return a.elapsed_time(b) / k

        for s in h:
            window(s, max(20, n // 10))                                 # warm-up
        ms = {s: [] for s in h}
        for _ in range(args.reps):
            for s in h:
                ms[s].append(window(s, n))
        r = dict(planes=nplanes, steps_per_window=n, **summary(ms))
        r["best_vs_never"] = {s: r["best"][s] / r["best"]["never"] for s in HANDLES}
        r["control_range"] = [min(ms["control"]), max(ms["control"])]
        cells = nplanes * h["profiles"].Ny * h["profiles"].Nz
        k = kernel_us(h["profiles"], dt, max(20, min(n, 200)))
        r["kernel_us"] = k
        r["hbm_fraction"] = BYTES_PER_CELL * cells / (k * 1e-6) / (HBM_TBS * 1e12) if k > 0 else None
        rec["workloads"][wname] = r
        print("%-24s ms/step never %.4f control %.4f cleared %.4f profiles %.4f (x%.3f) +N2 %.4f (x%.3f) +flux %.4f (x%.3f)  "
              "kernel %.2f us, HBM %.3f" %
              (wname, r["best"]["never"], r["best"]["control"], r["best"]["cleared"], r["best"]["profiles"], r["best_vs_never"]["profiles"],
               r["best"]["profiles_n2"], r["best_vs_never"]["profiles_n2"], r["best"]["profiles_flux"], r["best_vs_never"]["profiles_flux"],
               k, r["hbm_fraction"] or 0.0))
        print("    windows:", {s: [round(x, 4) for x in v] for s, v in ms.items()})
        for d in h.values():
            d.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
