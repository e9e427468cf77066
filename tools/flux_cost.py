"""tools/flux_cost.py -- what the inflow mass-flux correction (dfb_set_flux_correction) costs and what it does.

Step time: ms/step of four handles of one plane, alternating window by window in one process (best and median of the windows): a control
that never enabled the correction, a handle that enabled it and switched it off again, DFB_FLUX_MASS, and DFB_FLUX_MASS with N2 statistics
on; on the reference's default plane, a batch of 8 of those, and the 1024x2048 and 4096x8192 profile planes.
Kernel times: flux_rows_kernel and flux_apply_kernel from torch.profiler (CUDA activities) over the mass handle's steps in a run of their
own; the bytes they must move (rows: u' 8 B/cell; apply: u' read and u', T', rho' written, 32 B/cell) over the kernel time, against the
7.7 TB/s of the B200 data sheet.
Physics (default plane and 1024x2048 profile, 400 steps): the rms over the steps of m'_p / mean flux before the correction (what an
uncorrected handle delivers: filt_old and so the z-sweep's u' do not depend on the mode) and of the delivered sum A g u' / mean after it,
and the per-row ratio of the delivered R11 (N2 sums of u'^2 over the plane's row) with the correction to an uncorrected twin's.
Prints the device name and power limit, and writes a JSON record (default profiles/flux_cost.json).

    python tools/flux_cost.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from time_scales_cost import WORKLOADS, gpu_identity, plane_of, summary  # noqa: E402

HANDLES = ("control", "off", "mass", "mass_n2")
HBM_TBS = 7.7
PHYSICS = (("default_510x400", 1e-5), ("1024x2048_profile_N128", 1e-7))


def make(dfb, pl, nplanes, which):
    d = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=1), fetch=False, nplanes=nplanes)
    if which != "control":
        d.set_flux_correction(dfb.FLUX_MASS)
    if which == "off":
        d.set_flux_correction(dfb.FLUX_OFF)
    if which == "mass_n2":
        d.stats_enable(True)
    return d


def kernel_us(torch, d, dt, n):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(5):
        d.filter(dt)
    d.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            d.filter(dt)
        d.sync()
    out = {}
    for e in prof.key_averages():
        for k in ("flux_rows_kernel", "flux_apply_kernel"):
            if k in e.key:
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                out[k] = t / max(e.count, 1)
    return out


def physics(dfb, pl, dt, steps=400):
    a, b = (dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=3), fetch=False) for _ in range(2))
    a.set_flux_correction(dfb.FLUX_MASS)
    for d in (a, b):
        d.stats_enable(True)
    Ny, Nz = a.Ny, a.Nz
    Ms, rhos = a.table(7), a.table(6)
    w = ((rhos * (1.0 + 0.2 * Ms * Ms)) * np.diff(a.table(12, n=Ny + 1)))[:, None] * np.diff(a.table(13, n=Nz + 1))[None, :]
    before, after = [], []
    for s in range(steps):
        a.filter(dt)
        b.filter(dt)
        c, m, mean = a.flux_info(0)
        before.append(m / mean)
        if s % 10 == 0:
            after.append(float((w * a.get(0)).sum()) / mean)
    Ra, Rb = a.stats(0)[0].sum(1), b.stats(0)[0].sum(1)
    ratio = np.where(Rb > 0, Ra / np.where(Rb > 0, Rb, 1.0), 1.0)
    r = dict(steps=steps, dt=dt, rms_mflux_over_mean_uncorrected=float(np.sqrt(np.mean(np.square(before)))),
             max_abs_mflux_over_mean_uncorrected=float(np.max(np.abs(before))),
             rms_mflux_over_mean_corrected=float(np.sqrt(np.mean(np.square(after)))),
             R11_ratio_per_row=ratio.tolist(), R11_ratio_min=float(ratio.min()), R11_ratio_max=float(ratio.max()),
             R11_ratio_mean=float(ratio.mean()))
    a.close()
    b.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "flux_cost.json"))
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
                      "synchronise; the four handles alternate window by window; best and median of the windows.  kernels_us: "
                      "torch.profiler CUDA activities over the mass handle's steps, mean per launch.  hbm_fraction: bytes the kernel "
                      "must move (rows 8 B/cell, apply 32 B/cell) / kernel time / 7.7 TB/s (data sheet).",
               workloads={}, physics={})
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
        r["best_vs_control"] = {s: r["best"][s] / r["best"]["control"] for s in HANDLES}
        r["control_spread"] = (max(ms["control"]) - min(ms["control"])) / min(ms["control"])
        cells = nplanes * h["mass"].Ny * h["mass"].Nz
        k = kernel_us(torch, h["mass"], dt, max(20, min(n, 200)))
        r["kernels_us"] = k
        r["hbm_fraction"] = {kk: (8 if "rows" in kk else 32) * cells / (v * 1e-6) / (HBM_TBS * 1e12) for kk, v in k.items() if v > 0}
        rec["workloads"][wname] = r
        print("%-24s ms/step control %.4f off %.4f mass %.4f mass+N2 %.4f (x%.3f, x%.3f)  control spread %.3f  kernels us %s  HBM %s" %
              (wname, r["best"]["control"], r["best"]["off"], r["best"]["mass"], r["best"]["mass_n2"], r["best_vs_control"]["mass"],
               r["best_vs_control"]["mass_n2"], r["control_spread"], {kk: round(v, 2) for kk, v in k.items()},
               {kk: round(v, 3) for kk, v in r["hbm_fraction"].items()}))
        for d in h.values():
            d.close()
    for wname, dt in PHYSICS:
        p = physics(dfb, plane_of(wname), dt)
        rec["physics"][wname] = p
        print("%-24s rms m'/mean: uncorrected %.3e, corrected %.3e; delivered R11 ratio per row: min %.4f mean %.4f max %.4f" %
              (wname, p["rms_mflux_over_mean_uncorrected"], p["rms_mflux_over_mean_corrected"], p["R11_ratio_min"], p["R11_ratio_mean"],
               p["R11_ratio_max"]))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
