"""tools/corr_cost.py -- what the correlation statistics (dfb_corr_enable) cost per step, and the integral scales they measure.

Production ms/step of handles that alternate in one process: never enabled, enabled then switched off, z only, y only, t only
(L_t = 8), all on -- z and y at the filter's full support -- and a second never-enabled handle as the control of the spread, on the headline plane, the reference's default plane (alone and as a
batch of 8) and the 4096x8192 plane.  Per-kernel times from torch.profiler (a separate pass after the timed windows) and their share
of the roof: the FMAs of the products that count (include/dfb200.h) over the fp64 rate measured in the same run, the bytes of the
temporal pass over 6 453 GB/s.  Then the integral scales the headline plane delivers against the configured Iz and Lt.
Records the device name and power limit; writes a JSON record (default profiles/corr_cost.json).

    python tools/corr_cost.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import _dfb_import  # noqa: E402,F401
import digital_filtering_b200 as dfb  # noqa: E402
from digital_filtering_b200 import workloads as W  # noqa: E402
from oracle.oracle import stored_default_plane  # noqa: E402

HBM_GBS = 6453.0      # DESIGN.md section 5
S = dfb.DFB_CORR_SUPPORT
WORKLOADS = [  # name, plane, planes per handle, dt, timed steps per window
    ("1024x2048_profile_N128", lambda: W.NAMED["1024x2048_profile_N128"](), 1, 1e-7, 200),
    ("default_510x400", stored_default_plane, 1, 1e-5, 200),
    ("default_510x400_batch8", stored_default_plane, 8, 1e-5, 100),
    ("4096x8192_profile_N128", lambda: W.NAMED["4096x8192_profile_N128"](), 1, 1e-7, 30),
]
# never2: a second never-enabled handle, created last, is the control -- how far two identical handles differ from each other
MODES = [("never", None), ("off", "off"), ("z", (S, 0, 0)), ("y", (0, S, 0)), ("t8", (0, 0, 8)), ("all", (S, S, 8)), ("never2", None)]


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip()
    except Exception as e:               # the measurement still stands; the record says what could not be read
        smi = "nvidia-smi unavailable: %s" % e
    return name, smi


def window(df, st, dt, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(n):
        df.filter(dt)
    b.record(st)
    df.sync()
    return a.elapsed_time(b) / n


def work(df, nplanes):
    """useful FMAs of the z and y products and bytes of the temporal pass (steady state, L_t lags) per step"""
    Lz, Ly, Lt = df.corr_lags
    Ny, Nz, P = df.Ny, df.Nz, nplanes
    fz = 3 * P * Ny * sum((Nz if df.periodic_z else Nz - d) for d in range(Lz + 1))
    fy = 3 * P * Nz * sum(Ny - d for d in range(Ly + 1))
    bt = 3 * P * Ny * Nz * 8 * (Lt + 2) if Lt else 0        # f read, L_t ring slots read, one written
    return fz, fy, bt


def kernel_times(df, dt, n):
    from torch.profiler import ProfilerActivity, profile
    df.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            df.filter(dt)
        df.sync()
    out = {}
    for ev in prof.key_averages():
        if "corr_" in ev.key:
            key = ev.key.split("corr_")[1].split("_kernel")[0]
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            out[key] = out.get(key, 0.0) + t / 1e3 / n          # ms per step
    return out


def scales(dt=1e-7, steps=400):
    """integral scales of the headline plane against the configured ones (row medians over the rows with n = N_z/2 >= 4)"""
    plane = W.NAMED["1024x2048_profile_N128"]()
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=11), fetch=False)
    df.corr_enable(S, S, 64)
    for _ in range(steps):
        df.filter(dt)
    yc = df.table(8)
    Lt = df.table(10)
    sc = np.asarray(plane["scales"])
    rec = dict(steps=steps, dt=dt, lags=df.corr_lags, fields={})
    vz = df.table(13, n=plane["Nz"] + 1)
    wbar = (vz[-1] - vz[0]) / plane["Nz"]
    for f in range(3):
        Iz = sc[f, 0] + (sc[f, 1] - sc[f, 0]) * 0.5 * (1 + np.tanh((yc / plane["d_i"] - 0.2) / 0.03))
        nz = df.half_widths(f, 1)[:, 0] // 2
        ny = df.half_widths(f, 0)[:, 0] // 2
        keep = nz >= 4
        Lz, Ly, Ltm = (df.integral_scales(f, d) for d in range(3))
        rec["fields"]["uvw"[f]] = dict(
            rows=int(keep.sum()),
            z_over_n_cells=float(np.nanmedian(Lz[keep] / (nz[keep] * wbar))),
            z_over_Iz=float(np.nanmedian(Lz[keep] / Iz[keep])),
            y_over_n_cells=float(np.nanmedian(Ly[keep & (ny >= 4)] / (ny[keep & (ny >= 4)] * plane["dy"][keep & (ny >= 4)]))),
            y_over_067Iz=float(np.nanmedian(Ly[keep] / (0.67 * Iz[keep]))),
            t_over_Lt=float(np.nanmedian(Ltm[keep] * dt / Lt[f])))
        print("scales %s: Lz/(n dz) %.3f  Lz/Iz %.3f  Ly/(n dy) %.3f  Ly/(0.67 Iz) %.3f  Lt_meas/Lt %.3f" % (
            "uvw"[f], *[rec["fields"]["uvw"[f]][k] for k in ("z_over_n_cells", "z_over_Iz", "y_over_n_cells", "y_over_067Iz", "t_over_Lt")]))
    df.close()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "corr_cost.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    name, smi = gpu_identity()
    tflops, _ = dfb.measure_fp64_peak(0)
    print("device:", name, "|", smi, "| fp64 DFMA peak %.1f TFLOP/s" % tflops)
    rec = dict(device=name, nvidia_smi=smi, fp64_tflops_measured=tflops, hbm_gbs_roof=HBM_GBS, reps=args.reps,
               method="CUDA events around n production steps (fetch=False) on each handle's stream; the handles of a workload alternate "
                      "window by window; best and median of the windows.  Kernel times: torch.profiler over a separate pass.  Shares: "
                      "useful FMAs / kernel time / (measured fp64 rate / 2); temporal bytes / kernel time / HBM roof", workloads={})
    for wname, mk, nplanes, dt, n in WORKLOADS:
        plane = mk()
        h, st = {}, {}
        for mode, lags in MODES:
            h[mode] = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1), fetch=False, nplanes=nplanes)
            if lags == "off":
                h[mode].corr_enable(S, S, 8)
                h[mode].corr_enable(on=False)
            elif lags is not None:
                h[mode].corr_enable(*lags)
            st[mode] = torch.cuda.ExternalStream(h[mode].stream())
            window(h[mode], st[mode], dt, max(10, n // 10))          # warm-up
        ms = {m: [] for m, _ in MODES}
        for _ in range(args.reps):
            for m, _ in MODES:
                ms[m].append(window(h[m], st[m], dt, n))
        r = dict(planes=nplanes, steps_per_window=n, lags_all=h["all"].corr_lags, ms=ms,
                 best={m: min(v) for m, v in ms.items()}, median={m: sorted(v)[len(v) // 2] for m, v in ms.items()})
        kt = kernel_times(h["all"], dt, max(5, n // 10))
        fz, fy, bt = work(h["all"], nplanes)
        zt = kt.get("z", 0.0) + (kt.get("reduce", 0.0) if "z" in kt and "y" not in kt else 0.0)
        r["kernel_ms"] = kt
        r["useful_fma"] = dict(z=fz, y=fy)
        r["temporal_bytes"] = bt
        r["share_of_roof"] = dict(z=fz / (kt["z"] * 1e-3) / (tflops * 0.5e12) if kt.get("z") else None,
                                  y=fy / (kt["y"] * 1e-3) / (tflops * 0.5e12) if kt.get("y") else None,
                                  t=bt / (kt["t"] * 1e-3) / (HBM_GBS * 1e9) if kt.get("t") else None)
        rec["workloads"][wname] = r
        print("%-24s " % wname + "  ".join("%s %.4f" % (m, r["best"][m]) for m, _ in MODES) + " ms/step (best of %d)" % args.reps)
        print("%-24s kernels %s ms/step; share of roof %s" % ("", {k: round(v, 4) for k, v in kt.items()},
                                                              {k: (round(v, 3) if v else v) for k, v in r["share_of_roof"].items()}))
        for m, _ in MODES:
            h[m].close()
        torch.cuda.empty_cache()
    rec["integral_scales_1024x2048"] = scales()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
