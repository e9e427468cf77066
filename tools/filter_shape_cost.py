"""tools/filter_shape_cost.py -- what the Gaussian filter shape (dfb_set_filter_shape) costs: ms/step of an exponential and a Gaussian
handle of the same plane, alternating window by window in one process (best and median of the windows), and the per-kernel times of
each (timing mode: CUDA events around the noise, the y-sweep and the z-sweep of every step, the least over the steps), on the
reference's default plane, a batch of 8 of those, and the 1024x2048 and 4096x8192 profile planes.  The sweeps' share of the fp64 roof
is their useful multiply-adds (the taps sum_cells (2N + 1) of their direction) over the DFMA peak dfb_measure_fp64_peak measures in the
same run.  Prints the device name and power limit, and writes a JSON record (default profiles/filter_shape_cost.json).

    python tools/filter_shape_cost.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from time_scales_cost import WORKLOADS, gpu_identity, plane_of, summary  # noqa: E402

SHAPES = ("exponential", "gaussian")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "filter_shape_cost.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    import _dfb_import  # noqa: F401
    import digital_filtering_b200 as dfb
    name, smi = gpu_identity(torch)
    print("device:", name, "|", smi)
    peak_tflops, mhz = dfb.measure_fp64_peak(0)
    print("measured DFMA peak %.2f TFLOP/s (%.0f MHz at 64 DFMA/clk/SM)" % (peak_tflops, mhz))
    rec = dict(device=name, nvidia_smi=smi, reps=args.reps, fp64_peak_tflops=peak_tflops,
               method="ms/step: CUDA events around n steps per window on each handle's own stream (fetch=False), ended by a "
                      "synchronise; the two handles alternate window by window; best and median of the windows.  kernels_us: timing "
                      "mode (dfb_set_timing), CUDA events between the step's noise, y-sweep and z-sweep launches on the main stream "
                      "(no look-ahead noise), least over the steps of one window.  roof: useful multiply-adds of the sweep "
                      "(sum over fields, planes and cells of 2N+1 in its direction) x 2 flop over the measured DFMA peak, over the "
                      "kernel time; the executed multiply-adds (padding of band matrices and lane windows) are not counted.",
               workloads={})
    for wname, nplanes, dt, n in WORKLOADS:
        pl = plane_of(wname)
        h = {s: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=1, filter_shape=i), fetch=False, nplanes=nplanes)
             for i, s in enumerate(SHAPES)}
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
        r["best_gaussian_vs_exponential"] = r["best"]["gaussian"] / r["best"]["exponential"]
        r["forms"], r["kernels_us"], r["roof"] = {}, {}, {}
        for s, d in h.items():
            r["forms"][s] = dict(tuned=d.info(3), z_form=d.info(7), y_form=d.info(10))
            taps = [nplanes * sum(int((2 * d.half_widths(f, di) + 1).sum()) for f in range(3)) for di in (0, 1)]
            d.set_timing(True)
            best = [1e30] * 3
            for _ in range(max(20, n // 10)):
                d.filter(dt)
                t = d.last_ms()
                best = [min(best[i], t[k]) for i, k in enumerate(("noise", "ysweep", "zsweep_epilogue"))]
            d.set_timing(False)
            r["kernels_us"][s] = dict(noise=1e3 * best[0], y_sweep=1e3 * best[1], z_sweep=1e3 * best[2])
            r["roof"][s] = dict(y_sweep=2.0 * taps[0] / (best[1] * 1e-3) / (peak_tflops * 1e12),
                                z_sweep=2.0 * taps[1] / (best[2] * 1e-3) / (peak_tflops * 1e12), taps_y=taps[0], taps_z=taps[1])
        rec["workloads"][wname] = r
        print("%-24s ms/step exp %.4f gauss %.4f (x%.3f)  y-sweep us exp %.1f gauss %.1f  z-sweep us exp %.1f gauss %.1f  "
              "roof gauss y %.2f z %.2f" %
              (wname, r["best"]["exponential"], r["best"]["gaussian"], r["best_gaussian_vs_exponential"],
               r["kernels_us"]["exponential"]["y_sweep"], r["kernels_us"]["gaussian"]["y_sweep"],
               r["kernels_us"]["exponential"]["z_sweep"], r["kernels_us"]["gaussian"]["z_sweep"],
               r["roof"]["gaussian"]["y_sweep"], r["roof"]["gaussian"]["z_sweep"]))
        for d in h.values():
            d.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
