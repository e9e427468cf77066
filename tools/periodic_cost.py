"""tools/periodic_cost.py -- production ms/step with periodic_z off and on (dfb_config.periodic_z), the two handles of a workload
alternating in one process, on the headline plane, the reference's default plane (alone and as a batch of 8) and the 4096x8192
plane.  Prints the device name and power limit, and writes a JSON record (default profiles/periodic_cost.json).

    python tools/periodic_cost.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import _dfb_import  # noqa: E402,F401
import digital_filtering_b200 as dfb  # noqa: E402
from digital_filtering_b200 import workloads as W  # noqa: E402
from oracle.oracle import stored_default_plane  # noqa: E402

WORKLOADS = [  # name, plane, planes per handle, dt, timed steps per window
    ("1024x2048_profile_N128", lambda: W.NAMED["1024x2048_profile_N128"](), 1, 1e-7, 400),
    ("default_510x400", stored_default_plane, 1, 1e-5, 400),
    ("default_510x400_batch8", stored_default_plane, 8, 1e-5, 200),
    ("4096x8192_profile_N128", lambda: W.NAMED["4096x8192_profile_N128"](), 1, 1e-7, 60),
]


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "periodic_cost.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    name, smi = gpu_identity()
    print("device:", name, "|", smi)
    rec = dict(device=name, nvidia_smi=smi, reps=args.reps, method="CUDA events around n production steps (fetch=False) on the "
               "handle's stream; off / on windows alternate; best and median of the windows", workloads={})
    for wname, mk, nplanes, dt, n in WORKLOADS:
        plane = mk()
        h = {p: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1, periodic_z=p), fetch=False, nplanes=nplanes) for p in (0, 1)}
        st = {p: torch.cuda.ExternalStream(h[p].stream()) for p in (0, 1)}
        for p in (0, 1):
            window(h[p], st[p], dt, max(20, n // 10))                # warm-up
        ms = {0: [], 1: []}
        for _ in range(args.reps):
            for p in (0, 1):
                ms[p].append(window(h[p], st[p], dt, n))
        r = dict(planes=nplanes, steps_per_window=n, y_form=[h[p].info(10) for p in (0, 1)],
                 ms_off=ms[0], ms_on=ms[1], best_off=min(ms[0]), best_on=min(ms[1]),
                 median_off=sorted(ms[0])[len(ms[0]) // 2], median_on=sorted(ms[1])[len(ms[1]) // 2])
        r["ratio_best"] = r["best_on"] / r["best_off"]
        M = max(h[0].info(1, f) for f in range(3))
        r["extra_columns_estimate"] = 2 * M / plane["Nz"]             # noise + y-sweep columns added by the wrap, whole plane
        rec["workloads"][wname] = r
        print("%-24s off %.4f  on %.4f ms/step (best of %d; median %.4f / %.4f)  on/off %.3f  (+%.1f%% noise/y columns)"
              % (wname, r["best_off"], r["best_on"], args.reps, r["median_off"], r["median_on"], r["ratio_best"], 100 * r["extra_columns_estimate"]))
        for p in (0, 1):
            h[p].close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
