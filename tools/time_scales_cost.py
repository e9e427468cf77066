"""tools/time_scales_cost.py -- ms/step of handles with and without per-row time scales (dfb_set_time_scales), alternating in one
process: a handle that never set rows ("off"), a second one for the spread ("control"), one with rows at a constant dt ("on_const": the
blend constants are uploaded once) and one with rows and a dt that changes every step ("on_vary": one host computation and upload of
[3][Ny] pairs per step).  On the reference's default plane, a batch of 8 of those, the 1024x2048 and 4096x8192 profile planes, and
graph replays of one attached step on the default plane (rows off / on; the attached step computes its pairs on the device).  Prints
the device name and power limit, and writes a JSON record (default profiles/time_scales_cost.json).

    python tools/time_scales_cost.py [--out PATH] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKLOADS = [  # name, planes per handle, dt, timed steps per window
    ("default_510x400", 1, 1e-5, 1000),
    ("default_510x400_batch8", 8, 1e-5, 300),
    ("1024x2048_profile_N128", 1, 1e-7, 300),
    ("4096x8192_profile_N128", 1, 1e-7, 40),
]


def plane_of(name):
    from digital_filtering_b200 import workloads as W
    from oracle.oracle import stored_default_plane
    return W.NAMED[name]() if name[0] in "14" else stored_default_plane()


def gpu_identity(torch):
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip()
    except Exception as e:               # the measurement still stands; the record says what could not be read
        smi = "nvidia-smi unavailable: %s" % e
    return name, smi


def rows_for(df, pl):
    """a wall-normal profile of Lt: the plane's own Lt scaled from 0.25 at the wall to 1 in the freestream"""
    Lt = np.asarray(pl["scales"], dtype=np.float64)[:, 2]
    return Lt[:, None] * np.linspace(0.25, 1.0, df.Ny)[None, :]


def summary(ms):
    return dict(ms=ms, best={m: min(v) for m, v in ms.items()}, median={m: sorted(v)[len(v) // 2] for m, v in ms.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "time_scales_cost.json"))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    import torch
    import _dfb_import  # noqa: F401
    import digital_filtering_b200 as dfb
    name, smi = gpu_identity(torch)
    print("device:", name, "|", smi)
    rec = dict(device=name, nvidia_smi=smi, reps=args.reps,
               method="CUDA events around n steps per window on each handle's own stream (fetch=False), ended by a synchronise; the "
                      "handles of a workload alternate window by window; best and median of the windows.  off / control: two handles "
                      "that never set rows.  on_const: rows set, dt constant.  on_vary: rows set, dt = dt0 (1 + 0.01 (k mod 7)), a "
                      "new dt every step.  graph: dt in device memory, one replay of a graph holding one dfb_filter_dev per step.",
               workloads={})
    for wname, nplanes, dt, n in WORKLOADS:
        pl = plane_of(wname)
        h = {m: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=1), fetch=False, nplanes=nplanes)
             for m in ("off", "control", "on_const", "on_vary")}
        for m in ("on_const", "on_vary"):
            h[m].set_time_scales(rows_for(h[m], pl))
        st = {m: torch.cuda.ExternalStream(d.stream()) for m, d in h.items()}
        dts = {m: [dt * (1 + 0.01 * (k % 7)) if m == "on_vary" else dt for k in range(n)] for m in h}

        def window(m, k):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st[m])
            for i in range(k):
                h[m].filter(dts[m][i % n])
            b.record(st[m])
            h[m].sync()
            return a.elapsed_time(b) / k

        for m in h:
            window(m, max(20, n // 10))                                 # warm-up
        ms = {m: [] for m in h}
        for _ in range(args.reps):
            for m in h:
                ms[m].append(window(m, n))
        r = dict(planes=nplanes, steps_per_window=n, y_form=h["off"].info(10), z_form=h["off"].info(7), **summary(ms))
        r["best_vs_off"] = {m: r["best"][m] / r["best"]["off"] for m in ms}
        rec["workloads"][wname] = r
        print("%-24s off %.4f  control %.4f  on_const %.4f  on_vary %.4f ms/step (best of %d)" %
              (wname, *(r["best"][m] for m in ("off", "control", "on_const", "on_vary")), args.reps))
        for d in h.values():
            d.close()

    # graph replays of an attached step on the default plane, rows off and on
    wname, _, dt, n = WORKLOADS[0]
    pl = plane_of(wname)
    h = {m: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=1), fetch=False) for m in ("graph_off", "graph_control", "graph_on")}
    h["graph_on"].set_time_scales(rows_for(h["graph_on"], pl))
    s = {m: torch.cuda.Stream() for m in h}
    dtd = {m: torch.full((1,), dt, dtype=torch.float64, device="cuda") for m in h}
    torch.cuda.synchronize()
    g = {}
    for m in h:
        h[m].attach_stream(s[m])
        g[m] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g[m], stream=s[m]):
            h[m].filter_dev(dtd[m])

    def gwindow(m, k):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(s[m]):
            a.record()
            for _ in range(k):
                g[m].replay()
            b.record()
        s[m].synchronize()
        return a.elapsed_time(b) / k

    for m in h:
        gwindow(m, n // 10)
    ms = {m: [] for m in h}
    for _ in range(args.reps):
        for m in h:
            ms[m].append(gwindow(m, n))
    r = dict(planes=1, steps_per_window=n, **summary(ms))
    r["best_vs_off"] = {m: r["best"][m] / r["best"]["graph_off"] for m in ms}
    rec["workloads"][wname + "_graph"] = r
    print("%-24s graph off %.4f  control %.4f  on %.4f ms/step (best of %d)" %
          (wname + "_graph", r["best"]["graph_off"], r["best"]["graph_control"], r["best"]["graph_on"], args.reps))
    for m in h:
        h[m].attach_stream(None)
    g.clear()
    for d in h.values():
        d.close()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
