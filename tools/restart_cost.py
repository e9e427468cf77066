"""tools/restart_cost.py -- what a restart file costs: save and load times, and the step time around them.

For the headline 1024x2048 plane and the 4096x8192 plane, a handle with the N2 statistics on saves and loads (dfb_save_restart /
dfb_load_restart) its state alone and its state + N2 sums, to a file in a temporary directory on local disk (the calls are synchronous
and return when the file has been written into the page cache: no fsync).  Wall-clock time of each call, best and median of --reps.
Then the production ms/step of that handle (CUDA events around n steps) before any save, after the saves and after the loads, beside
a second handle that never saves, to show that nothing per step changed.  Records the device name and power limit; writes a JSON
record (default profiles/restart_cost.json).

    python tools/restart_cost.py [--out PATH] [--reps 3]
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
import _dfb_import  # noqa: E402,F401
import digital_filtering_b200 as dfb  # noqa: E402
from digital_filtering_b200 import workloads as W  # noqa: E402
from corr_cost import gpu_identity, window  # noqa: E402

WORKLOADS = [("1024x2048_profile_N128", 1e-7, 200), ("4096x8192_profile_N128", 1e-7, 30)]   # name, dt, timed steps per window


def timed(fn, reps):
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return dict(ms=t, best=min(t), median=sorted(t)[len(t) // 2])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "restart_cost.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    name, smi = gpu_identity()
    print("device:", name, "|", smi)
    tmp = tempfile.mkdtemp(prefix="dfb_restart_cost_")
    rec = dict(device=name, nvidia_smi=smi, reps=args.reps, file_dir=tmp,
               method="wall clock around each synchronous dfb_save_restart / dfb_load_restart call (file in a temporary directory on local "
                      "disk, written into the page cache, no fsync); step times: CUDA events around n production steps (fetch=False), "
                      "the saving handle and a control handle alternating window by window", workloads={})
    try:
        for wname, dt, n in WORKLOADS:
            plane = W.NAMED[wname]()
            h = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1), fetch=False)
            ctl = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1), fetch=False)
            st, sc = torch.cuda.ExternalStream(h.stream()), torch.cuda.ExternalStream(ctl.stream())
            for df in (h, ctl):
                df.stats_enable()
            window(h, st, dt, max(10, n // 10))
            window(ctl, sc, dt, max(10, n // 10))

            def step_ms():
                a, b = [], []
                for _ in range(args.reps):
                    a.append(window(h, st, dt, n))
                    b.append(window(ctl, sc, dt, n))
                return dict(handle=min(a), control=min(b))

            r = dict(steps_per_window=n, step_ms_before=step_ms())
            paths = {k: os.path.join(tmp, "%s_%s.dfbr" % (wname, k)) for k in ("state", "state_stats")}
            r["save_state"] = timed(lambda: h.save_restart(paths["state"]), args.reps)
            r["save_state_stats"] = timed(lambda: h.save_restart(paths["state_stats"], stats=True), args.reps)
            r["bytes"] = {k: os.path.getsize(p) for k, p in paths.items()}
            r["step_ms_after_save"] = step_ms()
            r["load_state"] = timed(lambda: h.load_restart(paths["state"]), args.reps)
            r["load_state_stats"] = timed(lambda: h.load_restart(paths["state_stats"], stats=True), args.reps)
            r["step_ms_after_load"] = step_ms()
            rec["workloads"][wname] = r
            print("%-24s save %.1f / %.1f ms, load %.1f / %.1f ms (state / state+N2, best of %d; %.0f / %.0f MB); ms/step before %.4f "
                  "after save %.4f after load %.4f, control %.4f %.4f %.4f" % (
                      wname, r["save_state"]["best"], r["save_state_stats"]["best"], r["load_state"]["best"], r["load_state_stats"]["best"],
                      args.reps, r["bytes"]["state"] / 1e6, r["bytes"]["state_stats"] / 1e6, r["step_ms_before"]["handle"],
                      r["step_ms_after_save"]["handle"], r["step_ms_after_load"]["handle"], r["step_ms_before"]["control"],
                      r["step_ms_after_save"]["control"], r["step_ms_after_load"]["control"]))
            for p in paths.values():
                os.unlink(p)
            h.close()
            ctl.close()
            torch.cuda.empty_cache()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
