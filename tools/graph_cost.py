"""tools/graph_cost.py -- ms/step of three ways of driving a handle, alternating in one process: host-driven dfb_filter, attached eager
dfb_filter_dev (dt in device memory, every launch on the caller's stream), and replays of a CUDA graph holding one dfb_filter_dev.  On the
reference's default plane, a batch of 8 of those, and the 1024x2048 profile plane.  With --parent-tree, the host-driven step time of
another built tree (the parent commit's, its library built) is measured in the same run, alternating with this tree's, to check that
the record pointer the kernels gained costs nothing host-driven.  Prints the device name and power limit, and writes a JSON record (default
profiles/graph_cost.json).

    python tools/graph_cost.py [--out PATH] [--reps 5] [--parent-tree PATH]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKLOADS = [  # name, planes per handle, dt, timed steps per window
    ("default_510x400", 1, 1e-5, 1000),
    ("default_510x400_batch8", 8, 1e-5, 300),
    ("1024x2048_profile_N128", 1, 1e-7, 300),
]


def plane_of(name):
    from digital_filtering_b200 import workloads as W
    from oracle.oracle import stored_default_plane
    return W.NAMED["1024x2048_profile_N128"]() if name.startswith("1024") else stored_default_plane()


def gpu_identity(torch):
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip()
    except Exception as e:               # the measurement still stands; the record says what could not be read
        smi = "nvidia-smi unavailable: %s" % e
    return name, smi


def host_window(torch, df, st, dt, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(n):
        df.filter(dt)
    b.record(st)
    df.sync()
    return a.elapsed_time(b) / n


def host_only(args):
    """--host-only: the package of tree --tree alone, host-driven windows; prints one JSON line of ms per workload and window"""
    sys.path.insert(0, args.tree)
    import torch
    import _dfb_import  # noqa: F401
    import digital_filtering_b200 as dfb
    out = {}
    for wname, nplanes, dt, n in WORKLOADS:
        df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane_of(wname), seed=1), fetch=False, nplanes=nplanes)
        st = torch.cuda.ExternalStream(df.stream())
        host_window(torch, df, st, dt, max(20, n // 10))
        out[wname] = [host_window(torch, df, st, dt, n) for _ in range(args.windows)]
        df.close()
    print("HOST_MS " + json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "graph_cost.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--tree", default=ROOT)
    ap.add_argument("--host-only", action="store_true")
    ap.add_argument("--windows", type=int, default=1)
    args = ap.parse_args()
    if args.host_only:
        return host_only(args)
    sys.path.insert(0, ROOT)
    import torch
    import _dfb_import  # noqa: F401
    import digital_filtering_b200 as dfb
    name, smi = gpu_identity(torch)
    print("device:", name, "|", smi)
    rec = dict(device=name, nvidia_smi=smi, reps=args.reps,
               method="CUDA events around n steps per window (fetch=False); the three modes use three handles of the workload and "
                      "alternate window by window; best and median of the windows.  host: dfb_filter on the handle's own streams.  "
                      "attached: dfb_filter_dev on one caller stream, dt rewritten in device memory before each step (a 1-element "
                      "fill kernel, timed with the step).  graph: the same fill + one replay of a graph holding one dfb_filter_dev.",
               workloads={})
    for wname, nplanes, dt, n in WORKLOADS:
        pl = plane_of(wname)
        h = {m: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(pl, seed=1), fetch=False, nplanes=nplanes) for m in ("host", "attached", "graph")}
        st_host = torch.cuda.ExternalStream(h["host"].stream())
        s_att, s_g = torch.cuda.Stream(), torch.cuda.Stream()
        dt_att = torch.full((1,), dt, dtype=torch.float64, device="cuda")
        dt_g = torch.full((1,), dt, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        h["attached"].attach_stream(s_att)
        h["graph"].attach_stream(s_g)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s_g):
            h["graph"].filter_dev(dt_g)

        def att_window(k):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s_att):
                a.record()
                for _ in range(k):
                    dt_att.fill_(dt)
                    h["attached"].filter_dev(dt_att)
                b.record()
            s_att.synchronize()
            return a.elapsed_time(b) / k

        def graph_window(k):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s_g):
                a.record()
                for _ in range(k):
                    dt_g.fill_(dt)
                    g.replay()
                b.record()
            s_g.synchronize()
            return a.elapsed_time(b) / k

        fns = dict(host=lambda k: host_window(torch, h["host"], st_host, dt, k), attached=att_window, graph=graph_window)
        for m in fns:
            fns[m](max(20, n // 10))                                   # warm-up
        ms = {m: [] for m in fns}
        for _ in range(args.reps):
            for m in fns:
                ms[m].append(fns[m](n))
        r = dict(planes=nplanes, steps_per_window=n, y_form=h["host"].info(10), ms=ms,
                 best={m: min(v) for m, v in ms.items()}, median={m: sorted(v)[len(v) // 2] for m, v in ms.items()})
        r["best_vs_host"] = {m: r["best"][m] / r["best"]["host"] for m in ms}
        rec["workloads"][wname] = r
        print("%-24s host %.4f  attached %.4f  graph %.4f ms/step (best of %d)  attached/host %.3f  graph/host %.3f"
              % (wname, r["best"]["host"], r["best"]["attached"], r["best"]["graph"], args.reps, r["best_vs_host"]["attached"],
                 r["best_vs_host"]["graph"]))
        h["attached"].attach_stream(None)
        h["graph"].attach_stream(None)
        del g
        for d in h.values():
            d.close()
    if args.parent_tree:
        # host-driven steps of the parent build against this build's: subprocesses alternate, one window each, so that both see the
        # same machine state; best and median over the reps
        trees = dict(parent=os.path.abspath(args.parent_tree), this=ROOT)
        par = {k: {w[0]: [] for w in WORKLOADS} for k in trees}
        for _ in range(args.reps):
            for k, tree in trees.items():
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--host-only", "--tree", tree], capture_output=True,
                                   text=True, timeout=900)
                line = [x for x in r.stdout.splitlines() if x.startswith("HOST_MS ")]
                if r.returncode != 0 or not line:
                    raise RuntimeError("host-only run failed for %s:\n%s\n%s" % (tree, r.stdout, r.stderr))
                for w, v in json.loads(line[0][8:]).items():
                    par[k][w] += v
        rec["host_driven_vs_parent"] = {w: dict(parent=par["parent"][w], this=par["this"][w], best_parent=min(par["parent"][w]),
                                                best_this=min(par["this"][w]), ratio_best=min(par["this"][w]) / min(par["parent"][w]))
                                        for w in par["this"]}
        for w, v in rec["host_driven_vs_parent"].items():
            print("%-24s host-driven: parent %.4f  this %.4f ms/step (best)  this/parent %.3f  spread parent %.4f-%.4f this %.4f-%.4f"
                  % (w, v["best_parent"], v["best_this"], v["ratio_best"], min(v["parent"]), max(v["parent"]), min(v["this"]), max(v["this"])))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(rec, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
