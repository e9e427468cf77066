#!/usr/bin/env python
"""bench.py -- inflow cell-updates/s per filter() step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one DIGITAL_FILTER::filter(dt) (df.cpp:449-468) over one synthetic plane: noise generation,
y-sweep, z-sweep, temporal blend, RST scaling, SRA -- all five outputs of every cell.
  value    whole-job cell-updates/s, state resident in HBM, CUDA events on the library's stream
  e2e      the same through the reference-facing call (dfb_filter_to_host: filter(dt) + the five
           fields copied into pinned HOST arrays, as the C++/Fortran facades do every step);
           e2e.facade: the C++ class itself (examples/facade_bench.cpp, its own page-locked std::vectors)
  roofline the dominant kernel and the step against the HBM roof (MEASURED_PEAKS.json) -- both sweeps evaluate the
           reference's exponential windows recursively and no longer execute its flops; the fp64-FMA roof (measured
           live by a DFMA microbenchmark: MEASURED_PEAKS.json has no fp64 entry) is reported as "equivalent"
  cpu_baseline  the reference's own df.cpp (oracle/_ref) on the box's host, bounded sample
  batched_planes  BASELINE config 5 on this rank's GPU: 8 reference-default planes behind one handle (dfb_create_batch)
N > 1 (torchrun): every rank filters its own independent plane (distinct RNG stream group = rank): weak scaling, no
data-path collective; time = max over ranks.  Additionally (`slab`) BASELINE config 4: ONE 4096x8192 plane in spanwise
slabs over the N ranks, halos regenerated locally, the library's NCCL hand-off of the finished plane to rank 0.
--impl reference: the reference's CPU filter() on all host cores (independent processes; the reference is
single-threaded with a process-wide RNG), same metric/config, bounded sample per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_WORKLOAD = "1024x2048_profile_N128"
SLAB_WORKLOAD = "4096x8192_profile_N128"
METRIC = "inflow cell-updates/sec per filter() step"
DT = 1e-7
NCU_SUMMARY = os.path.join("profiles", "ncu_full_r02b_summary.csv")


def common_config(plane):
    """the part of `config` both arms print, key for key (the driver compares them)"""
    from digital_filtering_b200 import workloads as WL
    sc = np.asarray(plane["scales"])
    ny, nz = WL._N_from_geometry(np.asarray(plane["yc"]), np.asarray(plane["dy"]), np.asarray(plane["dz"]), plane["d_i"], sc[0, 0], sc[0, 1])
    return dict(workload=plane["name"], plane=[int(plane["Ny"]), int(plane["Nz"])], max_half_width=[int(ny.max()), int(nz.max())], dt=DT)


def ncu_traffic(kernel, workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full summary
    (captured on the 1024x2048 profile workload); None for other workloads."""
    if workload != DEFAULT_WORKLOAD:
        return None
    try:
        import csv
        rows = list(csv.reader(open(os.path.join(ROOT, NCU_SUMMARY))))
        col = [i for i, h in enumerate(rows[0]) if kernel.split("<")[0] in h][0]
        tot = 0.0
        for r in rows[1:]:
            if r[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[r[1]]
                tot += float(r[col]) * scale
        return tot or None
    except Exception:
        return None


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML every
    2 ms from a thread (pynvml ships in the image)."""
    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40),
               ("hw_power_brake_slowdown", 0x80), ("sw_power_cap", 0x4))

    def __init__(self, gpu_index):
        self.idx, self.samples, self.stop_flag, self.t, self.h, self.nv = gpu_index, [], False, None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                     int(nv.nvmlDeviceGetCurrentClocksEventReasons(h)),
                                     float(nv.nvmlDeviceGetPowerUsage(h)) / 1e3))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        if not self.nv or not self.t:
            return None
        self.stop_flag = True
        self.t.join(timeout=1)
        if not self.samples:
            return None
        sm = [s[0] for s in self.samples]
        mask = 0
        for s in self.samples:
            mask |= s[1]
        reasons = [n for n, bit in self.REASONS if mask & bit]
        return dict(sm_mhz=float(np.median(sm)), sm_min_mhz=float(min(sm)), sm_max_mhz=self.max_mhz, reasons=reasons,
                    power_w_max=max(s[2] for s in self.samples), samples=len(sm))


# --------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own df.cpp on a bounded sample of the workload
# --------------------------------------------------------------------------------------------------
def sample_plane(plane, target_taps=4.0e8):
    """A spanwise sub-slab of the same plane (same rows, same half-width profile, fewer columns)
    sized for ~1 s of single-core CPU work per step."""
    from oracle import oracle as O
    p = dict(plane)
    O.half_widths(p)
    taps_per_col = float(sum((2 * p["N_y"][f][:, 0].astype(np.int64) + 1).sum() + (2 * p["N_z"][f][:, 0].astype(np.int64) + 1).sum() for f in range(3)))
    ncol = int(max(8, min(plane["Nz"], target_taps // taps_per_col)))
    s = dict(plane)
    s["Nz"] = ncol
    s["name"] = plane["name"] + f"[sample:{plane['Ny']}x{ncol}]"
    return s, taps_per_col * ncol


def _ref_worker(args):
    plane, steps, warmup = args
    from oracle import oracle as O
    R = O.RefFilter()
    R.reshape(plane)
    R.time_steps(DT, warmup)
    tot, st = R.time_steps(DT, steps)
    R.close()
    return tot


def cpu_reference_run(plane, steps, warmup, nproc):
    """nproc independent reference objects, one process each; returns (seconds for `steps` steps, kind)."""
    from oracle import oracle as O
    if O.have_ref():
        import multiprocessing as mp
        if nproc == 1:
            return _ref_worker((plane, steps, warmup)), "reference"
        with mp.get_context("fork").Pool(nproc) as pool:
            ts = pool.map(_ref_worker, [(plane, steps, warmup)] * nproc)
        return max(ts), "reference"
    # fall-back checker: the plain-C restatement (single instance, OpenMP over rows)
    p = dict(plane)
    O.half_widths(p)
    Ny, Nz = p["Ny"], p["Nz"]
    rys = [O.noise_rys(1, 0, f, 0, Ny, p["Ny_max"][f], Nz) for f in range(3)]
    hal = [O.noise_halo(1, 0, f, 0, Ny, p["Nz_max"][f]) for f in range(3)]
    fo = np.zeros((3, Ny, Nz))
    for _ in range(warmup):
        O.step(p, rys, hal, fo, DT)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.step(p, rys, hal, fo, DT)
    return time.perf_counter() - t0, "port"


def full_plane_check(plane):
    """ONE instance of the reference on the WHOLE plane (not the sub-slab sample), one step on one core, to show that the
    sample extrapolates.  The reference stores a private copy of the coefficients per cell (SURVEY quirk 7): 26 GB at
    1024x2048 / N = 128 -- only attempted when the host has the memory; says so otherwise."""
    try:
        import psutil
        from oracle import oracle as O
        if not O.have_ref():
            return dict(skipped="oracle/_ref did not travel")
        p = dict(plane)
        O.half_widths(p)
        need = 8.0 * 2 * sum(float((2 * p["N_y"][f].astype(np.int64) + 1).sum() + (2 * p["N_z"][f].astype(np.int64) + 1).sum()) for f in range(3)) / 2
        avail = float(psutil.virtual_memory().available)
        if need * 1.3 > avail:
            return dict(skipped=f"needs {need / 2**30:.0f} GiB of per-cell coefficient copies, host has {avail / 2**30:.0f} GiB available")
        R = O.RefFilter()
        t0 = time.perf_counter()
        R.reshape(plane)
        setup_s = time.perf_counter() - t0
        tot, _ = R.time_steps(DT, 1)
        R.close()
        cells = plane["Ny"] * plane["Nz"]
        return dict(cells=cells, ms_per_step=1e3 * tot, cell_updates_per_s_one_core=cells / tot, setup_s=setup_s,
                    note="one reference object on the whole plane, one step, one core")
    except Exception as e:
        return dict(skipped=str(e)[:200])


def run_reference_arm(args, plane):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    ncores = os.cpu_count() or 1
    nproc = max(1, min(ncores, 32))
    # bounded sample: ~100 s of wall clock for the whole --steps/--warmup run at ~0.4 G tap/s per core
    wu = min(args.warmup, 2)
    target = min(2.0e8, max(1.0e7, 0.4e9 * 100.0 / (args.steps + wu)))
    s, taps = sample_plane(plane, target_taps=target)
    # one instance in THIS process first: oracle/_ref/libdfref.so (the reference's own df.cpp) is loaded here, not only in the
    # forked workers, and gives the one-core rate of the sample
    one_core = None
    if O.have_ref():
        secs1 = _ref_worker((s, 2, 1))
        one_core = s["Ny"] * s["Nz"] * 2 / secs1
    secs, kind = cpu_reference_run(s, args.steps, wu, nproc)
    cells = s["Ny"] * s["Nz"] * nproc * args.steps
    value = cells / secs
    full = full_plane_check(plane) if not args.no_full_plane else dict(skipped="--no-full-plane")
    line = dict(impl="reference", metric=METRIC, value=value, unit="cell-updates/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=1e3 * secs / args.steps, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", config=common_config(plane),
                cpu_baseline=dict(value=value, unit="cell-updates/s", cores=nproc if kind == "reference" else ncores, kind=kind,
                                  library=os.path.relpath(os.path.join(O.REF_DIR, "libdfref.so"), ROOT) if kind == "reference" else "oracle/libdforacle.so",
                                  sample=f"{nproc} independent instances x ({s['Ny']}x{s['Nz']} sub-slab of the {plane['Ny']}x{plane['Nz']} plane, same rows/half-widths)"
                                         f" per step; the reference's five stage calls (df.cpp:453-461), no print/CSV",
                                  one_core_cell_updates_per_s=one_core, full_plane_one_core=full),
                e2e=dict(value=value, unit="cell-updates/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def facade_e2e(plane, steps, device):
    """e2e through the C++ class itself: builds examples/facade_bench.cpp against include/digital_filter.hpp and runs it"""
    import tempfile
    libdir = os.path.join(ROOT, "digital-filtering_b200", "lib")
    tmp = tempfile.mkdtemp(prefix="dfb_facade_")
    exe, pf = os.path.join(tmp, "facade_bench"), os.path.join(tmp, "plane.bin")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "facade_bench.cpp"),
                    "-L" + libdir, "-ldfb200", "-Wl,-rpath," + libdir, "-o", exe], check=True, capture_output=True)
    with open(pf, "wb") as fh:
        np.array([plane["Ny"], plane["Nz"]], dtype=np.int32).tofile(fh)
        for k in ("yc", "dy", "dz", "rows", "scales"):
            np.ascontiguousarray(plane[k], dtype=np.float64).tofile(fh)
    r = subprocess.run([exe, pf, str(steps), "3", str(device)], capture_output=True, text=True, timeout=600)
    if r.returncode != 0:
        raise RuntimeError(r.stderr[-300:])
    tok = [ln for ln in r.stdout.splitlines() if ln.startswith("FACADE ")][-1].split()
    return int(tok[1]) * int(tok[2]) / float(tok[3])


def batched_planes(dfb, torch, local, nplanes=8, steps=300):
    """BASELINE config 5 on one GPU: `nplanes` planes of the reference's default 510x400 geometry (its stored setup tables) behind ONE handle
    (dfb_create_batch: one launch set per step for all of them), dt = 1e-5; resident and with the five fields of every plane
    delivered to pinned host memory."""
    from oracle import oracle as O
    plane = O.stored_default_plane()
    out = {}
    for P in (1, nplanes):
        d = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=1, device=local, plane_id=100 * local), fetch=False, nplanes=P)
        st = torch.cuda.ExternalStream(d.stream(), device=local)
        for _ in range(10):
            d.filter(1e-5)
        d.sync()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(steps):
            d.filter(1e-5)
        b.record(st)
        d.sync()
        ms = a.elapsed_time(b) / steps
        rec = dict(planes=P, cells_per_plane=d.n_cells, ms_per_step=ms, us_per_plane_step=1e3 * ms / P, cell_updates_per_s=P * d.n_cells / (ms * 1e-3))
        if P == nplanes:
            host = [torch.empty(P * d.n_cells, dtype=torch.float64).pin_memory() for _ in range(5)]
            hp = [h.data_ptr() for h in host]
            L = dfb.lib()
            for _ in range(3):
                dfb._check(L.dfb_filter_to_host(d._h, 1e-5, *hp))
            t0 = time.perf_counter()
            for _ in range(100):
                dfb._check(L.dfb_filter_to_host(d._h, 1e-5, *hp))
            e = (time.perf_counter() - t0) / 100
            rec["e2e_us_per_plane_step"] = 1e6 * e / P
            rec["e2e_d2h_bytes_per_step"] = 40 * P * d.n_cells
        out["planes_%d" % P] = rec
        d.close()
    out["note"] = ("BASELINE config 5 = 64 such planes x 1000 steps over 8 GPUs: 8 planes per GPU, i.e. planes_%d x 1000 steps per GPU "
                   "(no collective; every rank runs this same job)" % nplanes)
    out["config5_seconds_per_gpu_1000_steps"] = out["planes_%d" % nplanes]["ms_per_step"]
    return out


def slab_job(dfb, torch, dist, rank, world, local, steps=20):
    """BASELINE config 4: ONE 4096x8192 plane, spanwise slabs over the ranks (halos regenerated locally, no exchange), the
    library's own NCCL hand-off of the finished plane to rank 0 (u', v', w' on the wire; T', rho' rebuilt there).
    Device-side timing (CUDA events on the library's compute / communication streams), max over ranks."""
    from digital_filtering_b200 import parallel as P, workloads as WL
    plane = WL.NAMED[SLAB_WORKLOAD]()
    seed = 20261018
    sf = P.SlabFilter(dist, plane["Nz"], lambda k0, k1: dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=seed, device=local, k_begin=k0, k_end=k1), fetch=False))
    cs = torch.cuda.ExternalStream(sf.filt.stream(), device=local)
    ms_ = torch.cuda.ExternalStream(sf.filt.comm_stream(), device=local)
    dev = torch.device("cuda", local)

    def reduce_max(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def fence():
        sf.filt.sync()
        torch.cuda.synchronize()
        dist.barrier()

    def timed(mode):
        # mode 0: filter only; 1: filter + gather, one after the other; 2: gather of step t under filter of step t+1
        def body(n):
            if mode == 0:
                for _ in range(n):
                    sf.filter(DT)
            elif mode == 1:
                for _ in range(n):
                    sf.filter(DT)
                    sf.gather_begin()
                    sf.gather_end()
            elif mode == 3:                                # the hand-off alone (staging + transfer + assembly of the same step again and again)
                for _ in range(n):
                    sf.gather_begin()
                    sf.gather_end()
            else:
                sf.filter(DT)
                sf.gather_begin()
                for _ in range(n - 1):
                    sf.filter(DT)
                    sf.gather_end()
                    sf.gather_begin()
                sf.gather_end()
        body(3)
        fence()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(cs)
        body(steps)
        if mode == 0:
            b.record(cs)
        else:
            ms_.wait_stream(cs)
            b.record(ms_)
        fence()
        return reduce_max(a.elapsed_time(b)) / steps

    t_no, t_sync, t_ovl, t_gather = timed(0), timed(1), timed(2), timed(3)
    wire = torch.tensor([float(sf.filt.gather_wire_bytes()) if rank != 0 else 0.0], dtype=torch.float64, device=dev)
    dist.all_reduce(wire, op=dist.ReduceOp.SUM)
    # slab == whole: the plane gathered now against the same plane filtered whole on rank 0's GPU (same number of steps)
    nsteps = int(sf.filt.step)
    sf.gather()
    rec = None
    if rank == 0:
        whole = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=seed, device=local), fetch=False)
        ws = torch.cuda.ExternalStream(whole.stream(), device=local)
        for _ in range(nsteps - 1 - 20):
            whole.filter(DT)
        whole.sync()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(ws)
        for _ in range(20):
            whole.filter(DT)
        b.record(ws)
        whole.sync()
        one_gpu_ms = a.elapsed_time(b) / 20
        same = all(bool(np.array_equal(sf.plane(w), whole.get(w))) for w in range(5))
        whole.close()
        cells = plane["Ny"] * plane["Nz"]
        rec = dict(workload=plane["name"], n_gpus=world, slabs=[list(b) for b in sf.bounds], steps=steps,
                   ms_per_step_no_gather=t_no, ms_per_step_with_gather=t_sync, ms_per_step_with_gather_overlapped=t_ovl, ms_gather_alone=t_gather,
                   one_gpu_ms_per_step=one_gpu_ms, speedup_no_gather=one_gpu_ms / t_no, speedup_with_gather_overlapped=one_gpu_ms / t_ovl,
                   cell_updates_per_s_with_gather_overlapped=cells / (t_ovl * 1e-3),
                   wire_bytes_per_step=int(wire.item()), wire_bytes_per_cell=24, gathered_equals_whole_plane_bitwise=bool(same),
                   transport={2: "peer-to-peer inside libdfb200.so (dfb_gather_begin/_end): CUDA IPC mapping of rank 0's plane, each sender's copy engine writes "
                                 "u', v', w' of its slab into the final layout over NVLink, stream memory operations order it; T', rho' rebuilt on rank 0",
                              1: "NCCL send/recv inside libdfb200.so (dfb_gather_begin/_end) + assembly kernel; u', v', w' on the wire, T', rho' rebuilt on rank 0"}.get(int(sf.filt.info(12)), "?"),
                   wire_gbs_gather_alone=wire.item() / (t_gather * 1e-3) / 1e9,
                   timing="CUDA events on the library's compute and communication streams, max over ranks")
    dist.barrier()
    sf.filt.close()
    return rec


DUMP_BYTES = 64 * 10 ** 6        # all files of --dump-outputs together, .npy headers included


def dump_outputs(dfb, df, out_dir):
    """The five fields a caller of filter(dt) receives after the last timed step, as <out_dir>/<field>.npy (float64).  With
    several GPUs only rank 0's plane (plane_id 0) is written; the other ranks' planes differ only in their noise streams.  When all
    five do not fit in DUMP_BYTES, every field is sampled at the same cells: a fixed-seed draw without replacement, in
    ascending row-major order."""
    names = dict(u_fluc=dfb.U_FLUC, v_fluc=dfb.V_FLUC, w_fluc=dfb.W_FLUC, T_fluc=dfb.T_FLUC, rho_fluc=dfb.RHO_FLUC)
    cells = df.n_cells
    n = min(cells, (DUMP_BYTES // len(names) - 1024) // 8)
    idx = None if n == cells else np.sort(np.random.default_rng(0).choice(cells, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, which in names.items():
        a = df.get(which).ravel()
        np.save(os.path.join(out_dir, name + ".npy"), a if idx is None else a[idx])


def run_b200(args, plane):
    import torch
    import _dfb_import  # noqa: F401
    import digital_filtering_b200 as dfb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version banner / warnings: not on stdout, where ONE JSON line goes
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    K, Wm = args.steps, max(args.warmup, 3)
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane, seed=20261018, plane_id=rank, device=local), fetch=False)
    assert df.tuned, "tuned sm_100a kernels must be the measured path"
    stream = torch.cuda.ExternalStream(df.stream(), device=local)
    cells = df.n_cells
    N_y = [df.half_widths(f, 0) for f in range(3)]
    N_z = [df.half_widths(f, 1) for f in range(3)]
    taps_y = int(sum((2 * a.astype(np.int64) + 1).sum() for a in N_y))
    taps_z = int(sum((2 * a.astype(np.int64) + 1).sum() for a in N_z))
    ws_bytes = 8 * (sum((plane["Ny"] + 2 * int(a.max())) * plane["Nz"] for a in N_y) + 3 * cells + 11 * cells)
    l2_bytes = 126 * 2 ** 20
    flush = ws_bytes < 2 * l2_bytes
    fbuf = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device="cuda") if flush else None

    # ---- value: device-resident steps, CUDA events on the library's stream ----
    for _ in range(Wm):
        df.filter(DT)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(K):
        if flush:
            with torch.cuda.stream(stream):
                fbuf.zero_()
        ev[i][0].record(stream)
        df.filter(DT)
        ev[i][1].record(stream)
    df.sync()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms = sum(a.elapsed_time(b) for a, b in ev)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(dfb, df, args.dump_outputs)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * cells * K / (ms_total * 1e-3)

    # ---- e2e: filter(dt) + five fields into pinned host arrays, every step ----
    host = [torch.empty(cells, dtype=torch.float64).pin_memory() for _ in range(5)]
    hp = [h.data_ptr() for h in host]
    L = dfb.lib()
    Ke = min(K, 500)
    for _ in range(2):
        dfb._check(L.dfb_filter_to_host(df._h, DT, *hp))
    barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        dfb._check(L.dfb_filter_to_host(df._h, DT, *hp))
    barrier()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * cells * Ke / float(te.item())

    # ---- e2e, pipelined variant of the same call (dfb_filter_to_host_begin / _end, two sets of pinned arrays): the copy of step t
    # runs under the compute of step t+1; every step's five fields still arrive in host memory.  Reported beside, not instead of, e2e.
    host2 = [torch.empty(cells, dtype=torch.float64).pin_memory() for _ in range(5)]
    sets = [hp, [h.data_ptr() for h in host2]]
    dfb._check(L.dfb_filter_to_host_begin(df._h, DT, *sets[0]))
    dfb._check(L.dfb_filter_to_host_begin(df._h, DT, *sets[1]))
    dfb._check(L.dfb_filter_to_host_end(df._h)); dfb._check(L.dfb_filter_to_host_end(df._h))
    barrier()
    t0 = time.perf_counter()
    dfb._check(L.dfb_filter_to_host_begin(df._h, DT, *sets[0]))
    for i in range(1, Ke):
        dfb._check(L.dfb_filter_to_host_begin(df._h, DT, *sets[i & 1]))
        dfb._check(L.dfb_filter_to_host_end(df._h))            # step i-1 is in host memory
    dfb._check(L.dfb_filter_to_host_end(df._h))
    barrier()
    tp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
    e2e_pipelined = world * cells * Ke / float(tp.item())

    # ---- config 4 (N > 1): one plane in slabs + the NCCL hand-off, every rank takes part ----
    slab = None
    if dist is not None and not args.no_slab:
        del host2
        try:
            slab = slab_job(dfb, torch, dist, rank, world, local)
        except Exception as e:
            slab = dict(error=str(e)[:300])

    if rank != 0:
        df.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- per-kernel times (CUDA events inside the library, one sync per step: explains, not the headline) ----
    df.set_timing(True)
    stage = []
    for _ in range(max(5, min(K, 20))):
        if flush:
            with torch.cuda.stream(stream):
                fbuf.zero_()
        df.filter(DT)
        stage.append(df.last_ms())
    df.set_timing(False)
    med = {k: float(np.median([s[k] for s in stage])) for k in stage[0]}
    fp64_peak, mhz = dfb.measure_fp64_peak(local)
    peaks = load_peaks()
    hbm_peak = peaks["hbm_gbs"] if peaks and "hbm_gbs" in peaks else 6650.0
    hbm_src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
    alg_bytes = 88 * cells                                    # SURVEY 8d: 5 outputs + filt_old r/w x3
    zmode = "recursive" if df.info(7) == 1 else "direct"
    y_form = {3: "run-recursive on the row blocks where it pays + dense band matrices on the rest", 2: "run-recursive",
              1: "chunk-recursive band matrices", 0: "dense band matrices"}[int(df.info(10))]
    launches_per_step = 4 if int(df.info(10)) == 3 else 3     # noise + y-sweep (two launches when both forms serve the plane) + z-sweep/epilogue
    y_bytes = 3 * 16 * cells                                  # y-sweep: r_ys read once, r_zs interior written once, per field
    yname = "ysweep_run_kernel" if df.info(10) >= 2 else "ysweep_tma_kernel"
    kern = {
        # y-sweep.  Run-recursive form: every row group through the exponential window, ~5x fewer flops than the reference's
        # 2*(2N_y+1) per cell -> its roof is the memory system; equivalent_tflops = reference-formulation flops / time, for comparison.
        yname: dict(ms=med["ysweep"], form=y_form, equivalent_tflops=2 * taps_y / (med["ysweep"] * 1e-3) / 1e12,
                    hbm_gbs=y_bytes / (med["ysweep"] * 1e-3) / 1e9, alg_bytes_per_cell=48),
        # z-sweep + epilogue: recursive form (about 13x fewer flops at N = 128): its roof is the memory system
        "zsweep_epilogue_kernel": dict(ms=med["zsweep_epilogue"], form=zmode, equivalent_tflops=2 * taps_z / (med["zsweep_epilogue"] * 1e-3) / 1e12,
                                       hbm_gbs=alg_bytes / (med["zsweep_epilogue"] * 1e-3) / 1e9, alg_bytes_per_cell=88),
        "noise_kernel": dict(ms=med["noise"], note="timed alone here; in the production step it runs on a low-priority stream beside the sweeps of the previous step"),
    }
    for k in (yname, "zsweep_epilogue_kernel"):
        kern[k]["frac_hbm"] = kern[k]["hbm_gbs"] / hbm_peak
        kern[k]["equivalent_frac_fp64"] = kern[k]["equivalent_tflops"] / fp64_peak
    step_ms = ms_total / K
    eq_tf = 2 * (taps_y + taps_z) / (step_ms * 1e-3) / 1e12
    step = dict(equivalent_tflops=eq_tf, equivalent_frac_fp64=eq_tf / fp64_peak,
                note="reference-formulation flops / step time; the recursive sweeps execute far fewer, so this is a speed-up figure, not a utilisation",
                hbm_gbs=alg_bytes / (step_ms * 1e-3) / 1e9, frac_hbm=alg_bytes / (step_ms * 1e-3) / 1e9 / hbm_peak, hbm_peak=hbm_peak, hbm_peak_source=hbm_src,
                fp64_peak_tflops=fp64_peak, fp64_peak_source="DFMA microbenchmark measured live in this run (dfb_measure_fp64_peak); MEASURED_PEAKS.json has no fp64 entry")
    dom = yname if med["ysweep"] >= med["zsweep_epilogue"] else "zsweep_epilogue_kernel"
    kd = kern[dom]
    # SURVEY 8d: t_roof = max(F_alg / P_fp64, B_alg / BW_hbm) with F_alg the REFERENCE-formulation flops (2 per tap) and B_alg the
    # algorithmic bytes; on this plane the fp64 term binds for either sweep (y: 34 us against 16 us).  `achieved` is therefore the
    # algorithmic TFLOP/s of the dominant kernel.  Both sweeps now evaluate the exponential windows recursively and EXECUTE ~5x (y) /
    # ~13x (z) fewer flops than F_alg, so this fraction measures speed against the reference formulation's roof, not pipe utilisation
    # (it can exceed 1: the z-sweep's does); the physical bound of the new formulation is HBM, reported beside it (`hbm_view`).
    alg_flops = 2 * (taps_y if dom == yname else taps_z)
    roofline = dict(bound="fp64", kernel=dom, achieved=kd["equivalent_tflops"], peak=fp64_peak, unit="TFLOP/s", frac=kd["equivalent_frac_fp64"],
                    definition="algorithmic (reference-formulation, SURVEY 8d) flops of one launch / launch duration (CUDA events) / measured DFMA peak",
                    alg_flops_per_launch=alg_flops, alg_flops_per_cell=alg_flops / cells,
                    traffic=ncu_traffic(dom, plane["name"]), traffic_source=NCU_SUMMARY + " (ncu --set full, one launch)",
                    peak_source=step["fp64_peak_source"],
                    hbm_view=dict(bound="hbm", achieved=kd["hbm_gbs"], peak=hbm_peak, unit="GB/s", frac=kd["frac_hbm"], alg_bytes_per_cell=kd["alg_bytes_per_cell"],
                                  peak_source=hbm_src),
                    step=step, kernels=kern)

    # ---- e2e through the C++ facade (its own page-locked std::vectors) ----
    facade = None
    if world == 1 and not args.no_facade:
        try:
            facade = dict(value=facade_e2e(plane, min(K, 300), local), unit="cell-updates/s",
                          call="DIGITAL_FILTER::filter(dt) of include/digital_filter.hpp (examples/facade_bench.cpp): five std::vector members filled every step")
        except Exception as e:
            facade = dict(error=str(e)[:200])

    # ---- cpu baseline: the reference's own df.cpp, 1 core, bounded sample ----
    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            s, _ = sample_plane(plane)
            nst = 25                  # ~10 s of one host core
            secs, kind = cpu_reference_run(s, nst, 1, 1)
            cpu = dict(value=s["Ny"] * s["Nz"] * nst / secs, unit="cell-updates/s", cores=1 if kind == "reference" else (os.cpu_count() or 1), kind=kind,
                       sample=f"{nst} steps of a {s['Ny']}x{s['Nz']} spanwise sub-slab of the {plane['Ny']}x{plane['Nz']} plane (same rows, same half-widths); "
                              f"the reference's five stage calls (df.cpp:453-461), 1 of {os.cpu_count()} host cores", ms_per_step_sample=1e3 * secs / nst)
        except Exception as e:   # the checker is optional for the bench; say so rather than die
            cpu = dict(value=None, unit="cell-updates/s", cores=0, kind="unavailable", sample=str(e)[:200])

    # ---- the other single-GPU configurations of BASELINE.json, briefly (parity-test cases; reported for context) ----
    sweep, batched = None, None
    if not args.no_sweep:
        try:
            batched = batched_planes(dfb, torch, local)
        except Exception as e:
            batched = dict(error=str(e)[:200])
    if world == 1 and not args.no_sweep:
        from digital_filtering_b200 import workloads as WL
        from oracle import oracle as O
        sweep = {}
        cases = [("1024x2048_saturated_N128", lambda: dfb.DFConfig.from_plane(WL.NAMED["1024x2048_saturated_N128"](), seed=1, device=local)),
                 ("512x512_N32", lambda: dfb.DFConfig.from_plane(WL.NAMED["512x512_N32"](), seed=1, device=local)),
                 ("reference_default_plane_510x400", lambda: dfb.DFConfig.from_plane(O.stored_default_plane(), seed=1, device=local))]
        for name, mk in cases:
            try:
                d2 = dfb.DIGITAL_FILTER(mk(), fetch=False)
                st2 = torch.cuda.ExternalStream(d2.stream(), device=local)
                for _ in range(5):
                    d2.filter(DT)
                d2.sync()
                n2 = 200
                a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a2.record(st2)
                for _ in range(n2):
                    d2.filter(DT)
                b2.record(st2)
                d2.sync()
                ms2 = a2.elapsed_time(b2) / n2
                taps2 = d2.taps_per_step
                sweep[name] = dict(cells=d2.n_cells, ms_per_step=ms2, cell_updates_per_s=d2.n_cells / (ms2 * 1e-3),
                                   equivalent_tflops=2 * taps2 / (ms2 * 1e-3) / 1e12,
                                   l2_note="back-to-back steps, no flush (context only)")
                d2.close()
            except Exception as e:
                sweep[name] = dict(error=str(e)[:160])

    cfg = common_config(plane)
    extra = dict(taps_per_cell=(taps_y + taps_z) / cells, noise="generate (counter-based pcg32, spec v2)",
                 l2="flushed between steps (256 MiB write)" if flush else f"per-step working set {ws_bytes / 2**20:.0f} MiB > 126 MiB L2, no flush",
                 parallelism=f"{world} independent plane(s), one per GPU")
    line = dict(metric=METRIC, value=value, unit="cell-updates/s", n_gpus=world, steps=K, warmup=Wm, ms_per_step=step_ms,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=cfg, workload_detail=extra,
                clocks=clocks, gpu_launches=launches_per_step * K, wall_ms_per_step=1e3 * t_wall / K,
                e2e=dict(value=e2e_value, unit="cell-updates/s", h2d_bytes_per_step=8, d2h_bytes_per_step=40 * cells, steps=Ke,
                         call="dfb_filter_to_host (filter(dt) + u',v',w',T',rho' into pinned host arrays); input is the scalar dt",
                         pipelined=dict(value=e2e_pipelined, unit="cell-updates/s",
                                        call="dfb_filter_to_host_begin/_end with two sets of pinned arrays: the copy of step t under the compute of step t+1"),
                         facade=facade),
                roofline=roofline, cpu_baseline=cpu, other_configs=sweep, batched_planes=batched, slab=slab)
    print(json.dumps(line), flush=True)
    df.close()
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sweep", action="store_true", help="skip the brief runs of the other named configurations and the batched planes")
    ap.add_argument("--no-slab", action="store_true", help="N > 1: skip the config-4 slab job")
    ap.add_argument("--no-facade", action="store_true", help="skip the C++ facade end-to-end leg")
    ap.add_argument("--no-full-plane", action="store_true", help="reference arm: skip the one whole-plane step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write u', v', w', T', rho' of the last timed step to DIR/<field>.npy "
                    "(float64, at most 64 MB in all: a fixed sample of the cells when the plane is larger; rank 0's plane only)")
    args = ap.parse_args()
    import _dfb_import  # noqa: F401
    from digital_filtering_b200 import workloads as W
    if args.workload not in W.NAMED:
        raise SystemExit(f"unknown workload {args.workload}; choose from {sorted(W.NAMED)}")
    plane = W.NAMED[args.workload]()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes what the B200 arm computed; the reference arm does not support it")
        run_reference_arm(args, plane)
    else:
        run_b200(args, plane)


if __name__ == "__main__":
    main()
