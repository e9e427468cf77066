"""Long generate-mode runs against the oracle, step by step, across every way of driving a handle.

A host model of a handle (Model, tests/oracle_harness.py) is driven in lock step with the library.  Per plane it holds the step
counter, filt_old, the last u', v', w', T', rho', the N2 sums and the correlation sums and ring; each step is oracle.step (or the
periodic restatement, periodic_step in tests/oracle_harness.py) on the oracle's noise for (seed, plane_id + p, field, step).  After
every operation the library's fields, state, noise and statistics must match the model.  Comparing one handle with another cannot
see an error in what run_step decides (which noise set a step reads, whether the prefetched set holds this step's noise, when N2
and the correlation sums accumulate), because both sides go through the same run_step; the oracle can.

CPU: the model against plain oracle.step chains, and the operation generator.  GPU (-m gpu): one scenario per decision of run_step /
dfb_set_state / dfb_generate_noise, seeded random sequences of ~40 operations, on every y-sweep form, simple kernels, periodic planes,
a batch of 3 planes and the look-ahead y-sweep; invalid dt is refused and changes nothing; dt = 0 and dt >> Lt give exact results."""
import ctypes as C

import numpy as np
import pytest

from conftest import normwise_close
from oracle_harness import Model, np_sums, periodic_step

gpu = pytest.mark.gpu
TOL = 1e-12
SEED = 29
PLANE_ID = 2
LAGS_A = (9, 7, 3)                   # (L_z, L_y, L_t)
LAGS_B = (4, 0, 5)                   # changed lags: y off, more time lags than some runs have steps
DT = (1e-7, 2e-7, 3e-7, 5e-8)        # Lt is 1.2e-6 (u) and 4.5e-7 (v, w): every step blends


# ---------------------------------------------------------------------------------------------
# operation sequences
# ---------------------------------------------------------------------------------------------
def random_ops(seed, n=40):
    """n operations drawn from numpy.random.default_rng(seed): every kind of call, with arguments relative to the counter at the
    time the operation runs (resolved by Driver.apply), never more than two pipelined copies outstanding; the outstanding ones
    are collected at the end."""
    rng = np.random.default_rng(seed)
    kinds = ["filter", "to_host", "begin", "end", "batch", "first", "set_state", "set_state_none", "generate", "timing", "stats",
             "corr", "get_noise"]
    w = np.array([8, 2, 3, 3, 2, 2, 3, 1, 3, 1, 2, 2, 1], dtype=float)
    ops, pending = [], 0
    while len(ops) < n:
        k = kinds[rng.choice(len(kinds), p=w / w.sum())]
        dt = float(DT[rng.integers(len(DT))])
        if k == "begin" and pending == 2 or k == "end" and pending == 0:
            continue
        pending += {"begin": 1, "end": -1}.get(k, 0)
        if k in ("filter", "to_host", "begin"):
            ops.append((k, dt))
        elif k == "batch":
            ops.append((k, [float(DT[i]) for i in rng.integers(len(DT), size=int(rng.integers(1, 4)))]))
        elif k in ("set_state", "set_state_none", "generate"):
            ops.append((k, int(rng.integers(-4, 5))))              # earlier, the same or a later step, either parity
        elif k == "stats":
            ops.append((k, bool(rng.integers(2))))
        elif k == "corr":
            ops.append((k, [LAGS_A, LAGS_B, None][rng.integers(3)]))
        else:
            ops.append((k,))
    ops += [("end",)] * pending
    return ops


class Driver:
    """A library handle and its model, advanced together; check() compares them after every operation."""

    def __init__(self, dfb, O, plane, nplanes=1, periodic=False, **kw):
        self.dfb, self.O = dfb, O
        cfg = dfb.DFConfig.from_plane(plane, seed=SEED, plane_id=PLANE_ID, periodic_z=int(periodic), **kw)
        self.df = dfb.DIGITAL_FILTER(cfg, fetch=False, nplanes=nplanes)
        self.m = Model(O, plane, SEED, PLANE_ID, nplanes=nplanes, periodic=periodic)
        self.m.first_step()                                         # the constructor's step
        self.P, self.n = nplanes, plane["Ny"] * plane["Nz"]
        self.pending = []                                           # pipelined copies: (host arrays, expected fields)
        self.history = {self.m.step: self.m.state_for_library()}    # filt_old after each step, by counter
        self.timing = False
        self.check("create")

    def close(self):
        self.df.close()

    # ---- the comparison ----
    def check(self, what):
        df, m = self.df, self.m
        for p in range(self.P):
            for i in range(5):
                ok, r = normwise_close(df.get(i, plane=p), m.out[p, i], TOL)
                assert ok, (what, "field", p, i, r)
        fo, step = df.get_state()
        assert step == m.step, (what, step, m.step)
        ok, r = normwise_close(fo, m.state_for_library(), TOL)
        assert ok, (what, "filt_old", r)
        if m.stats is not None:
            for p in range(self.P):
                for i in range(6):
                    got, cnt = df.stats(i, plane=p)
                    assert cnt == m.stats_count, (what, "N2 count", cnt, m.stats_count)
                    ok, r = normwise_close(got, m.stats[p, i], TOL)
                    assert ok, (what, "N2", p, i, r)
        if m.lags is not None:
            assert df.corr_lags == tuple(m.lags), (what, df.corr_lags, m.lags)
            for d in m.csum:
                for p in range(self.P):
                    for f in range(3):
                        S, pairs, cnt = df.corr(f, d, normalized=False, plane=p)
                        assert cnt == m.corr_count, (what, "corr count", cnt, m.corr_count)
                        assert np.array_equal(pairs, m.pairs(d)), (what, "pairs", d, pairs, m.pairs(d))
                        ok, r = normwise_close(S, m.csum[d][p, f], TOL)
                        assert ok, (what, "corr", d, p, f, r)

    def check_noise(self, what):
        """dfb_get_noise (whole-plane, single-plane handles) against the oracle noise of the step the model says was consumed or
        generated last, bit for bit"""
        if self.P != 1 or self.m.noise_step is None:
            return
        for f in range(3):
            rys, hal = self.df.get_noise(f)
            ref_rys, ref_hal = self.m.noise(0, f, self.m.noise_step)
            assert np.array_equal(rys, ref_rys), (what, "r_ys", f, self.m.noise_step)
            if ref_hal is not None:
                assert np.array_equal(hal, ref_hal), (what, "halo", f, self.m.noise_step)

    def _stepped(self, what):
        self.history[self.m.step] = self.m.state_for_library()
        self.check(what)
        self.check_noise(what)

    def _host(self):
        return [np.zeros((self.P, self.n)) for _ in range(5)]

    def _ptrs(self, arrs):
        return [a.ctypes.data_as(C.c_void_p) for a in arrs]

    def _expect_host(self, arrs, expect, what):
        for i in range(5):
            for p in range(self.P):
                ok, r = normwise_close(arrs[i][p].reshape(expect.shape[2:]), expect[p, i], TOL)
                assert ok, (what, p, i, r)

    # ---- the operations ----
    def filter(self, dt):
        self.df.filter(dt)
        self.m.filter(dt)
        self._stepped(("filter", dt))

    def to_host(self, dt):
        arrs = self._host()
        self.dfb._check(self.dfb.lib().dfb_filter_to_host(self.df._h, dt, *self._ptrs(arrs)))
        self.m.filter(dt)
        self._expect_host(arrs, self.m.out, ("to_host", dt))
        self._stepped(("to_host", dt))

    def begin(self, dt):
        arrs = self._host()
        self.dfb._check(self.dfb.lib().dfb_filter_to_host_begin(self.df._h, dt, *self._ptrs(arrs)))
        self.m.filter(dt)
        self.pending.append((arrs, self.m.out.copy()))
        self._stepped(("begin", dt))

    def end(self):
        self.dfb._check(self.dfb.lib().dfb_filter_to_host_end(self.df._h))
        arrs, expect = self.pending.pop(0)
        self._expect_host(arrs, expect, "end")

    def batch(self, dts):
        out = np.zeros((len(dts), 5, self.P, self.n))
        self.df.filter_batch(np.array(dts), out)
        for s, dt in enumerate(dts):
            self.m.filter(dt)
            self._expect_host(list(out[s]), self.m.out, ("batch", s, dt))
            self.history[self.m.step] = self.m.state_for_library()
        self._stepped(("batch", tuple(dts)))

    def first(self):
        self.df.first_step()
        self.m.first_step()
        self._stepped("first_step")

    def set_state(self, step, fo="history"):
        """fo: "history" = filt_old as it was after step `step` (the current one if the run never got there), None = counter only,
        or an array"""
        if isinstance(fo, str):
            fo = self.history.get(step, self.m.state_for_library())
        self.df.set_state(fo, step)
        self.m.set_state(fo, step)
        self.check(("set_state", step, fo is None))

    def generate(self, k):
        self.df.generate_noise(k)
        self.m.generate_noise(k)
        self.check(("generate_noise", k))
        self.check_noise(("generate_noise", k))

    def set_timing(self, on):
        self.df.set_timing(on)
        self.timing = on
        self.check(("timing", on))

    def stats_enable(self, on):
        self.df.stats_enable(on)
        self.m.stats_enable(on)
        self.check(("stats", on))

    def corr_enable(self, lags):
        if lags is None:
            self.df.corr_enable(on=False)
            self.m.corr_enable(False)
        else:
            self.df.corr_enable(*lags)
            self.m.corr_enable(True, lags)
        self.check(("corr", lags))

    def apply(self, op):
        k, a = op[0], op[1:]
        if k in ("set_state", "set_state_none"):
            self.set_state(max(0, self.m.step + a[0]), "history" if k == "set_state" else None)
        elif k == "generate":
            self.generate(max(0, self.m.step + a[0]))
        elif k == "timing":
            self.set_timing(not self.timing)
        elif k == "get_noise":
            self.check_noise("get_noise")
        else:
            {"filter": self.filter, "to_host": self.to_host, "begin": self.begin, "end": self.end, "batch": self.batch,
             "first": self.first, "stats": self.stats_enable, "corr": self.corr_enable}[k](*a)

    def drain(self):
        while self.pending:
            self.end()


# ---------------------------------------------------------------------------------------------
# CPU: the model against plain oracle.step chains; the generator
# ---------------------------------------------------------------------------------------------
def _chain(O, plane, fo, steps, plane_id=PLANE_ID):
    """plain oracle.step over [(counter, dt, first)] from filt_old `fo` [3][Ny][Nz]: the five fields after each step, with T' / rho'
    carried over a first step"""
    Ny, Nz = plane["Ny"], plane["Nz"]
    outs, T, rho = [], np.zeros((Ny, Nz)), np.zeros((Ny, Nz))
    for s, dt, first in steps:
        rys = [O.noise_rys(SEED, plane_id, f, s, Ny, plane["Ny_max"][f], Nz) for f in range(3)]
        hal = [O.noise_halo(SEED, plane_id, f, s, Ny, plane["Nz_max"][f]) for f in range(3)]
        o = O.step(plane, rys, hal, fo, dt, first_step=first)
        fo = o["filt_old"]
        if not first:
            T, rho = o["T"], o["rho"]
        outs.append(np.concatenate([o["fluc"], T[None], rho[None]]))
    return outs, fo


@pytest.fixture(scope="module")
def small(O, W):
    return O.half_widths(W.plane_profile(24, 40, 6, 6))


def test_model_rewinds_and_counter_moves_follow_oracle_chains(O, small):
    """set_state to an earlier step with that step's filt_old, set_state(None, later) and a first step in the middle of the run"""
    m = Model(O, small, SEED, PLANE_ID)
    m.first_step()
    m.filter(1e-7)
    saved = m.state_for_library().copy()                          # filt_old after step 1, counter 2
    m.filter(2e-7); m.filter(3e-7)
    m.set_state(saved, 2)
    m.filter(5e-8)
    outs, fo = _chain(O, small, np.zeros((3, 24, 40)), [(0, 0.0, True), (1, 1e-7, False), (2, 5e-8, False)])
    assert np.array_equal(m.out[0], outs[-1]) and np.array_equal(m.fo[0], fo) and m.step == 3
    m.set_state(None, 7)                                          # only the counter moves
    m.filter(1e-7)
    m.first_step()                                                # no blend, T' / rho' stay
    m.filter(2e-7)
    outs2, fo2 = _chain(O, small, fo, [(7, 1e-7, False), (8, 0.0, True), (9, 2e-7, False)])
    assert np.array_equal(m.out[0], outs2[-1]) and np.array_equal(m.fo[0], fo2) and m.step == 10
    assert np.array_equal(outs2[1][3:], outs2[0][3:]) and not np.array_equal(outs2[1][:3], outs2[0][:3])
    assert m.noise_step == 9


def test_model_statistics_across_first_step_and_set_state(O, small):
    """N2: every non-first step since dfb_stats_enable(1), across set_state.  Correlation sums: z and y over the same steps, t only
    between steps with no set_state in between (the ring empties), pairs counted from the steps the ring held"""
    m = Model(O, small, SEED, PLANE_ID)
    m.first_step()
    m.stats_enable(True)
    L = (5, 4, 3)
    m.corr_enable(True, L)
    m.filter(1e-7); m.filter(2e-7)
    m.first_step()                                                # counted by neither
    m.filter(1e-7)
    saved = m.state_for_library().copy()                          # counter 5
    m.filter(3e-7)
    m.set_state(saved, 5)
    m.filter(2e-7); m.filter(1e-7)
    steps = [(0, 0.0, True), (1, 1e-7, False), (2, 2e-7, False), (3, 0.0, True), (4, 1e-7, False)]
    outs, fo = _chain(O, small, np.zeros((3, 24, 40)), steps)
    assert np.array_equal(fo, saved)
    a = [outs[1], outs[2], outs[4]]                               # accumulated before the rewind (the first steps are not)
    outs_b, _ = _chain(O, small, saved, [(5, 3e-7, False)])
    outs_c, _ = _chain(O, small, saved, [(5, 2e-7, False), (6, 1e-7, False)])
    acc = a + outs_b + outs_c
    assert m.stats_count == 6
    ref = np.stack([sum(x[i] * x[i] for x in acc) for i in range(5)] + [sum(x[0] * x[1] for x in acc)])
    assert normwise_close(m.stats[0], ref, 1e-13)[0]
    for f in range(3):
        before = np_sums([x[f] for x in a + outs_b], L)
        after = np_sums([x[f] for x in outs_c], L)
        for d in range(3):
            ok, r = normwise_close(m.csum[d][0, f], before[d][0] + after[d][0], 1e-13)
            assert ok, (f, d, r)
            assert np.array_equal(m.pairs(d), before[d][1] + after[d][1]), (d, m.pairs(d))
    assert m.corr_count == 6
    m.stats_enable(False); m.corr_enable(False)
    m.filter(1e-7)
    assert m.stats_count == 6 and m.corr_count == 6              # off: kept, not accumulated
    m.stats_enable(True)
    assert m.stats_count == 0 and not m.stats.any()


def test_model_batch_planes_are_single_planes_and_periodic_uses_the_restatement(O, small):
    """plane p of a batch model is the single-plane model with plane_id + p; a periodic model steps through periodic_step"""
    b = Model(O, small, SEED, PLANE_ID, nplanes=2)
    s = Model(O, small, SEED, PLANE_ID + 1)
    for m in (b, s):
        m.first_step(); m.filter(1e-7); m.filter(2e-7)
    assert np.array_equal(b.out[1], s.out[0]) and not np.array_equal(b.out[0], b.out[1])
    pm = Model(O, small, SEED, PLANE_ID, periodic=True)
    pm.first_step(); pm.filter(1e-7)
    rys = lambda st: [O.noise_rys(SEED, PLANE_ID, f, st, 24, small["Ny_max"][f], 40) for f in range(3)]
    o0 = periodic_step(O, small, rys(0), np.zeros((3, 24, 40)), 0.0, first_step=True)
    o1 = periodic_step(O, small, rys(1), o0["filt_old"], 1e-7)
    assert np.array_equal(pm.out[0, :3], o1["fluc"]) and np.array_equal(pm.out[0, 3], o1["T"])


RANDOM_SEEDS = [2, 4]               # each of these draws every kind of operation


def test_random_sequences_are_fixed_and_cover_every_operation():
    a, b = random_ops(RANDOM_SEEDS[0]), random_ops(RANDOM_SEEDS[0])
    assert a == b and a != random_ops(RANDOM_SEEDS[1])
    for s in RANDOM_SEEDS:
        assert {op[0] for op in random_ops(s)} == {"filter", "to_host", "begin", "end", "batch", "first", "set_state", "set_state_none",
                                                   "generate", "timing", "stats", "corr", "get_noise"}, s
    for s in RANDOM_SEEDS:
        ops, pending = random_ops(s), 0
        for op in ops:
            pending += {"begin": 1, "end": -1}.get(op[0], 0)
            assert 0 <= pending <= 2
        assert pending == 0


# ---------------------------------------------------------------------------------------------
# GPU: configurations
# ---------------------------------------------------------------------------------------------
# name: (plane_profile arguments, environment, config keywords, batch size, y-sweep form dfb_info(10) must report)
CONFIGS = {
    "tuned-run": ((72, 530, 20, 16), {"DFB_Y_MODE": "2"}, {}, 1, 2),
    "tuned-dense": ((64, 130, 16, 12), {"DFB_Y_MODE": "0"}, {}, 1, 0),
    "tuned-chunk": ((72, 530, 20, 16), {"DFB_Y_MODE": "1"}, {}, 1, 1),
    "simple": ((64, 130, 16, 12), {}, {"kernel_variant": 1}, 1, -1),
    "periodic": ((64, 130, 16, 12), {"DFB_Y_MODE": "2"}, {"periodic_z": 1}, 1, 2),
    "batch3": ((64, 130, 16, 12), {"DFB_Y_MODE": "2"}, {}, 3, 2),
}


def _driver(dfb, O, W, monkeypatch, name):
    shape, env, kw, nplanes, form = CONFIGS[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)                                    # read when the handle is created
    plane = O.half_widths(W.plane_profile(*shape))
    kw = dict(kw)
    periodic = bool(kw.pop("periodic_z", 0))
    d = Driver(dfb, O, plane, nplanes=nplanes, periodic=periodic, **kw)
    assert d.df.info(10) == form, (name, d.df.info(10))
    assert d.df.periodic_z == periodic
    return d


# ---------------------------------------------------------------------------------------------
# GPU: one scenario per decision
# ---------------------------------------------------------------------------------------------
def sc_prefetch_every_step(d):
    """run_step: `buf_step[b] != H.step` -- a long run of plain steps, every one of them reading the set the look-ahead filled
    after the step before"""
    for i in range(12):
        d.filter(DT[i % 4])


def sc_generate_noise_then_filter(d):
    """dfb_generate_noise(k) writes set k & 1 and records buf_step = k: the next step must regenerate unless k is its own step,
    and the look-ahead into that set must come after it (ev_noise)"""
    s = d.m.step
    d.generate(s)                  # the next step's own noise: reused
    d.filter(1e-7)
    d.generate(s - 1)              # an earlier step, the other parity from the next one
    d.filter(2e-7)
    d.generate(d.m.step + 2)       # a later step of the next one's parity: overwrites the prefetched set
    d.filter(1e-7)
    d.generate(d.m.step + 1)       # a later step of the look-ahead's parity
    d.filter(3e-7)
    d.filter(1e-7)
    d.generate(d.m.step + 5)
    d.generate(d.m.step)
    d.filter(2e-7)


def sc_set_state_later_and_counter_only(d):
    """dfb_set_state: `step != h->step` drops both prefetched sets -- forward jumps of either parity, the same step (sets kept),
    and set_state(NULL, s), which moves only the counter"""
    d.filter(1e-7)
    d.set_state(d.m.step + 3)
    d.filter(2e-7)
    d.set_state(d.m.step + 2)
    d.filter(1e-7)
    d.set_state(d.m.step)
    d.filter(3e-7)
    d.set_state(d.m.step + 1, fo=None)
    d.filter(1e-7)
    d.filter(2e-7)


def sc_rewinds(d):
    """dfb_set_state back by one and by two steps (the second lands on the set the look-ahead is writing), and back to 0"""
    for _ in range(3):
        d.filter(1e-7)
    s = d.m.step
    d.filter(2e-7); d.filter(2e-7)
    d.set_state(s)
    d.filter(3e-7)
    d.set_state(s - 1)
    d.filter(1e-7); d.filter(1e-7)
    d.set_state(0, fo=None)
    d.filter(2e-7)


def sc_timing_on_and_off(d):
    """`!H.timing`: timing mode generates each step's noise on the main stream, no look-ahead; switched on and off mid-run, the
    first step after each switch reads what the previous mode left"""
    d.filter(1e-7)
    d.set_timing(True)
    d.filter(2e-7); d.filter(1e-7)
    d.generate(d.m.step)
    d.filter(1e-7)
    d.set_timing(False)
    d.filter(3e-7); d.filter(1e-7)
    d.set_timing(True)
    d.set_state(d.m.step - 2)
    d.filter(2e-7)
    d.set_timing(False)
    d.filter(1e-7)


def sc_first_step_with_statistics(d):
    """`accumulate = stats_on && !first` and `corr_on && !first`: dfb_first_step in the middle of a run accumulates neither N2 nor
    the correlation sums, and does not blend"""
    d.stats_enable(True)
    d.corr_enable(LAGS_A)
    d.filter(1e-7); d.filter(2e-7)
    d.first()
    d.filter(1e-7)
    d.first()
    d.first()
    d.filter(3e-7); d.filter(1e-7)


def sc_statistics_across_rewinds(d):
    """dfb_set_state keeps the N2 sums and empties the correlation ring (`corr.ring_count = 0`): no temporal pair reaches back
    across a rewind, forward jump or counter-only move"""
    d.stats_enable(True)
    d.corr_enable(LAGS_A)
    for _ in range(4):
        d.filter(1e-7)
    d.set_state(d.m.step - 2)
    d.filter(2e-7); d.filter(1e-7); d.filter(1e-7)
    d.set_state(d.m.step + 3, fo=None)
    d.filter(1e-7); d.filter(3e-7)
    d.set_state(d.m.step)
    d.filter(1e-7)


def sc_statistics_switches(d):
    """dfb_stats_enable / dfb_corr_enable on and off and with changed lags mid-run: (1) zeroes, (0) keeps and stops"""
    d.stats_enable(True)
    d.corr_enable(LAGS_A)
    d.filter(1e-7); d.filter(2e-7)
    d.stats_enable(False)
    d.corr_enable(None)
    d.filter(1e-7)
    d.corr_enable(LAGS_A)
    d.filter(1e-7)
    d.stats_enable(True)
    d.corr_enable(LAGS_B)
    d.filter(2e-7); d.filter(1e-7); d.filter(3e-7)


def sc_pipelined_and_batched(d):
    """dfb_filter_to_host_begin/_end (two in flight), dfb_filter_to_host and dfb_filter_batch between them: every path through
    run_step consumes the next step's noise"""
    d.begin(1e-7)
    d.begin(2e-7)
    d.end()
    d.filter(1e-7)
    d.begin(3e-7)
    d.end()
    d.end()
    d.batch([1e-7, 2e-7, 1e-7])
    d.to_host(2e-7)
    d.set_state(d.m.step - 3)
    d.batch([3e-7, 1e-7])


SCENARIOS = [sc_prefetch_every_step, sc_generate_noise_then_filter, sc_set_state_later_and_counter_only, sc_rewinds,
             sc_timing_on_and_off, sc_first_step_with_statistics, sc_statistics_across_rewinds, sc_statistics_switches,
             sc_pipelined_and_batched]


@gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("scenario", SCENARIOS, ids=lambda f: f.__name__[3:])
def test_scenario(dfb, O, W, monkeypatch, config, scenario):
    d = _driver(dfb, O, W, monkeypatch, config)
    scenario(d)
    d.drain()
    d.close()


@gpu
@pytest.mark.parametrize("config", list(CONFIGS))
@pytest.mark.parametrize("seed", RANDOM_SEEDS)
def test_random_sequence(dfb, O, W, monkeypatch, config, seed):
    d = _driver(dfb, O, W, monkeypatch, config)
    for i, op in enumerate(random_ops(seed)):
        try:
            d.apply(op)
        except AssertionError as e:
            raise AssertionError(f"operation {i} {op}: {e}") from None
    d.close()


# ---------------------------------------------------------------------------------------------
# GPU: dt
# ---------------------------------------------------------------------------------------------
def _snapshot(d):
    """everything a refused call must leave alone, as copied back from the library"""
    df, snap = d.df, {}
    for p in range(d.P):
        for w in range(8):
            snap["field", p, w] = df.get(w, plane=p)
    snap["state"] = df.get_state()
    if d.m.stats is not None:
        for p in range(d.P):
            for i in range(6):
                snap["N2", p, i] = df.stats(i, plane=p)
    if d.m.lags is not None:
        for dd in d.m.csum:
            for p in range(d.P):
                for f in range(3):
                    snap["corr", dd, p, f] = df.corr(f, dd, normalized=False, plane=p)
    if d.P == 1:
        for f in range(3):
            snap["noise", f] = df.get_noise(f)
    return snap


def _same(a, b):
    if isinstance(a, tuple):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    if isinstance(a, np.ndarray):
        return np.array_equal(a, b)
    return a == b


BAD_DT = [-1e-7, -1e300, float("nan"), float("inf"), float("-inf")]


@gpu
@pytest.mark.parametrize("entry", ["filter", "filter_f", "to_host", "to_host_f", "begin", "get_rms", "batch@0", "batch@1", "batch@2"])
@pytest.mark.parametrize("config", ["tuned-run", "batch3"])
def test_invalid_dt_is_refused_and_changes_nothing(dfb, O, W, monkeypatch, config, entry):
    """negative, NaN and infinite dt: DFB_ERR_ARG naming dt from every entry point that steps (dfb_filter_batch with the bad value
    at any position of its array), and the handle -- counter, fields, filt_old, noise, N2 and correlation sums and ring -- bitwise
    as it was; the next valid step matches the model"""
    d = _driver(dfb, O, W, monkeypatch, config)
    d.stats_enable(True)
    d.corr_enable(LAGS_A)
    d.filter(1e-7); d.filter(2e-7)
    L, h = dfb.lib(), d.df._h
    arrs = d._host()
    for bad in BAD_DT:
        before = _snapshot(d)
        if entry == "filter":
            rc = L.dfb_filter(h, bad)
        elif entry == "filter_f":
            rc = L.dfb_filter_f(C.byref(C.c_void_p(h.value)), C.byref(C.c_double(bad)))
        elif entry == "to_host":
            rc = L.dfb_filter_to_host(h, bad, *d._ptrs(arrs))
        elif entry == "to_host_f":
            rc = L.dfb_filter_to_host_f(C.byref(C.c_void_p(h.value)), C.byref(C.c_double(bad)), *d._ptrs(arrs))
        elif entry == "begin":
            rc = L.dfb_filter_to_host_begin(h, bad, *d._ptrs(arrs))
        elif entry == "get_rms":
            rc = L.dfb_get_rms(h, 3, bad)
        else:
            dts = np.array([1e-7, 2e-7, 3e-7])
            dts[int(entry[-1])] = bad
            out = np.zeros((3, 5, d.P, d.n))
            rc = L.dfb_filter_batch(h, 3, dts.ctypes.data_as(dfb.c_dp), out.ctypes.data_as(C.c_void_p))
        assert rc == dfb.ERR_ARG, (entry, bad, rc)
        assert b"dt" in L.dfb_last_error(), L.dfb_last_error()
        after = _snapshot(d)
        assert before.keys() == after.keys()
        for k in before:
            assert _same(before[k], after[k]), (entry, bad, k)
        if entry == "begin":
            assert L.dfb_filter_to_host_end(h) == dfb.ERR_STATE         # nothing was begun
    d.filter(1e-7)                                                      # the next valid step: the model's
    d.batch([1e-7, 2e-7])
    d.close()


@gpu
@pytest.mark.parametrize("config", ["tuned-run", "simple", "periodic"])
def test_dt_zero_and_dt_far_beyond_Lt_are_exact(dfb, O, W, monkeypatch, config):
    """dt = 0: alpha = 1, filt == filt_old, so after a step that was not a first step all five outputs repeat bit for bit, after a
    first step u', v', w' do.  dt >> Lt: alpha = 0, u', v', w' are those of the unblended step dfb_first_step gives at the same
    counter from the same filt_old"""
    d = _driver(dfb, O, W, monkeypatch, config)
    d.filter(1e-7); d.filter(2e-7)
    prev = [d.df.get(w) for w in range(5)]
    d.filter(0.0)
    for w in range(5):
        assert np.array_equal(d.df.get(w), prev[w]), ("dt = 0", w)
    d.first()
    prev = [d.df.get(w) for w in range(5)]
    d.filter(0.0)
    for w in range(3):
        assert np.array_equal(d.df.get(w), prev[w]), ("dt = 0 after a first step", w)
    fo, s = d.df.get_state()
    d.filter(1.0)                                                       # pi * 1 / Lt ~ 3e6: alpha = exp(-3e6) = 0
    far = [d.df.get(w) for w in range(3)]
    d.set_state(s, fo=fo)
    d.first()
    for w in range(3):
        assert np.array_equal(d.df.get(w), far[w]), ("dt >> Lt", w)
    d.filter(3e-7)
    d.close()
