"""The multi-frame ("fused") pixel model's schedules against the CPU oracle.

A chunk of `max_frames_per_step` frames first runs through the multi-frame kernels as one segment. When a frame
breaks their assumption (more than kFusedMaxN = 31 events of one pixel, more than iter_cap, or the refractory filter
active: refractory_period_s > dt / max_n), v2e_emu_collect splits the chunk at the offending frames and runs the
runs between them through the multi-frame kernels again, the rest frame by frame (emu.cu, v2e_emu_collect). The
clips below are scripted so that every frame's maximum is chosen: a smooth background making 0-2 events per pixel
and frame, and small patches whose level steps by a chosen number of thresholds (tests/helpers.py).

The CPU part pins, per scenario, the oracle's per-frame maxima, which frames break the assumption and the schedule
the rule produces (restated below, with the back-off). The GPU part runs generate_events_batch on the same frames
and compares rows, counters and state with the oracle bit for bit, and the schedule statistics of the handle with
the restatement: a run that quietly went frame by frame fails."""
import copy
import ctypes

import numpy as np
import pytest

from helpers import assert_events_equal, scripted_clip

K_FUSED_MAX_N = 31
SEED = 17
DT = 2.0 ** -6                 # dyadic frame interval: dt / max_n and the frame-time differences are exact
REFR = 2.0 ** -8               # refractory period of the refractory scenarios: the filter runs iff max_n > 4

SCALAR = dict(pos_thres=0.05, neg_thres=0.05, sigma_thres=0.0, cutoff_hz=0.0, leak_rate_hz=0.0,
              shot_noise_rate_hz=0.0)
# v2e's CLI defaults (v2e_args.py) with shot noise off and a deterministic leak
CLI = dict(pos_thres=0.2, neg_thres=0.2, sigma_thres=0.03, cutoff_hz=300.0, leak_rate_hz=0.01,
           leak_jitter_fraction=0.0, shot_noise_rate_hz=0.0, refractory_period_s=0.0005)


# ---- the rule of v2e_emu_collect, restated --------------------------------------------------------------------
def is_bad(m, dt, refr, iter_cap):
    """The plan's test of one frame (emu.cu emu_fused_plan_kernel; emulator.py:792, 830)."""
    return m > K_FUSED_MAX_N or m > iter_cap or (refr > 0 and m > 0 and refr > dt / m)


def segment(bad, a, b, fb):
    """Re-schedule the rejected segment [a, b): runs of bad frames (fb always counts as bad) go frame by frame
    (kind 1), runs of >= 2 good frames through the multi-frame kernels (kind 0); a lone good frame joins the
    frame-by-frame segment before it; adjacent frame-by-frame segments are merged. Returns (segments, n_bad)."""
    neu, n_bad, f = [], 0, a
    while f < b:
        e = f
        if f == fb or bad(f):
            while e < b and (e == fb or bad(e)):
                e += 1
                n_bad += 1
            neu.append([1, f, e])
        else:
            while e < b and not (e == fb or bad(e)):
                e += 1
            if e - f >= 2:
                neu.append([0, f, e])
            elif neu and neu[-1][0] == 1:
                neu[-1][2] = e
            else:
                neu.append([1, f, e])
        f = e
    merged = []
    for q in neu:
        if merged and merged[-1][0] == 1 and q[0] == 1:
            merged[-1][2] = q[2]
        else:
            merged.append(list(q))
    return merged, n_bad


class ScheduleModel:
    """What one emulator handle does with a sequence of chunks: back-off (the next 1, 2, 4 ... 64 chunks frame by
    frame after a chunk with more than a quarter of its frames bad, reset by a wholly accepted chunk), rejection
    rounds (a mispredicted frame costs another round) and the resulting counters of v2e_emu_fused_stats /
    v2e_emu_fused_frames."""

    def __init__(self, real_bad, predict):
        self.real_bad, self.predict = real_bad, predict
        self.skip = self.penalty = 0
        self.chunks = self.rejected = self.multi = self.single = 0
        self.log = []

    def chunk(self, g0, n):
        if n < 2:
            self.log.append("classic")
            return
        if self.skip > 0:
            self.skip -= 1
            self.log.append("skip")
            return
        self.chunks += 1
        sched, k = [[0, g0, g0 + n]], 0
        while True:
            k = next((i for i in range(k, len(sched)) if sched[i][0] == 0 and
                      any(self.real_bad(q) for q in range(sched[i][1], sched[i][2]))), None)
            if k is None:
                break
            _, a, b = sched[k]
            fb = next(q for q in range(a, b) if self.real_bad(q))
            pred_bad = self.predict(a, b)
            new, n_bad = segment(pred_bad, a, b, fb)
            self.rejected += 1
            sched[k:k + 1] = new
            if 4 * n_bad > b - a:
                self.penalty = min(2 * self.penalty, 64) if self.penalty else 1
                self.skip = self.penalty
        if sched == [[0, g0, g0 + n]]:
            self.penalty = 0
        for kind, a, b in sched:
            if kind == 0:
                self.multi += b - a
            else:
                self.single += b - a
        self.log.append(" ".join("%s%d-%d" % ("MS"[kind], a - g0, b - g0) for kind, a, b in sched))


# ---- scenarios ---------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, frames, ts, kw, chunk, calls=None, iter_cap=1024, hint=None, shard=False):
        self.frames, self.ts, self.kw, self.chunk = frames, np.asarray(ts, np.float64), kw, chunk
        self.calls = calls or [len(frames)]          # end frame of each generate_events_batch call
        self.iter_cap, self.hint, self.shard = iter_cap, hint, shard

    def chunk_starts(self):
        """(first frame, length) of every chunk, call by call (a fresh emulator's frame 0 only initialises)."""
        out, s = [], 1
        for e in self.calls:
            for f in range(s, e, self.chunk):
                out.append((f, min(self.chunk, e - f)))
            s = e
        return out


def _targets(T, at):
    t = [0] * T
    for k, v in at.items():
        t[k] = v
    return t


def _clip(T, at, H=24, W=40, at2=None, start=30, start2=30, **kw):
    patches = [(8, 12, 3, _targets(T, at), start)]
    if at2:
        patches.append((8, 26, 3, _targets(T, at2), start2))
    return scripted_clip(H, W, T, patches, **kw)


def _bad_at(chunk0, local, n=40):
    return {chunk0 + q: n for q in local}


def make_case(name):
    ts = lambda T: np.arange(T) * DT
    if name == "a_split":            # chunk 1: bad frame at position 4; chunk 2 accepted whole
        T = 21
        return Case(_clip(T, _bad_at(1, [4])), ts(T), SCALAR, 10)
    if name.startswith("b_"):
        local = {"b_first": [0], "b_last": [7], "b_lone": [1, 6], "b_adjacent": [3, 4],
                 "b_alternate": [1, 3, 5, 7]}[name]
        T = 25
        return Case(_clip(T, _bad_at(1, local)), ts(T), SCALAR, 8)
    if name == "c_mispredict":       # filter at position 3 passes 3 of 9 events: position 4 really bad, predicted good
        T = 13
        return Case(_clip(T, {4: 9}), ts(T), dict(SCALAR, refractory_period_s=REFR), 12)
    if name.startswith("d_"):        # back-off; chunk 3 is bad in every frame; d_calls: two generate_events_batch calls
        mixed, allbad = [1, 3, 6], list(range(8))
        bad = {1: mixed, 3: allbad, 6: mixed, 12: mixed}
        at = {}
        for c, local in bad.items():
            at.update(_bad_at(1 + 8 * (c - 1), local))
        T = 1 + 14 * 8
        return Case(_clip(T, at), ts(T), SCALAR, 8, calls=[25, T] if name == "d_calls" else None)
    if name.startswith("e_"):        # capacity abort: in a multi-frame segment after a frame-by-frame one, and back
        T = 17
        local = [0] if name == "e_in_multi" else [3]
        return Case(_clip(T, _bad_at(1, local)), ts(T), SCALAR, 8)
    if name == "f_31":
        T = 17
        return Case(_clip(T, {4: 31}), ts(T), SCALAR, 8)
    if name == "f_32":
        T = 17
        return Case(_clip(T, {4: 32}), ts(T), SCALAR, 8)
    if name == "f_63_64":            # the record's 6-bit count field saturates at 63
        T = 17
        return Case(_clip(T, {3: 63}, at2={6: 64}, start=0, start2=0), ts(T), SCALAR, 8)
    if name == "f_iter_cap":         # call 1: a frame at iter_cap (accepted); call 2: a frame above it
        T = 17
        return Case(_clip(T, {4: 8, 12: 9}), ts(T), SCALAR, 8, calls=[9, T], iter_cap=8)
    if name.startswith("g_"):        # dt / max_n == refractory_period_s: the filter does not run
        T = 17
        t = ts(T)
        if name == "g_shorter":
            t[4] -= 2.0 ** -10       # frame 4's dt one step of 2^-10 shorter: dt / 4 < refractory_period_s
        return Case(_clip(T, {4: 4}), t, dict(SCALAR, refractory_period_s=REFR), 8)
    if name.startswith("h_"):
        H, W, C, T, y, x, s = {"h_481px": (13, 37, 8, 17, 5, 17, 3), "h_63px": (7, 9, 8, 17, 2, 3, 2),
                               "h_1xN": (1, 301, 8, 17, 0, 150, 1), "h_Nx1": (211, 1, 8, 17, 100, 0, 1),
                               "h_T2": (24, 40, 8, 3, 8, 12, 3), "h_Tchunk1": (24, 40, 8, 10, 8, 12, 3)}[name]
        at = {} if T < 17 else _bad_at(1, [4])
        fr = scripted_clip(H, W, T, [(y, x, s, _targets(T, at), 30)])
        return Case(fr, ts(T), SCALAR, C)
    if name == "i_1280x720":         # v2e's CLI defaults at the headline size, one offending frame per chunk
        T, dt = 49, 2.0 ** -8
        tg = _targets(T, {1 + 17: 10, 25 + 19: 10})
        fr = scripted_clip(720, 1280, T, [(300, 600, 2, tg, 30)], th=0.2, cutoff_hz=300.0, dt=dt, seed=3)
        return Case(fr, np.arange(T) * dt, CLI, 24)
    if name == "j_sharded":          # pixel-sharded batched path: first bad frame at position 3 -> prefix replay
        T = 13
        return Case(_clip(T, _bad_at(1, [3]), H=50, W=64), ts(T), SCALAR, 6, shard=True)
    raise KeyError(name)


# per scenario: oracle maxima per frame, and what the schedule does with every chunk
EXPECT = {
    "a_split": dict(
        maxima=[0, 1, 2, 2, 2, 40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-4 S4-5 M5-10', 'M0-10']),
    "b_first": dict(
        maxima=[0, 40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['S0-1 M1-8', 'M0-8', 'M0-8']),
    "b_last": dict(
        maxima=[0, 1, 2, 2, 2, 2, 2, 2, 40, 2, 2, 2, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-7 S7-8', 'M0-8', 'M0-8']),
    "b_lone": dict(
        maxima=[0, 1, 40, 2, 2, 2, 2, 40, 2, 2, 2, 2, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['S0-2 M2-6 S6-8', 'M0-8', 'M0-8']),
    "b_adjacent": dict(
        maxima=[0, 1, 2, 2, 40, 40, 2, 2, 2, 2, 2, 2, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-3 S3-5 M5-8', 'M0-8', 'M0-8']),
    "b_alternate": dict(
        maxima=[0, 1, 40, 2, 40, 2, 40, 2, 40, 2, 2, 2, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['S0-8', 'skip', 'M0-8']),
    "c_mispredict": dict(
        maxima=[0, 1, 2, 2, 9, 6, 3, 2, 2, 2, 2, 2, 2],
        sched=['M0-3 S3-4 S4-5 M5-12']),
    "d_single": dict(
        maxima=[0, 1, 40, 2, 40, 2, 2, 40, 2, 2, 2, 1, 1, 1, 1, 1, 1, 40, 40, 40, 40, 40, 40, 40, 40, 1, 1, 1, 1, 1, 1,
                    1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 40, 2, 40, 2, 2, 40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2,
                    2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 40, 2, 40, 2, 2,
                    40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['S0-4 M4-6 S6-8', 'skip', 'S0-8', 'skip', 'skip', 'S0-4 M4-6 S6-8', 'skip', 'skip', 'skip', 'skip',
               'M0-8', 'S0-4 M4-6 S6-8', 'skip', 'M0-8']),
    "d_calls": dict(
        maxima=[0, 1, 40, 2, 40, 2, 2, 40, 2, 2, 2, 1, 1, 1, 1, 1, 1, 40, 40, 40, 40, 40, 40, 40, 40, 1, 1, 1, 1, 1, 1,
                    1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 40, 2, 40, 2, 2, 40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2,
                    2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 40, 2, 40, 2, 2,
                    40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['S0-4 M4-6 S6-8', 'skip', 'S0-8', 'skip', 'skip', 'S0-4 M4-6 S6-8', 'skip', 'skip', 'skip', 'skip',
               'M0-8', 'S0-4 M4-6 S6-8', 'skip', 'M0-8']),
    "e_in_multi": dict(
        maxima=[0, 40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['S0-1 M1-8', 'M0-8']),
    "e_in_single": dict(
        maxima=[0, 1, 2, 2, 40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-3 S3-4 M4-8', 'M0-8']),
    "f_31": dict(
        maxima=[0, 1, 2, 2, 31, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-8', 'M0-8']),
    "f_32": dict(
        maxima=[0, 1, 2, 2, 32, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-3 S3-4 M4-8', 'M0-8']),
    "f_63_64": dict(
        maxima=[0, 1, 2, 63, 2, 2, 64, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-2 S2-3 M3-5 S5-6 M6-8', 'M0-8']),
    "f_iter_cap": dict(
        maxima=[0, 1, 2, 2, 8, 2, 2, 2, 2, 2, 2, 2, 9, 2, 2, 2, 2],
        sched=['M0-8', 'M0-3 S3-4 M4-8']),
    "g_equal": dict(
        maxima=[0, 1, 2, 2, 4, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-8', 'M0-8']),
    "g_shorter": dict(
        maxima=[0, 1, 2, 2, 4, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-3 S3-4 M4-8', 'M0-8']),
    "h_481px": dict(
        maxima=[0, 1, 2, 2, 2, 40, 1, 2, 2, 2, 2, 2, 2, 1, 2, 2, 2],
        sched=['M0-4 S4-5 M5-8', 'M0-8']),
    "h_63px": dict(
        maxima=[0, 1, 2, 2, 2, 40, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-4 S4-5 M5-8', 'M0-8']),
    "h_1xN": dict(
        maxima=[0, 1, 2, 2, 2, 40, 1, 1, 2, 2, 1, 2, 2, 1, 2, 1, 1],
        sched=['M0-4 S4-5 M5-8', 'M0-8']),
    "h_Nx1": dict(
        maxima=[0, 0, 0, 1, 2, 40, 2, 2, 2, 2, 1, 1, 1, 1, 2, 2, 2],
        sched=['M0-4 S4-5 M5-8', 'M0-8']),
    "h_T2": dict(
        maxima=[0, 1, 2],
        sched=['M0-2']),
    "h_Tchunk1": dict(
        maxima=[0, 1, 2, 2, 2, 2, 1, 2, 2, 2],
        sched=['M0-8', 'classic']),
    "i_1280x720": dict(
        maxima=[0, 1, 2, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 12, 6, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1,
                    1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 10, 5, 1, 1, 1],
        sched=['M0-17 S17-18 M18-24', 'M0-19 S19-20 M20-24']),
    "j_sharded": dict(
        maxima=[0, 1, 2, 2, 40, 2, 2, 2, 2, 2, 2, 2, 2],
        sched=['M0-3 S3-4 M4-6', 'M0-6']),
}

SCENARIOS = list(EXPECT)


# ---- oracle ------------------------------------------------------------------------------------------------------
class OracleRun:
    """The CPU oracle over the case's frames: rows, per-frame maxima, final state; and the maxima the multi-frame
    kernels would predict from the real state at any frame (refractory filter skipped)."""

    def __init__(self, case):
        from emu_oracle import OracleEmulator
        self.case = case
        o = OracleEmulator(seed=SEED, shuffle=False, **case.kw)
        self.refr = case.kw.get("refractory_period_s", 0.0)
        tp = np.concatenate([[case.ts[0]], case.ts[:-1]])
        self.dt = case.ts - tp
        self.rows, self.maxima, self.snap = [], [], {}
        prev_bad = False
        for k, (f, t) in enumerate(zip(case.frames, case.ts)):
            s = copy.deepcopy(o) if self.refr > 0 else None
            ev = o.generate_events(f, t)
            self.rows.append(np.zeros((0, 4), np.float32) if ev is None else ev)
            self.maxima.append(int(o.last_max_n))
            bad = k > 0 and self.bad(k, self.maxima[k])
            if s is not None and (bad or prev_bad):
                self.snap[k] = s                       # state before frame k
            prev_bad = bad
        self.orc = o

    def bad(self, q, m):
        return is_bad(m, self.dt[q], self.refr, self.case.iter_cap)

    def real_bad(self, q):
        return self.bad(q, self.maxima[q])

    def predict(self, a, b):
        """bad(q) for q in [a, b) under the maxima of a multi-frame pass from the real state at a: exact up to the
        first really bad frame fb, then from a state where the refractory filter did not run."""
        fb = next((q for q in range(a, b) if self.real_bad(q)), b)
        pm = dict((q, self.maxima[q]) for q in range(a, min(fb + 1, b)))
        if fb + 1 < b:
            if self.refr > 0:
                o = copy.deepcopy(self.snap[fb])
                o.refractory_period_s = 0.0
                for q in range(fb, b):
                    o.generate_events(self.case.frames[q], self.case.ts[q])
                    pm[q] = int(o.last_max_n)
            else:
                pm.update((q, self.maxima[q]) for q in range(fb + 1, b))
        return lambda q: self.bad(q, pm[q])

    def model(self):
        m = ScheduleModel(self.real_bad, self.predict)
        for g0, n in self.case.chunk_starts():
            m.chunk(g0, n)
        return m


_ORACLE = {}


def oracle(name):
    if name not in _ORACLE:
        _ORACLE[name] = OracleRun(make_case(name))
    return _ORACLE[name]


def capacity_hint(name, run):
    """Initial event-buffer rows of the capacity scenarios: the first segment of the rescheduled chunk fits, the
    second does not."""
    if name == "e_in_multi":           # S0-1 fits, the abort lands in M1-8
        return len(run.rows[1]) + 1
    if name == "e_in_single":          # M0-3 fits, the abort lands in S3-4
        return sum(len(run.rows[k]) for k in (1, 2, 3)) + 1
    return None


# ---- CPU: the scripted clips make the situations they are named for ---------------------------------------------
@pytest.mark.parametrize("name", SCENARIOS)
def test_oracle_maxima_and_schedule(name):
    run = oracle(name)
    want = EXPECT[name]
    assert run.maxima == want["maxima"]
    m = run.model()
    assert m.log == want["sched"]
    assert m.multi > 0
    bad = [q for q in range(1, len(run.maxima)) if run.real_bad(q)]
    if name.startswith(("a_", "b_", "c_", "d_", "e_", "i_")):
        assert m.single > 0 and bad                    # mixed schedules
    if name == "c_mispredict":
        # frame 5 is really bad (the filter passed 3 of frame 4's 9 events), but a pass without the filter predicts it
        # good: the chunk needs a second rejection round
        assert bad == [4, 5] and not run.predict(1, 13)(5)
        assert m.rejected > m.chunks
    if name == "e_in_multi" or name == "e_in_single":
        hint = capacity_hint(name, run)
        cum = np.cumsum([len(r) for r in run.rows])
        # the first frame whose rows do not fit, and the kind of segment holding it
        first_over = int(np.argmax(cum > hint))
        assert (first_over, m.log[0]) == ((2, "S0-1 M1-8") if name == "e_in_multi" else (4, "M0-3 S3-4 M4-8"))
    if name == "f_iter_cap":
        assert bad == [12] and run.maxima[4] == run.case.iter_cap
    if name.startswith("g_"):
        assert run.maxima[4] == 4
        assert (run.dt[4] / 4 == REFR) == (name == "g_equal") and run.dt[4] / 4 <= REFR
    if name == "h_481px":
        assert (13 * 37) % 4 != 0
    if name == "j_sharded":
        assert bad == [4] and bad[0] - 1 >= 2           # first bad frame at position 3 of chunk [1, 7)


def test_segment_rule_by_hand():
    """The restated rule on maxima sequences written out by hand (chunk of 8, no refractory period)."""
    def sched(maxima, fb=None):
        bad = lambda q: maxima[q] > K_FUSED_MAX_N
        fb = next(q for q in range(8) if bad(q)) if fb is None else fb
        segs, _ = segment(bad, 0, 8, fb)
        return " ".join("%s%d-%d" % ("MS"[k], a, b) for k, a, b in segs)
    g, B = 2, 40
    assert sched([g, g, g, B, g, g, g, g]) == "M0-3 S3-4 M4-8"
    assert sched([B, g, g, g, g, g, g, g]) == "S0-1 M1-8"
    assert sched([g, B, g, g, g, g, B, g]) == "S0-2 M2-6 S6-8"
    assert sched([B, g, B, g, B, g, B, g]) == "S0-8"
    assert sched([g, g, g, g, g, g, g, 32]) == "M0-7 S7-8"


# ---- GPU: bit-exact against the oracle, and the schedule the handle really ran ----------------------------------
def _stats(em):
    v = [ctypes.c_longlong(0) for _ in range(4)]
    em._lib.v2e_emu_fused_stats(em._h, ctypes.byref(v[0]), ctypes.byref(v[1]))
    em._lib.v2e_emu_fused_frames(em._h, ctypes.byref(v[2]), ctypes.byref(v[3]))
    return dict(zip(("chunks", "rejected", "multi", "single"), (x.value for x in v)))


def _emulator(case):
    from v2e_b200 import EventEmulator
    return EventEmulator(device="cuda", seed=SEED, rng_mode="device", max_frames_per_step=case.chunk,
                         iter_cap=case.iter_cap, **case.kw)


def _compare_call(rows, offs, run, s, e, ctx):
    assert len(offs) == e - s + 1 and offs[0] == 0
    assert np.array_equal(np.diff(offs), [len(run.rows[k]) for k in range(s, e)]), ctx
    for k in range(s, e):
        assert_events_equal(rows[offs[k - s]:offs[k - s + 1]], run.rows[k], exact_order=False,
                            ctx="%s frame %d" % (ctx, k))


GPU_SCENARIOS = [n for n in SCENARIOS if n not in ("f_iter_cap", "j_sharded")]


@pytest.mark.gpu
@pytest.mark.parametrize("name", GPU_SCENARIOS)
def test_schedule_matches_oracle(name):
    """Rows per frame (canonical order, timestamps bit-exact), offsets, counters and final state equal to the oracle;
    the handle's schedule counters equal the restated rule's."""
    run = oracle(name)
    case, model = run.case, run.model()
    em = _emulator(case)
    em.event_rows_hint = capacity_hint(name, run)
    s = 0
    for e in case.calls:
        rows, offs = em.generate_events_batch(case.frames[s:e], case.ts[s:e])
        _compare_call(rows, offs, run, s, e, name)
        s = e
    assert (em.num_events_on, em.num_events_off) == (run.orc.num_events_on, run.orc.num_events_off)
    assert np.array_equal(em.lp_log_frame.cpu().numpy(), run.orc.lp)
    assert np.array_equal(em.base_log_frame.cpu().numpy(), run.orc.base)
    if case.kw.get("refractory_period_s", 0) > 0:
        assert np.array_equal(em.timestamp_mem.cpu().numpy(), run.orc.tmem)
    st = _stats(em)
    assert st == dict(chunks=model.chunks, rejected=model.rejected, multi=model.multi, single=model.single), st
    assert st["multi"] > 0


@pytest.mark.gpu
def test_iter_cap_accepted_at_the_cap_then_raises():
    """A frame with iter_cap events goes through the multi-frame kernels; one with iter_cap + 1 is rejected, replayed
    frame by frame, and the batch call raises instead of truncating."""
    from v2e_b200 import _lib
    run = oracle("f_iter_cap")
    case = run.case
    em = _emulator(case)
    rows, offs = em.generate_events_batch(case.frames[:9], case.ts[:9])
    _compare_call(rows, offs, run, 0, 9, "f_iter_cap")
    assert _stats(em) == dict(chunks=1, rejected=0, multi=8, single=0)
    with pytest.raises(_lib.V2eError):
        em.generate_events_batch(case.frames[9:], case.ts[9:])
    assert _stats(em)["rejected"] == 1


def _band_worker(rank, world, port, case, q):
    import os
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from v2e_b200 import EventEmulator
        from v2e_b200.parallel import row_band
        em = EventEmulator(device="cuda:0", seed=SEED, rng_mode="device", shard=(rank, world, None),
                           max_frames_per_step=case.chunk, **case.kw)
        y0, y1 = row_band(case.frames.shape[1], rank, world)
        rows, offs = em.generate_events_band_batch(np.ascontiguousarray(case.frames[:, y0:y1]), case.ts,
                                                   case.frames.shape[1])
        q.put((rank, rows, offs, em.num_events_total, _stats(em)))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_batched_prefix_replay_matches_oracle():
    """Two ranks, batched: the rejected chunk's accepted prefix (3 frames) runs through the multi-frame kernels again,
    the rest frame by frame; the union of the ranks' rows equals the oracle per frame."""
    import socket
    import torch.multiprocessing as mp
    run = oracle("j_sharded")
    case = run.case
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_band_worker, args=(r, 2, port, case, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(2):
        r, rows, offs, n, st = q.get(timeout=300)
        res[r] = (rows, offs, n, st)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert res[0][2] + res[1][2] == run.orc.num_events_total
    T = len(case.frames)
    for k in range(T):
        got = np.concatenate([res[r][0][res[r][1][k]:res[r][1][k + 1]] for r in (0, 1)])
        assert_events_equal(got, run.rows[k], exact_order=False, ctx="frame %d" % k)
    for r in (0, 1):
        # chunk [1, 7) rejected at frame 4, its prefix [1, 4) accepted on the second pass; chunk [7, 13) accepted
        assert res[r][3]["chunks"] == 3 and res[r][3]["rejected"] == 1, res[r][3]
