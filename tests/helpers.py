"""Shared test helpers: golden-fixture loading, the RNG tape, event comparators."""
import json
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

EMU_GOLDENS = ["emu_class_default", "emu_cli_noisy", "emu_clean", "emu_scalar_thres_f64",
               "emu_refractory_multi", "emu_float_frames", "emu_static_leak_shot",
               "emu_ragged_13x37", "emu_csdvs", "emu_csdvs_120x176"]
# optional pixel models: SCIDVS (emulator.py:58-80, 719-725), photoreceptor noise (emulator.py:694-703)
EMU_GOLDENS_OPT = ["emu_scidvs", "emu_scidvs_f32", "emu_prnoise", "emu_prnoise_scidvs_csdvs"]


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)
    g = {k: z[k] for k in z.files if not k.startswith("tape_0")}
    g["kwargs"] = json.loads(str(z["kwargs_json"]))
    if "tape_kinds" in z.files:
        g["tape"] = [(str(k), z["tape_%05d" % i]) for i, k in enumerate(z["tape_kinds"])]
    return g


class TapeRNG:
    """Replays the random draws the reference made when the golden was recorded
    (oracle/make_golden.py::Recorder), checking that the consumer asks for the same
    kind and size of draw in the same order."""

    def __init__(self, tape):
        self.tape = list(tape)
        self.pos = 0

    def _next(self, kind, shape=None):
        assert self.pos < len(self.tape), "RNG tape exhausted (asked for %s)" % kind
        k, arr = self.tape[self.pos]
        self.pos += 1
        assert k == kind, "draw %d: reference drew %s, consumer asked %s" % (self.pos - 1, k, kind)
        if shape is not None:
            assert tuple(arr.shape) == tuple(shape), (kind, arr.shape, shape)
        return torch.from_numpy(np.array(arr))

    def normal(self, mean, std, shape):
        return self._next("normal", shape)

    def randn(self, shape):
        return self._next("randn", shape)

    def rand(self, shape):
        return self._next("rand", shape)

    def randperm(self, n):
        t = self._next("randperm", (n,))
        return t.long()

    def exhausted(self):
        return self.pos == len(self.tape)


def smooth_background(H, W, T, seed=0, lo=90.0, hi=150.0):
    """Smooth low-contrast texture translating 1 px per frame: 0-2 events per pixel and frame at
    thresholds 0.05 (0-1 at 0.2)."""
    from bench import source_clip
    return source_clip(H, W, 2 * T + 1, seed=seed, px_per_frame=1, up=8, lo=lo, hi=hi)[:T]


def patch_codes(targets, th=0.05, cutoff_hz=0.0, dt=2.0 ** -6, start=30):
    """uint8 codes of one pixel, frame by frame, such that the CPU oracle (scalar threshold `th`, no noise, no
    refractory period) makes exactly targets[k] events in frame k. Frame 0 initialises the state. A target of 0
    keeps the code (the residual left after the last step is below one threshold); any other target is searched
    upwards from the current code, then downwards."""
    import copy
    from emu_oracle import OracleEmulator
    o = OracleEmulator(pos_thres=th, neg_thres=th, sigma_thres=0.0, cutoff_hz=cutoff_hz, leak_rate_hz=0.0,
                       shuffle=False)
    px = lambda c: np.full((1, 1), c, np.uint8)
    o.generate_events(px(start), 0.0)
    codes, code = [start], start
    for k, n in enumerate(targets[1:], 1):
        cands = [code] if n == 0 else list(range(code + 1, 256)) + list(range(code - 1, -1, -1))
        for c in cands:
            trial = copy.deepcopy(o)
            trial.generate_events(px(c), k * dt)
            if trial.last_max_n == n:
                break
        else:
            raise ValueError("no code makes %d events in frame %d" % (n, k))
        o.generate_events(px(c), k * dt)
        codes.append(c)
        code = c
    return codes


def scripted_clip(H, W, T, patches, th=0.05, cutoff_hz=0.0, dt=2.0 ** -6, seed=0, lo=90.0, hi=150.0):
    """Smooth background plus small square patches whose level steps so that each patch pixel makes a chosen
    number of events per frame. patches: [(y, x, size, targets, start_code)], targets[k] for frame k (length T)."""
    fr = smooth_background(H, W, T, seed=seed, lo=lo, hi=hi).copy()
    for y, x, s, targets, start in patches:
        assert len(targets) == T
        codes = patch_codes(targets, th=th, cutoff_hz=cutoff_hz, dt=dt, start=start)
        fr[:, y:y + s, x:x + s] = np.asarray(codes, np.uint8)[:, None, None]
    return fr


def split_events(events, counts):
    off = np.concatenate([[0], np.cumsum(counts)])
    return [events[off[i]:off[i + 1]] for i in range(len(counts))]


def canonical(ev):
    """Sort rows by (t, y, x, p) -- the order-insensitive form (SURVEY 8d parity criteria)."""
    if ev is None or len(ev) == 0:
        return np.zeros((0, 4), np.float32)
    k = np.lexsort((ev[:, 3], ev[:, 1], ev[:, 2], ev[:, 0]))
    return np.ascontiguousarray(ev[k])


def assert_events_equal(got, want, exact_order=True, t_tol=0.0, ctx=""):
    got = np.zeros((0, 4), np.float32) if got is None else got
    want = np.zeros((0, 4), np.float32) if want is None else want
    assert got.shape == want.shape, "%s: %s rows vs reference %s" % (ctx, got.shape, want.shape)
    if not exact_order:
        got, want = canonical(got), canonical(want)
    assert np.array_equal(got[:, 1:], want[:, 1:]), "%s: x/y/polarity differ" % ctx
    if t_tol == 0.0:
        assert np.array_equal(got[:, 0], want[:, 0]), "%s: timestamps differ" % ctx
    else:
        assert np.max(np.abs(got[:, 0] - want[:, 0]), initial=0.0) <= t_tol, "%s: timestamps" % ctx
