#!/usr/bin/env python
"""bench.py -- headline benchmark of the v2e hot path on B200 (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference_cuda]
                    [--workload headline|s|c3|c5] [--dump-outputs DIR]

Headline workload (BASELINE.json: "Mevents/s + interpolated-frames/s ... 1280x720 at 10x slowdown"):
one clip of 9 source frames (1280x720 uint8, smooth random texture translating 10 px per source
frame) -> SuperSloMo x10 (batch 8) -> 80 interpolated frames -> DVS pixel model with v2e's CLI-default
parameters -> events. A "step" is one pass of that whole path over one clip.
  value : events/s with the source frames already resident in HBM, events left in HBM
  e2e   : same, source frames in pinned host memory copied in and the packed event rows copied out
          (pinned staging, on every rank) inside the timed region, through V2EPipeline.run
With N>1 every rank processes its own clip (weak scaling, no data-path collective) and the event
streams are gathered with NCCL at the end of each step.

Secondary lines in the same JSON object (BASELINE.json configs, SURVEY.md 8d):
  secondary_346x260 (C2)  scripts/gradients.py's moving bump at 346x260, x10, CLI defaults -- on every N
  secondary_c3            1280x720 random 4x4-block texture, x20, 'noisy' pixel parameters (N = 1)
  replay_mode             the bit-exact mode (host-replayed torch draws, frame by frame) on the headline frames
  slomo_event_delta       events of the fp16 SloMo frames vs the float32 reference's frames, same pixel model
  config5 (--workload c5) ONE 1280x720 clip over the N ranks: SloMo sharded over frame pairs, all-to-all of row
                          bands, centre-surround pixel model sharded over pixel rows (halo exchange per Euler chunk)
`--impl reference` times the UNMODIFIED reference (oracle/_ref: the vendored v2ecore package) on the host cores.
One JSON line on stdout (rank 0).
`--dump-outputs DIR` (headline, rank 0) writes the events, frame offsets and frame times of the last timed step as
DIR/<name>.npy (bench.dump_outputs). Every input is seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

CLI_DEFAULTS = dict(pos_thres=0.2, neg_thres=0.2, sigma_thres=0.03, cutoff_hz=300.0, leak_rate_hz=0.01,
                    shot_noise_rate_hz=0.001, refractory_period_s=0.0005)   # v2e_args.py:150-204
# SURVEY.md 8(d) C3: the 'noisy' preset's leak / shot rates (emulator.py:525-535) on the CLI cutoff / refractory
C3_PARAMS = dict(pos_thres=0.2, neg_thres=0.2, sigma_thres=0.03, cutoff_hz=300.0, leak_rate_hz=0.1,
                 shot_noise_rate_hz=5.0, refractory_period_s=0.0005)
# SURVEY.md 8(d) C5: scripts/csdvs.sh:7-16
C5_PARAMS = dict(pos_thres=0.2, neg_thres=0.2, sigma_thres=0.03, cutoff_hz=100.0, leak_rate_hz=0.0,
                 shot_noise_rate_hz=0.0, refractory_period_s=0.001, cs_lambda_pixels=10, cs_tau_p_ms=0.5)
SRC_FPS = 30.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"],
                    bf16_tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def ncu_traffic():
    """DRAM bytes per launch from the committed ncu captures (profiles/r2_traffic.json, written by hand from
    `ncu --set full` of the same kernels; bench.py never runs under a profiler)."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def source_clip(H, W, n_src, seed=0, px_per_frame=10, up=16, lo=40.0, hi=215.0):
    """n_src source frames: smooth random texture (uniform noise, bicubic x16) translating
    `px_per_frame` px per source frame, forward then backward so that the clip loops seamlessly."""
    import torch
    rng = np.random.default_rng(seed)
    half = n_src // 2
    pw = W + px_per_frame * half + 2 * up
    base = torch.from_numpy(rng.uniform(lo, hi, (1, 1, H // up + 5, pw // up + 5)).astype(np.float32))
    big = torch.nn.functional.interpolate(base, scale_factor=up, mode="bicubic", align_corners=False)[0, 0]
    big = big.clamp(0, 255).round().to(torch.uint8).numpy()
    out = np.empty((n_src, H, W), np.uint8)
    for k in range(n_src):
        j = k if k <= half else n_src - 1 - k
        out[k] = big[up:up + H, j * px_per_frame:j * px_per_frame + W]
    return out


def gradient_clip(H=260, W=346, n_src=31, fps=SRC_FPS, contrast=2.0, speed_pps=300.0, bump_width=0.5, bg=127):
    """BASELINE config 2 input: scripts/gradients.py::im_function (:117-140) sampled at `fps`: a triangular bump of
    contrast 2 around the background level moving right at 300 px/s, with a 10-px bright bar ahead of it."""
    low = (bg * 2) / (contrast + 1)
    high = contrast * low
    diff = high - low
    w2 = (bump_width * W) / 2
    x = np.arange(W)
    out = np.empty((n_src, H, W), np.uint8)
    for k in range(n_src):
        p = w2 + (k / fps) * speed_pps
        p2 = p + w2 * 2
        g = np.ones((H, W)) * low
        ind = (x > p - w2) & (x < p)
        g[:, ind] = high + (-diff / w2) * (p - x[ind])
        ind = (x <= p + w2) & (x >= p)
        g[:, ind] = high + (-diff / w2) * (x[ind] - p)
        ind = (x > p2) & (x <= p2 + 10)
        g[:, ind] = high
        out[k] = np.uint8(g)
    return out


def block_texture_clip(H, W, n_src, seed=0, block=4, shift=(8, 4)):
    """SURVEY.md 8(d) C3 input: uniform random bytes in block x block squares, translated by `shift` px per source frame."""
    rng = np.random.default_rng(seed)
    pad_x, pad_y = shift[0] * n_src + block, shift[1] * n_src + block
    t0 = rng.integers(0, 256, ((H + pad_y) // block + 1, (W + pad_x) // block + 1), dtype=np.uint8)
    big = np.kron(t0, np.ones((block, block), np.uint8))
    return np.stack([np.ascontiguousarray(big[k * shift[1]:k * shift[1] + H, k * shift[0]:k * shift[0] + W])
                     for k in range(n_src)])


def unet_activation_bytes(in_ch, out_ch, H, W, B):
    """Algorithmic DRAM bytes of one UNet pass: every layer's input + output activations once (fp16 NHWC, channels
    padded to 16; the up blocks' first convolution charged with the LOW-resolution tensor it is a function of; fp32
    heads), weights excluded (19.8 M parameters, L2-resident)."""
    pad16 = lambda c: (c + 15) // 16 * 16
    ch = [32, 64, 128, 256, 512, 512]
    layers = [(in_ch, 32, 0), (32, 32, 0)]
    for d in range(5):
        layers += [(ch[d], ch[d + 1], d + 1), (ch[d + 1], ch[d + 1], d + 1)]
    uo, ui = [512, 256, 128, 64, 32], [512, 512, 256, 128, 64]
    for k in range(5):
        layers += [(ui[k], uo[k], 4 - k), (2 * uo[k], uo[k], 4 - k)]
    layers += [(32, out_ch, 0)]
    tot = 0.0
    for i, (ci, co, lvl) in enumerate(layers):
        inb = pad16(ci) * 2 / (4 if i in (12, 14, 16, 18, 20) else 1)
        outb = 32 if i == len(layers) - 1 else pad16(co) * 2
        tot += B * (H >> lvl) * (W >> lvl) * (inb + outb)
    return tot


DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, events, offsets, times, budget=DUMP_BYTES, seed=0):
    """--dump-outputs: what V2EPipeline.run returned for one clip, as <out_dir>/<name>.npy: events [M, 4] float32
    (t, x, y, p), offsets [T+1] and times [T] (float64). The order in which the pixel model emits the rows of one
    frame varies from run to run, so each frame's rows are written sorted by (t, y, x, p). When the files would
    exceed `budget` bytes, events is a seeded sample of those rows, kept in order, and events_rows [k] (float64)
    holds their row numbers."""
    os.makedirs(out_dir, exist_ok=True)
    ev = np.asarray(events, np.float32)
    frame = np.repeat(np.arange(len(offsets) - 1), np.diff(offsets))
    ev = ev[np.lexsort((ev[:, 3], ev[:, 1], ev[:, 2], ev[:, 0], frame))]
    out = {"offsets": np.asarray(offsets, np.float64), "times": np.asarray(times, np.float64)}
    room = budget - sum(a.nbytes for a in out.values()) - 4 * 4096        # .npy headers
    if ev.nbytes > room:
        rows = np.sort(np.random.default_rng(seed).choice(len(ev), room // (ev.itemsize * 4 + 8), replace=False))
        out["events_rows"] = rows.astype(np.float64)
        ev = ev[rows]
    out["events"] = ev
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def slomo_weights():
    """Seeded variance-preserving weights in the reference's checkpoint layout ('state_dictFC' /
    'state_dictAT'); the real SuperSloMo39.ckpt is not available offline (README.md:95-96)."""
    import slomo_ref
    # flow head gain 25 (flows of ~1.5 px, as in the parity tests and in round 1); V2E_BENCH_FLOW_GAIN overrides
    g = float(os.environ.get("V2E_BENCH_FLOW_GAIN", "25"))
    return {"state_dictFC": slomo_ref.make_test_weights(1234, 2, 4, head_gain=g),
            "state_dictAT": slomo_ref.make_test_weights(4321, 12, 5, head_gain=0.3)}


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md "clocks line")."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                for nm, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------
# the reference arm: the UNMODIFIED reference package (oracle/_ref, vendored by oracle/make_ref.py) through
# its own public API, on a bounded sample of the headline workload
# ---------------------------------------------------------------------------------------------------------
REF_SAMPLE = dict(n_src=3, batch=1)      # 2 frame pairs in 2 batches (the reference needs >= 2 batches, slomo.py:323)


def port_sample(frames, U, params):
    """Fallback of the CPU arm where the vendored reference (oracle/_ref) is missing: the oracle PORT of the same
    sample (float32 torch restatement of SuperSloMo + scalar C pixel model), kind "port"."""
    import torch
    import slomo_ref
    from emu_oracle import OracleEmulator
    wts = slomo_weights()
    t0 = time.perf_counter()
    out, times, _ = slomo_ref.interpolate_frames(frames, wts["state_dictFC"], wts["state_dictAT"], U, batch_size=1)
    t_slomo = time.perf_counter() - t0
    em = OracleEmulator(seed=1, **params)
    dt = 1.0 / (SRC_FPS * U)
    t1 = time.perf_counter()
    for i in range(out.shape[0]):
        em.generate_events(out[i], i * dt)
    t_emu = time.perf_counter() - t1
    return dict(events=em.num_events_total, interp_frames=int(out.shape[0]), seconds=t_slomo + t_emu, slomo_s=t_slomo,
                emu_s=t_emu, threads=torch.get_num_threads(), kind="port", slomo_device="cpu")


def reference_sample(H, W, U, params, device="cpu", seed=0):
    """3 source frames of the headline clip -> SuperSloMo.interpolate (x U, its .npy / .png folders) -> read_image
    -> EventEmulator.generate_events: the GPU arm's per-frame work (flow net amortised over U frames), 2U frames."""
    import ref_run
    import ref_shim
    if os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "v2ecore")):
        os.environ.setdefault("V2E_REFERENCE_ROOT", os.path.join(ROOT, "oracle", "_ref"))
    frames = source_clip(H, W, 9, seed=seed)[:REF_SAMPLE["n_src"]]
    if not (os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "v2ecore")) or ref_shim.reference_available()):
        return port_sample(frames, U, params)          # oracle/_ref was not built (python oracle/make_ref.py)
    return ref_run.run_reference(frames, SRC_FPS, U, REF_SAMPLE["batch"], params, slomo_weights(), seed=1,
                                 device=device)


def reference_arm(args, workload, H, W, U):
    import torch
    cuda = args.impl == "reference_cuda"
    if not cuda:
        # torchrun pins OMP_NUM_THREADS=1; the CPU arm uses every physical core (hyper-threads slow ATen's convs)
        torch.set_num_threads(max(1, min(64, (os.cpu_count() or 2) // 2)))
    reference_sample(64, 64, 2, CLI_DEFAULTS, device="cuda" if cuda else "cpu")      # page the libraries in
    budget = float(os.environ.get("V2E_REF_BUDGET_S", "200"))
    vals, t0 = [], time.perf_counter()
    while len(vals) < max(1, args.steps):
        vals.append(reference_sample(H, W, U, CLI_DEFAULTS, device="cuda" if cuda else "cpu"))
        spent = time.perf_counter() - t0
        if spent + spent / len(vals) > budget:
            break
    ev = sum(v["events"] for v in vals)
    sec = sum(v["seconds"] for v in vals)
    fr = sum(v["interp_frames"] for v in vals)
    v = ev / sec / 1e6
    kind = vals[0]["kind"]
    sample = ("%d source frames (2 pairs, batch 1) -> SuperSloMo.interpolate x%d -> %d frames (.npy in, .png out) -> "
              "read_image -> EventEmulator.generate_events, CLI defaults; SloMo on %s %.1f s + pixel model on %s %.1f s "
              "per sample; %d of the %d requested steps fit the %d s budget" % (
                  REF_SAMPLE["n_src"], U, vals[0]["interp_frames"], vals[0]["slomo_device"],
                  np.mean([x["slomo_s"] for x in vals]), "cuda" if cuda else "cpu",
                  np.mean([x["emu_s"] for x in vals]), len(vals), args.steps, int(budget)))
    line = {"impl": args.impl, "metric": "Mevents/s", "value": v, "unit": "Mevents/s", "n_gpus": args.gpus,
            "steps": args.steps, "steps_run": len(vals), "warmup": args.warmup,
            "ms_per_step": sec / len(vals) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 convs / f64 pixel state", "data": "synthetic", "config": {"workload": workload},
            "interp_frames_per_s": fr / sec,
            "cpu_baseline": {"value": v, "unit": "Mevents/s", "cores": vals[0]["threads"], "kind": kind,
                             "sample": sample, "interp_frames_per_s": fr / sec},
            "e2e": {"value": v, "unit": "Mevents/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference_cuda"])
    ap.add_argument("--workload", default="headline", choices=["headline", "s", "c3", "c5"])
    ap.add_argument("--height", type=int, default=720)
    ap.add_argument("--width", type=int, default=1280)
    ap.add_argument("--src-frames", type=int, default=9)
    ap.add_argument("--upsampling", type=int, default=10)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="development: skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the events, frame offsets and frame times of the last timed headline step to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "headline"):
        ap.error("--dump-outputs writes the headline workload of --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    H, W, NS, U = args.height, args.width, args.src_frames, args.upsampling
    n_interp = (NS - 1) * U
    clip_s = (NS - 1) / SRC_FPS
    workload = "%dx%d_smooth_texture_%dsrc_frames_slomo_x%d_b%d_emulator_cli_defaults" % (W, H, NS, U, args.batch)
    pk = peaks()
    Wd, Hd = int(W / 32) * 32, int(H / 32) * 32
    flops_per_interp = 2.0 * Hd * Wd * (330016 + 314048 / U)       # SURVEY 8(d)

    if args.impl != "b200":
        if args.impl == "reference":
            os.environ["CUDA_VISIBLE_DEVICES"] = ""        # the reference picks cuda:0 when it sees one (slomo.py:84-89)
        if rank != 0:
            return
        reference_arm(args, workload, H, W, U)
        return

    import torch
    import torch.distributed as dist
    from v2e_b200 import EventEmulator, SuperSloMo, V2EPipeline, _lib
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    devname = "cuda:%d" % local_rank
    if world > 1:
        # keep stdout to the one JSON line: NCCL prints its version banner there at the VERSION level
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    wts = slomo_weights()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_events(rows):
        """NCCL gather of the packed event streams to rank 0 (the only collective of the job): counts first
        (one small all-gather, read back with one sync -- the stream is already drained by the pixel model's own
        count read-back), rows padded to the largest count."""
        n = torch.tensor([rows.shape[0]], device=dev, dtype=torch.int64)
        ns = torch.empty((world,), device=dev, dtype=torch.int64)
        dist.all_gather_into_tensor(ns, n)
        mx = int(ns.max().item())
        pad = torch.empty((mx, 4), dtype=torch.float32, device=dev)
        pad[:rows.shape[0]] = rows
        out = torch.empty((world * mx, 4), dtype=torch.float32, device=dev) if rank == 0 else None
        dist.gather(pad, list(out.split(mx)) if rank == 0 else None, dst=0)

    def all_max_sum(ms, cnt):
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        c = torch.tensor([float(cnt)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
        return t.item(), c.item()

    def run_clips(src_host, src_dev, params, U_, batch, n_frames, rows_hint, steps, warmup, e2e, clip_seconds, seed,
                  last_step=None):
        """`steps` timed passes of SloMo + pixel model over this rank's clip. Returns (ms max over ranks, events
        summed over ranks, pipeline). A `last_step` list receives host copies of the (events, offsets, times) the
        last timed pass returned."""
        sl = SuperSloMo(model=None, auto_upsample=False, upsampling_factor=U_, batch_size=batch, device=devname,
                        state_dicts=wts)
        em = EventEmulator(device=devname, rng_mode="device", seed=seed, max_frames_per_step=n_frames, **params)
        em.event_rows_hint = rows_hint
        pipe = V2EPipeline(sl, em)
        k = 0
        last = None

        period = clip_seconds * n_frames / (n_frames - 1)      # the next pass starts one frame interval after the last frame

        def one():
            nonlocal k, last
            t0 = k * period
            k += 1
            if e2e:
                # host frames in (pinned), packed rows out through the emulator's pinned staging buffer on EVERY
                # rank; the device rows are still gathered to rank 0 (the merged stream stays in HBM there)
                fr = src_host.to(dev, non_blocking=True)
                ev, offs, t, nf = pipe.run(fr, clip_seconds, t_offset=t0, return_device=False, copy=False)
                if world > 1:
                    gather_events(em._ev_dev[:ev.shape[0]])
            else:
                ev, offs, t, nf = pipe.run(src_dev, clip_seconds, t_offset=t0, return_device=True)
                if world > 1:
                    gather_events(ev)
            last = (ev, offs, t)
            return ev.shape[0]
        for _ in range(warmup):
            one()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = 0
        for _ in range(steps):
            n += one()
        e1.record()
        barrier()
        if last_step is not None:
            ev, offs, t = last          # rows are views of buffers the next pass reuses: copy them now
            last_step.extend([ev.cpu().numpy() if torch.is_tensor(ev) else np.array(ev), np.array(offs), np.array(t)])
        ms, cnt = all_max_sum(e0.elapsed_time(e1), n)
        return ms, cnt, pipe

    def close(pipe):
        pipe.slomo.cleanup()
        pipe.emulator.cleanup()
        torch.cuda.empty_cache()

    # ------------------------------------------------------------------------------------------------
    # BASELINE config 5: one clip over all ranks, centre-surround pixel model
    # ------------------------------------------------------------------------------------------------
    if args.workload == "c5":
        from bench_c5 import run_config5
        line = run_config5(args, rank, world, local_rank, pk)
        if rank == 0:
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return

    def secondary_s(steps=3, warmup=2):
        """BASELINE config 2 size and input: 346x260 gradient clip, 31 source frames, x10; all pairs in one batch
        (batch_size is SuperSloMo's own knob, slomo.py:44-54: at 10x8-pixel deep levels a batch of 8 leaves SMs idle)."""
        H2, W2, NS2 = 260, 346, 31
        src = gradient_clip(H2, W2, NS2)
        if rank:
            src = np.ascontiguousarray(src[:, :, ::-1] if rank % 2 else src)        # other ranks: mirrored / same clip
        sh = torch.from_numpy(src).pin_memory()
        sd = sh.to(dev)
        nf = (NS2 - 1) * U
        ms, cnt, p2 = run_clips(sh, sd, CLI_DEFAULTS, U, NS2 - 1, nf, 16 * 1024 * 1024, steps, warmup, False,
                                (NS2 - 1) / SRC_FPS, 99 + rank)
        close(p2)
        ms_e, cnt_e, p3 = run_clips(sh, sd, CLI_DEFAULTS, U, NS2 - 1, nf, 16 * 1024 * 1024, steps, warmup, True,
                                    (NS2 - 1) / SRC_FPS, 99 + rank)
        close(p3)
        return {"workload": "346x260_gradients_py_bump_%dsrc_frames_slomo_x%d_b%d_emulator_cli_defaults" % (NS2, U, NS2 - 1),
                "value": cnt / (ms * 1e-3) / 1e6, "unit": "Mevents/s", "steps": steps, "ms_per_step": ms / steps,
                "interp_frames_per_s": world * steps * nf / (ms * 1e-3),
                "e2e": {"value": cnt_e / (ms_e * 1e-3) / 1e6, "unit": "Mevents/s", "ms_per_step": ms_e / steps,
                        "interp_frames_per_s": world * steps * nf / (ms_e * 1e-3)},
                "events_per_px_per_frame": cnt / steps / world / (nf * H2 * W2), "clips": world}

    if args.workload == "s":
        sec = secondary_s(args.steps, args.warmup)
        if rank == 0:
            sec.update({"metric": "Mevents/s", "n_gpus": world, "higher_is_better": True, "scaling": "weak",
                        "data": "synthetic", "config": {"workload": sec["workload"]}})
            print(json.dumps(sec))
        if world > 1:
            dist.destroy_process_group()
        return

    def secondary_c3(steps=2, warmup=1):
        """BASELINE config 3: 1280x720 random 4x4-block texture moving (8, 4) px per source frame, 17 source frames,
        x20 (320 frames), leak 0.1 Hz / shot 5 Hz ('noisy' preset rates), sigma 0.03, refractory 0.5 ms."""
        NS3, U3 = 17, 20
        src = block_texture_clip(H, W, NS3, seed=0)
        sh = torch.from_numpy(src).pin_memory()
        sd = sh.to(dev)
        nf = (NS3 - 1) * U3
        ms, cnt, p = run_clips(sh, sd, C3_PARAMS, U3, args.batch, nf, 160 * 1024 * 1024, steps, warmup, False,
                               (NS3 - 1) / SRC_FPS, 7)
        a, b = ctypes.c_longlong(0), ctypes.c_longlong(0)
        p.emulator._lib.v2e_emu_fused_stats(p.emulator._h, ctypes.byref(a), ctypes.byref(b))
        e, f = ctypes.c_longlong(0), ctypes.c_longlong(0)
        p.emulator._lib.v2e_emu_fused_frames(p.emulator._h, ctypes.byref(e), ctypes.byref(f))
        close(p)
        fl = 2.0 * Hd * Wd * (330016 + 314048 / U3)
        return {"workload": "1280x720_random_4x4_block_texture_%dsrc_frames_slomo_x%d_b%d_emulator_noisy" % (NS3, U3, args.batch),
                "value": cnt / (ms * 1e-3) / 1e6, "unit": "Mevents/s", "steps": steps, "ms_per_step": ms / steps,
                "interp_frames_per_s": steps * nf / (ms * 1e-3),
                "slomo_tflops": steps * nf * fl / (ms * 1e-3) / 1e12,
                "events_per_px_per_frame": cnt / steps / (nf * H * W),
                "pixel_model_chunks": {"chunks_through_multi_frame_path": a.value, "re_scheduling_rounds": b.value,
                                       "frames_in_multi_frame_segments": e.value, "frames_frame_by_frame": f.value},
                "params": C3_PARAMS}

    if args.workload == "c3":
        sec = secondary_c3(args.steps, args.warmup)
        sec.update({"metric": "Mevents/s", "n_gpus": 1, "higher_is_better": True, "data": "synthetic",
                    "config": {"workload": sec["workload"]}})
        print(json.dumps(sec))
        return

    # ------------------------------------------------------------------------------------------------
    # headline
    # ------------------------------------------------------------------------------------------------
    src_host = torch.from_numpy(source_clip(H, W, NS, seed=rank)).pin_memory()
    src_dev = src_host.to(dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last_step = [] if args.dump_outputs and rank == 0 else None
    ms_dev, ev_dev, pipe = run_clips(src_host, src_dev, CLI_DEFAULTS, U, args.batch, n_interp, 48 * 1024 * 1024,
                                     args.steps, args.warmup, False, clip_s, 1234 + rank, last_step)
    clocks = sampler.stop() if rank == 0 else None
    if last_step:
        dump_outputs(args.dump_outputs, *last_step)
    _a, _b = ctypes.c_longlong(0), ctypes.c_longlong(0)
    pipe.emulator._lib.v2e_emu_fused_stats(pipe.emulator._h, ctypes.byref(_a), ctypes.byref(_b))
    _c, _d = ctypes.c_int(0), ctypes.c_int(0)
    pipe.emulator._lib.v2e_emu_fused_last_reject(pipe.emulator._h, ctypes.byref(_c), ctypes.byref(_d))
    _e, _f = ctypes.c_longlong(0), ctypes.c_longlong(0)
    pipe.emulator._lib.v2e_emu_fused_frames(pipe.emulator._h, ctypes.byref(_e), ctypes.byref(_f))
    chunk_stats = {"chunks_through_multi_frame_path": _a.value, "re_scheduling_rounds": _b.value,
                   "frames_in_multi_frame_segments": _e.value, "frames_frame_by_frame": _f.value}
    if _b.value:
        chunk_stats["last_rejected_at"] = {"frame_in_chunk": _c.value, "max_events_of_one_pixel": _d.value}

    # ---- roofline of the dominant kernel (UNet convolutions, tensor pipe) and of the pixel model (HBM) ----
    prof = {}
    replay = None
    if rank == 0 and not args.no_profile:
        traffic = ncu_traffic()
        eng = pipe.slomo._engine
        em = pipe.emulator
        _lib.check(eng.lib.v2e_slomo_profile(eng._h, 1))
        k0 = args.steps + args.warmup
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        pipe.run(src_dev, clip_s, t_offset=k0 * clip_s * n_interp / (n_interp - 1), return_device=True)
        torch.cuda.synchronize()
        step_ms_prof = (time.perf_counter() - w0) * 1e3
        conv_ms, conv_n, conv_fl = ctypes.c_float(0), ctypes.c_int(0), ctypes.c_double(0)
        ms23, n23, fl23 = (ctypes.c_float * 23)(), (ctypes.c_int * 23)(), (ctypes.c_double * 23)()
        _lib.check(eng.lib.v2e_slomo_profile_read_layers(eng._h, ms23, n23, fl23, ctypes.byref(conv_ms),
                                                         ctypes.byref(conv_n), ctypes.byref(conv_fl), eng._stream()))
        _lib.check(eng.lib.v2e_slomo_profile(eng._h, 0))
        names = ["conv1", "conv2"] + ["down%d.conv%d" % (d, c) for d in range(1, 6) for c in (1, 2)] + \
                ["up%d.conv%d" % (d, c) for d in range(1, 6) for c in (1, 2)] + ["conv3"]
        layers = []
        for i in range(23):
            if n23[i]:
                tf = fl23[i] / (ms23[i] * 1e-3) / 1e12
                layers.append({"layer": names[i], "launches": n23[i], "ms": ms23[i], "tflops": tf,
                               "frac": tf / pk["bf16_tflops_sustained"]})
        big = max(range(23), key=lambda i: ms23[i])
        achieved = conv_fl.value / (conv_ms.value * 1e-3) / 1e12
        tr_conv = traffic.get("conv_all_layers_per_step")
        n_batches_p = -(-(NS - 1) // args.batch)
        # pixel model alone: the multi-frame path on a clean 1280x720 clip (the headline texture translating 1 px per
        # frame, CLI defaults, device RNG), K repetitions of one 80-frame chunk between one event pair. Measured on its
        # own clip because the headline's interpolated frames -- synthesised by a RANDOM-weight network -- flicker: in
        # a few frames of every chunk some pixel makes >= 7 events, the refractory filter engages there
        # (emulator.py:830), and the chunk is re-scheduled: those frames frame by frame, the runs between them through
        # the multi-frame kernels (config.pixel_model_chunks says how many of each).
        T = 80
        clean = torch.from_numpy(source_clip(H, W, T + 1, seed=11, px_per_frame=1)).to(dev)      # loops: frame T == frame 0
        emc = EventEmulator(device=devname, rng_mode="device", seed=77, max_frames_per_step=T, **CLI_DEFAULTS)
        emc.event_rows_hint = 48 * 1024 * 1024
        emc.generate_events_batch(clean, np.arange(T + 1) / (SRC_FPS * U), return_device=True)
        rows_c, _ = emc.generate_events_batch(clean[1:], (T + 1 + np.arange(T)) / (SRC_FPS * U), return_device=True)
        ca, cb = ctypes.c_longlong(0), ctypes.c_longlong(0)
        emc._lib.v2e_emu_fused_stats(emc._h, ctypes.byref(ca), ctypes.byref(cb))
        ts = (ctypes.c_double * T)(*[(2 * T + 1 + k) / (SRC_FPS * U) for k in range(T)])
        uc, uu = ctypes.c_float(0), ctypes.c_float(0)
        _lib.check(emc._lib.v2e_emu_time_fused(emc._h, ctypes.c_void_p(clean[1:].data_ptr()), 0, T, ts,
                                               float(emc.t_previous), ctypes.c_void_p(emc._ev_dev.data_ptr()),
                                               emc._ev_dev.shape[0], 10, ctypes.byref(uc), ctypes.byref(uu), emc._stream()))
        ev_clean = rows_c.shape[0] / T
        emc.cleanup()
        # what the headline step itself ran: per-kernel brackets of the frame-by-frame kernels (or of the chunk)
        em = pipe.emulator
        _lib.check(em._lib.v2e_emu_profile(em._h, 1))
        pipe.run(src_dev, clip_s, t_offset=(k0 + 1) * clip_s * n_interp / (n_interp - 1), return_device=True)
        ms4, n4 = (ctypes.c_float * 4)(), (ctypes.c_int * 4)()
        _lib.check(em._lib.v2e_emu_profile_read4(em._h, ms4, n4, em._stream()))
        _lib.check(em._lib.v2e_emu_profile(em._h, 0))
        ev_per_frame = ev_clean
        us_frame = uc.value / T
        bytes_frame = H * W * 53.0 + 16.0 * ev_per_frame                    # SURVEY 8(d): T = 1 form, per frame
        bytes_launch = H * W * (T * 1.0 + 52.0) + 16.0 * ev_per_frame * T   # SURVEY 8(d): one launch over T frames
        prof = {
            "roofline": {"kernel": "conv_strip2 / conv_strip2up / conv_tc kernels (all UNet convolutions of one step, summed)",
                         "bound": "tensor", "achieved": achieved, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": achieved / pk["bf16_tflops_sustained"], "traffic": tr_conv,
                         "peak_source": pk["source"] + " (sustained 16-bit dense; burst %.1f)" % pk["bf16_tflops"],
                         "algorithmic_bytes": n_batches_p * (unet_activation_bytes(2, 4, Hd, Wd, args.batch) +
                                                             U * unet_activation_bytes(12, 5, Hd, Wd, args.batch)),
                         "flops_per_step": conv_fl.value, "conv_ms_per_step": conv_ms.value,
                         "launches_per_step": conv_n.value, "share_of_step": conv_ms.value / step_ms_prof,
                         "largest_layer": {"layer": names[big], "ms_per_launch": ms23[big] / n23[big],
                                           "tflops": fl23[big] / (ms23[big] * 1e-3) / 1e12,
                                           "frac": fl23[big] / (ms23[big] * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
                                           "traffic": traffic.get(names[big])},
                         "layers": layers},
            "roofline_emulator": {
                "kernel": "emu_fused_update + count + plan + emit (multi-frame pixel model, one chunk of %d frames)" % T,
                "bound": "hbm", "achieved": bytes_frame / (us_frame * 1e-6) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": bytes_frame / (us_frame * 1e-6) / 1e9 / pk["hbm_gbs"],
                "traffic": traffic.get("emu_fused_chunk"),
                "bytes_per_frame": bytes_frame, "us_per_frame": us_frame, "frames_per_launch": T,
                "us_per_chunk": uc.value, "us_update_kernel": uu.value,
                "basis": "SURVEY 8(d) per-call figure (53 B/px + 16 B/event per frame: the frame-by-frame API's traffic) "
                         "over the chunk's device time / T",
                # the same launch against the bytes a T-frame launch really has to move (state once per chunk):
                "as_one_launch": {"bytes": bytes_launch, "achieved": bytes_launch / (uc.value * 1e-6) / 1e9,
                                  "frac": bytes_launch / (uc.value * 1e-6) / 1e9 / pk["hbm_gbs"],
                                  "note": "per-pixel state stays in registers across the chunk, so the launch moves "
                                          "H*W*(T+52)+16N bytes and is instruction-issue bound, not HBM bound"},
                "timing": "v2e_emu_time_fused: 10 repetitions of the chunk (update, count, plan, emit; no commit, state "
                          "untouched) between one CUDA-event pair on the launching stream",
                "clip": "1280x720 smooth texture translating 1 px per frame, %.3f events/px/frame; chunks accepted %d, "
                        "rejected %d" % (ev_clean / (H * W), ca.value - cb.value, cb.value),
                # the headline step's own pixel-model launches (CUDA-event brackets, one profiled step)
                "headline_step_kernels": {"update_ms": ms4[0], "update_launches": n4[0], "filter_or_count_ms": ms4[1],
                                          "filter_or_count_launches": n4[1], "emit_ms": ms4[2], "emit_launches": n4[2],
                                          "note": "launch counts of one profiled headline step: frame-by-frame kernels for the "
                                                  "frames that break the assumption, multi-frame kernels for the runs between "
                                                  "them (config.pixel_model_chunks)"}},
        }
        # the bit-exact mode (host-replayed torch draws, one frame per call) on the same frames
        em_r = EventEmulator(device=devname, rng_mode="replay", seed=5, **CLI_DEFAULTS)
        interp, _, _ = pipe.slomo.interpolate_frames(src_dev)
        fr_host = interp[:24].cpu().numpy()
        em_r.generate_events(fr_host[0], 0.0)
        em_r.generate_events(fr_host[1], 1 / 300.0)
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        nr = 0
        for i in range(2, 24):
            e = em_r.generate_events(fr_host[i], i / 300.0)
            nr += 0 if e is None else len(e)
        wall = time.perf_counter() - w0
        em_r.cleanup()
        replay = {"value": nr / wall / 1e6, "unit": "Mevents/s", "frames_per_s": 22 / wall,
                  "what": "EventEmulator.generate_events, rng_mode='replay' (rows bit-identical to the reference incl. "
                          "order): 22 frames 1280x720 from host uint8 arrays, torch CPU draws + upload + D2H per frame, wall clock"}
    close(pipe)
    del pipe

    if args.no_e2e:
        ms_e2e, ev_e2e = ms_dev, ev_dev
    else:
        ms_e2e, ev_e2e, pipe2 = run_clips(src_host, src_dev, CLI_DEFAULTS, U, args.batch, n_interp, 48 * 1024 * 1024,
                                          args.steps, max(1, args.warmup), True, clip_s, 1234 + rank)
        close(pipe2)

    secondary = secondary_s() if not args.no_secondary else None
    c3 = delta = None
    if rank == 0 and world == 1 and not args.no_secondary:
        c3 = secondary_c3()
        delta = slomo_event_delta(devname, wts)
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            # the reference picks cuda:0 when it sees one (slomo.py:84-89): the CPU leg runs in a child process with
            # the GPUs hidden -- one bounded sample of the --impl reference arm
            env = dict(os.environ, CUDA_VISIBLE_DEVICES="", V2E_REF_BUDGET_S="1")
            env.pop("OMP_NUM_THREADS", None)
            try:
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1",
                                      "--warmup", "0", "--height", str(H), "--width", str(W), "--upsampling", str(U)],
                                     env=env, capture_output=True, text=True, timeout=900)
                cpu = json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception as exc:
                cpu = {"value": None, "unit": "Mevents/s", "cores": 0, "kind": "_ref",
                       "sample": "the reference leg failed: %s" % exc}
        steps = args.steps
        value = ev_dev / (ms_dev * 1e-3) / 1e6
        e2e = ev_e2e / (ms_e2e * 1e-3) / 1e6
        n_batches = -(-(NS - 1) // args.batch)
        # SloMo: per batch resize + prep + 33 flow-net launches, per t 33 interp-net launches + pre/post + resize;
        # pixel model: first frame once, then per chunk update / count / plan / emit / commit
        launches_step = n_batches * (1 + 33 + U * (1 + 33 + 1 + 2) + 2) + 5 + 2
        line = {
            "metric": "Mevents/s", "value": value, "unit": "Mevents/s", "n_gpus": world, "steps": steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16 tensor-core convs (fp32 accumulate) + f64 pixel state",
            "data": "synthetic",
            "config": {"workload": workload, "interp_frames_per_step": n_interp, "clips": world,
                       "events_per_px_per_frame": ev_dev / steps / world / (n_interp * H * W),
                       "l2_policy": "activations of one UNet pass (>2 GB at batch 8) exceed L2",
                       "rng": "device philox",
                       "weights": "seeded random, reference checkpoint layout",
                       "pixel_model_chunks": chunk_stats,
                       "sharding": "one independent clip per GPU; NCCL gather of the event streams per step"},
            "interp_frames_per_s": world * n_interp * steps / (ms_dev * 1e-3),
            "slomo_flops_per_interp_frame": flops_per_interp,
            "e2e": {"value": e2e, "unit": "Mevents/s", "h2d_bytes_per_step": NS * H * W,
                    "d2h_bytes_per_step": int(16 * ev_e2e / steps / world), "ms_per_step": ms_e2e / steps,
                    "interp_frames_per_s": world * n_interp * steps / (ms_e2e * 1e-3),
                    "note": "every rank: pinned host frames in, its packed rows out through pinned staging"},
            "gpu_launches": int(steps * launches_step),
            "clocks": clocks,
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        line.update(prof)
        if secondary is not None:
            line["secondary_346x260"] = secondary
        if c3 is not None:
            line["secondary_c3"] = c3
        if replay is not None:
            line["replay_mode"] = replay
        if delta is not None:
            line["slomo_event_delta"] = delta
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def slomo_event_delta(devname, wts):
    """SURVEY.md 8(d) parity criterion "the induced event-count delta": the same source frames through (a) the fp16
    tensor-core SloMo and (b) the float32 torch restatement of the reference (oracle/slomo_ref.py, CPU), both frame
    sets through the same pixel model (CUDA, noise off so that nothing but the frames differs)."""
    import torch
    import slomo_ref
    from v2e_b200 import EventEmulator, SuperSloMo
    H2, W2, U2 = 260, 346, 10
    src = gradient_clip(H2, W2, 4)[1:4]                       # 2 pairs with the bump inside the frame
    sl = SuperSloMo(model=None, auto_upsample=False, upsampling_factor=U2, batch_size=2, device=devname, state_dicts=wts)
    got, times, _ = sl.interpolate_frames(src)
    got = got.cpu().numpy()
    sl.cleanup()
    want, _, _ = slomo_ref.interpolate_frames(src, wts["state_dictFC"], wts["state_dictAT"], U2, batch_size=2)
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    kw = dict(pos_thres=0.2, neg_thres=0.2, sigma_thres=0.0, cutoff_hz=300.0, leak_rate_hz=0.0,
              shot_noise_rate_hz=0.0, refractory_period_s=0.0005)
    ts = np.arange(got.shape[0]) / (SRC_FPS * U2)
    cnt = []
    for frames in (got, want):
        em = EventEmulator(device=devname, rng_mode="device", max_frames_per_step=got.shape[0], **kw)
        em.generate_events_batch(frames, ts)
        cnt.append((em.num_events_total, em.num_events_on, em.num_events_off))
        em.cleanup()
    (a, a_on, a_off), (b, b_on, b_off) = cnt
    return {"what": "346x260 gradients.py clip, 2 pairs x10 = 20 frames: fp16 tcgen05 SloMo vs float32 torch reference "
                    "frames, same pixel model (noise off)",
            "dn_abs_diff_hist": np.bincount(d.ravel(), minlength=4)[:8].tolist(), "dn_max": int(d.max()),
            "dn_mean": float(d.mean()),
            "events_fp16": a, "events_fp32": b, "delta_events": a - b, "delta_rel": (a - b) / max(b, 1),
            "delta_on": a_on - b_on, "delta_off": a_off - b_off}


if __name__ == "__main__":
    main()
