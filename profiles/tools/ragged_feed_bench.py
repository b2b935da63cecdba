"""Ragged list pushes (ewk_push_streams) with paced ticks (ewk_tick_ready) on one GPU, against today's uniform push.

    python profiles/tools/ragged_feed_bench.py [--out profiles/r05_ragged_feed.json] [--steps 30] [--warmup 5]

Bank: 4096 slots, 10 s int16 rings.  Each step every active slot receives its own length, drawn from U(0.5, 1.5) s
(1 s nominal), as one push_streams of pinned host memory, then tick_ready takes every tick that is due.  Active slots are
a scattered random subset at 100 %, 50 % and 10 % occupancy; idle slots get nothing.  Feeds: 16 kHz int16 and 8 kHz
mu-law.  For comparison in the same run: the uniform ewk_push / ewk_push_resampled of all 4096 slots (1 s each, ewk_tick),
and the list path at 100 % with equal 1 s lengths.  Step times are host clocks around steps that end in a synchronise;
H2D bytes are the packed input plus the row descriptors, computed from the lengths.  Kernel times per profiler class come
from ewk_profile in a separate pass."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

TOOLS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(TOOLS))
sys.path.insert(0, REPO)
sys.path.insert(0, TOOLS)

from easywakeword_b200 import _lib  # noqa: E402
from native_rate_bench import gpu_info, sm_clock_now  # noqa: E402

SLOTS, RING, SLACK = 4096, 160000, 32000
DESC_BYTES = 40                                     # one RowDesc per non-empty row
CLASSES = {"ring_push": 0, "tick_gate": 1, "resample_push": 7}


def make_ctx():
    ctx = _lib.Context(device=0, n_streams=SLOTS, ring_samples=RING, slack_samples=SLACK, pcm_format=_lib.PCM_I16,
                       max_events=8 * SLOTS)
    word = (np.sin(np.arange(12000) * 0.05) * 0.3).astype(np.float32)
    ctx.set_template(0, word)
    ctx.set_stream_params(-1, frame_size=1600, speech_duration_min=0.4, speech_duration_max=1.2)
    return ctx


def make_steps(rate, fmt, occupancy, equal, n_var, rng):
    """n_var step patterns: (streams, pinned buffer, offsets, lens, in_len)"""
    out = []
    n_act = int(round(occupancy * SLOTS))
    active = np.sort(rng.choice(SLOTS, n_act, replace=False)).astype(np.int32)
    for _ in range(n_var):
        lens = np.full(n_act, rate, np.int64) if equal else (rng.uniform(0.5, 1.5, n_act) * rate).astype(np.int64)
        offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
        total = int(lens.sum())
        dt = np.int16 if fmt == "i16" else np.uint8
        buf = _lib.PinnedArray((total,), dt)
        if fmt == "i16":
            buf.array[...] = (rng.standard_normal(total) * 1500).astype(np.int16)
        else:
            buf.array[...] = rng.integers(0, 256, total, dtype=np.uint8)
        out.append((active, buf, offs, lens, total))
    return out


def run_list(rate, fmt, occupancy, equal, steps, warmup, rng, profile=False):
    ctx = make_ctx()
    pats = make_steps(rate, fmt, occupancy, equal, 4, rng)
    esz = 2 if fmt == "i16" else 1
    law = "ulaw" if fmt == "ulaw" else None
    landed_s, h2d, times = 0, 0, []
    try:
        for i in range(warmup + steps):
            st, buf, offs, lens, total = pats[i % len(pats)]
            if profile and i == warmup:
                ctx.synchronize()
                ctx.profile(True)
            ctx.synchronize()
            t0 = time.perf_counter()
            landed = ctx.push_streams(st, (buf.ptr.value, offs, lens, total, buf.array.dtype), sr_in=rate, fmt=law)
            while ctx.tick_ready(64).max() == 64:
                pass
            ctx.poll()
            ctx.synchronize()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
                landed_s += int(landed.sum())
                h2d += total * esz + DESC_BYTES * len(st)
        prof = ctx.profile_read() if profile else None
    finally:
        ctx.close()
    t = float(np.sum(times))
    return {"step_ms_median": float(np.median(times)) * 1e3, "step_ms_mean": t / len(times) * 1e3,
            "active_audio_s_per_s": landed_s / 16000 / t, "h2d_bytes_per_step": h2d / len(times),
            "kernels": {k: prof[k] for k in CLASSES} if prof else None}


def run_uniform(rate, fmt, steps, warmup, rng, profile=False):
    ctx = make_ctx()
    dt = np.int16 if fmt == "i16" else np.uint8
    bufs = []
    for _ in range(4):
        b = _lib.PinnedArray((SLOTS, rate), dt)
        b.array[...] = (rng.standard_normal((SLOTS, rate)) * 1500).astype(np.int16) if fmt == "i16" else \
            rng.integers(0, 256, (SLOTS, rate), dtype=np.uint8)
        bufs.append(b)
    landed_s, ticks, times = 0, 0, []
    try:
        for i in range(warmup + steps):
            if profile and i == warmup:
                ctx.synchronize()
                ctx.profile(True)
            ctx.synchronize()
            t0 = time.perf_counter()
            x = bufs[i % len(bufs)].array
            if rate == 16000:
                ctx.push(x)
                n = rate
            else:
                n = ctx.push_resampled(x, rate, fmt="ulaw")
            landed_s += n
            due = landed_s // 1600 - ticks
            if due > 0:
                ctx.tick(due)
                ticks += due
            ctx.poll()
            ctx.synchronize()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        prof = ctx.profile_read() if profile else None
    finally:
        ctx.close()
    t = float(np.sum(times))
    esz = 2 if fmt == "i16" else 1
    return {"step_ms_median": float(np.median(times)) * 1e3, "step_ms_mean": t / len(times) * 1e3,
            "active_audio_s_per_s": SLOTS * steps / t, "h2d_bytes_per_step": SLOTS * rate * esz,
            "kernels": {k: prof[k] for k in CLASSES} if prof else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r05_ragged_feed.json"))
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"gpu": gpu_info(), "slots": SLOTS, "ring_samples": RING, "slack_samples": SLACK, "steps": a.steps,
           "warmup": a.warmup, "feeds": {}}
    rng = np.random.default_rng(2026)
    for name, rate, fmt in (("pcm16_16k_int16", 16000, "i16"), ("ulaw_8k", 8000, "ulaw")):
        r = {}
        r["uniform_push_all_slots"] = run_uniform(rate, fmt, a.steps, a.warmup, rng)
        r["list_equal_1s_occ100"] = run_list(rate, fmt, 1.0, True, a.steps, a.warmup, rng)
        for occ in (1.0, 0.5, 0.1):
            r[f"list_jitter_occ{int(occ * 100)}"] = run_list(rate, fmt, occ, False, a.steps, a.warmup, rng)
        # per-class kernel times, in passes of their own (event pairs around every launch)
        r["profile_uniform"] = run_uniform(rate, fmt, 10, 3, rng, profile=True)["kernels"]
        for occ in (1.0, 0.1):
            r[f"profile_list_jitter_occ{int(occ * 100)}"] = run_list(rate, fmt, occ, False, 10, 3, rng, profile=True)["kernels"]
        r["list_equal_vs_uniform_step"] = r["list_equal_1s_occ100"]["step_ms_median"] / r["uniform_push_all_slots"]["step_ms_median"]
        res["feeds"][name] = r
        print(json.dumps({name: r}), flush=True)
    res["gpu"]["sm_clock_mhz_at_end"] = sm_clock_now()
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
