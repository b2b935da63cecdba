"""Ragged dense scoring (ewk_dense_scores_streams) and paced dense scoring (ewk_dense_ready) on one GPU, against the uniform
ewk_dense_scores.

    python profiles/tools/ragged_dense_bench.py [--out profiles/r06_ragged_dense.json] [--reps 20]

Bank: 4096 slots, 10 s int16 rings of synthetic speech-like audio (synth.stream_batch), every output left on the device.
1. Equal hop ranges: 4096 streams x 100 hops through the uniform and the ragged entry point, alternated call by call in
   one process, for one template (the bundled word) and for bench.py's 4-template sweep set.
2. Occupancy: 100 / 50 / 10 % of the slots active (a scattered random subset), each with its own row of U(50, 150) hops
   (U(0.5, 1.5) s of audio), through ewk_dense_scores_streams (which runs the rows longest first: r06_ragged_dense.json
   measured that order against list order).
3. A live step at those occupancies: push_streams of U(0.5, 1.5) s per active slot from pinned host memory, tick_ready
   until nothing is due, dense_ready until nothing is due, poll.
Call and step times are host clocks around work that ends in a synchronise; K4 times per launch come from ewk_profile
(CUDA events around each launch) in passes of their own.  The card's name and power limit are read in the same run."""
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

from easywakeword_b200 import _lib, synth  # noqa: E402
from native_rate_bench import gpu_info, sm_clock_now  # noqa: E402
from bench import sweep_templates  # noqa: E402

SLOTS, RING, SLACK = 4096, 160000, 32000
AUDIO_S = 4


def load_word():
    return np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))["pcm_i16"].astype(np.float32) / np.float32(32768)


def make_ctx(tpls, live):
    ctx = _lib.Context(device=0, n_streams=SLOTS, ring_samples=RING, slack_samples=SLACK, pcm_format=_lib.PCM_I16,
                       max_templates=len(tpls), max_events=8 * SLOTS)
    for i, t in enumerate(tpls):
        ctx.set_template(i, t)
    ctx.set_stream_params(-1, frame_size=1600, speech_duration_min=0.4, speech_duration_max=1.2, live=1 if live else 0)
    return ctx


def timed(fn, ctx):
    ctx.synchronize()
    t0 = time.perf_counter()
    fn()
    ctx.synchronize()
    return time.perf_counter() - t0


def k4_profile(ctx, fn, n):
    ctx.synchronize()
    ctx.profile(True)
    for _ in range(n):
        fn()
    p = ctx.profile_read()["dense_score"]
    ctx.profile(False)
    return p["ms"] / max(1, p["launches"])


def equal_ranges(ctx, T, reps):
    out = torch.empty(SLOTS * 100 * T, dtype=torch.float32, device="cuda:0")
    st = np.arange(SLOTS, dtype=np.int32)
    h0, nh = np.full(SLOTS, 201, np.int64), np.full(SLOTS, 100, np.int32)

    def uni():
        ctx.dense_scores(201, 100, 0, T, out_device_ptr=out.data_ptr())

    def rag():
        ctx.dense_scores_streams(st, h0, nh, 0, T, out_device_ptr=out.data_ptr())

    for _ in range(3):
        uni(), rag()
    tu, tr = [], []
    for _ in range(reps):
        tu.append(timed(uni, ctx))
        tr.append(timed(rag, ctx))
    k4u, k4r = k4_profile(ctx, uni, 5), k4_profile(ctx, rag, 5)
    return {"uniform_call_ms_median": float(np.median(tu)) * 1e3, "ragged_call_ms_median": float(np.median(tr)) * 1e3,
            "uniform_k4_ms": k4u, "ragged_k4_ms": k4r, "ragged_over_uniform_k4": k4r / k4u,
            "ragged_over_uniform_call": float(np.median(tr) / np.median(tu))}


def occupancy(ctx, occ, reps, rng):
    n_act = int(round(occ * SLOTS))
    st = np.sort(rng.choice(SLOTS, n_act, replace=False)).astype(np.int32)
    nh = rng.integers(50, 151, n_act).astype(np.int32)
    h0 = (AUDIO_S * 100 - nh).astype(np.int64)                 # rows end at the newest hop
    out = torch.empty(int(nh.sum()), dtype=torch.float32, device="cuda:0")
    windows = int(nh.sum())

    def call():
        ctx.dense_scores_streams(st, h0, nh, 0, 1, out_device_ptr=out.data_ptr())

    times = [timed(call, ctx) for _ in range(reps + 2)][2:]
    k4 = k4_profile(ctx, call, 5)
    res = {"longest_first": {"call_ms_median": float(np.median(times)) * 1e3, "k4_ms": k4,
                             "windows_per_s_k4": windows / (k4 * 1e-3)}}
    res["active_streams"], res["windows"] = n_act, windows
    return res


def live_steps(word, occ, steps, warmup, rng):
    ctx = make_ctx([word], live=False)
    n_act = int(round(occ * SLOTS))
    active = np.sort(rng.choice(SLOTS, n_act, replace=False)).astype(np.int32)
    pats = []
    for _ in range(4):
        lens = (rng.uniform(0.5, 1.5, n_act) * 16000).astype(np.int64)
        offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
        buf = _lib.PinnedArray((int(lens.sum()),), np.int16)
        buf.array[...] = (rng.standard_normal(int(lens.sum())) * 1500).astype(np.int16)
        pats.append((buf, offs, lens))
    out = torch.empty(n_act * 200, dtype=torch.float32, device="cuda:0")
    times, hops = [], 0
    try:
        for i in range(warmup + steps):
            buf, offs, lens = pats[i % len(pats)]
            ctx.synchronize()
            t0 = time.perf_counter()
            ctx.push_streams(active, (buf.ptr.value, offs, lens, int(lens.sum()), np.int16))
            while ctx.tick_ready(64).max() == 64:
                pass
            n = 0
            while True:
                _, nh = ctx.dense_ready(active, 200, 0, 1, out_device_ptr=out.data_ptr())
                n += int(nh.sum())
                if nh.max() < 200:
                    break
            ctx.poll()
            ctx.synchronize()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
                hops += n
    finally:
        ctx.close()
    return {"step_ms_median": float(np.median(times)) * 1e3, "hops_per_step": hops / len(times),
            "active_streams": n_act}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r06_ragged_dense.json"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"gpu": gpu_info(), "slots": SLOTS, "ring_samples": RING, "reps": a.reps}
    word = load_word()
    rng = np.random.default_rng(2026)
    pcm = synth.stream_batch(7, SLOTS, float(AUDIO_S), word, as_int16=True, gain=(1.0, 4.0))
    sweep, _ = sweep_templates(word)
    for name, tpls in (("T1", [word]), ("T4_sweep_set", sweep)):
        ctx = make_ctx(tpls, live=True)
        ctx.push(np.ascontiguousarray(pcm))
        res[f"equal_4096x100_{name}"] = equal_ranges(ctx, len(tpls), a.reps)
        print(json.dumps({name: res[f"equal_4096x100_{name}"]}), flush=True)
        if name == "T1":
            for occ in (1.0, 0.5, 0.1):
                res[f"occupancy{int(occ * 100)}"] = occupancy(ctx, occ, a.reps, rng)
                print(json.dumps({occ: res[f"occupancy{int(occ * 100)}"]}), flush=True)
        ctx.close()
    for occ in (1.0, 0.5, 0.1):
        res[f"live_step_occupancy{int(occ * 100)}"] = live_steps(word, occ, a.steps, 4, rng)
        print(json.dumps({occ: res[f"live_step_occupancy{int(occ * 100)}"]}), flush=True)
    res["gpu"]["sm_clock_mhz_at_end"] = sm_clock_now()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
