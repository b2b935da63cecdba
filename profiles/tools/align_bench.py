"""Frame alignment on one GPU: 4096 ring segments of 0.6 .. 1.5 s against 1, 4 and 64 templates per row.

    python profiles/tools/align_bench.py [--out profiles/r11_align.json] [--runs 7] [--warmup 2]

One context: 4096 streams, 4096 template slots with stored frames (template_frames = 1), 3 s int16 rings.  Slot s holds
0.6 .. 1.5 s of stream s's own audio (ewk_set_templates_from_streams); row s aligns 0.6 .. 1.5 s of stream s against
slots [s', s' + T) with s' = min(s, 4096 - T).  Legs T = 1, 4, 64, alternated run by run.
  ms per call: a host clock around ewk_align_segments, which ends in a synchronise; median over the timed runs.
  K3 + K11 ms: ewk_profile's class-3 time of one call (K3 and K11 each bracketed by events), median, separate runs.
  DP cells per second: sum over rows and templates of n_i * m_j, over the call's time.
Launches per call from ewk_launch_count.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

TOOLS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(TOOLS))
sys.path.insert(0, REPO)

from easywakeword_b200 import _lib, synth  # noqa: E402

N, SR = 4096, 16000


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    return r.stdout.strip().splitlines()[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    rng = np.random.default_rng(11)
    bases = [synth.synthetic_word(seed=200 + i, duration=1.5) for i in range(64)]
    q = np.stack([synth.to_int16(np.concatenate([bases[s % 64] * np.float32(1.0 + (s % 7) / 7),
                                                 np.zeros(SR * 2 - len(bases[0]), np.float32)])) for s in range(N)])
    ctx = _lib.Context(device=0, n_streams=N, ring_samples=3 * SR, slack_samples=2 * SR, pcm_format=_lib.PCM_I16,
                       max_templates=N, max_events=8192, template_frames=True)
    ctx.set_stream_params(-1, frame_size=1600, live=1)
    ctx.push(q)
    streams = np.arange(N, dtype=np.int32)
    t_lens = rng.integers(int(0.6 * SR), int(1.5 * SR) + 1, N)
    ctx.set_templates_from_streams(streams, streams, np.zeros(N, np.int64), t_lens)
    s_lens = rng.integers(int(0.6 * SR), int(1.5 * SR) + 1, N)
    starts = rng.integers(0, 2 * SR - s_lens + 1).astype(np.int64)
    n_seg = 1 + s_lens // 160
    m_tmpl = 1 + t_lens // 160
    legs = {}
    for T in (1, 4, 64):
        first = np.minimum(streams, N - T).astype(np.int32)
        cells = int(sum(int(n_seg[i]) * int(m_tmpl[first[i]:first[i] + T].sum()) for i in range(N)))
        legs[T] = (first, cells)
    times = {T: [] for T in legs}
    launches, k11 = {}, {}
    for r in range(a.warmup + a.runs):
        for T, (first, _) in legs.items():
            l0 = ctx.launch_count()
            t0 = time.perf_counter()
            ctx.align_segments(streams, starts, s_lens, first, np.full(N, T, np.int32))
            dt = time.perf_counter() - t0
            launches[T] = ctx.launch_count() - l0
            if r >= a.warmup:
                times[T].append(dt * 1e3)
    # event-timed K3 + K11 of each leg (ewk_profile's class 3 holds both): a run of its own, profiling on
    ctx.profile(True)
    for T, (first, _) in legs.items():
        v = []
        for _ in range(a.runs):
            ctx.profile_read()
            ctx.align_segments(streams, starts, s_lens, first, np.full(N, T, np.int32))
            v.append(ctx.profile_read()["segment_batch"]["ms"])
        k11[T] = float(np.median(v))
    ctx.profile(False)
    res = {"gpu": gpu_info(), "rows": N, "segment_seconds": [0.6, 1.5], "template_seconds": [0.6, 1.5], "runs": a.runs,
           "warmup": a.warmup, "launches": {str(T): launches[T] for T in legs},
           "ms_median": {str(T): round(float(np.median(v)), 3) for T, v in times.items()},
           "ms_min": {str(T): round(float(np.min(v)), 3) for T, v in times.items()},
           "ms_max": {str(T): round(float(np.max(v)), 3) for T, v in times.items()},
           "k3_plus_k11_event_ms": {str(T): round(k11[T], 3) for T in legs},
           "dp_cells": {str(T): legs[T][1] for T in legs},
           "dp_cells_per_s_call": {str(T): float(f"{legs[T][1] / (np.median(times[T]) * 1e-3):.4g}") for T in legs}}
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")
    ctx.close()


if __name__ == "__main__":
    main()
