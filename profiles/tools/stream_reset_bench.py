"""Stream recycling on one GPU: K9 (ewk_reset_streams) against HBM bandwidth, a churn workload against the same workload
without resets, ewk_push_resampled_each against ewk_push_resampled at equal positions, and the uniform K8 of this build
against another build (--alt-lib, e.g. the parent commit's libewk.so) alternated in one run.

    python profiles/tools/stream_reset_bench.py [--alt-lib experiments/libewk_alt.so] [--out profiles/r04_stream_reset.json]

K9 times are the device durations of stream_reset_kernel from torch.profiler (CUDA activities), at the bench geometry:
10 s int16 rings + 1.2 s of slack.  Bytes are the ring rows plus the state, block-sum and chunk rows of each listed
stream.  Step times are host clocks around steps that end in a synchronise."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

TOOLS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(TOOLS))
sys.path.insert(0, REPO)
sys.path.insert(0, TOOLS)

from easywakeword_b200 import _lib, synth  # noqa: E402
from native_rate_bench import feed, gpu_info, sm_clock_now  # noqa: E402

RING, SLACK = 160000, 19200                      # WakeWordBank(buffer_seconds=10, max_push_seconds=1.0)
HBM_MEASURED, HBM_SHEET = 6.5e12, 7.7e12


def leg_k9(streams, counts, reps):
    ctx = _lib.Context(device=0, n_streams=streams, ring_samples=RING, slack_samples=SLACK, pcm_format=_lib.PCM_I16)
    P = (RING + SLACK + 63) // 64 * 64
    NB, chunk_cap = P // 1600, RING // 160
    per_stream = P * 2 + 8 * NB + 16 * chunk_cap + 128 + 8
    rng = np.random.default_rng(9)
    out = []
    try:
        for n in counts:
            lst = np.sort(rng.choice(streams, n, replace=False))
            for _ in range(3):
                ctx.reset_streams(lst)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    ctx.reset_streams(lst)
                ctx.synchronize()
            dur = [e.device_time for e in prof.events() if "stream_reset_kernel" in e.name]
            t = float(np.median(dur)) * 1e-6 if dur else float("nan")
            b = n * per_stream
            out.append({"streams": n, "kernels": len(dur), "kernel_us_median": t * 1e6, "bytes": b,
                        "tb_per_s": b / t / 1e12, "of_measured_6_5": b / t / HBM_MEASURED,
                        "of_datasheet_7_7": b / t / HBM_SHEET})
            print(json.dumps(out[-1]), flush=True)
    finally:
        ctx.close()
    return out


def leg_churn(streams, steps, warm, rounds, churn, word):
    from easywakeword_b200.bank import WakeWordBank
    rng = np.random.default_rng(4)
    codes = _lib.PinnedArray((streams, 8000), np.uint8)
    codes.array[...] = feed(8000, "ulaw", streams, torch.Generator().manual_seed(3)).numpy()
    banks = {k: WakeWordBank(streams, [word], sample_rate=8000, max_events=8 * streams) for k in ("steady", "churn")}
    times = {k: [] for k in banks}
    resets = 0
    try:
        def step(k):
            b = banks[k]
            if k == "churn":
                nonlocal resets
                lst = rng.choice(streams, max(1, int(round(churn * streams))), replace=False)
                b.reset(lst)
                resets += len(lst)
            b.push_g711(codes.array)
            due = b.samples_pushed // 1600 - b.ticks
            if due > 0:
                b.tick(due)
            b.poll()
        for k in banks:
            for _ in range(warm):
                step(k)
            banks[k].ctx.synchronize()
        for _ in range(rounds):
            for k in banks:
                t0 = time.perf_counter()
                for _ in range(steps):
                    step(k)
                banks[k].ctx.synchronize()
                times[k].append((time.perf_counter() - t0) / steps * 1e3)
        res = {k: {"ms_per_step": v, "median": float(np.median(v))} for k, v in times.items()}
        res["ratio_churn_over_steady"] = res["churn"]["median"] / res["steady"]["median"]
        res["streams_reset_per_step"] = max(1, int(round(churn * streams)))
        return res
    finally:
        for b in banks.values():
            b.close()
        codes.free()


def leg_each_vs_uniform(sr, kind, streams, steps, rounds):
    """equal positions: ewk_push_resampled_each against ewk_push_resampled, alternated, K8 time from ewk_profile"""
    x = feed(sr, kind, streams, torch.Generator().manual_seed(sr)).cuda()
    dev = (x.data_ptr(), streams, sr, sr, {"i16": np.int16, "ulaw": np.uint8}[kind])
    fmt = "ulaw" if kind == "ulaw" else None
    ctxs = {k: _lib.Context(device=0, n_streams=streams, ring_samples=RING, slack_samples=32000,
                            pcm_format=_lib.PCM_I16) for k in ("uniform", "each")}
    ms = {k: [] for k in ctxs}
    try:
        for c in ctxs.values():
            c.set_stream_params(-1, live=1)
        for _ in range(rounds):
            for k, c in ctxs.items():
                c.synchronize()
                c.profile(True)
                for _ in range(steps):
                    if k == "each":
                        c.push_resampled_each(dev, sr, where=_lib.DEVICE, fmt=fmt)
                    else:
                        c.push_resampled(dev, sr, where=_lib.DEVICE, fmt=fmt)
                r = c.profile_read()["resample_push"]
                c.profile(False)
                ms[k].append(r["ms"] / r["launches"])
        same = all(np.array_equal(ctxs["uniform"].read_last(s, RING), ctxs["each"].read_last(s, RING))
                   for s in range(0, streams, max(1, streams // 64)))
        return {"sr": sr, "kind": kind, "streams": streams, "k8_ms_per_push": ms,
                "median": {k: float(np.median(v)) for k, v in ms.items()}, "rings_equal_sampled_64": same}
    finally:
        for c in ctxs.values():
            c.close()


AB_CHILD = r"""
import ctypes, json, sys
class Tolerant(ctypes.CDLL):
    # a library without this build's newer entry points still declares the rest
    def __getattr__(self, name):
        try:
            return super().__getattr__(name)
        except AttributeError:
            if not name.startswith("ewk_"):
                raise
            f = ctypes.CFUNCTYPE(ctypes.c_int)(lambda *a: -1)
            setattr(self, name, f)
            return f
ctypes.CDLL = Tolerant
sys.path.insert(0, sys.argv[2]); sys.path.insert(0, sys.argv[3])
from easywakeword_b200 import _lib
_lib.LIB_PATH = sys.argv[1]
import torch
from native_rate_bench import leg_kernel
sm = torch.cuda.get_device_properties(0).multi_processor_count
print(json.dumps([leg_kernel(48000, "i16", 4096, 10, sm), leg_kernel(8000, "ulaw", 4096, 10, sm)]))
"""


def leg_ab(alt, rounds):
    libs = {"this": os.path.join(REPO, "easywakeword_b200", "libewk.so"), "alt": alt}
    out = {k: [] for k in libs}
    for _ in range(rounds):
        for k, path in libs.items():
            r = subprocess.run([sys.executable, "-c", AB_CHILD, path, REPO, TOOLS], capture_output=True, text=True)
            if r.returncode:
                raise RuntimeError(r.stderr[-2000:])
            legs = json.loads(r.stdout.strip().splitlines()[-1])
            out[k].append({str(l['sr_in']): l for l in legs})
    summary = {}
    for k, runs in out.items():
        summary[k] = {sr: [r[sr]["kernel_ms_per_step"] for r in runs] for sr in runs[0]}
    return {"runs": out, "kernel_ms_per_step": summary}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--alt-lib", default="")
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r04_stream_reset.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("stream_reset_bench needs a CUDA device")
    from easywakeword_b200 import build
    build.build()
    res = {"gpu": gpu_info()}
    word = synth.synthetic_word()
    res["k9"] = leg_k9(args.streams, [1, 64, 512, args.streams], 20)
    res["churn_8k_ulaw"] = leg_churn(args.streams, 5, 12, 3, 0.01, word)
    print(json.dumps({k: v for k, v in res["churn_8k_ulaw"].items() if k != "steady"}), flush=True)
    res["each_vs_uniform"] = [leg_each_vs_uniform(48000, "i16", args.streams, 10, 3),
                              leg_each_vs_uniform(8000, "ulaw", args.streams, 10, 3)]
    print(json.dumps(res["each_vs_uniform"]), flush=True)
    if args.alt_lib:
        res["uniform_k8_ab"] = leg_ab(args.alt_lib, 2)
        print(json.dumps(res["uniform_k8_ab"]["kernel_ms_per_step"]), flush=True)
    res["gpu"]["sm_clock_mhz_at_end"] = sm_clock_now()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"wrote": args.out}))


if __name__ == "__main__":
    main()
