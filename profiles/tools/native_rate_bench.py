"""K8 (ewk_push_resampled) on one GPU: the fused native-rate push against its FMA bound, against the two-step path
(ewk_resample device -> device, then ewk_push), end to end from a pinned host feed, and ewk_resample on its own shapes
(few rows, long inputs) beside a push of the same input.

    python profiles/tools/native_rate_bench.py [--streams 4096] [--steps 10] [--out profiles/r03_native_rate.json]

Every leg pushes 1.0 s of input per stream per step.  Kernel times are CUDA-event sums of ewk_profile (class 7
resample_push, 3 segment_batch for ewk_resample, 0 ring_push); step times are host clocks around steps that end in a
synchronise.  FMAs are computed from the shapes: landed outputs x 2W.  The FP32 FMA bound is 148 SMs x 128 lanes x the
SM clock read in the same run.  Inputs (>= 131 MB per step at 4096 streams) exceed the 126 MB L2."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)

from easywakeword_b200 import _lib  # noqa: E402
from easywakeword_b200.resample import ready_outputs  # noqa: E402

LANES_PER_SM = 128


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, pl, sm, smax = [v.strip() for v in r.stdout.strip().split(",")]
    return {"name": name, "power_limit_w": float(pl), "sm_clock_mhz_at_start": float(sm), "sm_clock_max_mhz": float(smax)}


def sm_clock_now():
    r = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    return float(r.stdout.strip())


def feed(sr, kind, streams, gen):
    """One second per stream of plausible audio at sr: band-limited noise bursts, int16 / uint8 G.711 / float32."""
    n = sr
    x = torch.randn(streams, n, generator=gen) * 0.05
    x = torch.clamp(x, -0.99, 0.99)
    if kind == "f32":
        return x.contiguous()
    q = torch.round(x * 32768).to(torch.int16)
    if kind == "i16":
        return q.contiguous()
    return torch.randint(0, 256, (streams, n), generator=gen, dtype=torch.uint8)   # G.711 codes: any byte is a code


def prof(ctx):
    r = ctx.profile_read()
    return {k: v for k, v in r.items() if v["launches"]}


def leg_kernel(sr, kind, streams, steps, sm_count):
    W, L, M = _lib.resample_info(sr)
    x = feed(sr, kind, streams, torch.Generator().manual_seed(sr)).cuda()
    ctx = _lib.Context(device=0, n_streams=streams, ring_samples=160000, slack_samples=32000, pcm_format=_lib.PCM_I16)
    ctx.set_stream_params(-1, live=1)
    fmt = {"ulaw": "ulaw"}.get(kind)
    dev = (x.data_ptr(), streams, sr, sr, {"i16": np.int16, "f32": np.float32, "ulaw": np.uint8}[kind])
    c = 0
    for _ in range(3):
        ctx.push_resampled(dev, sr, where=_lib.DEVICE, fmt=fmt)
        c += sr
    ctx.synchronize()
    ctx.profile(True)
    clk = []
    outs = 0
    for _ in range(steps):
        outs += ctx.push_resampled(dev, sr, where=_lib.DEVICE, fmt=fmt)
        c += sr
    clk.append(sm_clock_now())
    p = prof(ctx)
    ctx.profile(False)
    ctx.close()
    ms = p["resample_push"]["ms"]
    fma = float(outs) * streams * 2 * W
    clock = float(np.mean(clk))
    bound = sm_count * LANES_PER_SM * clock * 1e6
    return {"sr_in": sr, "input": kind, "L": L, "M": M, "taps": 2 * W, "streams": streams, "steps": steps,
            "path": "fast (register windows)" if L in (1, 2, 4, 8) and M <= 3 else "generic",
            "kernel_ms_per_step": ms / steps, "fma_per_step": fma / steps, "fma_per_s": fma / (ms * 1e-3),
            "sm_clock_mhz_during": clock, "fp32_fma_bound_per_s": bound, "share_of_fma_bound": fma / (ms * 1e-3) / bound,
            "audio_s_per_s": streams * steps / (ms * 1e-3)}


def leg_two_step(sr, streams, steps, rounds):
    """Fused K8 vs ewk_resample (device -> device) + ewk_push, alternating, f32 rings; the history the streaming
    ewk_resample call needs sits in place in front of the chunk (the feed repeats one chunk), so no copy is charged."""
    W, L, M = _lib.resample_info(sr)
    x = feed(sr, "i16", streams, torch.Generator().manual_seed(7))
    hist = 2 * W
    xx = torch.cat([x[:, -hist:], x], dim=1).contiguous().cuda()
    x = x.cuda()
    y = torch.empty(streams, 16000 + 16, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    A = _lib.Context(device=0, n_streams=streams, ring_samples=160000, slack_samples=32000, pcm_format=_lib.PCM_F32)
    B = _lib.Context(device=0, n_streams=streams, ring_samples=160000, slack_samples=32000, pcm_format=_lib.PCM_F32)
    for ctx in (A, B):
        ctx.set_stream_params(-1, live=1)
    st = {"c": 0, "o": 0}

    def fused():
        A.push_resampled((x.data_ptr(), streams, sr, sr, np.int16), sr, where=_lib.DEVICE)

    def two_step():
        c, o0 = st["c"], st["o"]
        o1 = ready_outputs(c + sr, W, L, M)
        if c == 0:
            ptr, in_first, n_in = x.data_ptr(), 0, sr
        else:                                                   # input [c - hist, c + sr) = tail of the chunk ++ chunk
            ptr, in_first, n_in = xx.data_ptr(), c - hist, hist + sr
        stride = sr if c == 0 else hist + sr
        B.resample((ptr, streams, n_in, stride, np.int16), sr, in_first=in_first, out_first=o0, n_out=o1 - o0,
                   out_device_ptr=y.data_ptr())
        # ewk_resample wrote rows n_out apart
        B.push((y.data_ptr(), streams, o1 - o0, o1 - o0), where=_lib.DEVICE)
        st["c"], st["o"] = c + sr, o1

    t = {"fused": [], "two_step": []}
    for r in range(rounds + 1):
        for name, fn, ctx in (("fused", fused, A), ("two_step", two_step, B)):
            ctx.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                fn()
            ctx.synchronize()
            if r:                                               # round 0 warms up
                t[name].append((time.perf_counter() - t0) / steps * 1e3)
    equal = all(np.array_equal(A.read_last(s, 160000), B.read_last(s, 160000)) for s in (0, streams // 2, streams - 1))
    # kernel times of one profiled step each
    A.profile(True); fused(); pa = prof(A); A.profile(False)
    B.profile(True); two_step(); pb = prof(B); B.profile(False)
    A.close(); B.close()
    return {"sr_in": sr, "streams": streams, "steps_per_round": steps, "rounds": rounds,
            "fused_ms_per_step": {"median": float(np.median(t["fused"])), "all": t["fused"]},
            "two_step_ms_per_step": {"median": float(np.median(t["two_step"])), "all": t["two_step"]},
            "speedup": float(np.median(t["two_step"]) / np.median(t["fused"])),
            "fused_kernels_one_step": pa, "two_step_kernels_one_step": pb, "rings_equal": bool(equal)}


def leg_end_to_end(sr, kind, streams, steps, word):
    """Pinned host feed, push + tick + poll per step (int16 rings, audio clock), against a plain H2D copy of the same bytes."""
    x = feed(sr, kind, streams, torch.Generator().manual_seed(11)).numpy()
    pin = _lib.PinnedArray(x.shape, x.dtype)
    pin.array[:] = x
    ctx = _lib.Context(device=0, n_streams=streams, ring_samples=160000, slack_samples=2 * 16000 + 3200,
                       pcm_format=_lib.PCM_I16, max_events=max(4096, 4 * streams))
    ctx.set_template(0, word)
    ctx.set_stream_params(-1, speech_duration_min=0.5, speech_duration_max=1.6, frame_size=1600)
    fmt = "ulaw" if kind == "ulaw" else None
    st = {"landed": 0, "ticks": 0}

    def step():
        st["landed"] += ctx.push_resampled(pin.array, sr, fmt=fmt)
        due = st["landed"] // 1600 - st["ticks"]
        if due > 0:
            ctx.tick(due)
            st["ticks"] += due
        ctx.poll()

    for _ in range(3):
        step()
    ctx.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    ctx.synchronize()
    step_ms = (time.perf_counter() - t0) / steps * 1e3
    ctx.profile(True)
    for _ in range(3):
        step()
    p = prof(ctx)
    ctx.profile(False)
    ctx.close()
    kern_ms = sum(v["ms"] for v in p.values()) / 3
    # plain H2D of the same bytes, CUDA events
    src = torch.from_numpy(x).pin_memory()
    dst = torch.empty_like(src, device="cuda")
    dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        dst.copy_(src, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    h2d_ms = e0.elapsed_time(e1) / steps
    pin.free()
    bound = "PCIe (H2D copy)" if h2d_ms >= kern_ms else "device kernels"
    return {"sr_in": sr, "input": kind, "streams": streams, "bytes_per_step": int(x.nbytes), "step_ms": step_ms,
            "audio_s_per_s": streams / (step_ms * 1e-3), "step_kernel_ms": kern_ms, "kernels_per_step": p,
            "h2d_copy_ms": h2d_ms, "h2d_gb_per_s": x.nbytes / (h2d_ms * 1e-3) / 1e9, "bound": bound}


def leg_few_rows(sr, seconds, rows, reps):
    """ewk_resample's own shape (one-shot, float32 rows out) beside ewk_push_resampled landing the same outputs in f32
    rings with one push of the whole input: the same FIR with and without the ring."""
    n = sr * seconds
    x = feed(sr, "f32", rows, torch.Generator().manual_seed(5))
    x = torch.cat([x] * seconds, dim=1).contiguous().cuda()
    n_out = int(_lib.load().ewk_resample_out_len(n, sr))
    y = torch.empty(rows, n_out, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    one = _lib.Context(device=0, n_streams=0)
    one.resample((x.data_ptr(), rows, n, n, np.float32), sr, out_device_ptr=y.data_ptr())      # table, smem attribute
    one.profile(True)
    for _ in range(reps):
        one.resample((x.data_ptr(), rows, n, n, np.float32), sr, out_device_ptr=y.data_ptr())
    p7 = prof(one)["segment_batch"]
    one.close()
    ms8, landed = [], 0
    for _ in range(reps):
        ctx = _lib.Context(device=0, n_streams=rows, ring_samples=16000 * (seconds + 1), slack_samples=16000,
                           pcm_format=_lib.PCM_F32)
        ctx.set_stream_params(-1, live=1)
        ctx.profile(True)
        landed = ctx.push_resampled((x.data_ptr(), rows, n, n, np.float32), sr, where=_lib.DEVICE)
        ms8.append(prof(ctx)["resample_push"]["ms"])
        ctx.close()
    return {"sr_in": sr, "rows": rows, "seconds": seconds, "ewk_resample_ms": p7["ms"] / p7["launches"],
            "ewk_resample_outputs": n_out, "push_resampled_ms": float(np.median(ms8)), "push_resampled_outputs": landed}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r03_native_rate.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("native_rate_bench needs a CUDA device")
    from easywakeword_b200 import build
    build.build()
    info = gpu_info()
    sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    info["sm_count"] = sm_count
    word = np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))["pcm_i16"].astype(np.float32) / 32768
    res = {"gpu": info, "kernel": [], "two_step": [], "end_to_end": [], "few_rows": []}
    for sr, kind in ((48000, "i16"), (8000, "ulaw"), (44100, "i16")):
        res["kernel"].append(leg_kernel(sr, kind, args.streams, args.steps, sm_count))
        print(json.dumps(res["kernel"][-1]), flush=True)
    for sr in (48000, 8000):
        res["two_step"].append(leg_two_step(sr, args.streams, args.steps, 3))
        print(json.dumps(res["two_step"][-1]), flush=True)
    for sr, kind in ((48000, "i16"), (8000, "ulaw")):
        res["end_to_end"].append(leg_end_to_end(sr, kind, args.streams, args.steps, word))
        print(json.dumps(res["end_to_end"][-1]), flush=True)
    for sr in (48000, 44100, 8000):
        res["few_rows"].append(leg_few_rows(sr, 30, 2, 5))
        print(json.dumps(res["few_rows"][-1]), flush=True)
    res["gpu"]["sm_clock_mhz_at_end"] = sm_clock_now()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"wrote": args.out}))


if __name__ == "__main__":
    main()
