"""Stream migration on one GPU: K10 (ewk_export_streams / ewk_import_streams) against HBM bandwidth, export + import
through a pinned host blob against the PCIe copy rate, and a rebalance loop of two banks against the same loop without
moves.

    python profiles/tools/stream_migrate_bench.py [--out profiles/r08_stream_migrate.json]

Geometry: 10 s int16 rings + 1.2 s of slack (WakeWordBank(buffer_seconds=10, max_push_seconds=1.0)), 4096 streams.
K10 times are the device durations of stream_export_kernel / stream_import_kernel from torch.profiler (CUDA activities),
median of 20, device blobs.  Bytes are the bulk rows (ring, block sums, chunk mean squares) plus the small state, each
read once and written once.  The reference rates are measured in the same run: a device-to-device torch copy of 1 GiB
(HBM) and pinned host <-> device copies of 1 GiB (PCIe).  Host-blob times are host clocks around the calls, which end in
a synchronise.  The rebalance loop feeds 8 kHz mu-law to two 4096-stream contexts (push_streams + tick_ready per 1 s
step) and moves 1 % of the streams from one to the other each step (export, poll, import, reset), alternated step by
step with the same loop without moves.  The card's name and power limit are read in the same run."""
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
from native_rate_bench import gpu_info  # noqa: E402

RING, SLACK, SLOTS, REPS = 160000, 19200, 4096, 20
HBM_SHEET = 7.7e12


def load_word():
    return np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))["pcm_i16"].astype(np.float32) / np.float32(32768)


def copy_rates():
    """bytes / s of a 1 GiB device-to-device copy (read + write counted) and of pinned H2D / D2H copies"""
    n = 1 << 30
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    h = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    out = {}
    for name, fn, factor in (("d2d", lambda: b.copy_(a), 2), ("h2d", lambda: a.copy_(h, non_blocking=True), 1),
                             ("d2h", lambda: h.copy_(a, non_blocking=True), 1)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out[name] = factor * n * 10 / (e0.elapsed_time(e1) * 1e-3)
    return out


def make_ctx(word, n=SLOTS):
    ctx = _lib.Context(device=0, n_streams=n, ring_samples=RING, slack_samples=SLACK, pcm_format=_lib.PCM_I16,
                       max_templates=1, max_events=8 * n)
    ctx.set_template(0, word)
    return ctx


def leg_kernels(word, counts, rates):
    ctx = make_ctx(word)
    L = _lib.stream_blob_layout(RING, SLACK, _lib.PCM_I16, 1, 0, 0)
    per_stream = L["bulk_row_bytes"] + 112 + 8 + 48                  # bulk row + StreamState, result, DetState
    cap = ctx.stream_blob_bytes(SLOTS)
    d = torch.empty(cap, dtype=torch.uint8, device="cuda")
    rng = np.random.default_rng(3)
    ctx.push(np.zeros((SLOTS, 16000), np.int16))
    ctx.tick(10)
    ctx.poll()
    out = []
    try:
        for n in counts:
            lst = rng.choice(SLOTS, n, replace=False).astype(np.int32)
            for _ in range(3):
                ctx.export_streams(lst, where=_lib.DEVICE, out=(d.data_ptr(), cap))
                ctx.import_streams(lst, (d.data_ptr(), cap), where=_lib.DEVICE)
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(REPS):
                    ctx.export_streams(lst, where=_lib.DEVICE, out=(d.data_ptr(), cap))
                    ctx.import_streams(lst, (d.data_ptr(), cap), where=_lib.DEVICE)
            row = {"streams": int(n), "bytes_read_and_written": 2 * n * per_stream}
            for k in ("stream_export_kernel", "stream_import_kernel"):
                dur = [e.device_time for e in prof.events() if k in e.name]
                t = float(np.median(dur)) * 1e-6
                tbs = 2 * n * per_stream / t / 1e12
                row[k] = {"median_us": t * 1e6, "launches": len(dur), "tb_per_s": tbs,
                          "share_of_measured_copy": tbs * 1e12 / rates["d2d"], "share_of_data_sheet": tbs * 1e12 / HBM_SHEET}
            out.append(row)
            print(json.dumps(row), flush=True)
    finally:
        ctx.close()
    return out


def leg_host(word, counts, rates):
    ctx = make_ctx(word)
    dst = make_ctx(word)
    cap = ctx.stream_blob_bytes(SLOTS)
    pin = _lib.PinnedArray((cap,), np.uint8)
    rng = np.random.default_rng(4)
    out = []
    import ctypes as C
    try:
        for n in counts:
            lst = rng.choice(SLOTS, n, replace=False).astype(np.int32)
            sp = lst.ctypes.data_as(C.POINTER(C.c_int32))
            te, ti = [], []
            for r in range(REPS + 3):
                t0 = time.perf_counter()
                ctx._ck(ctx.lib.ewk_export_streams(ctx.h, sp, n, pin.ptr, cap, _lib.HOST))
                t1 = time.perf_counter()
                dst._ck(dst.lib.ewk_import_streams(dst.h, sp, n, pin.ptr, cap, _lib.HOST))
                t2 = time.perf_counter()
                if r >= 3:
                    te.append(t1 - t0)
                    ti.append(t2 - t1)
            nbytes = int(pin.array[:96].view(_lib.STREAM_BLOB_HEADER_DTYPE)[0]["total_bytes"])
            row = {"streams": int(n), "blob_bytes": nbytes}
            for name, ts, ref in (("export_d2h", te, rates["d2h"]), ("import_h2d", ti, rates["h2d"])):
                t = float(np.median(ts))
                row[name] = {"median_ms": t * 1e3, "gb_per_s": nbytes / t / 1e9, "share_of_measured_pcie": nbytes / t / ref}
            out.append(row)
            print(json.dumps(row), flush=True)
    finally:
        pin.free()
        ctx.close()
        dst.close()
    return out


def leg_rebalance(word, steps):
    """two banks, 8 kHz mu-law; the 'move' pair moves 1 % of streams a -> b each step, the 'still' pair does not"""
    codes = synth.stream_batch(77, 64, 8.0, word, as_int16=True, gain=(2.0, 4.0))[:, ::2]     # 8 kHz (decimated)
    from easywakeword_b200.resample import ULAW_TABLE
    table = ULAW_TABLE.astype(np.int32)
    order = np.argsort(table, kind="stable")
    srt = table[order]
    i = np.clip(np.searchsorted(srt, codes.astype(np.int32)), 1, 255)
    codes = order[np.where(np.abs(srt[i] - codes) < np.abs(srt[i - 1] - codes), i, i - 1)].astype(np.uint8)
    pairs = {k: [make_ctx(word), make_ctx(word)] for k in ("move", "still")}
    for a, b in pairs.values():
        for c in (a, b):
            c.set_stream_params(-1, frame_size=1600, speech_duration_min=0.5, speech_duration_max=1.6)
    n_move = SLOTS // 100
    rng = np.random.default_rng(5)
    times = {"move": [], "still": []}
    allst = list(range(SLOTS))
    try:
        for step in range(steps):
            feed = [codes[s % 64, (step % 8) * 8000:(step % 8 + 1) * 8000] for s in range(SLOTS)]
            src = rng.choice(SLOTS, n_move, replace=False).tolist()
            dstl = rng.choice(SLOTS, n_move, replace=False).tolist()
            for kind in (("move", "still") if step % 2 == 0 else ("still", "move")):
                a, b = pairs[kind]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for c in (a, b):
                    c.push_streams(allst, feed, sr_in=8000, fmt="ulaw")
                    c.tick_ready(64)
                    c.poll()
                if kind == "move":
                    blob = a.export_streams(src)
                    b.import_streams(dstl, blob)
                    a.reset_streams(src)
                a.synchronize()
                b.synchronize()
                times[kind].append(time.perf_counter() - t0)
    finally:
        for a, b in pairs.values():
            a.close()
            b.close()
    res = {k: {"median_step_ms": float(np.median(v[2:])) * 1e3, "steps": len(v) - 2} for k, v in times.items()}
    res["streams_moved_per_step"] = n_move
    res["move_cost_ms"] = res["move"]["median_step_ms"] - res["still"]["median_step_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r08_stream_migrate.json"))
    ap.add_argument("--steps", type=int, default=12)
    args = ap.parse_args()
    word = load_word()
    res = {"gpu": gpu_info(), "geometry": {"ring_samples": RING, "slack_samples": SLACK, "pcm": "int16", "slots": SLOTS}}
    res["copy_rates_bytes_per_s"] = copy_rates()
    print(json.dumps(res), flush=True)
    res["k10_device_blob"] = leg_kernels(word, [1, 64, 512, 4096], res["copy_rates_bytes_per_s"])
    res["pinned_host_blob"] = leg_host(word, [1, 64, 512, 4096], res["copy_rates_bytes_per_s"])
    res["rebalance_8k_ulaw"] = leg_rebalance(word, args.steps)
    print(json.dumps({"rebalance_8k_ulaw": res["rebalance_8k_ulaw"]}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
