"""bench.py — audio-seconds per wall-second of the level-1/level-2 hot path at 4096 streams per B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--only sweep|config3] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A "step" pushes 1.0 s of new 16 kHz int16 audio into each of the 4096 device rings of a rank and runs
the 10 ticks it covers: K1 ring_push, K2 tick_gate (adaptive silence threshold, is_silent, timing state machine),
K3 segment_queue (fused MFCC + template match on every candidate the state machine cut).  That is the reference's
WakeWord loop (wakeword.py:454-517, 1036-1157) for 4096 rooms.  Streams shard across ranks (4096 per GPU, weak
scaling); the only exchange is the delivery of the 8-byte per-stream result records to every rank: a put-with-signal
by a sender kernel behind K3 over NVLink (--gather peer, the default when symmetric memory is available) or one NCCL
all-gather per step (--gather nccl).

Printed JSON (one line, rank 0).  W warm-up steps, then --repeats (5) blocks of exactly K steps, each bracketed by
barrier + synchronize and timed with CUDA events on the launching stream (max over ranks): the MEDIAN block is reported
and every block is listed.  `value` = whole-job audio-s/s with inputs resident in HBM; `e2e` = the same through the
public API with host (pinned) PCM, H2D copies and the event read-back inside the timed region; `roofline` for the
dominant kernel from CUDA-event timings taken inside this run; `cpu_baseline` = the reference's own classes (staged
under oracle/_ref by oracle/stage_ref.py; the oracle port when absent) on this box's cores, one single-threaded
process per core (N=1 only), with a best-effort C + OpenMP statement of the same semantics beside it
(`best_effort_c`, `e2e_vs_best_effort_c`); `e2e_g711` = the end-to-end step fed with G.711 codes; secondary legs:
`dense` (per-hop scoring, K4, 100 hops per step), `sweep` (BASELINE configs[4]: 1024 streams x 600 s, T = 4 and
T = 1 templates, 10 s chunks) and `config3` (BASELINE configs[3]: 8192 streams per GPU, NCCL gather).
`--impl reference` times the reference's CPU implementation on all host cores on a bounded sample of the same
workload (same `config`).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

N_STREAMS = 4096
RING_SECONDS = 10
STEP_SECONDS = 1.0
STEP_SAMPLES = 16000
TICKS_PER_STEP = 10
POOL_SECONDS = 12      # period of the synthetic feed per stream; deliberately NOT the ring length: with a 10 s feed in a 10 s
                       # ring every new 0.1 s chunk equals the chunk it replaces, the gate's order-statistic update and
                       # threshold recomputation degenerate to no-ops and K2 looks 10 us cheaper than on real audio
SEED0 = 1000
PARAMS = dict(frame_size=1600, similarity_threshold=75.0, pre_speech_silence=0.8, speech_duration_min=0.69,
              speech_duration_max=1.38, post_speech_silence=0.4, timeout=30.0)
METRIC = "audio-sec/sec MFCC+cosine-match @4096 streams, 1/2/4/8 B200; % HBM peak"
UNIT = "audio-s/s"


def load_word():
    p = os.path.join(REPO, "tests", "golden", "reference_word.npz")
    if os.path.exists(p):
        return np.load(p)["pcm_i16"].astype(np.float32) / np.float32(32768.0), "bundled reference_word.wav"
    from easywakeword_b200 import synth
    return synth.synthetic_word(), "synthetic word"


def make_pool(stream0, n_streams, word, out, as_f32=False):
    """out[POOL_SECONDS, n_streams, 16000] int16 <- synthetic streams (seed = SEED0 + global stream id), laid out
    so that one step (1.0 s of every stream) is one contiguous block, the layout a caller pushing [streams, n]
    arrays has."""
    from concurrent.futures import ThreadPoolExecutor
    from easywakeword_b200 import synth

    def one(s):
        x, _ = synth.stream(SEED0 + stream0 + s, POOL_SECONDS, word, noise_sigma=0.002, gain=(1.0, 4.0))
        q = synth.to_int16(x)                                       # the same 16-bit sample values in either format
        out[:, s, :] = (synth.from_int16(q) if as_f32 else q).reshape(POOL_SECONDS, STEP_SAMPLES)

    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 8)) as ex:
        list(ex.map(one, range(n_streams)))


class ClockSampler:
    """nvidia-smi in loop mode (100 ms) for the whole measured part of the run (B200_PROFILING.md clocks line)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw"

    def __init__(self, index):
        self.rows, self.proc, self.thread = [], None, None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def start(self):
        if self.thread:
            self.thread.start()

    def finish(self):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()
        def num(x):
            try:
                return float(x)
            except Exception:
                return None
        sm = [num(r[0]) for r in self.rows if r and num(r[0]) is not None]
        mx = [num(r[1]) for r in self.rows if len(r) > 1 and num(r[1]) is not None]
        pw = [num(r[6]) for r in self.rows if len(r) > 6 and num(r[6]) is not None]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].startswith("Active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference's own classes (oracle/_ref staged by oracle/stage_ref.py, driven by oracle/ref_harness.py under
# the fake clock) when present, else the oracle port — one stream per process on every host core
THREAD_ENV = ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS")


def cpu_kind():
    """'reference' when the reference's unmodified module is importable on this box, else 'port'."""
    from oracle import ref_harness
    return "reference" if ref_harness.reference_available() else "port"


def _cpu_check_threads(_):
    """Runs in every worker right after it starts: one BLAS / OpenMP thread per process, or the arm is oversubscribed."""
    bad = {k: os.environ.get(k) for k in THREAD_ENV if os.environ.get(k) != "1"}
    assert not bad, f"worker started without single-thread environment: {bad}"
    try:
        from threadpoolctl import threadpool_info
        import numpy as _np
        _np.ones((64, 64)) @ _np.ones((64, 64))            # make sure the BLAS pool exists before it is inspected
        info = threadpool_info()
        assert all(int(i.get("num_threads", 1)) == 1 for i in info), info
        return len(info)
    except ImportError:
        return -1


def _cpu_worker(args):
    seed, seconds, mode = args
    from easywakeword_b200 import synth
    word, _ = load_word()
    x, _ = synth.stream(seed, RING_SECONDS + seconds + 0.2, word, noise_sigma=0.002, gain=(1.0, 4.0))
    x = synth.from_int16(synth.to_int16(x))
    timing = {}
    p = {k: v for k, v in PARAMS.items() if k != "frame_size"}
    if mode == "reference":
        import contextlib
        from oracle import ref_harness
        with open(os.devnull, "w") as null, contextlib.redirect_stdout(null):   # the reference print()s device warnings
            r = ref_harness.run_reference_stream(x, word, block=PARAMS["frame_size"], timing=timing, keep_audio=False, **p)
    else:
        from oracle import ewk_oracle as O
        r = O.detect_stream(x, word, block=PARAMS["frame_size"], fast=(mode == "port_fast"), timing=timing, **p)
    return timing["t_end"] - timing["t_full"], timing["steady_ticks"] * 0.1, len(r["events"])


class CpuPool:
    """`procs` spawn-context workers that inherit *_NUM_THREADS=1 from the moment they start (numpy and its BLAS pool
    are imported while the worker re-imports this module, before any task runs: setting the variables inside a task is
    too late and left the round-1 arm 2-5x oversubscribed)."""

    def __init__(self, procs):
        import multiprocessing as mp
        self.procs = procs
        saved = {k: os.environ.get(k) for k in THREAD_ENV}
        for k in THREAD_ENV:
            os.environ[k] = "1"
        try:
            self.pool = mp.get_context("spawn").Pool(procs)
            self.blas_pools = self.pool.map(_cpu_check_threads, range(procs), chunksize=1)
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v

    def run(self, seconds_per_stream, mode, seed0=SEED0):
        """Every worker runs the CPU path over one stream (steady state timed, ring fill untimed).
        -> (audio_s, wall_s, events, wall_s of the slowest worker).  wall_s = audio / (sum of the workers' own rates):
        the time the cores would need with perfect load balance.  Streams differ in how many level-2 evaluations they
        hold, so the slowest worker of a round finishes well after the average one; charging that tail to the
        reference would understate what its cores deliver on thousands of independent streams."""
        res = self.pool.map(_cpu_worker, [(seed0 + i, seconds_per_stream, mode) for i in range(self.procs)], chunksize=1)
        audio = sum(a for _, a, _ in res)
        rate = sum(a / w for w, a, _ in res if w > 0)
        return audio, audio / rate, sum(e for _, _, e in res), max(w for w, _, _ in res)

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_throughput(seconds_per_stream, procs, mode, rounds=1, pool=None):
    """audio-s/s of `procs` processes each running the CPU path over one stream per round, all concurrently: the sum of
    the workers' own steady-state rates (CpuPool.run).  Returns (value, audio_s, wall_s, events)."""
    own = pool is None
    pool = pool or CpuPool(procs)
    tot_audio = tot_wall = 0.0
    events = 0
    try:
        for r in range(rounds):
            a, w, e, _ = pool.run(seconds_per_stream, mode, SEED0 + r * procs)
            tot_audio += a
            tot_wall += w
            events += e
    finally:
        if own:
            pool.close()
    return tot_audio / tot_wall, tot_audio, tot_wall, events


def cpu_best_effort_c(pool, word, cores, streams=1024, repeats=3, rounds=3):
    """SURVEY §8(d) CPU baseline (iii): the best-effort C statement of the same gated path (oracle/cpu_port, OpenMP over
    streams, pinned against the numpy oracle in tests/test_cpu_port.py) over `streams` streams of the bench pool,
    each POOL_SECONDS x repeats long.  Returns (audio-s/s, level-2 events, audio seconds)."""
    from easywakeword_b200 import synth
    from oracle import cpu_port
    streams = min(streams, pool.shape[1])
    q = np.ascontiguousarray(np.tile(pool[:, :streams, :].transpose(1, 0, 2).reshape(streams, -1), (1, repeats)))
    p = {k: v for k, v in PARAMS.items() if k != "frame_size"}
    cpu_port.load()
    cpu_port.detect_batch(q[:cores, :32000], synth.to_int16(word), threads=cores, **p)        # warm the threads
    t0 = time.perf_counter()
    for _ in range(rounds):                                         # ~1 GB of PCM per round: far beyond the host caches
        ev = cpu_port.detect_batch(q, synth.to_int16(word), threads=cores, **p)
    dt = time.perf_counter() - t0
    audio = rounds * streams * q.shape[1] / 16000.0
    return audio / dt, rounds * sum(len(e) for e in ev), audio


def cpu_dense_throughput(seconds=3.0):
    """A9 on one host core: the oracle's per-hop `calculate_similarity` (SURVEY §8(d) CPU baseline (ii)) over
    `seconds` of one synthetic stream.  Returns (audio-s/s, windows/s)."""
    from easywakeword_b200 import synth
    from oracle import ewk_oracle as O
    word, _ = load_word()
    x, _ = synth.stream(SEED0, RING_SECONDS + seconds, word, noise_sigma=0.002, gain=(1.0, 4.0))
    x = synth.from_int16(synth.to_int16(x))
    hops = np.arange(RING_SECONDS * 100, RING_SECONDS * 100 + int(seconds * 100))
    t0 = time.perf_counter()
    O.dense_scores(x, [word], hops)
    dt = time.perf_counter() - t0
    return seconds / dt, len(hops) / dt


def bench_config(n, pcm_name, world, word_name):
    """The workload both arms run (the GPU arm whole, the CPU arm on a bounded sample of it): `config` of the line."""
    esz = 4 if pcm_name == "float32" else 2
    return {"workload": ("configs[2]" if n == N_STREAMS else "configs[3] shard size" if n == 8192 else "custom") +
                        f": {n} streams per B200, 10 s {pcm_name} rings, 1.0 s of new audio per stream per step = 10 ticks of "
                        "the gated level-1+2 path (ring write, adaptive silence threshold, is_silent, timing state machine, "
                        "fused MFCC+match on every candidate segment)",
            "streams_per_gpu": n, "ring_seconds": RING_SECONDS, "step_seconds": STEP_SECONDS,
            "template": word_name, "pcm": pcm_name, "params": PARAMS,
            "l2": f"inputs larger than L2: {n * STEP_SAMPLES * esz / 1e6:.0f} MB of new PCM per step, "
                  f"{n * (RING_SECONDS * 16000 + int(2 * STEP_SECONDS * 16000) + 3200) * esz / 1e9:.2f} GB of rings per GPU "
                  "(10 s + 2.2 s slack)",
            "parallelism": f"streams sharded {n}/GPU x {world}" if world > 1 else "1 GPU"}


def run_reference(args):
    """The reference's CPU implementation of the path on every host core, on a bounded sample of the GPU arm's workload:
    per step every core runs the reference over `sample_s` seconds of one of the workload's streams (the streams are
    independent, so the 4096-stream step is this per-stream work repeated).  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    K, W = max(1, args.steps), args.warmup
    kind = cpu_kind()
    mode = "reference" if kind == "reference" else "port"
    sample_s = 64.0
    word, word_name = load_word()
    pool = CpuPool(cores)
    t0 = time.perf_counter()
    for _ in range(W):
        pool.run(1.0, mode)
    audio = wall = wall_slowest = 0.0
    ev = 0
    step_ms = []
    for k in range(K):
        a, w, e, ws = pool.run(sample_s, mode, SEED0 + k * cores)
        audio += a
        wall += w
        wall_slowest += ws
        ev += e
        step_ms.append(1e3 * w)
    pool.close()
    total_wall = time.perf_counter() - t0
    val = audio / wall
    what = ("the reference's own SoundBuffer / WordMatcher / WakeWord._detect_word (easywakeword/wakeword.py unmodified, "
            "staged by oracle/stage_ref.py, on the restated-librosa shim; fake clock of oracle/ref_harness.py)"
            if kind == "reference" else
            "oracle port in the reference's statement order (the reference module is not staged on this box)")
    pcm_name = "float32" if args.pcm == "f32" else "int16"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": 1e3 * wall / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.streams, pcm_name, max(1, args.gpus), word_name),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{cores} processes (one BLAS/OpenMP thread each, checked in every worker) x {sample_s} s "
                                   f"steady state of one workload stream each per step x {K} steps = {audio:.0f} audio-s; {what}",
                         "per_core": val / cores,
                         "timing": "value = sum over the workers of (audio / own steady-state wall time), i.e. perfect load "
                                   "balance over the cores; value_slowest_worker charges every step its slowest worker",
                         "value_slowest_worker": audio / wall_slowest},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": total_wall, "level2_events": ev,
        "ms_per_step_minmax": [min(step_ms), max(step_ms)],
    }
    # context, not the arm's value: what a tuned C + OpenMP statement of the same semantics reaches on these cores
    try:
        pool_pcm = np.empty((POOL_SECONDS, 256, STEP_SAMPLES), np.int16)
        make_pool(0, 256, word, pool_pcm)
        vc, evc, audio_c = cpu_best_effort_c(pool_pcm, word, cores, streams=256, repeats=3, rounds=4)
        line["best_effort_c"] = {"value": vc, "unit": UNIT, "cores": cores, "kind": "port (C, OpenMP over streams)",
                                 "sample": f"4 x 256 streams x {3 * POOL_SECONDS} s = {audio_c:.0f} audio-s, {evc} level-2 evaluations"}
    except Exception as e:
        line["best_effort_c"] = {"unavailable": f"{type(e).__name__}: {e}"[:160]}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# secondary legs of the GPU arm: BASELINE configs[4] (offline multi-template sweep) and configs[3] (65 536 / 8 streams per GPU)
SWEEP_STREAMS = 1024
SWEEP_CHUNK_SECONDS = 10
SWEEP_SECONDS = 600            # per stream, measured; the config's 3600 s are 6 x the same chunks (stated in the leg)


def sweep_templates(word):
    """SURVEY §8(d) config 5: the bundled word (1-word), a 2-word phrase built as word + 0.15 s gap + time-reversed word,
    and two pitch-shifted sines under a speech-like envelope."""
    phrase = np.concatenate([word, np.zeros(2400, np.float32), word[::-1]]).astype(np.float32)
    out = [word, phrase]
    for f, dur in ((440.0, 1.0), (440.0 * 2 ** (5 / 12), 0.6)):
        t = np.arange(int(dur * 16000)) / 16000.0
        out.append((0.3 * np.sin(2 * np.pi * f * t) * np.sin(np.pi * t / dur) ** 0.5).astype(np.float32))
    return out, ["bundled word (0.97 s)", "word + 0.15 s + reversed word (2.09 s)", "440 Hz tone (1.0 s)", "587 Hz tone (0.6 s)"]


def sweep_leg(torch, dist, dev, stream, local_rank, rank, world, word, hbm_peak, seconds=SWEEP_SECONDS):
    """configs[4]: 1024 streams per GPU, every hop scored against T = 4 templates (and T = 1), streamed in 10 s chunks:
    one ewk_push of the chunk (K1) + one ewk_dense_scores over its 1000 hops (K4; the window history of a chunk's first
    hops is the previous chunk's audio still in the ring: the (L_k + 352)-sample halo of SURVEY §8(d))."""
    from easywakeword_b200 import _lib, synth
    from easywakeword_b200.bank import WakeWordBank
    n, chunk = SWEEP_STREAMS, SWEEP_CHUNK_SECONDS * 16000
    tpls, names = sweep_templates(word)
    T = len(tpls)
    n_pool = 3                                                      # distinct 10 s chunks per stream, cycled
    pin = _lib.PinnedArray((n_pool, n, chunk), np.int16)
    from concurrent.futures import ThreadPoolExecutor

    def one(s_):
        x, _ = synth.stream(SEED0 + 100000 + rank * n + s_, n_pool * SWEEP_CHUNK_SECONDS, word, noise_sigma=0.002, gain=(1.0, 4.0))
        pin.array[:, s_, :] = synth.to_int16(x).reshape(n_pool, chunk)

    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 8)) as ex:
        list(ex.map(one, range(n)))
    host = torch.from_numpy(pin.array)
    pool = host.to(dev)
    bank = WakeWordBank(n, tpls, device=local_rank, buffer_seconds=SWEEP_CHUNK_SECONDS, pcm_dtype=np.int16, max_push_seconds=3.0,
                        cuda_stream=stream.cuda_stream, **PARAMS)
    ctx = bank.ctx
    ctx.set_stream_params(-1, live=1, **PARAMS)                     # no ticks in this mode: pushes run free of the gate's guard
    hops = chunk // 160
    out_dev = torch.empty(n * hops * T, dtype=torch.float32, device=dev)
    out_pin = _lib.PinnedArray((n, hops, T), np.float32)
    pushed = [0]

    scored = [0]

    def push_chunk(where):
        j = pushed[0] % n_pool
        src = pool if where == _lib.DEVICE else host
        bank.push((src.data_ptr() + j * n * chunk * 2, n, chunk, chunk), where=where)
        pushed[0] += 1

    def chunk_step(where, t_first, t_count, to_host):
        """push + score one chunk.  With host PCM the NEXT chunk's push is issued before this chunk is scored, so that its
        H2D copy runs beside K4 (every chunk still pays its own copy and its own read-back inside the timed region)."""
        if pushed[0] == scored[0]:
            push_chunk(where)
        hop0 = scored[0] * hops + 1
        scored[0] += 1
        if to_host:
            push_chunk(where)
            ctx._ck(ctx.lib.ewk_dense_scores(ctx.h, hop0, hops, t_first, t_count, out_pin.ptr, _lib.HOST))
        else:
            ctx.dense_scores(hop0, hops, t_first, t_count, out_device_ptr=out_dev.data_ptr())

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def run(where, t_count, to_host, chunks):
        for _ in range(2):
            chunk_step(where, 0, t_count, to_host)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(chunks):
            chunk_step(where, 0, t_count, to_host)
        e1.record(stream)
        sync_all()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    chunks = max(2, seconds // SWEEP_CHUNK_SECONDS)
    audio = n * SWEEP_CHUNK_SECONDS * chunks * world
    ms4 = run(_lib.DEVICE, T, False, chunks)
    ms1 = run(_lib.DEVICE, 1, False, chunks)
    ms4_e2e = run(_lib.HOST, T, True, max(2, chunks // 3))
    audio_e2e = n * SWEEP_CHUNK_SECONDS * max(2, chunks // 3) * world
    ctx.profile(True)
    for _ in range(3):
        chunk_step(_lib.DEVICE, 0, T, False)
    prof4 = ctx.profile_read()
    for _ in range(3):
        chunk_step(_lib.DEVICE, 0, 1, False)
    prof1 = ctx.profile_read()
    ctx.profile(False)
    k4_ms = prof4["dense_score"]["ms"] / max(1, prof4["dense_score"]["launches"])
    k1_ms = prof1["dense_score"]["ms"] / max(1, prof1["dense_score"]["launches"])
    pcm_bytes = n * chunk * 2
    leg = {
        "what": f"configs[4]: {n} streams per GPU, {seconds} s of audio per stream measured in {SWEEP_CHUNK_SECONDS} s chunks "
                f"(the config's 3600 s per stream are {3600 // seconds} x the same chunk loop: throughput is per chunk), every 10 ms hop "
                f"scored against T = {T} templates; per chunk one ewk_push (K1) + one ewk_dense_scores over {hops} hops (K4), "
                "scores left on the device",
        "templates": names, "streams_per_gpu": n, "seconds_per_stream": chunks * SWEEP_CHUNK_SECONDS, "chunk_seconds": SWEEP_CHUNK_SECONDS,
        "value": audio / (ms4 * 1e-3), "unit": UNIT, "ms_per_chunk": ms4 / chunks,
        "windows_per_s": n * hops * T * chunks * world / (ms4 * 1e-3),
        "t1": {"value": audio / (ms1 * 1e-3), "unit": UNIT, "ms_per_chunk": ms1 / chunks, "kernel_ms": k1_ms,
               "windows_per_s": n * hops * chunks * world / (ms1 * 1e-3)},
        "kernel_ms": k4_ms,
        "e2e": {"value": audio_e2e / (ms4_e2e * 1e-3), "unit": UNIT, "ms_per_chunk": ms4_e2e / max(2, chunks // 3),
                "h2d_bytes_per_chunk": pcm_bytes, "d2h_bytes_per_chunk": n * hops * T * 4,
                "what": "pinned host PCM -> H2D -> K1 -> K4 -> scores copied back into pinned host memory, every chunk"},
        "algorithmic_bytes_per_chunk": pcm_bytes + n * hops * T * 4,
        "hbm_frac": (pcm_bytes + n * hops * T * 4) / (k4_ms * 1e-3) / 1e9 / hbm_peak,
        "traffic": _traffic().get("dense_score_sweep_t4") if T == 4 else None,
        "geometry": "K4 chooses hops per sub-chunk / threads per CTA / CTAs per SM from shared memory (csrc/ewk_api.cu dense_plan)",
    }
    bank.close()
    pin.free()
    out_pin.free()
    return leg


def _traffic():
    """dram read+write bytes per launch from the committed `ncu --set full` captures (profiles/traffic.json)."""
    tp = os.path.join(REPO, "profiles", "traffic.json")
    return json.load(open(tp)) if os.path.exists(tp) else {}


def config3_leg(torch, dist, dev, stream, local_rank, rank, world, word, pool_dev, K, W, overlap):
    """configs[3]: 65 536 streams over 8 GPUs = 8192 streams per GPU (the same per-GPU shard at every N: weak scaling), the
    gated level-1+2 path, 8-byte result records gathered over NVLink with one NCCL all-gather per step."""
    from easywakeword_b200 import _lib
    from easywakeword_b200.bank import WakeWordBank
    n = 8192
    n0 = pool_dev.shape[1]
    reps = -(-n // n0)
    # streams beyond the pool are the pool's streams shifted by 3, 6, ... seconds (cheap stand-in for more seeds)
    big = torch.cat([pool_dev.roll(3 * r, dims=0) for r in range(reps)], dim=1)[:, :n, :].contiguous()
    bank = WakeWordBank(n, [word], device=local_rank, buffer_seconds=RING_SECONDS, pcm_dtype=np.int16,
                        max_push_seconds=2 * STEP_SECONDS, cuda_stream=stream.cuda_stream, max_events=1 << 18, **PARAMS)
    ctx = bank.ctx
    results = torch.zeros(n, 2, dtype=torch.int32, device=dev)
    ctx.set_results_buffer(results.data_ptr())
    ctx.set_overlap(overlap)
    gathered = torch.zeros(world * n, 2, dtype=torch.int32, device=dev) if world > 1 else None
    pushed = [0]
    stepped = [0]

    def push():
        j = pushed[0] % POOL_SECONDS
        pushed[0] += 1
        bank.push((big.data_ptr() + j * n * STEP_SAMPLES * 2, n, STEP_SAMPLES, STEP_SAMPLES), where=_lib.DEVICE)

    def step():
        if pushed[0] == stepped[0]:
            push()
        stepped[0] += 1
        bank.tick(TICKS_PER_STEP)
        if gathered is not None:
            if overlap:
                push()                                              # the next step's K1 beside this step's K3, ahead of the gather
            ctx.join()
            dist.all_gather_into_tensor(gathered, results)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    n_ev = 0
    for _ in range(RING_SECONDS + W):
        step()
        n_ev = len(bank.poll())
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(K):
        step()
    ctx.join()
    e1.record(stream)
    sync_all()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ev = bank.poll()
    KP = 2 * POOL_SECONDS                                           # whole periods of the feed, as in the main leg's profile pass
    ctx.set_overlap(False)
    ctx.profile(True)
    for _ in range(KP):
        step()
    prof = ctx.profile_read()
    ctx.profile(False)
    evp = bank.poll()
    evp = evp[evp["kind"] == _lib.EV_SCORED]
    leg = {"what": f"configs[3]: {n} streams per GPU x {world} GPU(s) = {n * world} streams (65 536 at 8 GPUs), gated level-1+2 path, "
                   "PCM resident in HBM, one NCCL all-gather of the 8-byte result records per step" + ("" if world > 1 else " (N > 1 only)"),
           "streams_per_gpu": n, "streams_total": n * world, "value": n * STEP_SECONDS * world * K / (ms * 1e-3), "unit": UNIT,
           "ms_per_step": ms / K, "level2_events_per_step": int((ev["kind"] == 2).sum()) / K,
           "kernel_ms_per_step": {k: v["ms"] / KP for k, v in prof.items() if v["launches"]},
           "profile_pass": {"steps": KP, "candidates_per_step": len(evp) / KP,
                            "candidate_frames_per_step": float((1 + evp["seg_len"] // 160).sum()) / KP},
           "rings_gb_per_gpu": n * (RING_SECONDS * 16000 + int(2 * STEP_SECONDS * 16000) + 3200) * 2 / 1e9}
    bank.close()
    del big
    return leg


def dump_outputs(out_dir, results, events, last_tick):
    """--dump-outputs: what the device-resident timed path computed in its last step, one DIR/<name>.npy per array:
    every stream's result record (`stream_score`, `stream_flags`: the caller's ewk_stream_result buffer) and each field
    of the events the step's ticks produced (`event_<field>`, in ewk_poll's order).  float32 values stay float32,
    integers become float64 (exact).  A score is NaN where none exists (a stream before its first level-2 evaluation,
    a timeout event): it is written as 0 with `<name>_valid` = 0 beside it, so that every value written is finite."""
    from easywakeword_b200 import _lib
    os.makedirs(out_dir, exist_ok=True)
    rec = results.cpu().numpy()
    origin = events["tick"] + (events["kind"] == _lib.EV_TIMEOUT)      # a timeout event carries the tick before the one that raised it
    ev = events[origin > last_tick - TICKS_PER_STEP]
    arrays = {"stream_score": rec[:, 0].copy().view(np.float32),
              "stream_flags": rec[:, 1].copy().view(np.uint32).astype(np.float64)}
    for f in _lib.EVENT_DTYPE.names:
        arrays[f"event_{f}"] = ev[f] if ev[f].dtype == np.float32 else ev[f].astype(np.float64)
    for name in ("stream_score", "event_score"):
        valid = np.isfinite(arrays[name])
        arrays[name] = np.where(valid, arrays[name], np.float32(0))
        arrays[f"{name}_valid"] = valid.astype(np.float32)
    for name, a in arrays.items():
        assert np.isfinite(a).all(), name
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ----------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from easywakeword_b200 import _lib
    from easywakeword_b200.bank import WakeWordBank

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # pinned staging memory is first-touched below: keep this rank on the CPUs next to its GPU (NUMA / PCIe root)
    from easywakeword_b200.dist import bind_host_near_gpu
    host_cpus = bind_host_near_gpu(local_rank) if world > 1 and not args.no_bind else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, max(3, args.warmup)
    word, word_name = load_word()

    n = args.streams
    f32 = args.pcm == "f32"                                         # the reference's native PortAudio dtype (wakeword.py:438-444)
    esz = 4 if f32 else 2
    pcm_name = "float32" if f32 else "int16"
    pool_pin = _lib.PinnedArray((POOL_SECONDS, n, STEP_SAMPLES), np.float32 if f32 else np.int16)
    make_pool(rank * n, n, word, pool_pin.array, as_f32=f32)
    pool_host = torch.from_numpy(pool_pin.array)
    pool_dev = pool_host.to(dev, non_blocking=False)

    # a real (non-legacy) stream: libewk launches on it and torch.cuda.Event times it
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    bank = WakeWordBank(n, [word], device=local_rank, buffer_seconds=RING_SECONDS, pcm_dtype=np.float32 if f32 else np.int16,
                        max_push_seconds=2 * STEP_SECONDS, cuda_stream=stream.cuda_stream, max_events=1 << 17, **PARAMS)
    ctx = bank.ctx
    results = torch.zeros(n, 2, dtype=torch.int32, device=dev)          # ewk_stream_result[n]: NCCL send buffer
    ctx.set_results_buffer(results.data_ptr())
    overlap = not args.no_overlap
    ctx.set_overlap(overlap)
    gathered = torch.zeros(world * n, 2, dtype=torch.int32, device=dev) if world > 1 and args.gather != "none" else None
    # multi-GPU result exchange: the producing kernels store every record into all ranks' copies over NVLink
    # (peer-mapped symmetric memory) and a step ends with a barrier behind K3; NCCL all-gather otherwise
    exchange, exchange_note = None, None
    if world > 1 and args.gather not in ("nccl", "none"):
        try:
            from easywakeword_b200.dist import PeerResultExchange
            exchange = PeerResultExchange(world * n, world, rank, dev)
        except Exception as e:                                      # no symmetric memory on this box
            exchange_note = f"{type(e).__name__}: {e}"[:200]
        ok = torch.tensor([1 if exchange is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            exchange = None
            if args.gather.startswith("peer"):
                raise SystemExit(f"bench.py: --gather peer requested but symmetric memory is unavailable: {exchange_note}")
        else:
            exchange.install(ctx)

    def slice_ptr(t, j):
        return (t.data_ptr() + j * n * STEP_SAMPLES * esz, n, STEP_SAMPLES, STEP_SAMPLES)

    step_no = [0]
    pushed = [0]

    def push_next(where):
        j = pushed[0] % POOL_SECONDS
        pushed[0] += 1
        bank.push(slice_ptr(pool_dev if where == _lib.DEVICE else pool_host, j), where=where)

    def step(where, read_back):
        """One step = push of 1.0 s for every stream + its 10 ticks (+ gather, + event read-back).
        The push of the NEXT step is issued before this step's ticks so that, for host PCM, its H2D copy
        (copy stream, double-buffered staging) overlaps this step's kernels; every step still pays its own copy."""
        if pushed[0] == step_no[0]:
            push_next(where)
        step_no[0] += 1
        if read_back and where == _lib.HOST:
            push_next(where)
        bank.tick(TICKS_PER_STEP)
        if gathered is not None:
            if overlap and where == _lib.DEVICE and pushed[0] == step_no[0]:
                push_next(where)                                    # next step's K1 goes beside this step's K3, ahead of the gather
            if exchange is not None:
                if args.gather == "peer-barrier":
                    exchange.barrier(ctx)                           # lock step: a barrier behind K3 on its stream
                # default: nothing to do — K2/K3 stored the records into every rank's copy and K3 releases the step's
                # sequence number into every rank's signal row when it is done
            else:
                ctx.join()                                          # the gather reads the records K3 writes
                dist.all_gather_into_tensor(gathered, results)
        return bank.poll() if read_back else None

    # fill the rings (10 s) so that every stream is past is_buffer_full and thresholds are adaptive
    for _ in range(RING_SECONDS):
        step(_lib.DEVICE, True)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    by_rank = []                                                    # per timed() call: every rank's own device time and enqueue time

    def timed(where, read_back, steps, repeats):
        """W warm-up steps, then `repeats` blocks of exactly `steps` steps, each bracketed by barrier + synchronize and
        timed with CUDA events on the launching stream (max over ranks).  Returns the MEDIAN block's ms plus every
        block's ms, the launches of one block and the level-2 events of the median block."""
        for _ in range(W):
            step(where, True)
        blocks = []
        for _ in range(repeats):
            if not read_back:
                bank.poll()         # untimed: the event queue holds one block's events, none of them dropped for lack of room
            gc.collect()
            gc.disable()            # a collection inside a 3 ms block stalls the enqueueing thread for longer than the queue is deep
            barrier()
            l0 = ctx.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_ev = 0
            e0.record(stream)
            c0 = time.perf_counter()
            for _ in range(steps):
                ev = step(where, read_back)
                if ev is not None:
                    n_ev += int((ev["kind"] == 2).sum())
            cpu_issue_ms = (time.perf_counter() - c0) * 1e3         # host time to enqueue the steps (not a result: a diagnostic)
            ctx.join()                                              # the last step's K3 belongs to the timed region
            if exchange is not None:
                if args.gather == "peer-barrier":
                    exchange.finish(stream)                         # ... and so does its barrier
                else:
                    exchange.wait(ctx)                              # ... and so does the arrival of every rank's last step
            e1.record(stream)
            barrier()
            gc.enable()
            ms = e0.elapsed_time(e1)
            br = {"ms_per_step": [ms / steps], "host_enqueue_ms_per_step": [cpu_issue_ms / steps]}
            if world > 1:
                allr = torch.zeros(world, 2, device=dev)
                dist.all_gather_into_tensor(allr, torch.tensor([[ms / steps, cpu_issue_ms / steps]], device=dev))
                br = {"ms_per_step": [round(float(v), 5) for v in allr[:, 0]],
                      "host_enqueue_ms_per_step": [round(float(v), 5) for v in allr[:, 1]]}
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            blocks.append((ms, ctx.launch_count() - l0, n_ev, br))
        order = sorted(range(repeats), key=lambda i: blocks[i][0])
        med = blocks[order[repeats // 2]]
        by_rank.append(med[3])
        return med[0], med[1], med[2], [b[0] for b in blocks]

    audio_per_step_all = n * STEP_SECONDS * world
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    R = max(1, args.repeats)
    ms_dev, launches, _, dev_blocks = timed(_lib.DEVICE, False, K, R)      # inputs resident in HBM
    ev_dev = bank.poll()
    if args.dump_outputs and rank == 0:
        if ctx.dropped:
            raise SystemExit(f"bench.py: the event queue dropped {ctx.dropped} events in the last timed block, so its "
                             "last step is incomplete and is not dumped; use fewer --steps")
        dump_outputs(args.dump_outputs, results, ev_dev, ctx.status(0).tick)
    ms_e2e, _, n_events, e2e_blocks = timed(_lib.HOST, True, K, R)         # host PCM -> rings -> events on host

    # the same end-to-end step fed with G.711 mu-law codes (ewk_push_g711: 1 byte per sample over PCIe, expanded on the
    # device).  A secondary figure: the audio is the pool after companding, so its events differ from the PCM16 run.
    g711 = None
    if not f32 and not args.no_g711:
        try:
            from easywakeword_b200.resample import ULAW_TABLE
            tab = torch.tensor(ULAW_TABLE.astype(np.int32), device=dev)
            srt, order = torch.sort(tab)
            codes_pin = _lib.PinnedArray((POOL_SECONDS, n, STEP_SAMPLES), np.uint8)
            codes_host = torch.from_numpy(codes_pin.array)
            for j in range(POOL_SECONDS):                           # nearest code of every pool sample, one pool second at a time
                x = pool_dev[j].to(torch.int32)
                i = torch.bucketize(x, srt).clamp_(1, 255)
                pick = torch.where((srt[i] - x).abs() < (srt[i - 1] - x).abs(), i, i - 1)
                codes_host[j].copy_(order[pick].to(torch.uint8))
                del x, i, pick
            torch.cuda.synchronize(dev)
            while pushed[0] > step_no[0]:                           # consume the PCM push the e2e loop issued ahead
                bank.tick(TICKS_PER_STEP)
                step_no[0] += 1
                bank.poll()
            gp = [0]

            def g_push():
                ptr = codes_host.data_ptr() + (gp[0] % POOL_SECONDS) * n * STEP_SAMPLES
                gp[0] += 1
                bank.push_g711((ptr, n, STEP_SAMPLES, STEP_SAMPLES), law="ulaw", where=_lib.HOST)

            def g_step():
                g_push()                                            # the NEXT step's codes: copy + expansion beside this step's kernels
                bank.tick(TICKS_PER_STEP)
                if gathered is not None and exchange is None:       # (peer publication needs no call: the tick sends the records)
                    ctx.join()
                    dist.all_gather_into_tensor(gathered, results)
                return bank.poll()

            g_push()
            for _ in range(W):
                g_step()
            barrier()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record(stream)
            for _ in range(K):
                g_step()
            ctx.join()
            q1.record(stream)
            barrier()
            ms_g = q0.elapsed_time(q1)
            if world > 1:
                t = torch.tensor([ms_g], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms_g = float(t.item())
            bank.tick(TICKS_PER_STEP)                               # the push issued ahead by the last step
            bank.poll()
            g711 = {"value": audio_per_step_all * K / (ms_g * 1e-3), "unit": UNIT, "ms_per_step": ms_g / K,
                    "h2d_bytes_per_step": n * STEP_SAMPLES, "h2d_gbs_per_gpu": n * STEP_SAMPLES / (ms_g / K * 1e-3) / 1e9,
                    "what": "e2e with the host feed as G.711 mu-law codes (pool after companding), K0 expansion on the copy stream"}
        except Exception as e:
            g711 = {"unavailable": f"{type(e).__name__}: {e}"[:200]}

    # the exchange on its own (SURVEY §8(d) config 4: "report gather latency separately"), and a self-check that the
    # peer-published copy equals an NCCL all-gather of the local records
    gather_info = {"mode": "none (--gather none: a diagnostic, the ranks exchange nothing)"} if world > 1 and gathered is None else None
    if world > 1 and gathered is not None:
        def per_call_us(fn, reps=50):
            for _ in range(5):
                fn()
            barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(stream)
            for _ in range(reps):
                fn()
            g1.record(stream)
            barrier()
            t = torch.tensor([g0.elapsed_time(g1) * 1e3 / reps], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        ctx.join()
        nccl_us = per_call_us(lambda: dist.all_gather_into_tensor(gathered, results))
        gather_info = {"mode": "nccl all_gather per step", "bytes_per_rank": n * 8, "nccl_all_gather_us": nccl_us,
                       "note": exchange_note}
        if exchange is not None:
            peer_us = per_call_us(lambda: exchange.hdl.barrier())
            step(_lib.DEVICE, False)
            ctx.join()
            exchange.finish(stream)
            exchange.wait(ctx)
            seqs, timed_out = exchange.published(ctx)
            if timed_out or not (seqs == ctx.publish_seq()).all():
                raise SystemExit(f"bench.py: peer signals incomplete: {seqs.tolist()} vs {ctx.publish_seq()} (timed out: {timed_out})")
            barrier()
            dist.all_gather_into_tensor(gathered, results)
            torch.cuda.synchronize(dev)
            same = bool(torch.equal(exchange.view(ctx.publish_parity()), gathered))
            flag = torch.tensor([1 if same else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) != 1:
                raise SystemExit("bench.py: peer-published records differ from the NCCL all-gather of the same step")
            gather_info.update({"mode": ("peer stores by K2/K3 over NVLink (symmetric memory) + one barrier per step behind K3"
                                         if args.gather == "peer-barrier" else
                                         "put-with-signal: K2/K3 write the call's local copy of the records, a sender kernel on a "
                                         "side stream behind K3 stores it into every rank's copy over NVLink (symmetric memory) and "
                                         "releases the step's sequence number; no collective, no per-step barrier, nothing of it on "
                                         "the next step's critical path; the timed region ends with a device-side wait for every "
                                         "rank's last step"),
                                "symm_barrier_us": peer_us, "peer_copy_equals_nccl_all_gather": True})

    # per-kernel device time (CUDA events on the launching stream), same workload, separate loop; sequential order
    # (no overlap) so that every kernel is timed alone
    # The pass covers whole periods of the feed (2 x POOL_SECONDS steps), so that it sees the feed's average step and
    # two passes see the same steps; the candidates it scored are read back afterwards: K3's algorithmic bytes and
    # frames are THEIR samples and frames, not an assumed mean.
    KP = 2 * POOL_SECONDS
    ctx.set_overlap(False)
    bank.poll()
    ctx.profile(True)
    for _ in range(KP):
        step(_lib.DEVICE, False)
    prof = ctx.profile_read()
    ctx.profile(False)
    ev_prof = bank.poll()
    ev_prof = ev_prof[ev_prof["kind"] == _lib.EV_SCORED]
    prof_cand = len(ev_prof) / KP                                   # candidates per K3 launch
    prof_samples = float(ev_prof["seg_len"].sum()) / KP             # their PCM samples per launch
    prof_frames = float((1 + ev_prof["seg_len"] // 160).sum()) / KP  # and frames (1 + len // hop each)
    prof_nopub = None
    if exchange is not None:
        # what the peer stores cost the kernels: the same loop (the same steps of the feed) with publication off
        ctx.set_results_peers([])
        ctx.profile(True)
        for _ in range(KP):
            step(_lib.DEVICE, False)
        prof_nopub = ctx.profile_read()
        ctx.profile(False)
        bank.poll()

    # dense mode (A9): per-hop scoring of every stream, same push, K4 instead of K2/K3
    dense_out = torch.empty(n * 100, dtype=torch.float32, device=dev)
    def dense_step():
        push_next(_lib.DEVICE)
        step_no[0] = pushed[0]
        hop_end = bank.samples_pushed // 160
        ctx.dense_scores(hop_end - 100, 100, 0, 1, out_device_ptr=dense_out.data_ptr())
    # no ticks in this arm: let pushes run free of the gate's "un-gated audio" guard
    ctx.set_stream_params(-1, live=1, **PARAMS)
    dense_steps = max(2, K // 2)
    for _ in range(2):
        dense_step()
    barrier()
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record(stream)
    for _ in range(dense_steps):
        dense_step()
    d1.record(stream)
    barrier()
    ms_dense = d0.elapsed_time(d1)
    if world > 1:
        t = torch.tensor([ms_dense], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_dense = float(t.item())
    ctx.profile(True)
    for _ in range(2):
        dense_step()
    prof_dense = ctx.profile_read()
    ctx.profile(False)

    pk = os.path.join(REPO, "MEASURED_PEAKS.json")
    peaks = json.load(open(pk)) if os.path.exists(pk) else {}
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    sweep = config3 = None
    if not args.no_extra and not f32:
        torch.cuda.synchronize(dev)
        try:
            sweep = sweep_leg(torch, dist, dev, stream, local_rank, rank, world, word, hbm_peak)
        except Exception as e:                                      # a secondary leg never takes the headline down with it
            sweep = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
        if n != 8192:
            try:
                config3 = config3_leg(torch, dist, dev, stream, local_rank, rank, world, word, pool_dev, K, W, overlap)
            except Exception as e:
                config3 = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    clocks = sampler.finish() if sampler else None
    audio_per_step = n * STEP_SECONDS * world
    value = audio_per_step * K / (ms_dev * 1e-3)
    e2e_val = audio_per_step * K / (ms_e2e * 1e-3)

    if rank == 0:
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
        kern = {k: v for k, v in prof.items() if v["launches"]}
        tot_ms = sum(v["ms"] for v in kern.values()) or 1.0
        dom = max(kern, key=lambda k: kern[k]["ms"])
        ev_per_step = n_events / max(1, K)                          # rank 0's own events (its 4096 streams)
        # ALGORITHMIC bytes per launch (SURVEY §8(d); DESIGN.md §4), one launch = one step of one rank:
        #  ring_push   (K1 fused): step PCM read once + written once into the rings + one 8-byte block sum per tick
        #  tick_gate   (K2): with K1's block sums it reads no PCM: 10 block sums + state in/out per stream;
        #              (host pushes: it reads the step's PCM once itself)
        #  segment_queue (K3): the PCM of every candidate segment of the profiled launches once + its 40-byte event
        alg_bytes = {"ring_push": n * (STEP_SAMPLES * esz * 2 + TICKS_PER_STEP * 8),
                     "tick_gate": n * (TICKS_PER_STEP * 8 + 2 * 104 + 72 + 2 * 1600),
                     "segment_queue": prof_samples * esz + prof_cand * 40}
        share = {k: v["ms"] / tot_ms for k, v in kern.items()}

        def kroof(name):
            if name not in kern:
                return None
            ms = kern[name]["ms"] / kern[name]["launches"]
            gbs = alg_bytes.get(name, 0.0) / (ms * 1e-3) / 1e9
            return {"avg_launch_ms": ms, "algorithmic_bytes": alg_bytes.get(name), "achieved_gbs": gbs, "frac": gbs / hbm_peak,
                    "traffic": traffic.get(name)}

        traffic = _traffic()
        avg_ms = kern[dom]["ms"] / kern[dom]["launches"]
        achieved = alg_bytes.get(dom, 0.0) / (avg_ms * 1e-3) / 1e9
        frames_per_step = prof_frames
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak, "traffic": traffic.get(dom), "peak_source": peak_src,
                    "avg_launch_ms": avg_ms, "share_of_kernel_time": share,
                    "note": "the dominant kernel (fused MFCC+match on candidate segments) does ~45 flop per PCM byte "
                            "(DESIGN.md §4) and is bound on the SM, not on HBM: ncu shows the shared-memory data pipe "
                            "(l1tex lsu wavefronts) at ~73 % of peak while an SM is busy (profiles/README.md); its HBM "
                            "fraction is small by construction.  `compute` gives its FP32 rate and `hbm_bound_kernel` "
                            "the roofline of the HBM-bound kernel of the step (K1 fused push+sums)",
                    "compute": {"frames_per_launch": frames_per_step, "flop_per_frame": 15300,
                                "achieved_tflops": frames_per_step * 15300 / (avg_ms * 1e-3) / 1e12 if dom == "segment_queue" else None,
                                "fp32_peak_tflops": 148 * 128 * 2 * 1.965e9 / 1e12},
                    "hbm_bound_kernel": dict(kernel="ring_push", **(kroof("ring_push") or {})),
                    "tick_gate": kroof("tick_gate"),
                    "whole_step_frac": (n * STEP_SAMPLES * esz) * K / (ms_dev * 1e-3) / 1e9 / hbm_peak}
        cpu = None
        best_c = None
        if world == 1 and not args.no_cpu:
            cores = os.cpu_count() or 1
            kind = cpu_kind()
            cpool = CpuPool(cores)
            CPU_S = 120.0           # ~1 s of reference work per core (~125 audio-s/s per core): ~16 core-seconds in all
            v, audio, wall, _ = cpu_throughput(CPU_S, cores, "reference" if kind == "reference" else "port", pool=cpool)
            vf, _, _, _ = cpu_throughput(CPU_S, cores, "port_fast", pool=cpool)
            cpool.close()
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "per_core": v / cores,
                   "sample": f"{cores} processes (one BLAS/OpenMP thread each, checked in every worker) x {CPU_S:.0f} s steady state of "
                             f"one workload stream each = {audio:.0f} audio-s, value = sum of the workers' own rates; " +
                             ("the reference's own SoundBuffer / WordMatcher / _detect_word (oracle/_ref, unmodified) under the fake clock"
                              if kind == "reference" else "oracle port in the reference's statement order") +
                             f"; vectorised oracle variant: {vf:.1f} audio-s/s",
                   "vectorised_port_value": vf}
            if pool_pin.array.dtype == np.int16:
                try:
                    vc, evc, audio_c = cpu_best_effort_c(pool_pin.array, word, cores)
                    best_c = {"value": vc, "unit": UNIT, "cores": cores, "kind": "port (C, OpenMP over streams)",
                              "sample": f"3 x 1024 streams x {3 * POOL_SECONDS} s of the bench pool = {audio_c:.0f} audio-s, "
                                        f"{evc} level-2 evaluations; not the reference's code path: what a "
                                        "tuned CPU implementation of the same semantics reaches on this host"}
                except Exception as e:                              # no gcc on the box: the baseline above stands alone
                    best_c = {"unavailable": f"{type(e).__name__}: {e}"[:160]}
                cpu["best_effort_c"] = best_c
        dense_cpu = None
        if world == 1 and not args.no_cpu:
            dv, dw = cpu_dense_throughput(3.0)
            dense_cpu = {"value": dv, "unit": UNIT, "cores": 1, "kind": "port", "windows_per_s": dw,
                         "sample": "300 hops (3.0 s) of one stream, oracle WordMatcher.calculate_similarity per hop"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "repeats": {"blocks": R, "steps_per_block": K, "reported": "median block",
                        "ms_per_step_blocks": [round(b / K, 5) for b in dev_blocks],
                        "e2e_ms_per_step_blocks": [round(b / K, 5) for b in e2e_blocks]},
            "config": bench_config(n, pcm_name, world, word_name),
            "execution": {"overlap": ("K3 of step i runs on a second stream beside K1 of step i+1 (ewk_set_overlap; K1 in its "
                                      "cp.async.bulk form); the timed region ends after the last K3 (ewk_join); per-kernel "
                                      "times are taken in sequential order, each kernel alone")
                          if overlap else "off: K1, K2, K3 in sequence on one stream",
                          "exchange": (("8 B/stream result records + completion signal put into every rank's copy over NVLink by a "
                                        "sender kernel behind K3 (side stream)" + (", one barrier per step" if args.gather == "peer-barrier" else
                                                                                   " (put-with-signal, no collective)") if exchange is not None else
                                        ("all_gather of 8 B/stream results per step" if gathered is not None else
                                         "none (--gather none)"))) if world > 1 else None},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": n * STEP_SAMPLES * esz,
                    "d2h_bytes_per_step": int(8 + ev_per_step * 40), "ms_per_step": ms_e2e / K,
                    "h2d_gbs_per_gpu": n * STEP_SAMPLES * esz / (ms_e2e / K * 1e-3) / 1e9,
                    "host_cpus_rank0": (f"{host_cpus[0]}-{host_cpus[-1]} ({len(host_cpus)})" if host_cpus else None),
                    "bound": f"host->device copy (PCIe): the PCM of a step is {n * STEP_SAMPLES * esz / 1e6:.0f} MB per GPU and every step pays its own "
                             "copy; kernels take ~10 % of the step and overlap the next copy"},
            "e2e_g711": g711,
            "gpu_launches": int(launches),
            "by_rank": {"device_resident": by_rank[0], "e2e": by_rank[1]},
            "gather": gather_info,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "best_effort_c": best_c,
            "e2e_vs_best_effort_c": (e2e_val / best_c["value"]) if best_c and "value" in best_c else None,
            "dense": {"what": f"A9 per-hop scoring: 100 hops x {n} streams per step, 4 FFT frames per hop (1 stream-grid + 3 "
                              "window-edge), K1 ring_push + K4 dense_score, scores left on the device",
                      "value": audio_per_step * dense_steps / (ms_dense * 1e-3), "unit": UNIT,
                      "ms_per_step": ms_dense / dense_steps,
                      "kernel_ms": prof_dense["dense_score"]["ms"] / max(1, prof_dense["dense_score"]["launches"]),
                      "windows_per_s": n * 100 * world * dense_steps / (ms_dense * 1e-3),
                      "traffic": traffic.get("dense_score"),
                      "hbm_frac": (n * STEP_SAMPLES * esz + n * 400) * dense_steps / (ms_dense * 1e-3) / 1e9 / hbm_peak,
                      "cpu_baseline": dense_cpu},
            "sweep": sweep,
            "config3": config3,
            "level2_events_per_step": ev_per_step,
            "profile_pass": {"steps": KP, "candidates_per_step": prof_cand, "candidate_samples_per_step": prof_samples,
                             "candidate_frames_per_step": prof_frames,
                             "what": "the per-kernel times and the roofline come from this separate pass: sequential order, whole "
                                     "periods of the feed, its own candidates counted"},
            "kernel_ms_per_step": {k: v["ms"] / KP for k, v in kern.items()},
            "kernel_ms_per_step_without_publication": ({k: v["ms"] / KP for k, v in prof_nopub.items() if v["launches"]}
                                                       if prof_nopub else None),
        }
        print(json.dumps(line), flush=True)
    bank.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_only(args):
    """`--only sweep|config3`: one secondary leg on its own (profiling, quick checks); prints {"<leg>": {...}}."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    word, _ = load_word()
    pk = os.path.join(REPO, "MEASURED_PEAKS.json")
    hbm_peak = float(json.load(open(pk)).get("hbm_gbs", 6650.0)) if os.path.exists(pk) else 6650.0
    if args.only == "sweep":
        leg = sweep_leg(torch, dist, dev, stream, local_rank, rank, world, word, hbm_peak, seconds=args.sweep_seconds)
    else:
        pool_pin = np.empty((POOL_SECONDS, N_STREAMS, STEP_SAMPLES), np.int16)
        make_pool(rank * N_STREAMS, N_STREAMS, word, pool_pin)
        pool_dev = torch.from_numpy(pool_pin).to(dev)
        leg = config3_leg(torch, dist, dev, stream, local_rank, rank, world, word, pool_dev, args.steps, max(3, args.warmup),
                          not args.no_overlap)
    if rank == 0:
        print(json.dumps({args.only: leg, "n_gpus": world}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=5,
                    help="timed blocks of exactly --steps steps; the line reports the median block (all blocks listed)")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary legs (sweep = configs[4], config3, dense)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--streams", type=int, default=N_STREAMS,
                    help="streams per GPU (default 4096 = BASELINE configs[2]; 8192 = the per-GPU shard of configs[3], 65536 / 8)")
    ap.add_argument("--pcm", default="int16", choices=["int16", "f32"],
                    help="ring / push sample format (int16: the wire format, default; f32: what PortAudio hands the reference)")
    ap.add_argument("--gather", default="auto", choices=["auto", "peer", "peer-barrier", "nccl", "none"],
                    help="multi-GPU result exchange: peer = K2/K3 store records and a completion signal into every rank's "
                         "copy over NVLink (no collective, no per-step barrier); peer-barrier = same stores, one "
                         "symmetric-memory barrier per step; nccl = all_gather per step; auto = peer when symmetric "
                         "memory is available")
    ap.add_argument("--no-g711", action="store_true", help="skip the secondary end-to-end leg fed with G.711 mu-law codes")
    ap.add_argument("--no-bind", action="store_true", help="multi-GPU: do not pin each rank to the CPUs next to its GPU")
    ap.add_argument("--no-overlap", action="store_true",
                    help="keep K3 on the context's stream (default: ewk_set_overlap(1), K3 beside the next push)")
    ap.add_argument("--only", default="all", choices=["all", "sweep", "config3"],
                    help="run one secondary leg on its own instead of the whole line")
    ap.add_argument("--sweep-seconds", type=int, default=SWEEP_SECONDS, help="audio seconds per stream the sweep leg measures")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline (device-resident) path computed for rank 0's "
                         "streams as DIR/<name>.npy: per-stream result records and that step's events")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.only != "all"):
        ap.error("--dump-outputs applies to the GPU line (--impl ours, --only all)")
    if args.impl == "reference":
        run_reference(args)
    elif args.only != "all":
        run_only(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
