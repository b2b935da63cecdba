"""Poison mode (EWK_POISON, include/ewk.h: ewk_debug_check): the library's own memory.

Each workload group runs three times in fresh contexts: with EWK_POISON unset, with 0xFF (NaN floats and doubles, -1
integers) and with 0x3C (float ~0.0115, double ~1e-17, a plausible value).  Poison mode fills every allocation of a
context with the byte before the library initialises it, allocates per-call workspaces at exactly the size a call needs
and refills them at every call, and puts a guard band of the byte behind every allocation.  So a kernel that reads memory
nobody wrote, or an index one past a valid range, changes an output; a write past a buffer's end damages a guard.  The
test requires every observable output to be equal byte for byte across the three runs, equal launch counts, and clean
guards after the group.

The groups together launch every __global__ kernel and template instance of csrc/; each names what it reaches.
profiles/tools/sanitize_workload.py runs the same list (WORKLOADS).
"""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

from conftest import REPO

PATTERNS = (None, 0xFF, 0x3C)


def _word():
    g = np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))
    return g["pcm_i16"].astype(np.float32) / np.float32(32768)


@contextlib.contextmanager
def _env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    try:
        for k, v in kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = str(v)
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _canon(v):
    """an output as comparable bytes"""
    if isinstance(v, np.ndarray):
        return ("nd", v.dtype.str, v.shape, np.ascontiguousarray(v).tobytes())
    if isinstance(v, C.Structure):
        return ("st", bytes(v))
    if isinstance(v, dict):
        return tuple((k, _canon(v[k])) for k in sorted(v))
    if isinstance(v, (list, tuple)):
        return tuple(_canon(x) for x in v)
    if isinstance(v, float):
        return ("f", np.float64(v).tobytes())
    return v


class Run:
    """One run of a group under one pattern: the contexts it creates and every output it records"""

    def __init__(self, pattern):
        self.pattern = pattern
        self.out = []
        self.ctxs = []
        self.prof = {}

    def ctx(self, **kw):
        from easywakeword_b200 import _lib
        c = _lib.Context(device=0, **kw)
        c.profile(True)
        self.ctxs.append(c)
        return c

    def add(self, name, v):
        self.out.append((name, _canon(v)))

    def events(self, name, c):
        ev = c.poll()
        self.add(name, sorted(e.tobytes() for e in ev))
        self.add(name + " dropped", c.dropped)
        return ev

    def bank_state(self, name, c):
        """everything a bank context shows: events, results, status and the whole visible ring of every stream"""
        self.events(name + " events", c)
        self.add(name + " results", c.results())
        for s in range(c.cfg.n_streams):
            self.add(f"{name} status {s}", c.status(s))
            self.add(f"{name} ring {s}", c.read_last(s, c.cfg.ring_samples))

    def check(self):
        """guards clean (poison runs), then launch counts, profile classes, close"""
        for i, c in enumerate(self.ctxs):
            if self.pattern is not None:
                c.debug_check()
            for k, v in c.profile_read().items():
                self.prof[k] = self.prof.get(k, 0) + v["launches"]
            self.add(f"launches of context {i}", c.launch_count())
            if self.pattern is not None:
                c.debug_check()
            c.close()


def _dev(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()
    return t


# -------------------------------------------------------------------------------------------------- workload groups
def level2(r, word):
    """reaches: segment_mfcc_match_kernel<false> (extract, set_template(s), similarity_batch incl. the b_ws spill),
    dense_template_features_kernel and dense_template_install_kernel (set_template / set_templates), template_vad_kernel
    (analyze_templates, set_templates want_vad), resample_push_kernel<0..3, false> (one-shot resample: every plan
    branch of the rates of test_gpu_resample_chain.py)"""
    from easywakeword_b200 import _lib, synth
    from test_gpu_resample_chain import RATES
    c = r.ctx(n_streams=0, max_templates=12)
    x, _ = synth.stream(5, 5.0, word, gain=(2.0, 3.0), inserts_per_10s=(1, 1), zero_gaps=1)
    x = synth.from_int16(synth.to_int16(x))
    r.add("extract", c.extract_mfcc(x[:24007], want_frames=True))
    d = _dev(x[:24007])
    m, s = np.empty(20, np.float32), np.empty(20, np.float32)
    fr = np.empty((1 + 24007 // 160, 20), np.float32)
    c._ck(c.lib.ewk_extract_mfcc(c.h, d.data_ptr(), 24007, _lib.DEVICE, _lib.f32ptr(m), _lib.f32ptr(s), _lib.f32ptr(fr), len(fr)))
    r.add("extract device", (m, s, fr))
    c.set_template(0, word)
    r.add("set_templates vad", c.set_templates([1, 2, 3, 4], [word[:1], word[:800], x[:60000], x[1:48001]], want_vad=True))
    lens = [1, 3000, 60000]
    dx = _dev(x[:sum(lens)])
    c.set_templates([5, 6, 7], (dx.data_ptr(), np.cumsum([0] + lens[:-1]), lens))
    for k in range(8):
        r.add(f"template {k}", c.get_template(k))
    offs, ln = [0, 8001, 100], [len(x), 20000, 64000]          # 80000 and 64000 samples: more frames than shared memory
    for pcm in (x, synth.to_int16(x)):
        r.add(f"similarity {pcm.dtype}", c.similarity_batch(0, pcm, offs, ln, want_features=True))
        dp = _dev(pcm)
        sc, mt, ft = np.empty(3, np.float32), np.empty(3, np.uint8), np.empty((3, 40), np.float32)
        o, l = np.asarray(offs, np.int64), np.asarray(ln, np.int64)
        c._ck(c.lib.ewk_similarity_batch(c.h, 0, dp.data_ptr(), _lib.PCM_I16 if pcm.dtype == np.int16 else _lib.PCM_F32,
                                         _lib.DEVICE, _lib.i64ptr(o), _lib.i64ptr(l), 3, 75.0, _lib.f32ptr(sc),
                                         _lib.u8ptr(mt), _lib.f32ptr(ft)))
        r.add(f"similarity {pcm.dtype} device", (sc, mt, ft))
    r.add("analyze", c.analyze_templates([word, x[:9000], np.zeros(700, np.float32)], want_rms=True))
    rng = np.random.default_rng(0)
    for sr in sorted(RATES):
        y = rng.standard_normal((2, max(64, sr // 5))).astype(np.float32)
        r.add(f"resample {sr}", c.resample(y, sr))
        r.add(f"resample {sr} i16 window", c.resample((y * 3000).astype(np.int16), sr, in_first=7, out_first=3, n_out=500))


def _bank(r, n, R, fmt, word, **kw):
    from easywakeword_b200 import _lib
    c = r.ctx(n_streams=n, ring_samples=R, slack_samples=kw.pop("slack", 16000),
              pcm_format=_lib.PCM_I16 if fmt == "i16" else _lib.PCM_F32, max_templates=kw.pop("max_templates", 4), **kw)
    c.set_template(0, word)
    c.set_stream_params(-1, frame_size=1600, timeout=3.0, speech_duration_min=0.3, speech_duration_max=2.0)
    return c


def _feed(seed, n, seconds, fmt, word):
    from easywakeword_b200 import synth
    q = synth.stream_batch(seed, n, seconds, word, zero_gaps=1, gain=(2.0, 4.0), distractor_prob=0.2)
    return q if fmt == "i16" else synth.from_int16(q)


def pushes(r, word, fmt):
    """reaches: ring_push_sums_kernel<T> (aligned host and device pushes), ring_push_kernel<T> + ring_commit_kernel
    (unaligned pushes), tick_gate_kernel<false> (presummed, staged and generic sums, traced), tick_gate_kernel<true>
    (tick_ready), g711_decode_kernel (push_g711 host and device, i16 rings), ring_push_list_kernel<T> (push_streams at
    16 kHz, PCM and G.711 codes), resample_push_kernel<M, false> (uniform K8 at 8, 44.1 and 48 kHz, the second rate grows
    the tails) and <M, true> (push_resampled_each, push_streams at 44.1 kHz), segment_queue_kernel<false> (ticks), and
    the queue overflow (16 event slots for 24 streams)"""
    T = np.int16 if fmt == "i16" else np.float32
    n = 8
    c = _bank(r, n, 48000, fmt, word)
    x = _feed(900, n, 6.0, fmt, word)
    c.push(np.ascontiguousarray(x[:, :16000]))
    r.add("trace 0", c.tick(10, trace=True))
    c.push(np.ascontiguousarray(x[:, 16000:24001]))                            # unaligned: scalar push, generic gate
    c.push(np.ascontiguousarray(x[:, 24001:32000]))
    r.add("trace 1", c.tick(10, trace=True))
    d = _dev(x[:, 32000:48000])
    c.push((d.data_ptr(), n, 16000, 16000), where=1)
    c.tick(10)
    if fmt == "i16":
        codes = np.random.default_rng(1).integers(0, 256, size=(n, 8000), dtype=np.uint8)
        c.push_g711(codes[:, :4800])
        dc = _dev(codes[:, 4800:])
        c.push_g711((dc.data_ptr(), n, 3200, 3200), where=1, law="alaw")
    rows = [np.ascontiguousarray(x[i, 48000:48000 + 1600 * (i % 3) + 333 * i]) for i in range(n)]
    r.add("push_streams", c.push_streams(list(range(n)), rows))
    if fmt == "i16":
        r.add("push_streams g711", c.push_streams([0, 3, 5], [np.arange(700, dtype=np.uint8)] * 3, fmt="ulaw"))
    r.add("tick_ready", c.tick_ready(30, trace=True))
    r.bank_state("16k", c)
    # native rates
    c = _bank(r, n, 48000, fmt, word)
    rng = np.random.default_rng(2)
    y8 = (rng.standard_normal((4, 8000)) * 2000).astype(np.int16)
    r.add("k8 8k", c.push_resampled(y8, 8000, stream0=0))
    y48 = (rng.standard_normal((4, 24000)) * 0.1).astype(np.float32)
    r.add("k8 48k", c.push_resampled(y48, 48000, stream0=4))
    r.add("k8 8k again", c.push_resampled(y8[:, ::-1].copy(), 8000, stream0=0))
    dy = _dev(y48)
    r.add("k8 48k device", c.push_resampled((dy.data_ptr(), 4, 24000, 24000, np.float32), 48000, stream0=4, where=1))
    c.tick_ready(20)
    r.events("native events", c)
    c.reset_streams([1, 2, 3])
    r.add("each", c.push_resampled_each(y8[:2], 8000, stream0=0))    # stream 0 goes on, stream 1 restarts at 0
    y44 = (rng.standard_normal((2, 4410 * 3)) * 0.1).astype(np.float32)
    r.add("k8 list 44.1k", c.push_streams([2, 3], [y44[0][:5000], y44[1]], sr_in=44100))
    r.add("tick_ready native", c.tick_ready(20, trace=True))
    r.bank_state("native", c)
    r.add("native blob", c.export_streams(list(range(n))))      # rings not yet full, K8 tails of three rates
    # queue overflow: more candidates than event slots
    c = _bank(r, 24, 32000, fmt, word, max_events=16)
    c.set_stream_params(-1, frame_size=1600, timeout=30.0, speech_duration_min=0.3, speech_duration_max=2.0,
                        similarity_threshold=0.0)
    x = _feed(300, 24, 4.0, fmt, word)
    for b in range(0, x.shape[1], 16000):
        c.push(np.ascontiguousarray(x[:, b:b + 16000]))
        c.tick(10)
    r.bank_state("overflow", c)


def tma(r, word, fmt):
    """reaches: ring_push_bulk_kernel<T> (device pushes beside K3 in overlap mode, 160 x 1 s = 1600 blocks per push)"""
    n = 160
    c = _bank(r, n, 96000, fmt, word)
    x = _feed(23, 12, 8.0, fmt, word)
    x = np.concatenate([x] * (n // 12 + 1))[:n]
    c.set_overlap(True)
    import torch
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for b in range(0, x.shape[1], 16000):
            d = _dev(x[:, b:b + 16000])
            c.push((d.data_ptr(), n, 16000, 16000), where=1)
            c.tick(10)
        c.synchronize()
    names = {e.name for e in prof.events()}
    assert any("ring_push_bulk_kernel" in k for k in names), "no push took the cp.async.bulk form"
    r.bank_state("tma", c)


def k3_forms(r, word):
    """reaches: segment_frames_kernel<false> (EWK_K3=2), segment_queue_kernel<false> without the log-mel workspace
    (EWK_SEG_LM=0), and with preemphasis=0.97, n_mfcc=13: segment_queue_kernel<true>, segment_frames_kernel<true>,
    segment_mfcc_match_kernel<true> (set_template, similarity_batch)"""
    for env, cfg in ((dict(EWK_K3=2), {}), (dict(EWK_SEG_LM=0), {}), ({}, dict(preemphasis=0.97, n_mfcc=13)),
                     (dict(EWK_K3=2), dict(preemphasis=0.97, n_mfcc=13))):
        with _env(**env):
            c = _bank(r, 6, 48000, "i16", word, **cfg)
        c.set_stream_params(-1, frame_size=1600, timeout=3.0, speech_duration_min=0.3, speech_duration_max=2.0,
                            similarity_threshold=0.0)
        x = _feed(77, 6, 6.0, "i16", word)
        for b in range(0, x.shape[1], 16000):
            c.push(np.ascontiguousarray(x[:, b:b + 16000]))
            c.tick(10)
        name = f"{sorted(env.items())} {sorted(cfg.items())}"
        r.bank_state(name, c)
        if cfg:
            r.add(name + " similarity", c.similarity_batch(0, x[0], [0, 1000], [30000, 52000], want_features=True))


def dense(r, word):
    """reaches: dense_score_kernel<false, false, false> (dense_scores at every geometry ewk_dense_plan can choose),
    <false, true, false> (dense_scores_streams with an empty row, rows in descending hop order and rows that overlap in
    hops; dense_ready; geometry groups of the _sets forms whose rows share one set), <false, true, true> (a _sets call
    with three sets of one geometry), dense_detect_kernel (dense_detect, dense_detect_sets), and with preemphasis the
    <true, ...> instances; calls whose DG differs from the previous call's; a set switch and a template change that
    rebuilds cached sets"""
    import helpers
    from easywakeword_b200 import _lib, synth
    geo = helpers.dense_geometry_sets(_lib.dense_plan)
    src = synth.stream_batch(8100, 1, 4.0, word)[0].astype(np.float32) / 32768
    c = _bank(r, 3, 64000, "i16", word, max_templates=8)
    x = _feed(81, 3, 3.0, "i16", word)
    c.push(np.ascontiguousarray(x))
    for g in sorted(geo):
        lens = geo[g]
        c.set_templates(list(range(len(lens))), [np.resize(src, L) for L in lens])
        r.add(f"geometry {g}", (c.dense_scores(3, 40, 0, len(lens)), c.dense_last_plan()))
    for pre in (0.0, 0.97):
        c = _bank(r, 4, 64000, "i16", word, max_templates=8, preemphasis=pre)
        c.set_templates([1, 2, 3], [word[:9000], np.resize(src, 30000), np.resize(src, 1001)])
        c.set_stream_params(-1, frame_size=1600, similarity_threshold=0.0)
        x = _feed(82, 4, 4.0, "i16", word)
        c.push(np.ascontiguousarray(x[:, :32000]))
        r.add(f"{pre} scores", c.dense_scores(1, 50, 0, 2))
        r.add(f"{pre} streams", c.dense_scores_streams([3, 0, 1, 2], [40, 5, 30, 7], [25, 0, 25, 3], 1, 3))
        r.add(f"{pre} ready", c.dense_ready([2, 0], 60, 0, 4))
        r.add(f"{pre} detect", c.dense_detect(None, 80, 0, 2, scores=True))
        c.push(np.ascontiguousarray(x[:, 32000:]))
        r.add(f"{pre} streams DG", c.dense_scores_streams([1], [3], [60], 2, 1))
        c.set_stream_params(0, frame_size=1600, template_first=0, template_count=2, similarity_threshold=0.0)
        c.set_stream_params(1, frame_size=1600, template_first=1, template_count=3, similarity_threshold=0.0)
        r.add(f"{pre} sets", c.dense_scores_sets([0, 1, 2], [4, 4, 4], [30, 30, 30]))
        r.add(f"{pre} sets one geometry", c.dense_scores_sets([0, 1, 2], [4, 4, 4], [30, 30, 30], [0, 1, 3], [1, 1, 1]))
        r.add(f"{pre} ready sets", c.dense_ready_sets(None, 50))
        r.add(f"{pre} detect sets", c.dense_detect_sets(None, 80, scores=True))
        c.set_template(2, word[::-1].copy())                 # rebuilds the cached sets that contain slot 2
        c.set_stream_params(2, frame_size=1600, template_first=2, template_count=2, similarity_threshold=0.0)
        r.add(f"{pre} sets after change", c.dense_scores_sets([0, 1, 2, 3], [2, 2, 2, 2], [60, 60, 60, 60]))
        r.add(f"{pre} detect sets after change", c.dense_detect_sets(None, 100, scores=True))
        for k in range(4):
            r.add(f"{pre} template {k}", c.get_template(k))


ARMED = 1                                  # DetState mode (oracle/dense_detect.py)


def _detector_modes(c, streams):
    """the dense detector's mode of each stream, from its exported meta record"""
    from easywakeword_b200 import _lib
    raw = c.export_streams(streams)
    mo = int(raw[:_lib.STREAM_BLOB_HEADER_DTYPE.itemsize].view(_lib.STREAM_BLOB_HEADER_DTYPE)[0]["meta_offset"])
    return [int(raw[mo + i * _lib.STREAM_META_BYTES + 256:][:4].view(np.int32)[0]) for i in range(len(streams))]


def lifecycle(r, word):
    """reaches: segment_prepare_kernel (K5, host and device output), ring_gather_kernel + segment_mfcc_match_kernel
    (set_templates_from_streams), stream_reset_kernel (K9 on streams whose dense detector holds an ARMED run, asserted
    from the exported detector state), stream_export_kernel (K10 export, host and device) and stream_import_kernel
    (import into a second context, host and device blob)"""
    import torch
    from easywakeword_b200 import _lib
    n = 6
    c = _bank(r, n, 48000, "f32", word, max_templates=8)
    c.set_stream_params(-1, frame_size=1600, timeout=3.0, speech_duration_min=0.3, speech_duration_max=2.0,
                        similarity_threshold=0.0)           # every scored hop arms the detector; hold keeps the run open
    x = _feed(91, n, 5.0, "f32", word)
    for b in range(0, 64000, 16000):
        c.push(np.ascontiguousarray(x[:, b:b + 16000]))
        c.tick(10)
        r.add(f"detect {b}", c.dense_detect(None, 100, hold_hops=1000, refractory_hops=10))
    segs = ([0, 2, 5], [20000, 47000, 30000], [1600, 9000, 333])
    r.add("k5 host", c.prepare_segments(*segs))
    st, a, ln = (np.asarray(v, t) for v, t in zip(segs, (np.int32, np.int64, np.int64)))
    offs = np.array([3, 2000, 12000], np.int64)
    out = torch.full((12500,), 7.0, dtype=torch.float32, device="cuda")
    c._ck(c.lib.ewk_prepare_segments(c.h, 3, st.ctypes.data_as(C.POINTER(C.c_int32)), _lib.i64ptr(a), _lib.i64ptr(ln),
                                     _lib.i64ptr(offs), C.cast(out.data_ptr(), C.POINTER(C.c_float)), 12500, _lib.DEVICE))
    torch.cuda.synchronize()
    r.add("k5 device", out.cpu().numpy())
    r.add("enrol from streams", c.set_templates_from_streams([4, 5], [1, 3], [30000, 40000], [16000, 7000], want_vad=True))
    for k in (4, 5):
        r.add(f"template {k}", c.get_template(k))
    c.push(np.ascontiguousarray(x[:, 64000:72000]))
    c.tick(5)
    r.add("detect before reset", c.dense_detect(None, 100, hold_hops=1000, refractory_hops=10))
    modes = _detector_modes(c, [0, 2, 3])
    r.add("detector modes before reset", modes)
    assert ARMED in modes, f"no stream to reset holds an ARMED run: {modes}"
    r.add("status before reset", [c.status(s).state for s in range(n)])
    r.events("before reset", c)
    c.reset_streams([0, 2, 3])
    c.push_resampled((np.random.default_rng(3).standard_normal((2, 8000)) * 0.1).astype(np.float32), 8000, stream0=2)
    blob = c.export_streams([1, 0, 4])
    r.add("blob host", blob)
    cap = c.stream_blob_bytes(3)
    dblob = torch.zeros(cap + 64, dtype=torch.uint8, device="cuda")
    c.export_streams([1, 0, 4], where=_lib.DEVICE, out=(dblob.data_ptr(), cap))
    torch.cuda.synchronize()
    r.add("blob device", dblob.cpu().numpy())
    c2 = _bank(r, 4, 48000, "f32", word, max_templates=8)
    c2.import_streams([3, 0, 1], blob)
    c2.import_streams([2], c.export_streams([5]))
    c2.tick_ready(10)
    r.bank_state("imported", c2)
    c3 = _bank(r, 3, 48000, "f32", word, max_templates=8)
    c3.import_streams([0, 1, 2], (dblob.data_ptr(), cap), where=_lib.DEVICE)
    r.bank_state("imported device", c3)
    c.tick_ready(10)
    r.bank_state("source", c)


def publish(r, word):
    """reaches: publish_records_kernel (set_results_peers onto local destinations with stride, offset and signals, in
    overlap mode), peer_wait_kernel (wait_published), the results buffer (set_results_buffer)"""
    import torch
    n = 40
    c = _bank(r, n, 48000, "i16", word)
    dests = [torch.full((2, 64, 2), -7, dtype=torch.int32, device="cuda") for _ in range(2)]
    sigs = [torch.zeros(2, 16, dtype=torch.int64, device="cuda") for _ in range(2)]
    c.set_results_peers([d.data_ptr() for d in dests], stride_records=64, offset_records=5,
                        signals=[g.data_ptr() for g in sigs], slot=0)
    own = torch.full((n, 2), -3, dtype=torch.int32, device="cuda")
    c.set_results_buffer(own.data_ptr())
    c.set_overlap(True)
    x = _feed(95, n, 4.0, "i16", word)
    for b in range(0, x.shape[1], 16000):
        c.push(np.ascontiguousarray(x[:, b:b + 16000]))
        c.tick(10)
        c.wait_published(1, c.publish_seq())
        c.synchronize()
        r.add(f"published {b}", [d.cpu().numpy() for d in dests] + [g.cpu().numpy() for g in sigs] + [own.cpu().numpy()])
        r.events(f"events {b}", c)
    r.add("published seq", c.published_seq(c.publish_parity(), 2))
    c.set_results_peers([])
    r.bank_state("publish", c)


WORKLOADS = {
    "level2": level2,
    "push_i16": lambda r, w: pushes(r, w, "i16"),
    "push_f32": lambda r, w: pushes(r, w, "f32"),
    "tma_i16": lambda r, w: tma(r, w, "i16"),
    "tma_f32": lambda r, w: tma(r, w, "f32"),
    "k3_forms": k3_forms,
    "dense": dense,
    "lifecycle": lifecycle,
    "publish": publish,
}


def run_workload(name, pattern, word=None):
    """run one group with EWK_POISON = pattern (None: unset) -> the Run"""
    r = Run(pattern)
    with _env(EWK_POISON=None if pattern is None else hex(pattern)):
        try:
            WORKLOADS[name](r, _word() if word is None else word)
            r.check()
        finally:
            for c in r.ctxs:
                c.close()
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("group", list(WORKLOADS))
def test_poison_patterns_agree(group, word):
    runs = [run_workload(group, p, word) for p in PATTERNS]
    base = runs[0]
    for r in runs[1:]:
        assert len(r.out) == len(base.out)
        for (name, a), (_, b) in zip(base.out, r.out):
            assert a == b, f"{group}: '{name}' differs with EWK_POISON={r.pattern:#04x}"


@pytest.mark.gpu
def test_groups_reach_every_profile_class(word):
    """ewk_profile_read summed over one run of every group: launches in every profiling class some call site records"""
    total = {}
    for g in WORKLOADS:
        for k, v in run_workload(g, None, word).prof.items():
            total[k] = total.get(k, 0) + v
    assert len(total) == 8 and all(v > 0 for v in total.values()), total


@pytest.mark.gpu
def test_debug_check_needs_poison_mode():
    from easywakeword_b200 import _lib
    with _env(EWK_POISON=None):
        c = _lib.Context(device=0, n_streams=0, max_templates=1)
    try:
        with pytest.raises(RuntimeError, match="poison mode is off"):
            c.debug_check()
    finally:
        c.close()
    with _env(EWK_POISON="256"), pytest.raises(ValueError, match="EWK_POISON"):
        _lib.Context(device=0, n_streams=0, max_templates=1)
