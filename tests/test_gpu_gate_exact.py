"""The level-1 gate (K2, tick_gate_kernel) against oracle/gate_model.py bit for bit: every trace cell (silent, state,
threshold and RMS as float64 bits), every event (stream, kind, tick, seg_start, seg_len), every ewk_stream_status field
and bits 1-4 and 8.. of the result flags.  The model knows nothing of K2's plan, so each case says which of K2's paths
(and which of K1's sum sources) it reaches, by construction:

* presummed: whole-tick pushes on a ring with P % 1600 == 0 — K1 forms the per-block sums, K2 reads no PCM;
* staged: half-tick pushes (no block sums) on such a ring — K2 stages every tick through shared memory (cp.async.bulk);
* generic: P % 1600 != 0, any frame size but 1600, ring wraps, first-full and heavy ticks, live streams — K2 sums the
  samples itself (warp_sumsq, vector or scalar path by the physical start);
* TMA push: overlap mode with >= 1184 blocks per push — K1's cp.async.bulk form forms the sums;
* list pushes (K1L) and native-rate pushes (K8), which leave no block sums.

The EWK_* switches are read once per process, so no case relies on them."""
import numpy as np
import pytest

from easywakeword_b200 import synth
from oracle import gate_model as G

pytestmark = pytest.mark.gpu


def _lib():
    from easywakeword_b200 import _lib as L
    return L


def feed(seed, n_streams, seconds, fmt, word=None, noise=0.01):
    """[n_streams, seconds * 16000] speech-like feeds in the ring's dtype (f32: not int16-representable)"""
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(n_streams):
        x, _ = synth.stream(seed * 97 + i, seconds, word if word is not None else _tone(), noise_sigma=noise,
                            gain=(1.0, 5.0), zero_gaps=1, distractor_prob=0.3)
        q = synth.to_int16(x)
        if fmt == "i16":
            rows.append(q)
        else:
            rows.append((synth.from_int16(q) + rng.standard_normal(q.size).astype(np.float32) * np.float32(3e-5))
                        .astype(np.float32))
    return np.stack(rows)


def _tone():
    t = np.arange(9000) / 16000.0
    return (0.3 * np.sin(2 * np.pi * 440 * t) * np.hanning(9000)).astype(np.float32)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


class Pair:
    """one context and the model, driven with the same calls; the model covers streams [0, n_model)"""

    def __init__(self, R, slack, fmt, params, n_model=None, max_events=4096):
        L = _lib()
        self.L, self.fmt, self.R = L, fmt, R
        self.ctx = L.Context(device=0, n_streams=len(params), ring_samples=R, slack_samples=slack,
                             pcm_format=L.PCM_I16 if fmt == "i16" else L.PCM_F32, max_templates=1, max_events=max_events)
        for i, p in enumerate(params):
            self.ctx.set_stream_params(i, **p)
        self.nm = len(params) if n_model is None else n_model
        self.model = G.GateModel(R, G.physical_ring(R, slack), fmt, params[:self.nm])
        self.events, self.dropped, self.cells = [], 0, 0

    def push(self, x, stream0=0, device=False):
        x = np.ascontiguousarray(x)
        if device:
            import torch
            t = torch.from_numpy(x).cuda()
            torch.cuda.synchronize()
            self.ctx.push((t.data_ptr(), x.shape[0], x.shape[1], x.shape[1]), stream0=stream0, where=self.L.DEVICE)
            self.ctx.synchronize()
        else:
            self.ctx.push(x, stream0=stream0)
        for r in range(x.shape[0]):
            if stream0 + r < self.nm:
                self.model.push(stream0 + r, x[r])

    def push_list(self, streams, rows):
        self.ctx.push_streams(streams, rows)
        for s, r in zip(streams, rows):
            if s < self.nm:
                self.model.push(s, r)

    def push_resampled(self, x, sr):
        """K8: the landed 16 kHz samples are read back from the ring (K8 itself is pinned by its own tests)"""
        before = [self.ctx.status(s).written for s in range(self.nm)]
        landed = self.ctx.push_resampled(x, sr)
        for s in range(self.nm if landed else 0):
            y = self.ctx.read_segment(s, before[s], landed)
            self.model.push(s, synth.to_int16(y) if self.fmt == "i16" else y)
        return landed

    def _poll(self):
        e = self.ctx.poll().copy()
        self.dropped += self.ctx.dropped
        self.events.append(e)

    def _check_trace(self, tr, mt, paced):
        n = self.nm
        for k in ("silent", "state"):
            a = tr[k][:n]
            b = mt[k] if paced else (mt[k].astype(bool) if k == "silent" else mt[k])
            assert np.array_equal(a, b), (k, np.argwhere(a != b)[:5])
        for k in ("thr", "rms"):
            a, b = _bits(tr[k][:n]), _bits(mt[k])
            assert np.array_equal(a, b), (k, np.argwhere(a != b)[:5], tr[k][:n][a != b][:3], mt[k][a != b][:3])
        self.cells += mt["thr"].size

    def tick(self, n, trace=True, poll=True):
        if trace:
            tr = self.ctx.tick(n, trace=True)
        else:
            self.ctx.tick(n)
        _, mt = self.model.tick(n)
        if trace:
            self._check_trace(tr, mt, False)
        if poll:
            self._poll()

    def ready(self, n):
        taken, tr = self.ctx.tick_ready(n, trace=True)
        mtaken, mt = self.model.tick(n, paced=True)
        assert np.array_equal(taken[:self.nm], mtaken)
        self._check_trace(tr, mt, True)
        self._poll()
        return taken

    def reset(self, streams):
        self.ctx.reset_streams(streams)
        self.model.reset([s for s in streams if s < self.nm])

    def check(self, exact_events=True):
        """events, status and result flags of the modelled streams"""
        ev = np.concatenate(self.events) if self.events else np.zeros(0, self.L.EVENT_DTYPE)
        ev = ev[ev["stream"] < self.nm]
        dev = np.stack([ev["stream"], ev["kind"], ev["tick"], ev["seg_start"], ev["seg_len"]], 1).astype(np.int64)
        dev = dev[np.lexsort((dev[:, 1], dev[:, 2], dev[:, 0]))] if len(dev) else dev.reshape(0, 5)
        mod = self.model.event_array()
        if exact_events:
            assert np.array_equal(dev, mod), (dev[:8], mod[:8])
        res = self.ctx.results()
        for s in range(self.nm):
            st, ms = self.ctx.status(s), self.model.status(s)
            for f, _ in st._fields_:
                a, b = getattr(st, f), ms[f]
                if isinstance(b, float):
                    assert _bits([a])[0] == _bits([b])[0], (s, f, a, b)
                elif exact_events or f != "n_events":
                    assert a == b, (s, f, a, b)
            if exact_events:
                assert int(res["flags"][s]) & ~1 == self.model.flags(s), (s, hex(int(res["flags"][s])), hex(self.model.flags(s)))
        return dev, mod

    def close(self):
        self.ctx.close()


def _params(fs=1600, **kw):
    p = dict(frame_size=fs, timeout=4.0, speech_duration_min=0.3, speech_duration_max=2.0)
    p.update(kw)
    return p


# ------------------------------------------------------------------------------------ sum sources x formats
@pytest.mark.parametrize("fmt", ["i16", "f32"])
@pytest.mark.parametrize("source", ["presummed", "staged", "generic", "list", "native"])
def test_sum_sources(source, fmt, word):
    n = 6
    if source == "generic":
        R, slack = 16000, 2000                                  # P = 18048: blocks straddle the physical wrap
    else:
        R, slack = 16000, 16000                                 # P = 32000 = 20 blocks
    pr = Pair(R, slack, fmt, [_params(timeout=3.0 + 0.1 * i) for i in range(n)])
    x = feed(11, n, 14.0, fmt, word)
    try:
        if source == "presummed":                              # 1 s device pushes: K1's fused sums, K2 reads none
            for b in range(0, x.shape[1], 16000):
                pr.push(x[:, b:b + 16000], device=True)
                pr.tick(10)
        elif source == "staged":                               # half-tick pushes: no sums, K2 stages its ticks
            for b in range(0, x.shape[1], 8000):
                for h in range(0, 8000, 800):
                    pr.push(x[:, b + h:b + h + 800])
                pr.tick(5)
        elif source == "generic":
            for b in range(0, x.shape[1], 1600):
                pr.push(x[:, b:b + 1600])
                pr.tick(1)
        elif source == "list":                                 # K1L rows of ragged lengths, ticks paced by the audio
            rng = np.random.default_rng(3)
            pos = np.zeros(n, np.int64)
            while (pos < x.shape[1]).any():
                ln = np.minimum(rng.integers(0, 9000, n), x.shape[1] - pos)
                pr.push_list(list(range(n)), [x[s, pos[s]:pos[s] + ln[s]] for s in range(n)])
                pos += ln
                pr.ready(7)
        else:                                                  # K8 at 48 kHz
            x48 = np.repeat(x.astype(np.float32) / (32768.0 if fmt == "i16" else 1.0), 3, axis=1).astype(np.float32)
            for b in range(0, x48.shape[1], 24000):
                pr.push_resampled(np.ascontiguousarray(x48[:, b:b + 24000]), 48000)
                pr.ready(16)
        dev, _ = pr.check()
        assert pr.cells >= n * 130 and (dev[:, 1] == G.EV_SCORED).sum() + (dev[:, 1] == G.EV_TIMEOUT).sum() >= 6
    finally:
        pr.close()


@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_tma_push_form(fmt, word):
    """overlap mode, 160 streams x 1 s device pushes (1600 blocks >= 4 x SMs x 2 warps): the pushes that run beside K3
    take K1's cp.async.bulk form; its sums feed K2 (presummed).  Traced ticks would keep K3 off the side stream, so the
    comparison is the final state of the first 12 streams"""
    n = 160
    pr = Pair(96000, 16000, fmt, [_params(timeout=5.0)] * n, n_model=12)
    x = feed(23, 12, 14.0, fmt, word)
    x = np.concatenate([x] * (n // 12 + 1))[:n]
    pr.ctx.set_overlap(True)
    try:
        for b in range(0, x.shape[1], 16000):
            pr.push(x[:, b:b + 16000], device=True)
            pr.tick(10, trace=False, poll=False)             # a poll would join K3: the next push would not overlap it
        pr._poll()
        dev, _ = pr.check()
        assert (dev[:, 1] == G.EV_SCORED).sum() >= 4
    finally:
        pr.close()


# ------------------------------------------------------------------------------------ frame sizes
@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_mixed_frame_sizes_in_one_cta(fmt, word):
    """333 (tail, odd starts: scalar paths), 512, 1000 (chunks straddle ticks), 1600, 4800 (ticks with no new samples),
    fs == R (one chunk), and frame size 0 latched by a first push of 640 — seven streams, so CTAs mix chunk counts"""
    R = 16000
    fss = [333, 512, 1000, 1600, 4800, R, 0]
    pr = Pair(R, 24000, fmt, [_params(fs) for fs in fss])         # frame size R holds up to R + a push un-gated
    x = feed(31, len(fss), 12.0, fmt, word)
    try:
        pr.push(x[6:7, :640], stream0=6)
        pr.push(x[:6, :640])
        for b in range(640, x.shape[1] - 4800, 4800):
            pr.push(x[:, b:b + 4800])
            pr.tick(3)
        pr.tick(2)
        pr.check()
        assert pr.model.status(6)["frame_size"] == 640
    finally:
        pr.close()


@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_few_chunks(fmt, word):
    """n_chunks 1..5: every fractional class of the percentile's virtual index"""
    R = 16000
    fss = [16000, 8000, 5333, 4000, 3200]
    pr = Pair(R, 24000, fmt, [_params(fs) for fs in fss])
    x = feed(37, len(fss), 10.0, fmt, word)
    try:
        for b in range(0, x.shape[1], 8000):
            pr.push(x[:, b:b + 8000])
            pr.tick(5)
        pr.check()
    finally:
        pr.close()


@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_2048_chunks(fmt, word):
    """frame size 160 at R = 327680: 2048 chunks, what a K2 warp holds in shared memory (the two-buffer replace of more
    than 128 chunks); 2049 are refused"""
    R = 327680
    pr = Pair(R, 32000, fmt, [_params(160, timeout=30.0), _params(1600), _params(160, timeout=30.0)])
    x = feed(41, 3, 23.0, fmt, word)
    try:
        pr.push(x[:, :R])
        pr.tick(R // 1600)
        for b in range(R, x.shape[1], 3200):
            pr.push(x[:, b:b + 3200])
            pr.tick(2)
        pr.check()
    finally:
        pr.close()
    L = _lib()
    ctx = L.Context(device=0, n_streams=1, ring_samples=R + 160, slack_samples=16000, pcm_format=L.PCM_I16)
    try:
        ctx.set_stream_params(0, frame_size=160)
        ctx.push(np.zeros((1, 1600), np.int16))
        with pytest.raises(ValueError, match="2049 chunks"):
            ctx.tick(1)
    finally:
        ctx.close()


# ------------------------------------------------------------------------------------ geometry
GEOMETRY = [(16000, 16000, 0), (16800, 2400, 0), (16800, 16000, 0), (20000, 2400, 0), (20000, 800, 1), (24800, 2400, 0),
            (24800, 16000, 0)]


@pytest.mark.parametrize("fmt", ["i16", "f32"])
@pytest.mark.parametrize("R,slack,live", GEOMETRY)
def test_ring_geometry(R, slack, live, fmt, word):
    """rings that are not whole ticks (the tick whose new samples cover the tail and the start of chunk 0), P % 1600 == 0
    (whole-tick pushes: presummed; half-tick pushes: staged) and not (generic), live streams at slack 800"""
    n = 5
    pr = Pair(R, slack, fmt, [_params(live=live, timeout=3.0)] * n)
    x = feed(R + slack, n, 9.0, fmt, word)
    try:
        for b in range(0, 4 * 16000, 1600):                    # whole ticks
            pr.push(x[:, b:b + 1600])
            pr.tick(1)
        for b in range(4 * 16000, x.shape[1], 1600):           # half ticks
            pr.push(x[:, b:b + 800])
            pr.push(x[:, b + 800:b + 1600])
            pr.tick(1)
        pr.check()
    finally:
        pr.close()


# ------------------------------------------------------------------------------------ pacing
@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_pacing(fmt, word):
    """1 / 16 / 17 / 40 ticks per call, ticks that run ahead of the audio and catch up (by more than GATE_MAXP chunks at
    frame size 160, and by more than a whole ring), a live stream, paced calls with ragged budgets, and a reset"""
    R = 16000
    fss = [1600, 160, 512, 1000, 333]
    params = [_params(fs, timeout=2.5) for fs in fss] + [_params(1600, live=1)]
    n = len(params)
    pr = Pair(R, 40000, fmt, params)
    x = feed(53, n, 30.0, fmt, word)
    pos = 0
    try:
        def push(m):
            nonlocal pos
            pr.push(x[:, pos:pos + m])
            pos += m
        push(24000)
        push(24000)
        pr.tick(17)
        pr.tick(16)
        pr.tick(1)
        push(16000)
        pr.tick(40)                                            # runs ahead: the audio covers 6 of the 40 ticks
        push(R + 4800)                                         # catching up: a jump of more than a whole ring
        pr.tick(1)
        push(3200)
        pr.tick(1)                                             # 2 ticks behind the clock: frame size 160 -> 20+ chunks
        push(4000)
        pr.ready(3)
        pr.reset([2, 5])
        for step in range(12):
            m = [1600, 2400, 6400, 800, 3200, 1600][step % 6]
            push(m)
            pr.ready(16 if step % 3 else 5)
        for k in (1, 16, 17):
            push(k * 1600)
            pr.tick(k)
        pr.check()
    finally:
        pr.close()


@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_ragged_budgets(fmt, word):
    """ewk_tick_ready over streams with different amounts of audio: a different budget per stream in one call"""
    n = 9
    pr = Pair(16000, 64000, fmt, [_params(1600 if i % 3 else 1000) for i in range(n)])
    x = feed(59, n, 16.0, fmt, word)
    rng = np.random.default_rng(59)
    pos = np.zeros(n, np.int64)
    try:
        for step in range(14):
            ln = np.minimum(rng.integers(0, 16000, n) * (rng.random(n) < 0.7), x.shape[1] - pos)
            pr.push_list(list(range(n)), [x[s, pos[s]:pos[s] + ln[s]] for s in range(n)])
            pos += ln
            pr.ready(40 if step % 2 else 9)
        pr.check()
    finally:
        pr.close()


# ------------------------------------------------------------------------------------ ties, duplicates, segment edges
def blocks(levels, n=1600):
    return np.concatenate([np.full(n, v, np.int16) for v in levels])


def _as(fmt, q):
    return q if fmt == "i16" else synth.from_int16(q)


@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_ties_and_duplicates(fmt):
    """rms == thr == 3/32768 (constants 2 and 3), 1.5 P25 == min_threshold, digital silence, a feed whose period is the
    ring (every replacement equal), replacements inside runs of equal values, and each duration compare at its edge and
    one double past it"""
    from test_gate_model import DUR_EDGES, duration_feed, duration_params
    R = 16000
    rng = np.random.default_rng(61)
    period = (rng.standard_normal(R) * 2000).astype(np.int16)
    feeds, params = [], []
    lv = [2] * 10 + [3] + [2] * 4 + [3, 3, 2, 2, 3] * 4
    feeds.append(blocks(lv)); params.append(_params(min_threshold=0.0))
    feeds.append(blocks([2] * 35)); params.append(_params(min_threshold=3 / 32768))
    feeds.append(np.zeros(35 * 1600, np.int16)); params.append(_params())
    feeds.append(np.tile(period, 4)[:35 * 1600]); params.append(_params(min_threshold=0.0))
    feeds.append(blocks([5] * 6 + [7] * 6 + [5] * 6 + [9] * 3 + [5] * 14)); params.append(_params(min_threshold=0.0))
    for name in sorted(DUR_EDGES):
        for side in (0, 1):
            feeds.append(blocks(duration_feed())); params.append(dict(duration_params(name, side), timeout=30.0))
    N = min(len(f) for f in feeds)
    x = np.stack([_as(fmt, f[:N]) for f in feeds])
    pr = Pair(R, 16000, fmt, params)
    try:
        for b in range(0, N, 1600):
            pr.push(x[:, b:b + 1600])
            pr.tick(1)
        dev, _ = pr.check()
        assert (dev[:, 1] == G.EV_SCORED).sum() >= 4
        assert pr.model.s[0].thr == 3 / 32768
    finally:
        pr.close()


@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_segment_cut_edges(fmt):
    """n_back > R on a short ring (clamped), len < 1 (no event), len > 48000 (no event), timeouts"""
    cases = []
    # R = 16000: 1.5 s of sound -> n_back = (1.5 + 0.4 + 0.05) * 16000 > R
    cases.append((16000, [0] * 20 + [1000] * 15 + [0] * 10, _params(pre_speech_silence=0.5, post_speech_silence=0.4)))
    # post_speech_silence 1.2 at R = 16000: n_drop > n_back -> len < 1
    cases.append((16000, [0] * 20 + [1000] * 5 + [0] * 20, _params(pre_speech_silence=0.5, post_speech_silence=1.2)))
    # R = 80000: 3.2 s of sound with speech_duration_max 4 -> len > 48000
    cases.append((80000, [0] * 60 + [1000] * 32 + [0] * 10 + [1000] * 10 + [0] * 10,
                  _params(pre_speech_silence=0.4, speech_duration_max=4.0)))
    # timeouts every 1.5 s
    cases.append((16000, [0] * 12 + ([1000] * 3 + [0] * 9) * 4, _params(pre_speech_silence=0.5, timeout=1.5)))
    n_ev = 0
    for R, lv, p in cases:
        pr = Pair(R, 16000, fmt, [p] * 3)
        x = np.stack([_as(fmt, blocks(lv))] * 3)
        try:
            for b in range(0, x.shape[1], 1600):
                pr.push(x[:, b:b + 1600])
                pr.tick(1)
            dev, mod = pr.check()
            n_ev += len(dev)
        finally:
            pr.close()
    assert n_ev >= 6


def test_queue_overflow(word):
    """more candidates in one call than the queue holds: which are kept depends on atomics, so only events + dropped
    is compared with the model's count"""
    n = 40
    pr = Pair(16000, 160000, "i16", [_params(1600, timeout=1.0, pre_speech_silence=0.3)] * n, max_events=16)
    lv = ([0] * 6 + [1000] * 4) * 10
    x = np.stack([blocks(lv)] * n)
    try:
        pr.push(x[:, :160000])
        pr.tick(100)
        dev, mod = pr.check(exact_events=False)
        assert len(mod) > 16 and len(dev) <= 16 and len(dev) + pr.dropped == len(mod)
    finally:
        pr.close()
