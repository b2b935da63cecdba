"""Native-rate ingest (ewk_push_resampled, K8): 8 / 44.1 / 48 kHz feeds converted to 16 kHz on the device as they land.
The rings must hold exactly what the two-step path gives — a one-shot ewk_resample of the whole feed, quantised like
the ring, pushed with ewk_push in the same per-call counts — and events, result records and gate traces must follow."""
import math

import numpy as np
import pytest

from easywakeword_b200 import synth
from easywakeword_b200.resample import ALAW_TABLE, ULAW_TABLE, ready_outputs

N_STREAMS, SECS, RING_S = 12, 24, 5


def _ctx(ring_fmt, n=N_STREAMS, word=None, **prm):
    from easywakeword_b200 import _lib
    ctx = _lib.Context(device=0, n_streams=n, ring_samples=RING_S * 16000, slack_samples=2 * 16000, pcm_format=ring_fmt,
                       max_templates=1, max_events=4096)
    if word is not None:
        ctx.set_template(0, word)
    ctx.set_stream_params(-1, speech_duration_min=0.5, speech_duration_max=1.6, **prm)
    return ctx


def _encode(q, law):
    """16-bit samples -> nearest G.711 code."""
    table = (ULAW_TABLE if law == "ulaw" else ALAW_TABLE).astype(np.int32)
    order = np.argsort(table, kind="stable")
    srt = table[order]
    i = np.clip(np.searchsorted(srt, q.astype(np.int32)), 1, 255)
    pick = np.where(np.abs(srt[i] - q) < np.abs(srt[i - 1] - q), i, i - 1)
    return order[pick].astype(np.uint8)


def _feed(word, sr, kind, n=N_STREAMS, seed=8300):
    """-> (what is pushed, the float32 values K7 reads from it): speech + word, brought to sr with resample_poly."""
    from scipy.signal import resample_poly
    pcm = synth.stream_batch(seed, n, float(SECS), word, as_int16=False, gain=(2.0, 4.0))
    g = math.gcd(sr, 16000)
    y = np.clip(resample_poly(pcm.astype(np.float64), sr // g, 16000 // g, axis=1), -0.99, 0.99)
    if kind == "f32":
        x = np.ascontiguousarray(y, dtype=np.float32)
        return x, x
    q = synth.to_int16(y)
    if kind == "i16":
        return q, q.astype(np.float32) / np.float32(32768)
    codes = _encode(q, kind)
    return codes, (ULAW_TABLE if kind == "ulaw" else ALAW_TABLE)[codes].astype(np.float32) / np.float32(32768)


def _chunks(sr, total):
    """Irregular push sizes: 20 ms packets, odd sizes, one 1-sample push, up to about 0.5 s."""
    cyc = [sr // 50, sr // 50, 1, 997, sr // 5 + 7, 3 * sr // 50 + 1, sr // 2 + 11]
    out, pos, i = [], 0, 0
    while pos < total:
        k = min(cyc[i % len(cyc)], total - pos)
        out.append(k)
        pos += k
        i += 1
    return out


def _run(ctx, pushes, trace=True):
    """pushes: list of callables, each pushing one call and returning its landed count.  Ticks as the landed audio
    allows.  -> (landed counts, events, results, thr trace, ring contents)."""
    landed, pushed, ticks, thr = [], 0, 0, []
    for push in pushes:
        m = push()
        landed.append(m)
        pushed += m
        due = pushed // 1600 - ticks
        if due > 0:
            tr = ctx.tick(due, trace=trace)
            if trace:
                thr.append(tr["thr"])
            ticks += due
    ev = ctx.poll().copy()
    res = ctx.results()
    ring = np.stack([ctx.read_last(s, RING_S * 16000) for s in range(ctx.cfg.n_streams)])
    return landed, ev, res, (np.concatenate(thr, axis=1) if thr else None), ring


def _reference(word, ring_fmt, sr, xf, landed, first_frame):
    """Two-step path: one-shot resample of the whole feed, quantised like the ring, pushed in the same counts."""
    from easywakeword_b200 import _lib
    ctx = _ctx(ring_fmt, word=word, frame_size=first_frame)
    y = ctx.resample(xf, sr)
    ring_y = synth.to_int16(y) if ring_fmt == _lib.PCM_I16 else y
    pos = [0]

    def push(m):
        def f():
            if m:
                ctx.push(np.ascontiguousarray(ring_y[:, pos[0]:pos[0] + m]))
            pos[0] += m
            return m
        return f
    try:
        return _run(ctx, [push(m) for m in landed]), ring_y
    finally:
        ctx.close()


def _assert_same(a, b):
    (l0, e0, r0, t0, g0), (l1, e1, r1, t1, g1) = a, b
    assert l0 == l1
    assert np.array_equal(g0, g1)
    assert len(e0) == len(e1)
    for f in e0.dtype.names:
        assert np.array_equal(e0[f], e1[f], equal_nan=e0[f].dtype.kind == "f"), f
    for f in r0.dtype.names:
        assert np.array_equal(r0[f], r1[f], equal_nan=r0[f].dtype.kind == "f"), f
    if t0 is not None:
        # bit for bit on either ring format: K1's block sums (the reference's fused path) and K2's own sums of the
        # samples K8 landed add a block's squares in one order (oracle/gate_model.py)
        assert np.array_equal(np.asarray(t0, np.float64).view(np.int64), np.asarray(t1, np.float64).view(np.int64))


CASES = [(8000, "ulaw", "i16"), (8000, "alaw", "i16"), (8000, "i16", "i16"), (44100, "i16", "i16"), (48000, "f32", "f32"),
         (48000, "i16", "f32")]


@pytest.mark.gpu
@pytest.mark.parametrize("sr,kind,ring", CASES, ids=[f"{a}-{b}-into-{c}" for a, b, c in CASES])
def test_equals_two_step_path(word, sr, kind, ring):
    from easywakeword_b200 import _lib
    ring_fmt = _lib.PCM_I16 if ring == "i16" else _lib.PCM_F32
    x, xf = _feed(word, sr, kind)
    sizes = _chunks(sr, x.shape[1])
    fmt = kind if kind in ("ulaw", "alaw") else None
    ctx = _ctx(ring_fmt, word=word)
    pos = [0]

    def push(k):
        def f():
            m = ctx.push_resampled(x[:, pos[0]:pos[0] + k], sr, fmt=fmt)
            pos[0] += k
            return m
        return f
    try:
        got = _run(ctx, [push(k) for k in sizes])
        assert ctx.status(0).frame_size == _lib.load().ewk_resample_out_len(sizes[0], sr)
    finally:
        ctx.close()
    ref, ring_y = _reference(word, ring_fmt, sr, xf, got[0], int(_lib.load().ewk_resample_out_len(sizes[0], sr)))
    _assert_same(got, ref)
    assert (got[1]["kind"] == 2).sum() >= 6
    V = sum(got[0]) // 1600 * 1600                               # what the last tick saw (frame size 320)
    want = ring_y[:, V - RING_S * 16000:V]
    assert np.array_equal(got[4], want.astype(np.float32) / np.float32(32768) if ring == "i16" else want)


@pytest.mark.gpu
@pytest.mark.parametrize("sr,kind", [(8000, "ulaw"), (44100, "i16"), (48000, "f32")])
def test_counts_and_stream_input(word, sr, kind):
    from easywakeword_b200 import _lib
    from easywakeword_b200.resample import StreamResampler
    x, xf = _feed(word, sr, kind, n=2)
    x, xf = x[:, :3 * sr], xf[:, :3 * sr]
    rng = np.random.default_rng(sr)
    sizes = [sr // 10] + [int(v) for v in rng.integers(1, sr // 4, size=400)]
    ctx = _ctx(_lib.PCM_F32, n=2, live=1)
    rs = StreamResampler(sr, 2, ctx=ctx, dtype=np.float32)
    pos, total = 0, 0
    try:
        assert ctx.stream_input(0) == (0, 0)
        for k in sizes:
            if pos >= x.shape[1]:
                break
            m = ctx.push_resampled(x[:, pos:pos + k], sr, fmt=kind if kind in ("ulaw", "alaw") else None)
            emitted = rs.push(xf[:, pos:pos + k])
            pos += min(k, x.shape[1] - pos)
            total += m
            assert m == emitted.shape[1] == ready_outputs(pos, *_lib.resample_info(sr)) - (total - m)
            assert ctx.stream_input(1) == (sr, pos)
        assert ctx.status(0).frame_size == _lib.load().ewk_resample_out_len(sizes[0], sr)
        assert ctx.status(1).written == total
        whole = ctx.resample(xf[:, :pos], sr)[:, :total]
        n = min(total, RING_S * 16000)
        ctx.tick(1)
        for s in range(2):
            assert np.array_equal(ctx.read_last(s, n), whole[s, total - n:])
    finally:
        ctx.close()


@pytest.mark.gpu
def test_mixed_rate_bank(word):
    """Streams 0-5: 8 kHz G.711 mu-law, streams 6-11: 48 kHz int16, two calls per step into int16 rings."""
    from easywakeword_b200 import _lib
    h = N_STREAMS // 2
    xa, xfa = _feed(word, 8000, "ulaw", n=h, seed=8300)
    xb, xfb = _feed(word, 48000, "i16", n=h, seed=9100)
    steps = SECS * 5                                             # 200 ms per step
    ctx = _ctx(_lib.PCM_I16, word=word)
    ref = _ctx(_lib.PCM_I16, word=word, frame_size=3200)
    ya = synth.to_int16(ref.resample(xfa, 8000))
    yb = synth.to_int16(ref.resample(xfb, 48000))
    pa = pb = 0
    try:
        def step(i):
            ma = ctx.push_resampled(xa[:, i * 1600:(i + 1) * 1600], 8000, stream0=0, fmt="ulaw")
            mb = ctx.push_resampled(xb[:, i * 9600:(i + 1) * 9600], 48000, stream0=h)
            return ma, mb
        outs, ticks, la, lb = [], 0, 0, 0
        for i in range(steps):
            ma, mb = step(i)
            if ma:
                ref.push(np.ascontiguousarray(ya[:, la:la + ma]), stream0=0)
            if mb:
                ref.push(np.ascontiguousarray(yb[:, lb:lb + mb]), stream0=h)
            la += ma
            lb += mb
            due = min(la, lb) // 1600 - ticks
            if due > 0:
                for c in (ctx, ref):
                    outs.append(c.tick(due, trace=True)["thr"])
                ticks += due
        assert ctx.stream_input(0) == (8000, steps * 1600) and ctx.stream_input(h) == (48000, steps * 9600)
        assert ctx.status(0).frame_size == ctx.status(h).frame_size == 3200
        e0, e1 = ctx.poll(), ref.poll()
        assert len(e0) == len(e1) and (e0["kind"] == 2).sum() >= 6
        for f in e0.dtype.names:
            assert np.array_equal(e0[f], e1[f], equal_nan=e0[f].dtype.kind == "f"), f
        r0, r1 = ctx.results(), ref.results()
        assert r0.tobytes() == r1.tobytes()
        for a, b in zip(outs[0::2], outs[1::2]):
            assert np.array_equal(a, b)
        for s in range(N_STREAMS):
            assert np.array_equal(ctx.read_last(s, RING_S * 16000), ref.read_last(s, RING_S * 16000))
    finally:
        ctx.close()
        ref.close()


@pytest.mark.gpu
def test_overlap_and_device_feed_match(word):
    """Overlap mode on equals off (host pinned feed); a device-resident feed equals the host feed."""
    import torch
    from easywakeword_b200 import _lib
    sr = 48000
    x, _ = _feed(word, sr, "i16", n=8)
    pin = _lib.PinnedArray(x.shape, np.int16)
    pin.array[:] = x
    dev = torch.from_numpy(x).cuda()
    torch.cuda.synchronize()
    sizes = _chunks(sr, x.shape[1])
    outs = []
    for mode in ("pinned", "pinned-overlap", "device"):
        ctx = _ctx(_lib.PCM_I16, n=8, word=word)
        if mode == "pinned-overlap":
            ctx.set_overlap(True)
        pos = [0]

        def push(k, ctx=ctx, mode=mode):
            def f():
                p = pos[0]
                pos[0] += k
                if mode == "device":
                    return ctx.push_resampled((dev.data_ptr() + 2 * p, 8, k, x.shape[1], np.int16), sr, where=_lib.DEVICE)
                return ctx.push_resampled(pin.array[:, p:p + k], sr)
            return f
        try:
            outs.append(_run(ctx, [push(k) for k in sizes], trace=False))
        finally:
            ctx.close()
    pin.free()
    assert (outs[0][1]["kind"] == 2).sum() >= 4
    _assert_same(outs[0], outs[1])
    _assert_same(outs[0], outs[2])


@pytest.mark.gpu
def test_errors_leave_context_usable():
    from easywakeword_b200 import _lib
    ctx = _ctx(_lib.PCM_I16, n=4, live=1)
    z8 = np.zeros((1, 60), np.int16)                                             # fewer than W = 94 inputs at 8 kHz
    try:
        ctx.push(np.zeros((1, 320), np.int16), stream0=0)                       # stream 0: 16 kHz
        with pytest.raises(_lib.EwkError, match="already takes 16000"):
            ctx.push_resampled(z8, 8000, stream0=0)                              # resampled push onto a 16 kHz stream
        assert ctx.push_resampled(z8, 8000, stream0=1) == 0                      # stream 1: 8 kHz, nothing lands yet
        with pytest.raises(_lib.EwkError, match="ewk_push_resampled"):
            ctx.push(np.zeros((1, 320), np.int16), stream0=1)
        with pytest.raises(_lib.EwkError, match="ewk_push_resampled"):
            ctx.push_g711(np.zeros((1, 320), np.uint8), stream0=1)
        with pytest.raises(_lib.EwkError, match="already takes 8000"):
            ctx.push_resampled(np.zeros((1, 480), np.int16), 48000, stream0=1)   # another rate
        with pytest.raises(_lib.EwkError, match="same position"):
            ctx.push_resampled(np.zeros((2, 160), np.int16), 8000, stream0=1)    # streams 1 and 2 at different counts
        with pytest.raises(ValueError, match="not a supported input rate"):
            ctx.push_resampled(z8, 16000, stream0=2)
        with pytest.raises(ValueError, match="not a supported input rate"):
            ctx.push_resampled(z8, 44101, stream0=2)
        with pytest.raises(ValueError):
            ctx.push_resampled(z8.astype(np.uint8), 8000, stream0=2)             # uint8 without a G.711 law
        assert ctx.stream_input(2) == (0, 0) and ctx.stream_input(0) == (16000, 320)
        # still usable: stream 1 continues, stream 2 starts at 8 kHz, stream 0 takes 16 kHz pushes
        rng = np.random.default_rng(1)
        x = (rng.standard_normal((1, 4000)) * 3000).astype(np.int16)
        m = ctx.push_resampled(x, 8000, stream0=1)
        assert ctx.push_resampled(np.concatenate([z8, x], axis=1), 8000, stream0=2) == m
        ctx.push(np.zeros((1, 320), np.int16), stream0=0)
        ctx.tick(1)
        assert np.array_equal(ctx.read_last(1, m), ctx.read_last(2, m))
        assert ctx.stream_input(1) == ctx.stream_input(2) == (8000, 4060)
    finally:
        ctx.close()


# ------------------------------------------------------------------------------------------------ no GPU
def test_new_exports_in_symbol_table():
    from easywakeword_b200 import _lib, build
    build.build()
    lib = _lib.load()
    for name in ("ewk_push_resampled", "ewk_stream_input"):
        assert hasattr(lib, name) and name in lib._protos


@pytest.mark.parametrize("sr", [8000, 11025, 44100, 48000, 96000])
def test_landed_count_rule(sr):
    """ready_outputs(c), the rule StreamResampler emits by and ewk_push_resampled lands by, counts the outputs n with
    floor(n M / L) + W <= c - 1: all 2W taps of n are present after c inputs."""
    from easywakeword_b200 import _lib
    W, L, M = _lib.resample_info(sr)
    rng = np.random.default_rng(sr)
    for c in [0, 1, W - 1, W, W + 1, 2 * W + 3] + [int(v) for v in rng.integers(0, 10 * sr, 200)]:
        brute = 0 if c <= W else int(np.searchsorted(np.arange(c * L // M + L + 2) * M // L + W, c, side="left"))
        assert ready_outputs(c, W, L, M) == brute, c
