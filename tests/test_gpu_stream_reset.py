"""Stream recycling (ewk_reset_streams, K9) and native-rate pushes with streams at their own input positions
(ewk_push_resampled_each).  A reset stream must behave exactly like the same stream of a new context given the same
calls from then on; the streams that were not reset exactly like a run without the reset."""
import math

import numpy as np
import pytest

from easywakeword_b200 import synth
from easywakeword_b200.resample import ALAW_TABLE, ULAW_TABLE, landed_counts

N, RING_S = 12, 5
RESET = [0, 3, 4, 8, 11]                       # non-contiguous, with the first and the last stream


def _lib():
    from easywakeword_b200 import _lib as L
    return L


def _ctx(ring, n=N, word=None, **prm):
    L = _lib()
    ctx = L.Context(device=0, n_streams=n, ring_samples=RING_S * 16000, slack_samples=2 * 16000,
                    pcm_format=L.PCM_I16 if ring == "i16" else L.PCM_F32, max_templates=1, max_events=4096)
    if word is not None:
        ctx.set_template(0, word)
    ctx.set_stream_params(-1, speech_duration_min=0.5, speech_duration_max=1.6, timeout=4.0, **prm)
    return ctx


def _encode(q, law):
    """16-bit samples -> nearest G.711 code."""
    table = (ULAW_TABLE if law == "ulaw" else ALAW_TABLE).astype(np.int32)
    order = np.argsort(table, kind="stable")
    srt = table[order]
    i = np.clip(np.searchsorted(srt, q.astype(np.int32)), 1, 255)
    pick = np.where(np.abs(srt[i] - q) < np.abs(srt[i - 1] - q), i, i - 1)
    return order[pick].astype(np.uint8)


def _audio(kind, ring, word, seed, secs):
    """[N, secs * rate] feed of `kind`: ("pcm",) 16 kHz in the ring's dtype, ("g711",) 16 kHz mu-law codes, or
    ("rs", sr, fmt) native-rate f32 / i16 / ulaw."""
    from scipy.signal import resample_poly
    pcm = synth.stream_batch(seed, N, float(secs), word, as_int16=False, gain=(2.0, 4.0))
    if kind[0] == "pcm":
        return synth.to_int16(pcm) if ring == "i16" else pcm
    if kind[0] == "g711":
        return _encode(synth.to_int16(pcm), "ulaw")
    sr, fmt = kind[1], kind[2]
    g = math.gcd(sr, 16000)
    y = np.clip(resample_poly(pcm.astype(np.float64), sr // g, 16000 // g, axis=1), -0.99, 0.99)
    if fmt == "f32":
        return np.ascontiguousarray(y, dtype=np.float32)
    q = synth.to_int16(y)
    return q if fmt == "i16" else _encode(q, fmt)


def _rate(kind):
    return kind[1] if kind[0] == "rs" else 16000


def _push(ctx, kind, x, stream0, pinned=False):
    """One push call of rows x onto streams [stream0, stream0 + len(x)); -> landed count per stream."""
    L = _lib()
    x = np.ascontiguousarray(x)
    buf = None
    if pinned:
        buf = L.PinnedArray(x.shape, x.dtype)
        buf.array[...] = x
        x = buf.array
    if kind[0] == "pcm":
        ctx.push(x, stream0=stream0)
        out = np.full(len(x), x.shape[1], np.int64)
    elif kind[0] == "g711":
        ctx.push_g711(x, stream0=stream0)
        out = np.full(len(x), x.shape[1], np.int64)
    else:
        out = ctx.push_resampled_each(x, kind[1], stream0=stream0, fmt=kind[2] if kind[2] in ("ulaw", "alaw") else None)
    return out, buf


def _runs(kinds):
    """contiguous runs of streams with the same feed kind: [(stream0, n, kind)]"""
    out, s0 = [], 0
    for s in range(1, len(kinds) + 1):
        if s == len(kinds) or kinds[s] != kinds[s0]:
            out.append((s0, s - s0, kinds[s0]))
            s0 = s
    return out


class Log:
    """A context and what its ticks and polls returned.  Traced ticks run K3 behind the gate, so a context in overlap
    mode ticks without traces."""

    def __init__(self, ctx, traced=True):
        self.ctx, self.traced, self.events = ctx, traced, []
        self.trace = {k: [] for k in ("thr", "rms", "silent", "state")} if traced else {}

    def tick(self, n):
        if n > 0:
            tr = self.ctx.tick(n, trace=self.traced)
            for k in self.trace:
                self.trace[k].append(tr[k])

    def poll(self):
        self.events.append(self.ctx.poll().copy())

    def state(self, streams):
        ctx = self.ctx
        ev = np.concatenate(self.events) if self.events else np.zeros(0, _lib().EVENT_DTYPE)
        ev = ev[np.isin(ev["stream"], streams)]
        tr = {k: np.concatenate(v, axis=1)[streams] for k, v in self.trace.items()}
        st = [tuple(getattr(ctx.status(s), f[0]) for f in ctx.status(s)._fields_) for s in streams]
        return dict(ev=ev, tr=tr, status=st, res=ctx.results()[streams], inp=[ctx.stream_input(s) for s in streams],
                    ring=np.stack([ctx.read_last(s, RING_S * 16000) for s in streams]))


def _assert_same(a, b):
    assert len(a["ev"]) == len(b["ev"])
    for f in a["ev"].dtype.names:
        x, y = a["ev"][f], b["ev"][f]
        if x.dtype.kind == "f":
            x, y = x.view(np.int32), y.view(np.int32)                  # scores by bits
        assert np.array_equal(x, y), f
    assert np.array_equal(a["res"].view(np.int32), b["res"].view(np.int32))
    assert a["status"] == b["status"]
    assert a["inp"] == b["inp"]
    assert np.array_equal(a["ring"], b["ring"])
    assert a["tr"].keys() == b["tr"].keys()
    for k in ("silent", "state"):
        if k in a["tr"]:
            assert np.array_equal(a["tr"][k], b["tr"][k]), k
    for k in ("thr", "rms"):
        if k not in a["tr"]:
            continue
        # bit for bit on either ring format: whether one context's K1 formed block sums and the other's gate summed the
        # samples itself, a block's squares add in one order (oracle/gate_model.py)
        assert np.array_equal(a["tr"][k].view(np.int64), b["tr"][k].view(np.int64)), k


PCM, G711 = ("pcm",), ("g711",)
U8K, I48K, I44K = ("rs", 8000, "ulaw"), ("rs", 48000, "i16"), ("rs", 44100, "i16")
CASES = {
    "pcm16-i16": dict(ring="i16", pre=PCM),
    "pcm16-f32": dict(ring="f32", pre=PCM),
    "g711-16k": dict(ring="i16", pre=G711),
    "ulaw-8k": dict(ring="i16", pre=U8K),
    "i16-48k-into-f32": dict(ring="f32", pre=I48K),
    "i16-44k1": dict(ring="i16", pre=I44K),
    "48k-then-8k": dict(ring="i16", pre=I48K, post=U8K),
    "native-then-16k": dict(ring="i16", pre=I48K, post=PCM),
    "frame-size-0": dict(ring="i16", pre=PCM, prm=dict(frame_size=0), post_secs=0.8),
    "live": dict(ring="i16", pre=U8K, prm=dict(live=1)),
    "overlap": dict(ring="i16", pre=PCM, overlap=True),
    "pinned-pending": dict(ring="i16", pre=U8K, pending=True),
    "between-push-and-tick": dict(ring="f32", pre=PCM, between=True),
    "all-streams": dict(ring="i16", pre=U8K, reset=list(range(N))),
}


def _scenario(word, ring, pre, post=None, prm=None, overlap=False, pending=False, between=False, reset=RESET,
              pre_steps=9, post_steps=14, post_secs=1.0, publish=False):
    """A: pre-phase, reset, post-phase.  B: a new context given A's post-phase calls.  C: A without the reset."""
    post = post or pre
    prm = prm or {}
    keep = [s for s in range(N) if s not in reset]
    ctxs = [_ctx(ring, word=word, **prm) for _ in range(3 if keep else 2)]
    dests, pins = [], []
    try:
        if overlap:
            for c in ctxs:
                c.set_overlap(True)
        A, B = Log(ctxs[0], not overlap), Log(ctxs[1], not overlap)
        C = Log(ctxs[2], not overlap) if keep else None
        x_pre = _audio(pre, ring, word, 7100, pre_steps + 1)
        k_pre = _rate(pre)
        clock, ticks = 0, 0
        for step in range(pre_steps + (1 if pending or between else 0)):
            last = step == pre_steps
            for lg in [A, C] if C else [A]:
                m, buf = _push(lg.ctx, pre, x_pre[:, step * k_pre:(step + 1) * k_pre], 0, pinned=last and pending)
                pins.append(buf)
            clock += int(m.max())
            if not last:
                lg_due = clock // 1600 - ticks
                for lg in [A, C] if C else [A]:
                    lg.tick(lg_due)
                ticks += lg_due
        for lg in [A, C] if C else [A]:
            lg.poll()
        n_before = sum(len(e) for e in A.events)
        assert n_before > 0
        for lg in [A, C] if C else [A]:                                # compare the post-phase only
            lg.events, lg.trace = [], {k: [] for k in lg.trace}
        if publish:
            import torch
            for c in (A.ctx, B.ctx):
                d = torch.full((2, N, 2), -7, dtype=torch.int32, device="cuda:0")
                c.set_results_peers([d.data_ptr()], stride_records=N, offset_records=0)
                dests.append(d)
        A.ctx.reset_streams(reset)
        # post-phase: the same calls to A, B and C (C skips feeds at a rate its old sessions do not take)
        kinds = [post if s in reset else pre for s in range(N)]
        x_post = {k: _audio(k, ring, word, 9100, math.ceil(post_steps * post_secs) + 1) for k in set(kinds)}
        clock, ticks = 0, 0
        if between or pending:                                         # the old sessions' last, un-ticked push
            for lg in [A, B, C] if C else [A, B]:
                lg.tick(10)
            clock, ticks = 16000, 10
        for step in range(post_steps):
            landed = np.zeros(N, np.int64)
            for s0, n, kind in _runs(kinds):
                k = int(round(_rate(kind) * post_secs))
                rows = x_post[kind][s0:s0 + n, step * k:(step + 1) * k]
                landed[s0:s0 + n], _ = _push(A.ctx, kind, rows, s0)
                _push(B.ctx, kind, rows, s0)
                if C and kind == pre:
                    _push(C.ctx, kind, rows, s0)
            clock += int(landed.max())
            due = max(0, clock // 1600 - ticks)
            for lg in [A, B, C] if C else [A, B]:
                lg.tick(due)
                lg.poll()
            ticks += due
        got = A.state(reset)
        _assert_same(got, B.state(reset))
        if C:
            _assert_same(A.state(keep), C.state(keep))
        assert len(got["ev"]) >= 2                                     # the new sessions produced events
        if publish:
            recs = []
            for lg, d in zip((A, B), dests):
                lg.ctx.results()                                       # joins K3 and synchronises
                h = d.cpu().numpy()
                recs.append(h[lg.ctx.publish_parity(), reset])
            assert np.array_equal(recs[0], recs[1])
            assert np.array_equal(recs[0], B.ctx.results()[reset].view(np.int32).reshape(-1, 2))
        return got
    finally:
        for c in ctxs:
            if publish:
                c.set_results_peers([])
            c.close()
        for b in pins:
            if b is not None:
                b.free()


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
def test_reset_equals_new_context(word, case):
    _scenario(word, **CASES[case])


@pytest.mark.gpu
def test_published_records_after_reset(word):
    _scenario(word, ring="i16", pre=PCM, publish=True)


@pytest.mark.gpu
def test_dense_after_reset_uses_no_stale_rows(word):
    """K4 carries the newest grid rows of a stream between calls; after a reset they belong to the old session."""
    x = synth.stream_batch(4300, 1, 9.0, word, gain=(2.0, 4.0))
    y = synth.stream_batch(4400, 1, 9.0, word, gain=(2.0, 4.0))
    A, B = _ctx("i16", n=1, word=word, live=1), _ctx("i16", n=1, word=word, live=1)
    try:
        A.push(np.ascontiguousarray(x[:, :64000]))
        A.dense_scores(300, 100)                                       # carries rows up to hop 399 of the old session
        A.reset_streams([0])
        for c in (A, B):
            c.push(np.ascontiguousarray(y[:, :72000]))
        a, b = A.dense_scores(400, 40), B.dense_scores(400, 40)        # the carried range would serve this window
        assert np.array_equal(a.view(np.int32), b.view(np.int32))
        assert np.isfinite(a).all()
    finally:
        A.close()
        B.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sr,fmt,device", [(8000, "ulaw", False), (44100, "i16", False), (48000, "i16", True),
                                           (48000, "f32", False)])
def test_each_equals_group_pushes(word, sr, fmt, device):
    import torch
    L = _lib()
    kind = ("rs", sr, fmt)
    x = _audio(kind, "i16", word, 5500, 3)[:8]
    k1, k2, n_in = sr // 3 + 17, sr // 2 + 5, sr // 2 + 123
    # streams 0-1 never pushed, 2-4 at k1, 5-7 at k1 + k2
    hist = [((2, 3), [x[:, :k1]]), ((5, 3), [x[:, :k1], x[:, k1:k1 + k2]])]
    pos = np.array([0, 0, k1, k1, k1, k1 + k2, k1 + k2, k1 + k2])
    new = np.ascontiguousarray(x[:, k1 + k2:k1 + k2 + n_in])
    new2 = np.ascontiguousarray(x[:, k1 + k2 + n_in:k1 + k2 + 2 * n_in])
    g711 = fmt if fmt in ("ulaw", "alaw") else None
    X, Y = _ctx("i16", n=8, live=1), _ctx("i16", n=8, live=1)
    pinned = None
    try:
        for c in (X, Y):
            for (s0, n), chunks in hist:
                for ch in chunks:
                    c.push_resampled(np.ascontiguousarray(ch[s0:s0 + n]), sr, stream0=s0, fmt=g711)
            c.status(0)                                                # lands the last of them
        X.profile(True)
        before = X.launch_count()
        if device:
            t = torch.from_numpy(new).cuda()
            landed = X.push_resampled_each((t.data_ptr(), 8, n_in, n_in, new.dtype), sr, fmt=g711, where=L.DEVICE)
            torch.cuda.synchronize()
        else:
            pinned = PinnedCopy(new)
            landed = X.push_resampled_each(pinned.array, sr, fmt=g711)
        X.status(0)                                                    # lands a pending host push
        assert X.launch_count() - before == 1                          # one K8 for all positions
        assert X.profile_read()["resample_push"]["launches"] == 1
        assert landed.tolist() == landed_counts(pos, n_in, sr).tolist()
        ref = []
        for s0, n in [(0, 2), (2, 3), (5, 3)]:                          # one call per group of equal positions
            ref += [Y.push_resampled(np.ascontiguousarray(new[s0:s0 + n]), sr, stream0=s0, fmt=g711)] * n
        assert landed.tolist() == ref
        # a second push: the tails K8 left behind must be the groups' tails as well
        l2 = X.push_resampled_each(new2, sr, fmt=g711)
        for s0, n in [(0, 2), (2, 3), (5, 3)]:
            Y.push_resampled(np.ascontiguousarray(new2[s0:s0 + n]), sr, stream0=s0, fmt=g711)
        assert l2.tolist() == landed_counts(pos + n_in, n_in, sr).tolist()
        for s in range(8):
            w = X.status(s).written
            assert w == Y.status(s).written and X.stream_input(s) == Y.stream_input(s)
            assert np.array_equal(X.read_segment(s, 0, w).view(np.int32), Y.read_segment(s, 0, w).view(np.int32))
    finally:
        X.close()
        Y.close()
        if pinned is not None:
            pinned.buf.free()


class PinnedCopy:
    def __init__(self, a):
        self.buf = _lib().PinnedArray(a.shape, a.dtype)
        self.buf.array[...] = a
        self.array = self.buf.array


@pytest.mark.gpu
def test_each_errors(word):
    import ctypes as C
    L = _lib()
    ctx = _ctx("i16", n=4, live=1)
    try:
        ctx.push_resampled(np.zeros((2, 480), np.int16), 48000, stream0=0)
        with pytest.raises(L.EwkError, match="already takes 48000"):
            ctx.push_resampled_each(np.zeros((4, 160), np.uint8), 8000, fmt="ulaw")
        ctx.push(np.zeros((1, 320), np.int16), stream0=3)
        with pytest.raises(L.EwkError, match="already takes 16000"):
            ctx.push_resampled_each(np.zeros((2, 480), np.int16), 48000, stream0=2)
        with pytest.raises(ValueError, match="not a supported input rate"):
            ctx.push_resampled_each(np.zeros((1, 480), np.int16), 16000, stream0=2)
        z = np.zeros((1, 480), np.int16)
        rc = ctx.lib.ewk_push_resampled_each(ctx.h, 2, 1, z.ctypes.data, L.PCM_I16, 480, 480, L.HOST, 48000, None)
        assert rc == L.EWK_ERR_ARG and "landed" in ctx.lib.ewk_last_error(ctx.h).decode()
        # the same-position rule of ewk_push_resampled stays
        ctx.push_resampled(z, 48000, stream0=2)
        ctx.push_resampled(z, 48000, stream0=2)                        # streams 0, 1 at 480 inputs, stream 2 at 960
        with pytest.raises(L.EwkError, match="same position"):
            ctx.push_resampled(np.zeros((3, 480), np.int16), 48000, stream0=0)
        assert ctx.push_resampled_each(np.zeros((3, 480), np.int16), 48000, stream0=0).shape == (3,)
    finally:
        ctx.close()


@pytest.mark.gpu
def test_reset_errors(word):
    L = _lib()
    ctx = _ctx("i16", n=4, word=word)
    try:
        x = synth.stream_batch(600, 4, 12.0, word, gain=(2.0, 4.0))
        for b in range(0, x.shape[1], 16000):
            ctx.push(np.ascontiguousarray(x[:, b:b + 16000]))
            ctx.tick(10)
        assert ctx.status(0).n_events + ctx.status(1).n_events + ctx.status(2).n_events + ctx.status(3).n_events > 0
        with pytest.raises(L.EwkError, match="poll first"):
            ctx.reset_streams([1])
        assert len(ctx.poll()) > 0
        with pytest.raises(ValueError):
            ctx.reset_streams([4])
        with pytest.raises(ValueError):
            ctx.reset_streams([-1])
        rc = ctx.lib.ewk_reset_streams(ctx.h, None, 2)
        assert rc == L.EWK_ERR_ARG
        ctx.reset_streams([])                                          # no-op
        ctx.reset_streams([2, 2, 1])                                   # duplicates are harmless
        assert ctx.status(2).written == 0 and ctx.status(1).tick == 0 and ctx.status(0).tick > 0
    finally:
        ctx.close()
    empty = L.Context(device=0, n_streams=0)
    try:
        with pytest.raises(L.EwkError, match="n_streams = 0"):
            empty.reset_streams([0])
    finally:
        empty.close()


@pytest.mark.gpu
def test_bank_staggered_resets_8k(word):
    """An 8 kHz bank whose streams restart at different steps: one push (one K8) per step for the whole bank, and the
    recycled stream's events are those of a new one-stream bank given the same blocks and ticks."""
    from easywakeword_b200.bank import WakeWordBank
    kw = dict(buffer_seconds=5, speech_duration_min=0.5, speech_duration_max=1.6, timeout=4.0, sample_rate=8000)
    n, steps = 8, 26
    codes = _encode(synth.to_int16(np.clip(_resample(synth.stream_batch(3300, n, steps, word, as_int16=False,
                                                                         gain=(2.0, 4.0)), 8000), -0.99, 0.99)), "ulaw")
    big = WakeWordBank(n, [word], **kw)
    one = None
    try:
        big.ctx.profile(True)
        drained, mine = [], []
        for step in range(steps):
            blk = np.ascontiguousarray(codes[:, step * 8000:(step + 1) * 8000])
            if step == 9:
                drained.append(big.reset([2]))
            if step == 12:
                drained.append(big.reset([5], similarity_threshold=70.0))
                one = WakeWordBank(1, [word], **kw)
                one.set_stream(0, similarity_threshold=70.0)
            t0 = big.ticks
            big.push_g711(blk)
            due = big.samples_pushed // 1600 - big.ticks
            if due > 0:
                big.tick(due)
            ev = big.poll() if step not in (8, 11) else None             # events stay queued for the resets
            if one is not None:
                one.push_g711(np.ascontiguousarray(blk[5:6]))
                if big.ticks > t0:
                    one.tick(big.ticks - t0)
                mine.append((ev[ev["stream"] == 5], one.poll()))
        assert big.ctx.profile_read()["resample_push"]["launches"] == steps
        assert sum(len(d) for d in drained) > 0                        # reset handed back the queued events
        a = np.concatenate([m[0] for m in mine])
        b = np.concatenate([m[1] for m in mine])
        assert len(a) == len(b) >= 1
        for f in a.dtype.names:
            if f != "stream":
                x, y = a[f], b[f]
                if x.dtype.kind == "f":
                    x, y = x.view(np.int32), y.view(np.int32)
                assert np.array_equal(x, y), f
        assert big.status(5).written < big.status(0).written            # its own count, from the reset
        assert big.ctx.stream_input(5)[1] == (steps - 12) * 8000
    finally:
        big.close()
        if one is not None:
            one.close()


def _resample(pcm, sr):
    from scipy.signal import resample_poly
    g = math.gcd(sr, 16000)
    return resample_poly(pcm.astype(np.float64), sr // g, 16000 // g, axis=1)


# ------------------------------------------------------------------------------------------------ no GPU
def test_reset_exports_in_symbol_table():
    from easywakeword_b200 import _lib as L, build
    build.build()
    lib = L.load()
    for name in ("ewk_reset_streams", "ewk_push_resampled_each"):
        assert hasattr(lib, name) and name in lib._protos


def test_sharded_reset_routing():
    from easywakeword_b200.dist import local_streams, owner_of, shard_range
    n_total, world = 23, 4
    g = [22, 0, 5, 6, 11, 12, 17, 18, 6]
    seen = []
    for r in range(world):
        a, b = shard_range(n_total, world, r)
        loc = local_streams(g, n_total, world, r)
        assert loc == [s - a for s in g if a <= s < b]
        assert all(owner_of(a + i, n_total, world) == (r, i) for i in loc)
        seen += [a + i for i in loc]
    assert sorted(seen) == sorted(g)
    with pytest.raises(ValueError):
        local_streams([23], n_total, world, 0)


@pytest.mark.parametrize("sr", [8000, 44100, 48000])
def test_landed_counts_per_position(sr):
    """Per stream, a push lands ready(c + n) - ready(c): what a group push at that position lands, and consecutive
    pushes add up to ready of the total."""
    from easywakeword_b200 import _lib as L
    from easywakeword_b200.resample import ready_outputs
    W, up, down = L.resample_info(sr)
    rng = np.random.default_rng(sr)
    pos = np.array([0, 1, W - 1, W, W + 1] + [int(v) for v in rng.integers(0, 5 * sr, 40)])
    n_in = sr // 3 + 7
    got = landed_counts(pos, n_in, sr)
    for c, m in zip(pos, got):
        assert m == landed_counts([c], n_in, sr)[0] == ready_outputs(c + n_in, W, up, down) - ready_outputs(c, W, up, down)
    second = landed_counts(pos + n_in, n_in, sr)
    assert ((got + second) == [ready_outputs(c + 2 * n_in, W, up, down) - ready_outputs(c, W, up, down) for c in pos]).all()
