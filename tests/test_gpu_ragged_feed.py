"""Ragged list pushes (ewk_push_streams) and ticks paced by each stream's own audio (ewk_tick_ready).  The same audio must
give the same events, records, traces, status and rings however it was split into pushes, whatever the other streams
received; a slot that is not fed takes no ticks."""
import math

import numpy as np
import pytest

from easywakeword_b200 import synth
from easywakeword_b200.resample import ALAW_TABLE, ULAW_TABLE, due_ticks, landed_counts

N, RING_S, SECS = 12, 5, 12
MAXT = 24


def _lib():
    from easywakeword_b200 import _lib as L
    return L


def _ctx(ring, word, n=N, **prm):
    L = _lib()
    ctx = L.Context(device=0, n_streams=n, ring_samples=RING_S * 16000, slack_samples=2 * 16000,
                    pcm_format=L.PCM_I16 if ring == "i16" else L.PCM_F32, max_templates=1, max_events=4096)
    ctx.set_template(0, word)
    prm.setdefault("frame_size", 1600)       # frame_size 0 would latch each split's first row length
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


# feed kinds: (rate, format); format "ring" = the rings' dtype
PCM, G711 = (16000, "ring"), (16000, "ulaw")
U8K, F44K, I48K = (8000, "ulaw"), (44100, "f32"), (48000, "i16")


def _audio(kind, ring, word, seed, secs, n=N):
    from scipy.signal import resample_poly
    pcm = synth.stream_batch(seed, n, float(secs), word, as_int16=False, gain=(2.0, 4.0))
    sr, fmt = kind
    if sr != 16000:
        g = math.gcd(sr, 16000)
        pcm = np.clip(resample_poly(pcm.astype(np.float64), sr // g, 16000 // g, axis=1), -0.99, 0.99)
    if fmt == "ring":
        fmt = "i16" if ring == "i16" else "f32"
    if fmt == "f32":
        return np.ascontiguousarray(pcm, dtype=np.float32)
    q = synth.to_int16(pcm)
    return q if fmt == "i16" else _encode(q, fmt)


def _law(kind):
    return kind[1] if kind[1] in ("ulaw", "alaw") else None


def _push_uniform(ctx, kind, x, stream0=0):
    """today's calls: ewk_push / ewk_push_g711 / ewk_push_resampled of rows x onto [stream0, stream0 + len(x))"""
    if kind[0] == 16000:
        if _law(kind):
            ctx.push_g711(x, stream0=stream0, law=kind[1])
        else:
            ctx.push(x, stream0=stream0)
        return np.full(len(x), x.shape[1], np.int64)
    return np.full(len(x), ctx.push_resampled(x, kind[0], stream0=stream0, fmt=_law(kind)), np.int64)


class Run:
    """A context and what its ticks and polls returned; traces are kept per stream (the cells of the ticks it took)."""

    def __init__(self, ctx, traced=True):
        self.ctx, self.traced, self.events = ctx, traced, []
        self.tr = [{k: [] for k in ("thr", "rms", "silent", "state")} for _ in range(ctx.cfg.n_streams)]
        self.taken = np.zeros(ctx.cfg.n_streams, np.int64)

    def tick(self, n):
        if n > 0:
            tr = self.ctx.tick(n, trace=self.traced)
            if self.traced:
                for s in range(len(self.tr)):
                    for k in self.tr[s]:
                        self.tr[s][k].append(np.asarray(tr[k][s], dtype=np.uint8 if k == "silent" else None))
            self.taken += n
        self.events.append(self.ctx.poll().copy())

    def ready(self, check_budget=False):
        """tick_ready until nothing is due; checks `taken` against the due rule when asked"""
        while True:
            if check_budget:
                st = [self.ctx.status(s) for s in range(len(self.tr))]
                want = due_ticks([x.written for x in st], [x.tick for x in st], MAXT)
            if self.traced:
                taken, tr = self.ctx.tick_ready(MAXT, trace=True)
                for s in range(len(self.tr)):
                    t = int(taken[s])
                    for k in self.tr[s]:
                        self.tr[s][k].append(tr[k][s, :t])
                    assert (tr["state"][s, t:] == 255).all() and (tr["silent"][s, t:] == 255).all()
                    assert np.isnan(tr["thr"][s, t:]).all() and np.isnan(tr["rms"][s, t:]).all()
            else:
                taken = self.ctx.tick_ready(MAXT)
            if check_budget:
                assert np.array_equal(taken, want)
            self.taken += taken
            self.events.append(self.ctx.poll().copy())
            if taken.max() < MAXT:
                return

    def state(self, streams, ring_s=RING_S):
        ctx = self.ctx
        ev = np.concatenate(self.events) if self.events else np.zeros(0, _lib().EVENT_DTYPE)
        out = {}
        for s in streams:
            e = ev[ev["stream"] == s]
            e = e[np.lexsort((e["kind"], e["tick"]))]
            tr = {k: np.concatenate(v) if v else np.zeros(0) for k, v in self.tr[s].items()} if self.traced else {}
            st = ctx.status(s)
            out[s] = dict(ev=e, tr=tr, status={f[0]: getattr(st, f[0]) for f in st._fields_},
                          res=ctx.results()[s:s + 1].copy(), inp=ctx.stream_input(s),
                          ring=ctx.read_last(s, ring_s * 16000))
        return out


def _same(a, b, bit4=False):
    """a, b: Run.state of the same streams, bit for bit on either ring format: K1's block sums and the gate's own sums
    of a block add in one order (oracle/gate_model.py), so thresholds and RMS agree to the last bit."""
    for s in a:
        x, y = a[s], b[s]
        assert len(x["ev"]) == len(y["ev"]), s
        for f in x["ev"].dtype.names:
            u, v = x["ev"][f], y["ev"][f]
            if u.dtype.kind == "f":
                u, v = u.view(np.int32), v.view(np.int32)
            assert np.array_equal(u, v), (s, f)
        mask = np.uint32(0xFFFFFFFF if bit4 else ~np.uint32(16))
        assert np.array_equal(x["res"]["score"].view(np.int32), y["res"]["score"].view(np.int32)), s
        assert np.array_equal(x["res"]["flags"] & mask, y["res"]["flags"] & mask), s
        for k in x["status"]:
            u, v = x["status"][k], y["status"][k]
            if isinstance(u, float):
                u, v = np.float64(u).view(np.int64), np.float64(v).view(np.int64)
            assert u == v, (s, k)
        assert x["inp"] == y["inp"], s
        assert np.array_equal(x["ring"], y["ring"]), s
        for k in x["tr"]:
            u, v = x["tr"][k], y["tr"][k]
            if k in ("thr", "rms"):
                u, v = np.asarray(u, np.float64).view(np.int64), np.asarray(v, np.float64).view(np.int64)
            assert np.array_equal(u, v), (s, k)


def _pieces(rng, total, rate, n_steps_max=200, p_active=0.7):
    """random ragged split of `total` samples per stream: list of steps, each a list of (stream, a, b)"""
    cur = np.zeros(len(total), np.int64)
    steps = []
    while (cur < total).any():
        assert len(steps) < n_steps_max
        step = []
        for s in rng.permutation(len(total)):
            if rng.random() > p_active:
                continue
            n = 0 if rng.random() < 0.1 else int(rng.uniform(0.5, 1.5) * rate)
            n = int(min(n, total[s] - cur[s]))
            step.append((int(s), int(cur[s]), int(cur[s] + n)))
            cur[s] += n
        steps.append(step)
    return steps


CASES = {
    "pcm-i16": dict(ring="i16", kind=PCM),
    "pcm-i16-fs512": dict(ring="i16", kind=PCM, prm=dict(frame_size=512)),
    "pcm-f32": dict(ring="f32", kind=PCM),
    "g711-16k": dict(ring="i16", kind=G711),
    "ulaw-8k": dict(ring="i16", kind=U8K),
    "f32-44k1": dict(ring="i16", kind=F44K),
    "i16-48k-into-f32": dict(ring="f32", kind=I48K),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_jitter_invariance(word, case):
    """A: uniform ewk_push + ewk_tick.  B: the same audio in random ragged pieces to random subsets through
    ewk_push_streams + ewk_tick_ready.  C: B's rows pushed one stream at a time with today's calls, same ticks."""
    c = CASES[case]
    ring, kind, prm = c["ring"], c["kind"], c.get("prm", {})
    rate = kind[0]
    x = _audio(kind, ring, word, 4200, SECS)
    A, B, C = (Run(_ctx(ring, word, **prm)) for _ in range(3))
    # A: one second per step to every stream
    clock = 0
    for step in range(SECS):
        m = _push_uniform(A.ctx, kind, x[:, step * rate:(step + 1) * rate])
        clock += int(m[0])
        A.tick(clock // 1600 - int(A.taken[0]))
    steps = _pieces(np.random.default_rng(list(CASES).index(case)), np.full(N, x.shape[1]), rate)
    pos = np.zeros(N, np.int64)
    for i, step in enumerate(steps):
        streams = [s for s, _, _ in step]
        rows = [x[s, a:b] for s, a, b in step]
        landed = B.ctx.push_streams(streams, rows, sr_in=rate, fmt=_law(kind))
        if rate != 16000:
            for j, (s, a, b) in enumerate(step):
                assert landed[j] == landed_counts([a], b - a, rate)[0]
        else:
            assert np.array_equal(landed, [b - a for _, a, b in step])
        for s, a, b in step:
            if b > a:
                _push_uniform(C.ctx, kind, x[s:s + 1, a:b], stream0=s)
        B.ready(check_budget=i % 4 == 0)
        C.ready()
        for s, a, b in step:
            pos[s] = b
    assert (pos == x.shape[1]).all()
    sa, sb, sc = A.state(range(N)), B.state(range(N)), C.state(range(N))
    assert sum(len(v["ev"]) for v in sa.values()) > 0
    assert any((v["ev"]["kind"] == 1).any() for v in sa.values())           # timeouts occur
    assert any((v["ev"]["kind"] == 2).any() for v in sa.values())           # level-2 evaluations occur
    _same(sa, sb)
    _same(sc, sb, bit4=True)
    # the K8 tails: one more identical push lands the same samples everywhere
    extra = _audio(kind, ring, word, 99, 1)
    _push_uniform(A.ctx, kind, extra)
    B.ctx.push_streams(list(range(N)), list(extra), sr_in=rate, fmt=_law(kind))
    for s in range(N):
        assert np.array_equal(A.ctx.read_last(s, RING_S * 16000), B.ctx.read_last(s, RING_S * 16000)), s


@pytest.mark.gpu
def test_parked_slots(word):
    """never-pushed slots, slots that stop being fed, and slots reset and left unfed take no ticks and raise nothing;
    the other streams equal a bank without them"""
    ring, rate = "i16", 16000
    never, stop, reset = [2, 5], [7, 10], [0, 9]
    active = [s for s in range(N) if s not in never]
    x = _audio(PCM, ring, word, 5100, SECS)
    B = Run(_ctx(ring, word))
    E = Run(_ctx(ring, word, n=len(active) - len(reset)))            # the streams that stay fed, alone
    fed = [s for s in active if s not in reset]
    rng = np.random.default_rng(3)
    steps = _pieces(rng, np.full(N, x.shape[1]), rate)
    before, n_ev = {}, 0
    for i, step in enumerate(steps):
        if i == len(steps) // 2:
            before = {s: (B.ctx.status(s).tick, B.ctx.status(s).written, B.ctx.results()[s].copy()) for s in stop}
            B.events.append(B.ctx.poll().copy())
            n_ev = len(B.events)
            B.ctx.reset_streams(reset)
        half = i >= len(steps) // 2
        rows = [(s, a, b) for s, a, b in step if s in active and not (half and s in stop + reset)]
        B.ctx.push_streams([s for s, _, _ in rows], [x[s, a:b] for s, a, b in rows])
        er = [(fed.index(s), a, b) for s, a, b in rows if s in fed]
        E.ctx.push_streams([s for s, _, _ in er], [x[fed[s], a:b] for s, a, b in er])
        B.ready(check_budget=True)
        E.ready()
    res = B.ctx.results()
    late = np.concatenate(B.events[n_ev:])
    for s in never + reset:
        st = B.ctx.status(s)
        assert st.tick == 0 and st.written == 0, s
        assert not (late["stream"] == s).any(), s
        assert np.isnan(res[s]["score"]), s
    assert not np.isin(np.concatenate(B.events)["stream"], never).any()
    for s in stop:
        t0, w0, r0 = before[s]
        st = B.ctx.status(s)
        assert st.written == w0 and st.tick == t0 == w0 // 1600, s
        assert res[s]["score"].view(np.int32) == r0["score"].view(np.int32), s
        assert not (late["stream"] == s).any(), s
    sb = B.state(fed)
    se = E.state(range(len(fed)))
    for i in range(len(fed)):
        se[i]["ev"]["stream"] = fed[i]
    _same({s: sb[s] for s in fed}, {fed[i]: se[i] for i in range(len(fed))})


@pytest.mark.gpu
def test_recycle_at_another_rate(word):
    """streams reset in the middle of a ragged 16 kHz run restart at 8 kHz mu-law; each equals the same stream of a new
    context given the same calls from the reset on"""
    ring, reset = "i16", [1, 4, 11]
    x16 = _audio(PCM, ring, word, 6100, SECS)
    x8 = _audio(U8K, ring, word, 6200, SECS - 4)
    B, F = Run(_ctx(ring, word)), Run(_ctx(ring, word))
    rng = np.random.default_rng(11)
    steps16 = _pieces(rng, np.full(N, x16.shape[1]), 16000)
    steps8 = _pieces(rng, np.full(N, x8.shape[1]), 8000)
    cut = 6
    for i, step in enumerate(steps16):
        if i == cut:
            B.events.append(B.ctx.poll().copy())
            B.ctx.reset_streams(reset)
            B.tr = [{k: [] for k in t} if s in reset else t for s, t in enumerate(B.tr)]
            B.events = [e[~np.isin(e["stream"], reset)] for e in B.events]
        rows = [(s, a, b) for s, a, b in step if not (i >= cut and s in reset)]
        B.ctx.push_streams([s for s, _, _ in rows], [x16[s, a:b] for s, a, b in rows])
        if i >= cut and i - cut < len(steps8):
            r8 = [(s, a, b) for s, a, b in steps8[i - cut] if s in reset]
            for ctx in (B.ctx, F.ctx):
                ctx.push_streams([s for s, _, _ in r8], [x8[s, a:b] for s, a, b in r8], sr_in=8000, fmt="ulaw")
        B.ready()
        if i >= cut:
            F.ready()
    _same(B.state(reset), F.state(reset))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["pinned", "device", "overlap"])
def test_input_paths(word, path):
    """pinned input (each push still pending when ewk_tick_ready lands it; then one pending at ewk_tick),
    device-resident input and overlap mode: all equal the pageable run"""
    import torch
    L = _lib()
    ring, rate = "i16", 16000
    x = _audio(PCM, ring, word, 7300, SECS)
    R = Run(_ctx(ring, word), traced=False)
    T = Run(_ctx(ring, word), traced=False)
    if path == "overlap":
        T.ctx.set_overlap(True)
    steps = _pieces(np.random.default_rng(5), np.full(N, x.shape[1]), rate)
    keep = []
    for step in steps:
        streams = [s for s, _, _ in step]
        rows = [x[s, a:b] for s, a, b in step]
        R.ctx.push_streams(streams, rows)
        R.ready()
        lens = np.array([len(r) for r in rows], np.int64)
        offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
        flat = np.concatenate(rows) if rows else np.zeros(0, np.int16)
        if path == "device":
            t = torch.from_numpy(flat.copy()).cuda()
            torch.cuda.synchronize()
            T.ctx.push_streams(streams, (t.data_ptr(), offs, lens, len(flat), np.int16), where=L.DEVICE)
            keep.append(t)
        elif path == "overlap":
            T.ctx.push_streams(streams, rows)
        else:
            buf = L.PinnedArray((max(1, len(flat)),), np.int16)
            buf.array[:len(flat)] = flat
            keep.append(buf)
            T.ctx.push_streams(streams, (buf.ptr.value, offs, lens, len(flat), np.int16))
        T.ready()
    _same(R.state(range(N)), T.state(range(N)))
    if path == "pinned":
        # a pinned list push left pending, then ewk_tick: every stream moves, and the pushed samples are what it sees
        flat = x[:, :1600].reshape(-1)
        buf = L.PinnedArray(flat.shape, np.int16)
        buf.array[...] = flat
        lens = np.full(N, 1600, np.int64)
        for ctx in (R.ctx, T.ctx):
            ctx.push_streams(list(range(N)), (buf.ptr.value, np.arange(N) * 1600, lens, len(flat), np.int16))
        R.ctx.synchronize()
        R.ctx.tick(3)
        T.ctx.tick(3)
        for s in range(N):
            assert R.ctx.status(s).tick == T.ctx.status(s).tick
            assert np.array_equal(R.ctx.read_last(s, 16000), T.ctx.read_last(s, 16000))
        keep.append(buf)


@pytest.mark.gpu
def test_publication_every_record_every_call(word):
    """peer publication to a local destination: after every ewk_tick_ready, every stream's record is at the call's
    parity, streams that took no tick included"""
    import torch
    ring, rate = "i16", 16000
    x = _audio(PCM, ring, word, 8300, 8)
    ctx = _ctx(ring, word)
    d = torch.full((2, N, 2), -7, dtype=torch.int32, device="cuda:0")
    ctx.set_results_peers([d.data_ptr()], stride_records=N, offset_records=0)
    steps = _pieces(np.random.default_rng(9), np.full(N, x.shape[1]), rate, p_active=0.4)
    zero_seen = False
    for step in steps:
        ctx.push_streams([s for s, _, _ in step], [x[s, a:b] for s, a, b in step])
        ctx.synchronize()
        torch.cuda.synchronize()
        d.fill_(-7)
        torch.cuda.synchronize()
        taken = ctx.tick_ready(MAXT)
        zero_seen |= bool((taken == 0).any())
        ctx.synchronize()
        torch.cuda.synchronize()
        got = d[ctx.publish_parity()].cpu().numpy()
        want = ctx.results()
        assert np.array_equal(got[:, 0], want["score"].view(np.int32))
        assert np.array_equal(got[:, 1].view(np.uint32), want["flags"])
    assert zero_seen
    ctx.set_results_peers([])


@pytest.mark.gpu
def test_bank_step_streams(word):
    """WakeWordBank.step_streams leaves no due tick behind, at 16 kHz and at 8 kHz"""
    from easywakeword_b200.bank import WakeWordBank
    for sr in (16000, 8000):
        bank = WakeWordBank(6, [word], buffer_seconds=5, sample_rate=sr, max_push_seconds=2.0)
        rng = np.random.default_rng(sr)
        for _ in range(6):
            streams = [int(s) for s in rng.choice(6, 4, replace=False)]
            blocks = [(rng.standard_normal(int(rng.uniform(0.2, 1.8) * sr)) * 300).astype(np.int16) for _ in streams]
            taken = bank.step_streams(streams, blocks)
            for s in range(6):
                st = bank.status(s)
                assert st.written // 1600 == st.tick
            assert taken.shape == (6,)
        bank.close()


def _err(fn, exc, *words):
    with pytest.raises(exc) as e:
        fn()
    for w in words:
        assert w in str(e.value), str(e.value)


@pytest.mark.gpu
def test_errors(word):
    L = _lib()
    ctx = _ctx("i16", word)
    f32 = _ctx("f32", word)
    z = np.zeros(100, np.int16)
    _err(lambda: ctx.push_streams([N], [z]), ValueError, "stream 12")
    _err(lambda: ctx.push_streams([-1], [z]), ValueError, "stream -1")
    _err(lambda: ctx.push_streams([3, 3], [z, z]), ValueError, "stream 3", "twice")
    buf = np.zeros(200, np.int16)
    _err(lambda: ctx.push_streams([4], (buf.ctypes.data, [150], [100], 200, np.int16)), ValueError, "stream 4", "outside")
    _err(lambda: ctx.push_streams([4], (buf.ctypes.data, [0], [-1], 200, np.int16)), ValueError, "stream 4")
    _err(lambda: ctx.push_streams([4], (buf.ctypes.data, [-1], [10], 200, np.int16)), ValueError, "stream 4")
    st = np.array([1], np.int32)
    off, ln = np.zeros(1, np.int64), np.full(1, 10, np.int64)
    rc = ctx.lib.ewk_push_streams(ctx.h, st.ctypes.data_as(L._p(L.C.c_int32)), 1, buf.ctypes.data, L.PCM_I16,
                                  L.i64ptr(off), L.i64ptr(ln), 200, L.HOST, 16000, None)
    assert rc == L.EWK_ERR_ARG and "landed is NULL" in ctx.lib.ewk_last_error(ctx.h).decode()
    _err(lambda: ctx.push_streams([1], [z], sr_in=300), ValueError, "300 Hz")
    _err(lambda: f32.push_streams([1], [np.zeros(10, np.uint8)], fmt="ulaw"), ValueError, "G.711")
    _err(lambda: ctx.push_streams([1], [np.zeros(10, np.float32)]), ValueError, "in_format")
    _err(lambda: ctx.push_streams([2], [np.zeros(RING_S * 16000 + 1, np.int16)]), ValueError, "stream 2", "exceed the ring")
    ctx.push_streams([5], [np.zeros(8000, np.uint8)], sr_in=8000, fmt="ulaw")
    _err(lambda: ctx.push_streams([5], [z]), L.EwkError, "stream 5", "Hz")
    _err(lambda: ctx.push_streams([5], [np.zeros(480, np.int16)], sr_in=48000), L.EwkError, "stream 5", "8000 Hz")
    ctx.push_streams([6], [np.zeros(60000, np.int16)])
    ctx.push_streams([6], [np.zeros(30000, np.int16)])
    _err(lambda: ctx.push_streams([6], [np.zeros(30000, np.int16)]), L.EwkError, "stream 6", "first full tick")
    for _ in range(3):
        ctx.tick_ready(MAXT)
    assert ctx.status(6).tick == 90000 // 1600
    _err(lambda: ctx.push_streams([6], [np.zeros(34000, np.int16)]), L.EwkError, "stream 6", "un-gated")
    _err(lambda: ctx.tick_ready(0), ValueError, "max_ticks")
    assert np.array_equal(ctx.push_streams([], []), np.zeros(0, np.int64))
    assert np.array_equal(ctx.push_streams([7, 8], [z[:0], z[:0]]), [0, 0])
    assert ctx.status(7).written == 0 and ctx.stream_input(7) == (0, 0)


# ---------------------------------------------------------------------------------------------------------- CPU
def test_due_ticks_brute_force():
    """tick k is due once 1600 k samples have landed: count them one by one"""
    rng = np.random.default_rng(0)
    written = rng.integers(0, 100000, 500)
    ticks = rng.integers(0, 80, 500)
    for cap in (None, 1, 7, 16, 4096):
        got = due_ticks(written, ticks, cap)
        for w, t, g in zip(written, ticks, got):
            k, n = int(t), 0
            while 1600 * (k + 1) <= w and (cap is None or n < cap):
                k, n = k + 1, n + 1
            assert g == n


class _FakeLib:
    def __init__(self):
        self.calls = []

    def ewk_push_streams(self, h, st, n, ptr, code, off, ln, in_len, where, sr, landed):
        import ctypes as C
        self.calls.append(dict(streams=[st[i] for i in range(n)], ptr=ptr, code=code, off=[off[i] for i in range(n)],
                               lens=[ln[i] for i in range(n)], in_len=in_len, where=where, sr=sr,
                               data=C.string_at(ptr, in_len * 2) if ptr else b""))
        for i in range(n):
            landed[i] = ln[i]
        return 0


def test_push_streams_packing():
    """rows of any length, zeros included, are packed back to back into one buffer with their offsets"""
    L = _lib()
    ctx = object.__new__(L.Context)
    ctx.lib, ctx.h = _FakeLib(), None
    ctx.cfg = L.Config(4, 16000, 1600, L.PCM_I16, 1, 16, 0.0, 20, 0, 0)
    rows = [np.arange(5, dtype=np.int16), np.zeros(0, np.int16), np.arange(100, 103, dtype=np.int16)]
    landed = ctx.push_streams([3, 0, 1], rows)
    c = ctx.lib.calls[-1]
    assert c["streams"] == [3, 0, 1] and c["off"] == [0, 5, 5] and c["lens"] == [5, 0, 3] and c["in_len"] == 8
    assert np.array_equal(np.frombuffer(c["data"], np.int16), np.concatenate(rows))
    assert c["code"] == L.PCM_I16 and c["sr"] == 16000 and c["where"] == L.HOST
    assert np.array_equal(landed, [5, 0, 3])
    ctx.push_streams([2], [np.zeros(4, np.uint8)], sr_in=8000, fmt="alaw")
    assert ctx.lib.calls[-1]["code"] == L.IN_ALAW and ctx.lib.calls[-1]["sr"] == 8000
    with pytest.raises(TypeError):
        ctx.push_streams([0, 1], [np.zeros(2, np.int16), np.zeros(2, np.float32)])
    with pytest.raises(ValueError):
        ctx.push_streams([0, 1], [np.zeros(2, np.int16)])


def test_sharded_step_streams_routing():
    """every rank takes the whole list and keeps its own rows, with local ids"""
    from easywakeword_b200.dist import ShardedBank, shard_range

    class _Bank:
        def step_streams(self, streams, rows):
            self.got = (streams, rows)

    n_total, world = 10, 3
    g = [9, 0, 4, 3, 7, 1]
    blocks = [np.full(3, v, np.int16) for v in g]
    seen = []
    for rank in range(world):
        sb = object.__new__(ShardedBank)
        sb.n_total, sb.world, sb.rank, sb.bank = n_total, world, rank, _Bank()
        sb.first, sb.last = shard_range(n_total, world, rank)
        sb.step_streams(g, blocks)
        streams, rows = sb.bank.got
        for s, r in zip(streams, rows):
            assert 0 <= s < sb.last - sb.first and r[0] == sb.first + s
            seen.append(sb.first + s)
    assert sorted(seen) == sorted(g)
