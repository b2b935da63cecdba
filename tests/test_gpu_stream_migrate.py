"""Stream migration (ewk_export_streams / ewk_import_streams, K10).  A stream exported from context A mid-run and
imported into slots of context B must go on in B exactly as it goes on in A given the same calls: events (ids mapped),
result records, tick traces, status, input counts, the whole ring, segments of events raised before the move, dense
scores and detections, all bit for bit.  Export must leave A exactly as a run without it (A0), and the slots of B that
were not imported exactly as a run without the import (B0)."""
import math

import numpy as np
import pytest

from easywakeword_b200 import synth
from easywakeword_b200.resample import ALAW_TABLE, ULAW_TABLE

N, RING_S = 12, 5
X = [1, 4, 6, 11]              # exported from A (11 is never fed before the move)
Y = [10, 2, 7, 0]              # their slots in B: a permutation of other ids
IDLE = N - 1


def _lib():
    from easywakeword_b200 import _lib as L
    return L


def _ctx(ring, n=N, word=None, n_mfcc=0, preemphasis=0.0, slack_s=2, ring_s=RING_S, max_templates=1, **prm):
    L = _lib()
    ctx = L.Context(device=0, n_streams=n, ring_samples=ring_s * 16000, slack_samples=slack_s * 16000,
                    pcm_format=L.PCM_I16 if ring == "i16" else L.PCM_F32, max_templates=max_templates, max_events=4096,
                    n_mfcc=n_mfcc, preemphasis=preemphasis)
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


def _audio(kind, ring, word, seed, secs, n=N):
    """[n, secs * rate] feed of `kind`: ("pcm",) 16 kHz in the ring's dtype, ("g711",) 16 kHz mu-law codes, or
    ("rs", sr, fmt) native-rate f32 / i16 / ulaw."""
    from scipy.signal import resample_poly
    pcm = synth.stream_batch(seed, n, float(secs), word, as_int16=False, gain=(2.0, 4.0))
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


def _g711(kind):
    return "ulaw" if kind[0] == "g711" or (kind[0] == "rs" and kind[2] == "ulaw") else None


def _push(ctx, kind, x, stream0, pinned=False):
    """One uniform push of rows x onto streams [stream0, stream0 + len(x)); -> landed count per stream."""
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
        out = ctx.push_resampled_each(x, kind[1], stream0=stream0, fmt=_g711(kind))
    return out, buf


class Log:
    """A context and what its ticks and polls returned.  Traced ticks run K3 behind the gate, so a context in overlap
    mode ticks without traces."""

    def __init__(self, ctx, traced=True):
        self.ctx, self.traced, self.events = ctx, traced, []
        self.trace = {k: [] for k in ("thr", "rms", "silent", "state")} if traced else {}
        self.mark = (0, 0)

    def tick(self, n):
        if n > 0:
            tr = self.ctx.tick(n, trace=self.traced)
            for k in self.trace:
                self.trace[k].append(tr[k].astype(np.uint8) if k == "silent" else tr[k])

    def tick_ready(self, cap=64):
        if self.traced:
            taken, tr = self.ctx.tick_ready(cap, trace=True)
            for k in self.trace:
                self.trace[k].append(tr[k])
        else:
            taken = self.ctx.tick_ready(cap)
        assert taken.max() < cap
        return taken

    def poll(self):
        self.events.append(self.ctx.poll().copy())

    def set_mark(self):
        self.mark = (len(self.events), len(next(iter(self.trace.values()))) if self.trace else 0)

    def state(self, streams, since_mark=False):
        ctx = self.ctx
        e0, t0 = self.mark if since_mark else (0, 0)
        evs = self.events[e0:]
        ev = np.concatenate(evs) if evs else np.zeros(0, _lib().EVENT_DTYPE)
        ev = ev[np.isin(ev["stream"], streams)]
        ev = ev[np.lexsort((ev["kind"], [streams.index(s) for s in ev["stream"]], ev["tick"]))] if len(ev) else ev
        tr = {k: np.concatenate(v[t0:], axis=1)[streams] for k, v in self.trace.items() if v[t0:]}
        st = [tuple(getattr(ctx.status(s), f[0]) for f in ctx.status(s)._fields_) for s in streams]
        return dict(ev=ev, tr=tr, status=st, res=ctx.results()[streams], inp=[ctx.stream_input(s) for s in streams],
                    ring=np.stack([ctx.read_last(s, RING_S * 16000) for s in streams]))


def _assert_same(a, b, ids=None):
    """b's streams are a's under the map ids (a's id -> b's id) when given."""
    assert len(a["ev"]) == len(b["ev"])
    for f in a["ev"].dtype.names:
        x, y = a["ev"][f], b["ev"][f]
        if f == "stream" and ids is not None:
            x = np.array([ids[int(s)] for s in x], dtype=x.dtype)
        if x.dtype.kind == "f":
            x, y = x.view(np.int32), y.view(np.int32)                  # scores by bits
        assert np.array_equal(x, y), f
    assert np.array_equal(a["res"].view(np.int32), b["res"].view(np.int32))
    assert a["status"] == b["status"]
    assert a["inp"] == b["inp"]
    assert np.array_equal(a["ring"].view(np.int32), b["ring"].view(np.int32))
    assert a["tr"].keys() == b["tr"].keys()
    for k in ("silent", "state"):
        if k in a["tr"]:
            assert np.array_equal(a["tr"][k], b["tr"][k]), k
    for k in ("thr", "rms"):
        if k in a["tr"]:
            assert np.array_equal(a["tr"][k].view(np.int64), b["tr"][k].view(np.int64)), k


def _export(ctx, streams, form):
    """Export in one of the blob forms -> (blob argument of import_streams, where, host bytes of the blob)."""
    import ctypes as C
    import torch
    L = _lib()
    if form in ("pageable", "file"):
        b = ctx.export_streams(streams)
        return b, L.HOST, b
    cap = ctx.stream_blob_bytes(len(streams))
    st = np.ascontiguousarray(streams, dtype=np.int32)
    if form == "pinned":
        pin = L.PinnedArray((cap,), np.uint8)
        ctx._ck(ctx.lib.ewk_export_streams(ctx.h, st.ctypes.data_as(C.POINTER(C.c_int32)), len(st), pin.ptr, cap, L.HOST))
        n = int(pin.array[:96].view(L.STREAM_BLOB_HEADER_DTYPE)[0]["total_bytes"])
        return pin, L.HOST, pin.array[:n].copy()
    d = torch.zeros(cap, dtype=torch.uint8, device=f"cuda:{ctx.device}")
    ctx.export_streams(streams, where=L.DEVICE, out=(d.data_ptr(), cap))
    h = d.cpu().numpy()
    n = int(h[:96].view(L.STREAM_BLOB_HEADER_DTYPE)[0]["total_bytes"])
    return d, L.DEVICE, h[:n]


def _import(ctx, streams, blob, where):
    import ctypes as C
    L = _lib()
    if where == L.DEVICE:
        ctx.import_streams(streams, (blob.data_ptr(), blob.numel()), where=L.DEVICE)
    elif isinstance(blob, L.PinnedArray):
        st = np.ascontiguousarray(streams, dtype=np.int32)
        ctx._ck(ctx.lib.ewk_import_streams(ctx.h, st.ctypes.data_as(C.POINTER(C.c_int32)), len(st), blob.ptr,
                                           blob.array.size, L.HOST))
    else:
        ctx.import_streams(streams, blob)


def _meta(blob_bytes, i):
    L = _lib()
    h = blob_bytes[:96].view(L.STREAM_BLOB_HEADER_DTYPE)[0]
    o = int(h["meta_offset"]) + i * L.STREAM_META_BYTES
    return blob_bytes[o:o + L.STREAM_META_BYTES]


def _gate_state(blob_bytes, i):
    return int(_meta(blob_bytes, i)[212:216].view(np.int32)[0])


PCM, G711 = ("pcm",), ("g711",)
U8K, I48K = ("rs", 8000, "ulaw"), ("rs", 48000, "i16")
CASES = {
    "pcm16-i16": dict(ring="i16", kind=PCM),
    "pcm16-f32": dict(ring="f32", kind=PCM),
    "g711-16k": dict(ring="i16", kind=G711),
    "ulaw-8k": dict(ring="i16", kind=U8K),
    "i16-48k-into-f32": dict(ring="f32", kind=I48K),
    "frame-size-0": dict(ring="i16", kind=PCM, prm=dict(frame_size=0)),
    "frame-size-512": dict(ring="i16", kind=PCM, prm=dict(frame_size=512)),
    "live": dict(ring="i16", kind=U8K, prm=dict(live=1)),
    "preemphasis-n13": dict(ring="f32", kind=PCM, cfg=dict(n_mfcc=13, preemphasis=0.97)),
    "overlap": dict(ring="i16", kind=PCM, overlap=True),
    "pending-at-export": dict(ring="i16", kind=U8K, pend_export=True),
    "pending-at-import": dict(ring="f32", kind=PCM, pend_import=True),
    "wrapped-many-times": dict(ring="i16", kind=G711, pre_steps=40),
    "pinned-blob": dict(ring="i16", kind=U8K, form="pinned"),
    "device-blob": dict(ring="f32", kind=I48K, form="device"),
    "saved-blob": dict(ring="i16", kind=PCM, form="file"),
}


def _scenario(word, ring, kind, prm=None, cfg=None, overlap=False, pend_export=False, pend_import=False, pre_steps=9,
              post_steps=10, form="pageable", xs=X, ys=Y, tmp_path=None):
    """A, A0: pre-phase (stream IDLE never fed), export xs from A mid-run (not from A0); B, B0: their own feed, then
    import into ys of B (not B0); then the same post-phase calls to A, A0 and B, B0 (B's ys get A's xs' audio)."""
    prm, cfg = prm or {}, cfg or {}
    ctxs = [_ctx(ring, word=word, **cfg, **prm) for _ in range(4)]
    pins = []
    try:
        if overlap:
            for c in ctxs:
                c.set_overlap(True)
        A, A0, B, B0 = (Log(c, not overlap) for c in ctxs)
        k = _rate(kind)
        x_pre = _audio(kind, ring, word, 7100, pre_steps + 1)
        y_pre = _audio(kind, ring, word, 8200, pre_steps + 1)
        fed = N - 1                                                    # streams [0, N - 1): IDLE stays empty
        clock = ticks = 0
        for step in range(pre_steps):
            last = step == pre_steps - 1
            for lg in (A, A0):
                m, buf = _push(lg.ctx, kind, x_pre[:fed, step * k:(step + 1) * k], 0, pinned=last and pend_export)
                pins.append(buf)
            clock += int(m.max())
            if not (last and pend_export):
                due = clock // 1600 - ticks
                for lg in (A, A0):
                    lg.tick(due)
                ticks += due
        clock = ticks = 0
        for step in range(pre_steps - 3):
            last = step == pre_steps - 4
            for lg in (B, B0):
                m, buf = _push(lg.ctx, kind, y_pre[:, step * k:(step + 1) * k], 0, pinned=last and pend_import)
                pins.append(buf)
            clock += int(m.max())
            if not (last and pend_import):
                due = clock // 1600 - ticks
                for lg in (B, B0):
                    lg.tick(due)
                ticks += due
        for lg in (B, B0):
            lg.poll()
        # export with A's queue not drained: its events stay in A with A's ids
        blob, where, raw = _export(A.ctx, xs, form)
        pins.append(blob if isinstance(blob, _lib().PinnedArray) else None)
        if form == "file":
            np.save(tmp_path / "blob.npy", blob)
            blob = np.load(tmp_path / "blob.npy")
        for lg in (A, A0):
            lg.poll()
        pre_ev = np.concatenate(A.events)
        pre_ev = pre_ev[np.isin(pre_ev["stream"], xs) & (pre_ev["kind"] == 2)]
        _import(B.ctx, ys, blob, where)
        ids = dict(zip(xs, ys))
        for e in pre_ev:                                               # segments raised before the move, still in the ring
            s, a0, n = int(e["stream"]), int(e["seg_start"]), int(e["seg_len"])
            if A.ctx.status(s).written - a0 <= RING_S * 16000:
                assert np.array_equal(A.ctx.read_segment(s, a0, n).view(np.int32),
                                      B.ctx.read_segment(ids[s], a0, n).view(np.int32))
        for lg in (A, A0, B, B0):
            lg.set_mark()
            lg.tick_ready()                                            # a push left un-ticked before the move
            lg.poll()
        # post-phase: one ragged push and one paced tick per step; B's ys get A's xs' audio
        x_post = _audio(kind, ring, word, 9100, post_steps + 1)
        y_post = _audio(kind, ring, word, 9300, post_steps + 1)
        for step in range(post_steps):
            rows_a = [x_post[s, step * k:(step + 1) * k] for s in range(N)]
            rows_b = [y_post[s, step * k:(step + 1) * k] for s in range(N)]
            for xi, yi in zip(xs, ys):
                rows_b[yi] = rows_a[xi]
            for lg, rows in ((A, rows_a), (A0, rows_a), (B, rows_b), (B0, rows_b)):
                lg.ctx.push_streams(list(range(N)), rows, sr_in=k, fmt=_g711(kind))
                lg.tick_ready()
                lg.poll()
        got = A.state(xs, since_mark=True)
        _assert_same(got, B.state(ys, since_mark=True), ids)
        _assert_same(A.state(list(range(N))), A0.state(list(range(N))))
        rest = [s for s in range(N) if s not in ys]
        if rest:
            _assert_same(B.state(rest), B0.state(rest))
        assert sum(len(e) for e in A.events) >= 2
        return raw
    finally:
        for c in ctxs:
            c.close()
        for b in pins:
            if b is not None:
                b.free()


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
def test_moved_stream_equals_unmoved(word, case, tmp_path):
    _scenario(word, tmp_path=tmp_path, **CASES[case])


@pytest.mark.gpu
def test_every_gate_state_moves(word):
    """All streams of A into B in reverse order: they sit in several gate states at the export, IDLE in none"""
    raw = _scenario(word, ring="i16", kind=PCM, pre_steps=12, xs=list(range(N)), ys=list(range(N))[::-1])
    states = {_gate_state(raw, i) for i in range(N)}
    assert len(states) >= 3, states


@pytest.mark.gpu
def test_blob_forms_are_identical(word):
    """pageable, pinned and device blobs of one export hold the same bytes; export is repeatable"""
    ctx = _ctx("i16", word=word)
    pin = None
    try:
        x = _audio(U8K, "i16", word, 5100, 4)
        for step in range(3):
            _push(ctx, U8K, x[:, step * 8000:(step + 1) * 8000], 0)
            ctx.tick(10)
        _, _, a = _export(ctx, [3, 0, 5], "pageable")
        pin, _, b = _export(ctx, [3, 0, 5], "pinned")
        _, _, c = _export(ctx, [3, 0, 5], "device")
        assert np.array_equal(a, b) and np.array_equal(a, c)
        L = _lib()
        h = a[:96].view(L.STREAM_BLOB_HEADER_DTYPE)[0]
        W, up, down = L.resample_info(8000)
        tf = int(h["tail_floats"])
        assert 0 < tf <= (2 * W + 3) // 4 * 4 and tf % 4 == 0
        lay = L.stream_blob_layout(RING_S * 16000, 2 * 16000, L.PCM_I16, 3, 1, tf)
        for f in ("ids_offset", "meta_offset", "template_offset", "bulk_offset", "bulk_row_bytes", "total_bytes"):
            assert int(h[f]) == lay[f], f
        assert ctx.stream_blob_bytes(3) == L.stream_blob_layout(RING_S * 16000, 2 * 16000, L.PCM_I16, 3, 1,
                                                                (2 * W + 3) // 4 * 4)["total_bytes"]
        for i, s in enumerate([3, 0, 5]):                              # the live tail inputs [t0, c), zeros beyond
            c = ctx.stream_input(s)[1]
            ready = max(0, -(-(c - W) * up // down))
            t0 = max(0, ready * down // up - W + 1)
            tl = int(_meta(a, i)[56:60].view(np.int32)[0])
            assert tl == c - t0 and 0 < tl <= 2 * W
            row = a[lay["bulk_offset"] + i * lay["bulk_row_bytes"]:][:lay["bulk_row_bytes"]]
            tail = row[lay["tail_off"]:lay["tail_off"] + 4 * tf].view(np.float32)
            assert not tail[tl:].any() and tail[:tl].any()
        assert a[96:108].view(np.int32).tolist() == [3, 0, 5]
    finally:
        ctx.close()
        if pin is not None:
            pin.free()


@pytest.mark.gpu
def test_each_gate_state_moves(word):
    """One stream moved in each gate state (waiting, in_silence, in_sound, after_sound), tick by tick: from the move on
    its status equals the unmoved stream's at every tick, and its events, record and ring at the end"""
    n = 8
    A = _ctx("i16", n=n, word=word)
    B = _ctx("i16", n=4, word=word)
    x = synth.stream_batch(7300, n, 40.0, word, gain=(2.0, 4.0))
    moved = {}                                                         # gate state -> (A's stream, B's slot, tick)
    ev_a, ev_b = [], []
    stat = lambda c, s: tuple(getattr(c.status(s), f[0]) for f in c.status(s)._fields_)    # noqa: E731
    try:
        for k in range(x.shape[1] // 1600):
            blk = x[:, k * 1600:(k + 1) * 1600]
            A.push(np.ascontiguousarray(blk))
            A.tick(1)
            ev_a.append(A.poll())
            if moved:
                B.push_streams([b for _, b, _ in moved.values()], [blk[a] for a, _, _ in moved.values()])
                B.tick_ready(8)
                ev_b.append(B.poll())
                for a, b, _ in moved.values():
                    assert stat(A, a) == stat(B, b)
            if k < 55 or len(moved) == 4:                              # the 5 s ring is full from tick 50
                continue
            for s in range(n):
                st = A.status(s).state
                if st not in moved and s not in [a for a, _, _ in moved.values()]:
                    ev_b.append(B.poll())
                    B.import_streams([st], A.export_streams([s]))
                    moved[st] = (s, st, k)
        assert sorted(moved) == [0, 1, 2, 3], sorted(moved)
        ea, eb = np.concatenate(ev_a), np.concatenate(ev_b)
        n_ev = 0
        for a, b, k in moved.values():
            x_a = ea[(ea["stream"] == a) & (ea["tick"] > k)]
            x_b = eb[eb["stream"] == b]
            assert len(x_a) == len(x_b)
            n_ev += len(x_a)
            for f in ea.dtype.names:
                if f != "stream":
                    p, q = x_a[f], x_b[f]
                    if p.dtype.kind == "f":
                        p, q = p.view(np.int32), q.view(np.int32)
                    assert np.array_equal(p, q), f
            assert np.array_equal(A.read_last(a, RING_S * 16000), B.read_last(b, RING_S * 16000))
            assert A.results()[a].tobytes() == B.results()[b].tobytes()
        assert n_ev >= 1
    finally:
        A.close()
        B.close()


def _dense_feed(word, seed, secs):
    return synth.stream_batch(seed, 1, float(secs), word, gain=(2.0, 4.0))[0]


@pytest.mark.gpu
def test_dense_and_detector_move(word):
    """dense_ready scores and dense_detect records of a moved stream equal the unmoved stream's, with a run ARMED at
    the export and a dense cursor that lags the audio"""
    L = _lib()
    A = _ctx("i16", n=3, word=word, live=1, similarity_threshold=60.0)
    B = _ctx("i16", n=4, word=word, live=1, similarity_threshold=60.0)
    try:
        x = np.stack([_dense_feed(word, 4700 + i, 30.0) for i in range(3)])
        z = np.stack([_dense_feed(word, 4800 + i, 30.0) for i in range(4)])
        armed = None
        for step in range(60):                                         # 0.25 s steps until stream 1 is ARMED
            A.push(np.ascontiguousarray(x[:, step * 4000:(step + 1) * 4000]))
            A.dense_detect(None, 30, hold_hops=40, refractory_hops=10)
            if step % 2 == 0:
                A.dense_ready([0, 1], 45)                              # the dense cursor lags the audio
            raw = A.export_streams([1])
            if int(_meta(raw, 0)[256:260].view(np.int32)[0]) == 1:
                armed = step
                break
        assert armed is not None, "no ARMED run to move"
        assert int(_meta(raw, 0)[24:32].view(np.int64)[0]) < A.status(1).written // 160 + 1
        B.push(np.ascontiguousarray(z[:, :64000]))
        B.import_streams([2], raw)                                     # B has no detector state yet: import allocates it
        det_a, det_b, sc_a, sc_b = [], [], [], []
        for step in range(armed + 1, armed + 30):
            blk = x[1, step * 4000:(step + 1) * 4000]
            A.push_streams([1], [blk])
            B.push_streams([2], [blk])
            if step % 4 == 0:
                sc_a.append(A.dense_ready([1], 120)[1][0])
                sc_b.append(B.dense_ready([2], 120)[1][0])
            det_a.append(A.dense_detect([1], 40, hold_hops=40, refractory_hops=10))
            det_b.append(B.dense_detect([2], 40, hold_hops=40, refractory_hops=10))
        da, db = np.concatenate(det_a), np.concatenate(det_b)
        assert len(da) >= 1 and len(da) == len(db)
        assert (db["stream"] == 2).all()
        for f in da.dtype.names:
            if f != "stream":
                assert np.array_equal(da[f].view(np.int32) if da[f].dtype.kind == "f" else da[f],
                                      db[f].view(np.int32) if db[f].dtype.kind == "f" else db[f]), f
        assert np.array_equal(np.concatenate(sc_a).view(np.int32), np.concatenate(sc_b).view(np.int32))
        assert sum(len(s) for s in sc_a) > 0
    finally:
        A.close()
        B.close()


def _busy(word, ring="i16", n=4, seed=600, secs=12, **kw):
    ctx = _ctx(ring, n=n, word=word, **kw)
    x = synth.stream_batch(seed, n, float(secs), word, gain=(2.0, 4.0))
    if ring == "f32":
        x = synth.from_int16(x)
    for b in range(0, x.shape[1], 16000):
        ctx.push(np.ascontiguousarray(x[:, b:b + 16000]))
        ctx.tick(10)
    return ctx


@pytest.mark.gpu
def test_same_context_swap_and_round_trip(word):
    """[a, b] -> [b, a] after a poll, and export / reset / import into the same slot, equal an untouched context"""
    A, U = _busy(word), _busy(word)
    try:
        for c in (A, U):
            c.poll()
        A.import_streams([3, 1], A.export_streams([1, 3]))
        raw = A.export_streams([2])
        A.reset_streams([2])
        A.import_streams([2], raw)
        x = synth.stream_batch(601, 4, 6.0, word, gain=(2.0, 4.0))
        ea, eu = [], []
        for b in range(0, x.shape[1], 16000):
            blk = np.ascontiguousarray(x[:, b:b + 16000])
            A.push_streams([0, 3, 2, 1], [blk[0], blk[1], blk[2], blk[3]])     # streams 1 and 3 swapped
            U.push_streams([0, 1, 2, 3], list(blk))
            A.tick_ready(64)
            U.tick_ready(64)
            ea.append(A.poll())
            eu.append(U.poll())
        ea, eu = np.concatenate(ea), np.concatenate(eu)
        swap = {0: 0, 1: 3, 2: 2, 3: 1}
        key = lambda e: (int(e["tick"]), int(e["stream"]), int(e["kind"]))       # noqa: E731
        bits = lambda e: int(np.float32(e["score"]).view(np.int32))                 # noqa: E731  (NaN scores too)
        ma = sorted((key(e)[0], swap[key(e)[1]], key(e)[2], bits(e)) for e in ea)
        mu = sorted((key(e)[0], key(e)[1], key(e)[2], bits(e)) for e in eu)
        assert ma == mu and len(ma) >= 1
        for s in range(4):
            assert tuple(getattr(A.status(swap[s]), f[0]) for f in A.status(0)._fields_) == \
                tuple(getattr(U.status(s), f[0]) for f in U.status(0)._fields_)
            assert np.array_equal(A.read_last(swap[s], RING_S * 16000), U.read_last(s, RING_S * 16000))
        assert np.array_equal(A.results()[[0, 3, 2, 1]].view(np.int32), U.results().view(np.int32))
    finally:
        A.close()
        U.close()


@pytest.mark.gpu
def test_published_record_after_import(word):
    """with peer publication on, the imported stream's record reaches the destination copy at the next tick"""
    import torch
    A, B = _busy(word), _busy(word, seed=650)
    try:
        d = torch.full((2, 4, 2), -7, dtype=torch.int32, device="cuda:0")
        B.set_results_peers([d.data_ptr()], stride_records=4, offset_records=0)
        A.poll()
        B.poll()
        raw = A.export_streams([0])
        B.import_streams([3], raw)
        assert np.array_equal(B.results()[3:4].view(np.int32), A.results()[0:1].view(np.int32))
        for c in (A, B):
            c.tick(1)
        B.results()
        h = d.cpu().numpy()[B.publish_parity(), 3]
        assert np.array_equal(h, A.results()[0:1].view(np.int32).reshape(-1))
        B.set_results_peers([])
    finally:
        A.close()
        B.close()


def _snapshot(ctx, n):
    """everything a stream carries: status, input counts, records, rings, and a (read-only) export of every stream,
    whose bytes hold the cursors, latches, parameters, gate state, detector state, block sums, chunk mean squares and
    K8 tails as well"""
    return ([tuple(getattr(ctx.status(s), f[0]) for f in ctx.status(s)._fields_) for s in range(n)],
            [ctx.stream_input(s) for s in range(n)], ctx.results().view(np.int32).copy(),
            np.stack([ctx.read_last(s, RING_S * 16000) for s in range(n)]).view(np.int32),
            ctx.export_streams(list(range(n))))


def _same_snapshot(a, b):
    assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    assert np.array_equal(a[4], b[4])


# (field, byte offset in the meta record, dtype, new value from the old one)
META_MUTATIONS = [
    ("written", 0, "<i8", lambda v: v + 1),
    ("ss_from", 240, "<i8", lambda v: -1),
    ("visible", 144, "<i8", lambda v: 1 << 40),
    ("tick", 16, "<i8", lambda v: -1),
    ("frame_size", 48, "<i4", lambda v: 100),
    ("state", 212, "<i4", lambda v: 4),
    ("dense cursor", 24, "<i8", lambda v: 0),
    ("detect cursor", 32, "<i8", lambda v: 1 << 40),
    ("rate", 52, "<i4", lambda v: 999),
    ("inputs", 40, "<i8", lambda v: v + 1),
    ("tail_len", 56, "<i4", lambda v: 8),
    ("detector mode", 256, "<i4", lambda v: 3),
    ("template range", 124, "<i4", lambda v: 99),
    ("stream parameters", 72, "<f8", lambda v: -1.0),
]


@pytest.mark.gpu
def test_errors_change_nothing(word):
    L = _lib()
    src = _busy(word, n=2, seed=650)
    dst = _busy(word)
    others = []
    try:
        src.poll()
        raw = src.export_streams([1])
        h = raw[:96].view(L.STREAM_BLOB_HEADER_DTYPE)[0]
        before = _snapshot(dst, 4)
        # a non-empty destination queue
        assert dst.status(0).n_events + dst.status(1).n_events + dst.status(2).n_events + dst.status(3).n_events > 0
        with pytest.raises(L.EwkError, match="poll first"):
            dst.import_streams([2], raw)
        _same_snapshot(before, _snapshot(dst, 4))
        dst.poll()

        def refused(blob, streams=(2,), err=ValueError, match=None):
            with pytest.raises(err, match=match):
                dst.import_streams(list(streams), blob)
            _same_snapshot(before, _snapshot(dst, 4))

        refused(raw, (4,), match="bad stream")
        refused(src.export_streams([0, 1]), (2, 2), match="listed twice")
        refused(raw, (2, 3), match="holds 1 streams")
        refused(raw[:-1], match="below")
        refused(raw[:50], match="no blob header")
        for f, v in (("magic", 0x1234), ("version", 2)):
            b = raw.copy()
            b[:96].view(L.STREAM_BLOB_HEADER_DTYPE)[f] = v
            refused(b, match="not a stream blob")
        b = raw.copy()
        b[:96].view(L.STREAM_BLOB_HEADER_DTYPE)["bulk_offset"] += 16
        refused(b, match="section offsets")
        for name, off, dt, fn in META_MUTATIONS:
            b = raw.copy()
            o = int(h["meta_offset"]) + off
            cell = b[o:o + np.dtype(dt).itemsize].view(dt)
            cell[0] = fn(cell[0])
            refused(b, match=f"blob stream 0: {name} is outside")
        # fingerprint: a context that differs in one field each
        for field, kw in (("ring_samples", dict(ring_s=6)), ("slack_samples", dict(slack_s=3)),
                          ("pcm_format", dict(ring="f32")), ("n_mfcc", dict(n_mfcc=13)),
                          ("preemphasis", dict(preemphasis=0.97))):
            o = _ctx(kw.pop("ring", "i16"), n=4, word=word, **kw)
            others.append(o)
            snap = _snapshot(o, 4)
            with pytest.raises(ValueError, match=f"blob's {field}"):
                o.import_streams([0], raw)
            _same_snapshot(snap, _snapshot(o, 4))
        # a template slot that differs in one bit
        o = _ctx("i16", n=4)
        others.append(o)
        mean, std = src.get_template(0)[:2]
        mean = mean.copy()
        mean.view(np.uint32)[3] ^= 1
        o.set_template_features(0, mean, std, src.get_template(0)[2])
        snap = _snapshot(o, 4)
        with pytest.raises(L.EwkError, match="template slot 0"):
            o.import_streams([1], raw)
        _same_snapshot(snap, _snapshot(o, 4))
        # export errors
        with pytest.raises(ValueError, match="listed twice"):
            src.export_streams([1, 1])
        import ctypes as C
        st = np.array([1], np.int32)
        small = np.zeros(64, np.uint8)
        assert src.lib.ewk_export_streams(src.h, st.ctypes.data_as(C.POINTER(C.c_int32)), 1, small.ctypes.data, 64,
                                          L.HOST) == L.EWK_ERR_ARG
        assert "blob_cap" in src.lib.ewk_last_error(src.h).decode()
        empty = L.Context(device=0, n_streams=0)
        others.append(empty)
        with pytest.raises(L.EwkError, match="n_streams = 0"):
            empty.import_streams([0], raw)
        # and the blob still imports
        dst.import_streams([2], raw)
        assert dst.status(2).written == src.status(1).written
    finally:
        for c in [src, dst] + others:
            c.close()


@pytest.mark.gpu
def test_bank_move_streams(word):
    """WakeWordBank.move_streams between two banks at 8 kHz equals the unmoved bank's stream"""
    from easywakeword_b200.bank import WakeWordBank
    kw = dict(buffer_seconds=5, speech_duration_min=0.5, speech_duration_max=1.6, timeout=4.0, sample_rate=8000)
    pcm = _audio(("rs", 8000, "i16"), "i16", word, 3300, 20, n=4)
    a, b, u = WakeWordBank(4, [word], **kw), WakeWordBank(4, [word], **kw), WakeWordBank(4, [word], **kw)
    try:
        ev_u, ev_b = [], []
        for step in range(8):
            blk = np.ascontiguousarray(pcm[:, step * 8000:(step + 1) * 8000])
            for bank in (a, u):
                bank.step(blk)
        ev_u.append(u.poll())
        src_ev, dst_ev = a.move_streams([2], b, [0])
        assert np.array_equal(src_ev, ev_u[0])
        assert a.status(2).written == 0                                # the source slot was recycled
        for step in range(8, 20):
            blk = pcm[2, step * 8000:(step + 1) * 8000]
            b.step_streams([0], [blk])
            u.step_streams([2], [blk])
            ev_b.append(b.poll())
            ev_u.append(u.poll())
        eb, eu = np.concatenate(ev_b), np.concatenate(ev_u[1:])
        eu = eu[eu["stream"] == 2]
        assert len(eb) == len(eu) >= 1
        for f in eb.dtype.names:
            if f != "stream":
                x, y = eb[f], eu[f]
                if x.dtype.kind == "f":
                    x, y = x.view(np.int32), y.view(np.int32)
                assert np.array_equal(x, y), f
        other = WakeWordBank(1, [word], buffer_seconds=5)
        try:
            with pytest.raises(ValueError, match="takes 8000 Hz"):
                other.import_streams([0], a.export_streams([0]))
        finally:
            other.close()
    finally:
        for bank in (a, b, u):
            bank.close()


@pytest.mark.gpu
def test_move_across_gpus(word):
    """cuda:0 -> cuda:1 through a host blob and through a device blob copied with torch"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L = _lib()
    A = _busy(word)
    B = L.Context(device=1, n_streams=4, ring_samples=RING_S * 16000, slack_samples=2 * 16000, pcm_format=L.PCM_I16,
                  max_templates=1, max_events=4096)
    try:
        B.set_template(0, word)
        A.poll()
        raw = A.export_streams([1, 2])
        B.import_streams([0, 1], raw)
        cap = A.stream_blob_bytes(2)
        d0 = torch.zeros(cap, dtype=torch.uint8, device="cuda:0")
        A.export_streams([1, 2], where=L.DEVICE, out=(d0.data_ptr(), cap))
        d1 = d0.to("cuda:1")
        torch.cuda.synchronize(1)
        B.import_streams([3, 2], (d1.data_ptr(), cap), where=L.DEVICE)
        x = synth.stream_batch(601, 2, 4.0, word, gain=(2.0, 4.0))
        for b in range(0, x.shape[1], 16000):
            A.push_streams([1, 2], list(x[:, b:b + 16000]))
            B.push_streams([0, 1, 3, 2], list(x[:, b:b + 16000]) * 2)
            A.tick_ready(64)
            B.tick_ready(64)
        for sa, sbs in ((1, (0, 3)), (2, (1, 2))):
            for sb in sbs:
                assert np.array_equal(A.read_last(sa, RING_S * 16000), B.read_last(sb, RING_S * 16000))
                assert A.status(sa).silence_threshold == B.status(sb).silence_threshold
                assert A.status(sa).n_events == B.status(sb).n_events
    finally:
        A.close()
        B.close()
