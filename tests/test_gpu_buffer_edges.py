"""The caller's memory: every entry point that takes a caller pointer, with that buffer placed inside a larger allocation.

* Device inputs: the bytes around each row, and between rows when the stride exceeds the length, hold NaN (f32),
  0x7FFF / 0x8000 (int16) or arbitrary codes (G.711).  Results must equal, bit for bit, the same call on host input.
* Device outputs: the buffer is pre-filled with a canary no kernel produces.  Afterwards exactly the cells the header
  assigns have changed, they equal the host-output result, and every other byte keeps the canary.
* Host outputs (through the C ABI): arrays padded with guard bytes, each call made twice with two different pre-fills.
  Declared cells do not depend on the pre-fill; bytes outside them do not change.
* Error paths that the header says write nothing leave the canary intact.

Poison mode (test_gpu_poison.py) guards the library's own allocations; these tests guard the caller's.
"""
import ctypes as C

import numpy as np
import pytest

CANARY = np.int32(0x7FA5A5A5)        # a signalling-NaN payload: no kernel stores it (kernels produce quiet NaNs)
PAD = 64                             # elements of neighbourhood on each side of a device row


def _L():
    from easywakeword_b200 import _lib
    return _lib


def _torch():
    import torch
    return torch


def _fill_for(dtype, shape, seed=0):
    """the neighbourhood of a device input: NaN, alternating 0x7FFF / 0x8000, or arbitrary G.711 codes"""
    if dtype == np.float32:
        return np.full(shape, np.nan, np.float32)
    if dtype == np.int16:
        f = np.full(shape, 0x7FFF, np.int16)
        f.reshape(-1)[1::2] = -0x8000
        return f
    return np.random.default_rng(seed).integers(0, 256, size=shape, dtype=np.uint8)


class DevRows:
    """rows [r][n] at column `lead` of a [r][stride] device buffer surrounded by PAD elements of the fill"""

    def __init__(self, rows, stride, lead):
        rows = np.ascontiguousarray(rows)
        r, n = rows.shape
        assert stride >= lead + n
        big = _fill_for(rows.dtype, (r * stride + 2 * PAD,), seed=r * n)
        for i in range(r):
            big[PAD + i * stride + lead:PAD + i * stride + lead + n] = rows[i]
        torch = _torch()
        self.t = torch.from_numpy(big).cuda()
        torch.cuda.synchronize()
        self.ptr = self.t.data_ptr() + (PAD + lead) * rows.itemsize
        self.stride = stride


class Canary:
    """a device output of n 4-byte cells at offset PAD inside a canary-filled int32 buffer"""

    def __init__(self, n):
        torch = _torch()
        self.n = n
        self.t = torch.full((n + 2 * PAD,), int(CANARY), dtype=torch.int32, device="cuda")
        self.ptr = self.t.data_ptr() + PAD * 4

    def read(self):
        _torch().cuda.synchronize()
        a = self.t.cpu().numpy()
        assert (a[:PAD] == CANARY).all() and (a[PAD + self.n:] == CANARY).all(), "write outside the buffer"
        return a[PAD:PAD + self.n]


def assert_cells(got_i32, written, want_f32, what):
    """cells where `written` is set equal want (bit for bit); all others keep the canary"""
    got = got_i32.view(np.float32)
    assert np.array_equal(got[written].view(np.int32), np.ascontiguousarray(want_f32, np.float32).view(np.int32)), what
    assert (got_i32[~written] == CANARY).all(), f"{what}: a cell the call does not own changed"


def _bank(fmt="i16", n=4, R=48000, **kw):
    L = _L()
    c = L.Context(device=0, n_streams=n, ring_samples=R, slack_samples=16000,
                  pcm_format=L.PCM_I16 if fmt == "i16" else L.PCM_F32, max_templates=4, **kw)
    return c


def _word():
    from test_gpu_poison import _word
    return _word()


def _feed(seed, n, seconds, fmt):
    from test_gpu_poison import _feed
    return _feed(seed, n, seconds, fmt, _word())


def _setup(c):
    c.set_template(0, _word())
    c.set_template(1, _word()[:9000])
    c.set_stream_params(-1, frame_size=1600, timeout=3.0, speech_duration_min=0.3, speech_duration_max=2.0,
                        similarity_threshold=0.0)


def _state(c):
    ev = c.poll()
    return (sorted(e.tobytes() for e in ev), c.results().tobytes(),
            [bytes(c.status(s)) for s in range(c.cfg.n_streams)],
            [c.read_last(s, c.cfg.ring_samples).tobytes() for s in range(c.cfg.n_streams)])


# -------------------------------------------------------------------------------------------------- device inputs
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_device_push_reads_only_its_rows(fmt):
    """ewk_push from device rows with stride > n and NaN / 0x7FFF-0x8000 around them == the host push; aligned rows take
    the fused K1, a lead of one element the unaligned path"""
    x = _feed(11, 4, 4.0, fmt)
    a, b = _bank(fmt), _bank(fmt)
    try:
        for c in (a, b):
            _setup(c)
        for k, (p0, p1, lead) in enumerate([(0, 16000, 8), (16000, 24001, 1), (24001, 48000, 3), (48000, 64000, 0)]):
            blk = np.ascontiguousarray(x[:, p0:p1])
            a.push(blk)
            d = DevRows(blk, blk.shape[1] + 40, lead)
            b.push((d.ptr, 4, blk.shape[1], d.stride), where=_L().DEVICE)
            a.tick(10)
            b.tick(10)
            assert _state(a) == _state(b), f"push {k}"
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_device_g711_reads_only_its_rows():
    codes = np.random.default_rng(5).integers(0, 256, size=(4, 16000), dtype=np.uint8)
    a, b = _bank(), _bank()
    try:
        for law in ("ulaw", "alaw"):
            a.push_g711(codes[:, :8000] if law == "ulaw" else codes[:, 8000:], law=law)
            blk = np.ascontiguousarray(codes[:, :8000] if law == "ulaw" else codes[:, 8000:])
            d = DevRows(blk, 8000 + 13, 5)
            b.push_g711((d.ptr, 4, 8000, d.stride), where=_L().DEVICE, law=law)
        a.tick(10)
        b.tick(10)
        assert _state(a) == _state(b)
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", [np.float32, np.int16])
def test_device_native_rate_reads_only_its_rows(dt):
    """push_resampled, push_resampled_each and push_streams (K8) from padded device rows == host input"""
    rng = np.random.default_rng(7)
    y = rng.standard_normal((4, 9000)) * 0.2
    y = (y * 20000).astype(np.int16) if dt == np.int16 else y.astype(np.float32)
    a, b = _bank("f32"), _bank("f32")
    try:
        la = a.push_resampled(y[:, :4410], 44100)
        d = DevRows(y[:, :4410], 4410 + 21, 3)
        lb = b.push_resampled((d.ptr, 4, 4410, d.stride, dt), 44100, where=_L().DEVICE)
        assert la == lb
        la = a.push_resampled_each(y[:, 4410:6000], 44100)
        d = DevRows(y[:, 4410:6000], 1590 + 7, 2)
        lb = b.push_resampled_each((d.ptr, 4, 1590, d.stride, dt), 44100, where=_L().DEVICE)
        assert np.array_equal(la, lb)
        rows = [y[0, 6000:6001], y[2, 6000:9000], y[1, 6000:6500], y[3, 6000:6000]]
        la = a.push_streams([0, 2, 1, 3], rows, sr_in=44100)
        offs, lens, pos = [], [], 5
        for r_ in rows:                                      # packed with gaps of fill between and around rows
            offs.append(pos)
            lens.append(len(r_))
            pos += len(r_) + 9
        buf = _fill_for(np.dtype(dt).type, (pos,), seed=3)
        for o, r_ in zip(offs, rows):
            buf[o:o + len(r_)] = r_
        d = DevRows(buf.reshape(1, -1), len(buf), 0)
        lb = b.push_streams([0, 2, 1, 3], (d.ptr, offs, lens, len(buf), dt), sr_in=44100, where=_L().DEVICE)
        assert np.array_equal(la, lb)
        a.tick_ready(10)
        b.tick_ready(10)
        assert _state(a) == _state(b)
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_level2_device_inputs_read_only_their_ranges():
    """similarity_batch, set_templates (+ VAD), extract_mfcc and resample on device input surrounded by NaN / int16
    extremes == host input"""
    L = _L()
    from easywakeword_b200 import synth
    word = _word()
    x = synth.from_int16(synth.to_int16(synth.stream(5, 4.0, word, gain=(2.0, 3.0))[0]))
    c = L.Context(device=0, n_streams=0, max_templates=8)
    try:
        c.set_template(0, word)
        offs, lens = [100, 9000, 30000], [8000, 50000, 1601]
        for pcm in (x, synth.to_int16(x)):
            want = c.similarity_batch(0, pcm, offs, lens, want_features=True)
            d = DevRows(pcm.reshape(1, -1), len(pcm), 0)
            buf = np.asarray(d.t.cpu().numpy())               # blank everything outside the segments
            keep = np.zeros(len(buf), bool)
            for o, n in zip(offs, lens):
                keep[PAD + o:PAD + o + n] = True
            fill = _fill_for(pcm.dtype.type, buf.shape)
            buf[~keep] = fill[~keep]
            d.t.copy_(_torch().from_numpy(buf))
            sc, mt, ft = np.empty(3, np.float32), np.empty(3, np.uint8), np.empty((3, 40), np.float32)
            o, l = np.asarray(offs, np.int64), np.asarray(lens, np.int64)
            c._ck(c.lib.ewk_similarity_batch(c.h, 0, d.ptr, L.PCM_I16 if pcm.dtype == np.int16 else L.PCM_F32, L.DEVICE,
                                             L.i64ptr(o), L.i64ptr(l), 3, 75.0, L.f32ptr(sc), L.u8ptr(mt), L.f32ptr(ft)))
            assert np.array_equal(sc.view(np.int32), want[0].view(np.int32))
            assert np.array_equal(ft.view(np.int32), want[2].view(np.int32))
        # templates from NaN-separated device audio == host templates, VAD too
        segs = [x[:1], x[500:3500], x[4000:52000]]
        vh = c.set_templates([1, 2, 3], segs, want_vad=True)
        th = [c.get_template(k) for k in (1, 2, 3)]
        buf = _fill_for(np.float32, (3 + sum(len(s) for s in segs) + 3 * 11,))
        offs, pos = [], 3
        for s in segs:
            buf[pos:pos + len(s)] = s
            offs.append(pos)
            pos += len(s) + 11
        d = DevRows(buf.reshape(1, -1), len(buf), 0)
        vd = c.set_templates([4, 5, 6], (d.ptr, offs, [len(s) for s in segs]), want_vad=True)
        assert vh.tobytes() == vd.tobytes()
        for k, t in zip((4, 5, 6), th):
            got = c.get_template(k)
            assert got[2] == t[2] and got[0].tobytes() == t[0].tobytes() and got[1].tobytes() == t[1].tobytes()
        # extract_mfcc
        seg = x[1000:25007]
        m0, s0, f0 = c.extract_mfcc(seg, want_frames=True)
        d = DevRows(seg.reshape(1, -1), len(seg) + 17, 5)
        m, s, fr = np.empty(20, np.float32), np.empty(20, np.float32), np.empty_like(f0)
        c._ck(c.lib.ewk_extract_mfcc(c.h, d.ptr, len(seg), L.DEVICE, L.f32ptr(m), L.f32ptr(s), L.f32ptr(fr), len(fr)))
        assert m.tobytes() == m0.tobytes() and s.tobytes() == s0.tobytes() and fr.tobytes() == f0.tobytes()
        # resample: rows with stride > n_in, fill between them
        for dt in (np.float32, np.int16):
            y = np.random.default_rng(2).standard_normal((3, 4801))
            y = (y * 9000).astype(np.int16) if dt == np.int16 else y.astype(np.float32)
            want = c.resample(y, 48000)
            d = DevRows(y, 4801 + 30, 7)
            got = np.empty_like(want)
            c._ck(c.lib.ewk_resample(c.h, d.ptr, L.PCM_I16 if dt == np.int16 else L.PCM_F32, L.DEVICE, 3, 4801, d.stride,
                                     48000, 0, 0, want.shape[1], got.ctypes.data, want.shape[1], L.HOST))
            assert got.tobytes() == want.tobytes()
    finally:
        c.close()


@pytest.mark.gpu
def test_device_blob_import_reads_only_the_blob():
    """import from a device blob followed by garbage == import of the host blob"""
    torch = _torch()
    L = _L()
    src = _bank("f32")
    a, b = _bank("f32"), _bank("f32")
    try:
        for c in (src, a, b):
            _setup(c)
        x = _feed(13, 4, 2.0, "f32")
        src.push(np.ascontiguousarray(x))
        src.tick(10)
        src.poll()
        blob = src.export_streams([2, 0])
        t = torch.from_numpy(np.concatenate([blob, np.full(4096, 0xA5, np.uint8)])).cuda()
        torch.cuda.synchronize()
        a.import_streams([1, 3], blob)
        b.import_streams([1, 3], (t.data_ptr(), len(blob)), where=L.DEVICE)
        a.tick_ready(10)
        b.tick_ready(10)
        assert _state(a) == _state(b)
    finally:
        for c in (src, a, b):
            c.close()


# -------------------------------------------------------------------------------------------------- device outputs
@pytest.mark.gpu
def test_k5_device_output_writes_only_its_segments():
    """ewk_prepare_segments: segments at offsets with gaps; the gaps and the neighbourhood keep the canary"""
    L = _L()
    c = _bank("f32")
    try:
        x = _feed(17, 4, 3.0, "f32")
        for b0 in range(0, 48000, 16000):
            c.push(np.ascontiguousarray(x[:, b0:b0 + 16000]))
            c.tick(10)
        st, a, ln = [0, 3, 1], [20000, 1000, 40000], [1600, 333, 7000]
        want = c.prepare_segments(st, a, ln)
        offs = np.array([5, 1700, 2100], np.int64)
        out = Canary(9200)
        s32, a64, l64 = np.asarray(st, np.int32), np.asarray(a, np.int64), np.asarray(ln, np.int64)
        c._ck(c.lib.ewk_prepare_segments(c.h, 3, s32.ctypes.data_as(C.POINTER(C.c_int32)), L.i64ptr(a64), L.i64ptr(l64),
                                         L.i64ptr(offs), C.cast(out.ptr, C.POINTER(C.c_float)), out.n, L.DEVICE))
        got = out.read()
        written = np.zeros(out.n, bool)
        for o, n in zip(offs, ln):
            written[o:o + n] = True
        assert_cells(got, written, np.concatenate(want), "K5 device output")
        # an overwritten segment is an error, and a failed call writes nothing
        for b0 in range(0, 48000, 16000):
            c.push(np.ascontiguousarray(x[:, b0:b0 + 16000]))
            c.tick(10)
        out2 = Canary(9200)
        rc = c.lib.ewk_prepare_segments(c.h, 3, s32.ctypes.data_as(C.POINTER(C.c_int32)), L.i64ptr(a64), L.i64ptr(l64),
                                        L.i64ptr(offs), C.cast(out2.ptr, C.POINTER(C.c_float)), out2.n, L.DEVICE)
        assert rc == L.EWK_ERR_STATE
        assert (out2.read() == CANARY).all()
    finally:
        c.close()


@pytest.mark.gpu
def test_dense_device_outputs_write_only_their_rows():
    """every dense form with out_cap larger than needed: the packed rows equal the host output, the rest keeps the canary;
    a failed call writes nothing"""
    a, b = _bank("i16"), _bank("i16")
    try:
        x = _feed(19, 4, 3.0, "i16")
        for c in (a, b):
            _setup(c)
            c.push(np.ascontiguousarray(x))
        # dense_scores: the full [n_streams][n_hops][T] grid
        want = a.dense_scores(5, 30, 0, 2)
        out = Canary(want.size + 100)
        b.dense_scores(5, 30, 0, 2, out_device_ptr=out.ptr)
        w = np.zeros(out.n, bool)
        w[:want.size] = True
        assert_cells(out.read(), w, want.reshape(-1), "dense_scores")
        # dense_scores_streams
        st, h0, nh = [3, 1, 0], [40, 2, 9], [20, 0, 33]
        want = np.concatenate([r.reshape(-1) for r in a.dense_scores_streams(st, h0, nh, 0, 2)])
        out = Canary(want.size + 77)
        b.dense_scores_streams(st, h0, nh, 0, 2, out_device_ptr=out.ptr, out_cap=out.n)
        w = np.zeros(out.n, bool)
        w[:want.size] = True
        assert_cells(out.read(), w, want, "dense_scores_streams")
        # dense_ready and dense_detect: cursors move alike in both contexts
        ha, rows = a.dense_ready([2, 0], 50, 0, 2)
        want = np.concatenate([r.reshape(-1) for r in rows])
        out = Canary(2 * 50 * 2 + 31)
        hb, nb = b.dense_ready([2, 0], 50, 0, 2, out_device_ptr=out.ptr, out_cap=out.n)
        assert np.array_equal(ha, hb)
        w = np.zeros(out.n, bool)
        w[:want.size] = True
        assert_cells(out.read(), w, want, "dense_ready")
        da, (ha, rows) = a.dense_detect(None, 60, 0, 2, scores=True)
        want = np.concatenate([r.reshape(-1) for r in rows])
        out = Canary(4 * 60 * 2 + 13)
        db, (hb, nb) = b.dense_detect(None, 60, 0, 2, out_device_ptr=out.ptr, out_cap=out.n)
        assert da.tobytes() == db.tobytes() and np.array_equal(ha, hb)
        w = np.zeros(out.n, bool)
        w[:want.size] = True
        assert_cells(out.read(), w, want, "dense_detect scores")
        # error: a row whose hops are not pushed yet scores nothing
        out = Canary(500)
        with pytest.raises(RuntimeError):
            b.dense_scores_streams([0], [290], [40], 0, 2, out_device_ptr=out.ptr, out_cap=out.n)
        assert (out.read() == CANARY).all()
    finally:
        a.close()
        b.close()


@pytest.mark.gpu
def test_resample_device_output_with_stride():
    L = _L()
    c = L.Context(device=0, n_streams=0, max_templates=1)
    try:
        y = np.random.default_rng(4).standard_normal((3, 2205)).astype(np.float32)
        want = c.resample(y, 22050, in_first=4, out_first=2, n_out=1500)
        stride = 1500 + 37
        out = Canary(3 * stride)
        c._ck(c.lib.ewk_resample(c.h, y.ctypes.data, L.PCM_F32, L.HOST, 3, 2205, 2205, 22050, 4, 2, 1500, out.ptr, stride,
                                 L.DEVICE))
        w = np.zeros(out.n, bool)
        for r in range(3):
            w[r * stride:r * stride + 1500] = True
        assert_cells(out.read(), w, want.reshape(-1), "resample out_device_ptr")
    finally:
        c.close()


@pytest.mark.gpu
def test_export_into_a_larger_buffer():
    """the device blob equals the host blob; bytes past total_bytes keep the canary; a too-small cap writes nothing"""
    torch = _torch()
    L = _L()
    c = _bank("f32")
    try:
        _setup(c)
        c.push(np.ascontiguousarray(_feed(23, 4, 2.0, "f32")))
        want = c.export_streams([3, 1])
        cap = c.stream_blob_bytes(2) + 256
        buf = torch.full((cap + 64,), 0xA5, dtype=torch.uint8, device="cuda")
        c.export_streams([3, 1], where=L.DEVICE, out=(buf.data_ptr(), cap))
        torch.cuda.synchronize()
        got = buf.cpu().numpy()
        assert got[:len(want)].tobytes() == want.tobytes()
        assert (got[len(want):] == 0xA5).all()
        buf.fill_(0xA5)
        with pytest.raises(ValueError):
            c.export_streams([3, 1], where=L.DEVICE, out=(buf.data_ptr(), len(want) - 16))
        torch.cuda.synchronize()
        assert (buf.cpu().numpy() == 0xA5).all()
    finally:
        c.close()


@pytest.mark.gpu
def test_results_buffer_and_peer_destinations_write_only_their_records():
    """set_results_buffer inside a larger allocation, and set_results_peers with stride and offset: only the records of
    the streams change, and they equal ewk_stream_results"""
    torch = _torch()
    n = 6
    c = _bank("i16", n=n)
    try:
        _setup(c)
        own = Canary(2 * n)
        c.set_results_buffer(own.ptr)
        stride, off = 20, 7
        dest = Canary(2 * 2 * stride)
        c.set_results_peers([dest.ptr], stride_records=stride, offset_records=off)
        x = _feed(29, n, 3.0, "i16")
        for b0 in range(0, x.shape[1], 16000):
            c.push(np.ascontiguousarray(x[:, b0:b0 + 16000]))
            c.tick(10)
        c.synchronize()
        torch.cuda.synchronize()
        res = c.results().view(np.int32)
        assert np.array_equal(own.read(), res)
        d = dest.read().reshape(2, stride, 2)
        par = c.publish_parity()
        mine = np.zeros((2, stride), bool)
        mine[:, off:off + n] = True
        assert (d[~mine] == CANARY).all(), "a peer record outside [offset, offset + n) changed"
        assert np.array_equal(d[par, off:off + n].reshape(-1), res)
        c.set_results_peers([])
    finally:
        c.close()


# -------------------------------------------------------------------------------------------------- host outputs
def _guarded(n, dtype, byte):
    """(raw bytes, view of n cells) with 64 guard bytes on each side, all pre-filled with `byte`"""
    item = np.dtype(dtype).itemsize
    raw = np.full(n * item + 128, byte, np.uint8)
    return raw, raw[64:64 + n * item].view(dtype)


def _guards_ok(raw, byte):
    return (raw[:64] == byte).all() and (raw[-64:] == byte).all()


@pytest.mark.gpu
def test_host_outputs_write_only_declared_cells():
    """read_last, read_segment, get_template and stream_results, each twice with two pre-fills"""
    L = _L()
    c = _bank("f32")
    try:
        _setup(c)
        c.push(np.ascontiguousarray(_feed(31, 4, 2.0, "f32")))
        c.tick(10)
        got = {}
        for byte in (0x00, 0xFF):
            raw, v = _guarded(5000, np.float32, byte)
            c._ck(c.lib.ewk_read_last(c.h, 2, 5000, C.cast(v.ctypes.data, C.POINTER(C.c_float))))
            assert _guards_ok(raw, byte)
            raw2, v2 = _guarded(777, np.float32, byte)
            c._ck(c.lib.ewk_read_segment(c.h, 1, 20000, 777, C.cast(v2.ctypes.data, C.POINTER(C.c_float))))
            assert _guards_ok(raw2, byte)
            rm, m = _guarded(20, np.float32, byte)
            rs, s = _guarded(20, np.float32, byte)
            rn, nn = _guarded(1, np.int64, byte)
            c._ck(c.lib.ewk_get_template(c.h, 1, C.cast(m.ctypes.data, C.POINTER(C.c_float)),
                                         C.cast(s.ctypes.data, C.POINTER(C.c_float)), C.cast(nn.ctypes.data, C.POINTER(C.c_int64))))
            assert _guards_ok(rm, byte) and _guards_ok(rs, byte) and _guards_ok(rn, byte)
            rr, res = _guarded(4, L.RESULT_DTYPE, byte)
            c._ck(c.lib.ewk_stream_results(c.h, res.ctypes.data))
            assert _guards_ok(rr, byte)
            got[byte] = (v.tobytes(), v2.tobytes(), m.tobytes(), s.tobytes(), nn.tobytes(), res.tobytes())
        assert got[0x00] == got[0xFF]
    finally:
        c.close()


@pytest.mark.gpu
def test_poll_trace_and_detect_records_write_only_declared_cells():
    """ewk_poll with cap below the event count, ewk_tick_trace / ewk_tick_ready with NULL pointers and ewk_dense_detect
    records: two contexts fed alike, one pre-fill each; declared cells agree, guards stay"""
    L = _L()
    ctxs = [_bank("i16", n=8, max_events=64), _bank("i16", n=8, max_events=64)]
    try:
        x = _feed(37, 8, 4.0, "i16")
        out = []
        for c, byte in zip(ctxs, (0x00, 0xFF)):
            _setup(c)
            rec = []
            for b0 in range(0, 48000, 16000):
                c.push(np.ascontiguousarray(x[:, b0:b0 + 16000]))
                rst, state = _guarded(8 * 10, np.uint8, byte)
                rrm, rms = _guarded(8 * 10, np.float64, byte)
                c._ck(c.lib.ewk_tick_trace(c.h, 10, None, state.ctypes.data, None, rms.ctypes.data))
                assert _guards_ok(rst, byte) and _guards_ok(rrm, byte)
                rec.append((state.tobytes(), rms.tobytes()))
            c.push(np.ascontiguousarray(x[:, 48000:]))
            rtk, taken = _guarded(8, np.int32, byte)
            rth, thr = _guarded(8 * 12, np.float64, byte)
            c._ck(c.lib.ewk_tick_ready(c.h, 12, taken.ctypes.data_as(C.POINTER(C.c_int32)), None, None, thr.ctypes.data, None))
            assert _guards_ok(rtk, byte) and _guards_ok(rth, byte)
            rec.append((taken.tobytes(), thr.tobytes()))
            cap = 3
            rev, ev = _guarded(cap, L.EVENT_DTYPE, byte)
            dropped = C.c_int(-5)
            k = c.lib.ewk_poll(c.h, ev.ctypes.data, cap, C.byref(dropped))
            assert 0 <= k <= cap and _guards_ok(rev, byte)
            rec.append((k, ev[:k].tobytes(), (ev.view(np.uint8)[k * L.EVENT_DTYPE.itemsize:] == byte).all()))
            det_cap = 8 * 25
            rdt, det = _guarded(det_cap, L.DETECTION_DTYPE, byte)
            h0, nh = np.zeros(8, np.int64), np.zeros(8, np.int32)
            k = c.lib.ewk_dense_detect(c.h, None, 8, 50, 0, 2, 20, 50, det.ctypes.data, det_cap, L.i64ptr(h0),
                                       nh.ctypes.data_as(C.POINTER(C.c_int32)), None, 0, L.HOST)
            assert k >= 0 and _guards_ok(rdt, byte)
            assert (det.view(np.uint8)[k * L.DETECTION_DTYPE.itemsize:] == byte).all(), "records past the count changed"
            rec.append((k, det[:k].tobytes(), h0.tobytes(), nh.tobytes()))
            out.append(rec)
        assert out[0] == out[1]
    finally:
        for c in ctxs:
            c.close()
