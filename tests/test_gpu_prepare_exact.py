"""K5 (segment_prepare_kernel, ewk_prepare_segments): the level-3 hand-off pinned bit for bit.

int16 rings: every sample is a multiple of 2^-15, so a segment's double sum (at most a whole ring) is exact in any
order, and K5's mean, subtraction, division, x1.5 and clip are the IEEE operations of the reference's float64 formula
(oracle.ewk_oracle.prepare_for_level3).  The output is that formula's result rounded to float32, bit for bit.
f32 rings: the double sum is not exact in general, so the output is compared with a model of K5's summation order
(prep_model): 256-thread strided double partial sums, a xor tree per warp, the 8 warp sums in order, / len.

Edges: lengths 1 .. a whole ring, segments across the ring end, constant segments (max |x - mean| = 0: zeros),
full-scale runs (the clip), many segments packed with gaps in one call, host and device output, segments from gated
events and from dense_detect records, and every error, each of which leaves the output buffer untouched."""
import ctypes as C

import numpy as np
import pytest

from easywakeword_b200 import synth
from oracle import ewk_oracle as O

SENTINEL = np.uint32(0x7FC0BEEF)                             # a NaN no computation produces
LANE = np.arange(32)


def k5_mean(v):
    """K5's mean of a float64 segment: thread t adds v[t], v[t + 256], ... from 0.0; each warp's 32 partials go through
    a xor butterfly (offsets 16, 8, 4, 2, 1) and lane 0's value is the warp sum; the 8 warp sums are added in order
    from 0.0; the total is divided by the length."""
    v = np.asarray(v, np.float64)
    part = np.zeros(256)
    for i in range(0, len(v), 256):
        seg = v[i:i + 256]
        part[:len(seg)] = part[:len(seg)] + seg
    t = 0.0
    for w in range(8):
        s = part[32 * w:32 * w + 32]
        for o in (16, 8, 4, 2, 1):
            s = s + s[LANE ^ o]
        t = t + s[0]
    return t / float(len(v))


def prep_model(v):
    """K5 on a float64 segment: x - mean (k5_mean), / max |x - mean| when > 0, * 1.5, clip to [-1, 1], float32."""
    d = np.asarray(v, np.float64) - k5_mean(v)
    mx = np.max(np.abs(d))
    if mx > 0:
        d = d / mx
    return np.clip(d * 1.5, -1.0, 1.0).astype(np.float32)


def want_for(vals, fmt):
    return O.prepare_for_level3(vals).astype(np.float32) if fmt == "i16" else prep_model(vals)


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


# ---------------------------------------------------------------------------------------------------- CPU: the model
def test_model_is_the_reference_formula_on_int16_values():
    """On multiples of 2^-15 the model's mean is exact, so the model is the reference formula bit for bit."""
    rng = np.random.default_rng(1)
    for n in (1, 31, 32, 255, 256, 257, 1000, 48000):
        q = rng.integers(-32768, 32768, n).astype(np.float64) / 32768.0
        assert np.array_equal(bits(prep_model(q)), bits(O.prepare_for_level3(q).astype(np.float32))), n


def test_model_against_the_reference_formula_on_float32_values():
    """On general float32 values the order of the double sum shows: the mean may differ in its last bits, and after
    rounding to float32 an output differs from the formula's by at most one ulp."""
    rng = np.random.default_rng(2)
    n_diff = n_all = 0
    for k in range(60):
        n = int(rng.integers(1, 48001))
        x = (rng.standard_normal(n) * np.exp(rng.uniform(-20, 2, n)) + rng.uniform(-0.5, 0.5)).astype(np.float32)
        a, b = bits(prep_model(x.astype(np.float64))), bits(O.prepare_for_level3(x.astype(np.float64)).astype(np.float32))
        d = np.abs(a.astype(np.int64) - b.astype(np.int64))
        assert d.max() <= 1, k
        n_diff += int(np.sum(d != 0))
        n_all += n
    print(f"K5 model vs reference formula on float32 values: {n_diff} of {n_all} samples differ by one ulp")


# ---------------------------------------------------------------------------------------------------- GPU
RING, SLACK = 48000, 16000


class Fed:
    """A context whose streams hold known audio: vals[s] is what stream s's ring received (float64)."""

    def __init__(self, fmt, pcm, templates=(), ring=RING, slack=SLACK, on_chunk=None):
        """pcm: [n_streams, n] in the ring's dtype (int16 for "i16", float32 for "f32")."""
        from easywakeword_b200 import _lib
        self.fmt, self._lib = fmt, _lib
        self.ctx = _lib.Context(device=0, n_streams=len(pcm), ring_samples=ring, slack_samples=slack,
                                pcm_format=_lib.PCM_I16 if fmt == "i16" else _lib.PCM_F32, max_templates=4)
        self.P = (ring + slack + 63) // 64 * 64
        for i, t in enumerate(templates):
            self.ctx.set_template(i, t)
        self.ctx.set_stream_params(-1, frame_size=1600, template_count=1, live=0)
        pcm = np.asarray(pcm)
        assert pcm.dtype == (np.int16 if fmt == "i16" else np.float32)
        self.vals = pcm.astype(np.float64) / (32768.0 if fmt == "i16" else 1.0)
        self.written = 0
        self.events = []
        self.n_checked = self.n_off_ref = 0          # f32 rings: samples checked, and those one ulp off the formula
        for p in range(0, pcm.shape[1], 16000):
            blk = np.ascontiguousarray(pcm[:, p:p + 16000])
            self.ctx.push(blk)
            self.written += blk.shape[1]
            self.ctx.tick(blk.shape[1] // 1600)
            self.events.append(self.ctx.poll().copy())
            if on_chunk is not None:
                on_chunk(self)

    def raw(self, streams, starts, lens, offs, out, out_len, where):
        st = np.ascontiguousarray(streams, np.int32)
        a, ln, of = (np.ascontiguousarray(v, np.int64) for v in (starts, lens, offs))
        from easywakeword_b200._lib import i64ptr
        return self.ctx.lib.ewk_prepare_segments(self.ctx.h, len(st), st.ctypes.data_as(C.POINTER(C.c_int32)),
                                                  i64ptr(a), i64ptr(ln), i64ptr(of), C.cast(out, C.POINTER(C.c_float)),
                                                  int(out_len), where)

    def prepare(self, segs, where="host", gap=0, lead=0):
        """segs: [(stream, start, len)] -> (list of outputs, whole buffer as uint32).  Segments are packed from `lead`
        with `gap` sentinel floats between them; the sentinel must survive everywhere outside the segments."""
        lens = [l for _, _, l in segs]
        offs = lead + np.concatenate([[0], np.cumsum(np.asarray(lens) + gap)[:-1]]).astype(np.int64)
        out_len = int(offs[-1] + lens[-1] + gap)
        buf = np.full(out_len, SENTINEL, np.uint32)
        if where == "host":
            rc = self.raw([s for s, _, _ in segs], [a for _, a, _ in segs], lens, offs, buf.ctypes.data, out_len,
                          self._lib.HOST)
            got = buf
        else:
            import torch
            t = torch.from_numpy(buf.view(np.int32)).cuda()
            torch.cuda.synchronize()
            rc = self.raw([s for s, _, _ in segs], [a for _, a, _ in segs], lens, offs, t.data_ptr(), out_len,
                          self._lib.DEVICE)
            got = t.cpu().numpy().view(np.uint32)
        assert rc == 0, (rc, self.ctx.lib.ewk_last_error(self.ctx.h))
        outside = np.ones(out_len, bool)
        for o, l in zip(offs, lens):
            outside[o:o + l] = False
        assert np.all(got[outside] == SENTINEL), f"{where}: {int(np.sum(got[outside] != SENTINEL))} floats outside the segments changed"
        return [got[o:o + l].view(np.float32) for o, l in zip(offs, lens)]

    def check(self, segs, **kw):
        outs = self.prepare(segs, **kw)
        for (s, a, l), g in zip(segs, outs):
            w = want_for(self.vals[s, a:a + l], self.fmt)
            if not np.array_equal(bits(g), bits(w)):
                bad = np.flatnonzero(bits(g) != bits(w))
                raise AssertionError(f"{self.fmt} stream {s} [{a}, +{l}) {kw}: {len(bad)} of {l} samples differ, e.g. "
                                     f"{[(int(i), float(g[i]), float(w[i])) for i in bad[:4]]}")
            if self.fmt == "f32":
                ref = bits(O.prepare_for_level3(self.vals[s, a:a + l]).astype(np.float32)).astype(np.int64)
                d = np.abs(bits(g).astype(np.int64) - ref)
                assert d.max() <= 1, (s, a, l)
                self.n_checked += l
                self.n_off_ref += int(np.sum(d != 0))
        return outs

    def close(self):
        self.ctx.close()


def to_ring(xs, fmt):
    return np.stack([synth.to_int16(x) if fmt == "i16" else np.asarray(x, np.float32) for x in xs])


N_FIX = 116800                                               # 7.3 s: each ring lapped almost twice
CONST_AT, FULL_AT = N_FIX - 14000, N_FIX - 8000              # both still in the ring at the end


@pytest.fixture(scope="module", params=["i16", "f32"])
def fed(request):
    """Three streams of noise with a DC offset (the mean matters), a constant stretch of 3000 samples at CONST_AT
    (max |x - mean| = 0 for segments inside it) and a full-scale run of 700 samples at FULL_AT (-32768 on int16 rings,
    -1.0 on f32 rings) followed by 20 samples at 0.9."""
    fmt = request.param
    rng = np.random.default_rng(11)
    xs = [(rng.standard_normal(N_FIX) * rng.uniform(0.001, 0.3) + rng.uniform(-0.2, 0.2)).astype(np.float32)
          for _ in range(3)]
    pcm = to_ring(xs, fmt)
    full = -32768 if fmt == "i16" else -1.0
    pcm[:, CONST_AT:CONST_AT + 3000] = pcm[:, CONST_AT:CONST_AT + 1]
    pcm[:, FULL_AT:FULL_AT + 700] = full
    pcm[:, FULL_AT + 700:FULL_AT + 720] = 29491 if fmt == "i16" else 0.9
    f = Fed(fmt, pcm)
    yield f
    f.close()


def edge_segments(f, rng):
    """(stream, start, len) at every edge class, all still in the ring."""
    w, Pp = f.written, f.P
    lo = w - Pp                                                  # oldest sample still held
    segs = []
    for s in range(f.vals.shape[0]):
        for l in (1, 31, 32, 33, 255, 256, 257, 511, 4097, 48000):
            segs.append((s, int(rng.integers(lo, w - l + 1)), l))
        segs.append((s, lo, Pp))                                # a whole ring
        wrap = (w // Pp) * Pp                                    # absolute sample at physical position 0
        for l in (2, 257, 9000):
            for before in (1, l // 2, l - 1):
                a = wrap - before
                if a >= lo and a + l <= w:
                    segs.append((s, a, l))                      # across the ring end
    return segs


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["host", "device"])
def test_edges_bit_for_bit(fed, where):
    rng = np.random.default_rng(3 if where == "host" else 4)
    segs = edge_segments(fed, rng)
    fed.check(segs, where=where, gap=3, lead=5)                 # many segments in one call, packed with gaps
    if fed.fmt == "f32":
        print(f"f32 ring, {where} output: {fed.n_off_ref} of {fed.n_checked} samples differ by one ulp from the "
              "reference formula (float64, numpy's pairwise mean)")


@pytest.mark.gpu
def test_constant_and_full_scale_segments(fed):
    """Constant segments give zeros (max |x - mean| = 0 skips the division).  Segments holding the full-scale run
    drive the clip: in [FULL_AT, +720) the 20 samples at 0.9 are the farthest from the mean, land on 1.5 and clip to
    1.0; in [FULL_AT - 100, +800) the louder part of the noise before the run clips."""
    assert fed.written - fed.P < CONST_AT
    segs = []
    for s in range(3):
        segs += [(s, CONST_AT, 1), (s, CONST_AT, 3000), (s, CONST_AT + 10, 257), (s, CONST_AT + 700, 256)]
        segs += [(s, FULL_AT - 100, 800), (s, FULL_AT, 720), (s, FULL_AT - 3000, 4000), (s, FULL_AT, 700)]
    outs = fed.check(segs, gap=2)
    for (s, a, l), o in zip(segs, outs):
        if a >= CONST_AT and a + l <= CONST_AT + 3000 or (a, l) == (FULL_AT, 700):
            assert np.all(bits(o) == 0), (s, a, l)
        if (a, l) == (FULL_AT, 720):
            assert np.sum(o == 1.0) == 20 and np.all(o[700:] == 1.0), s
        if (a, l) == (FULL_AT - 100, 800):
            assert np.sum(o == 1.0) >= 20, (s, int(np.sum(o == 1.0)))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_segments_of_gated_events_and_dense_detections(fmt, word):
    """What a caller hands on: the segments of the gate's scored events (poll) and of dense_detect records, prepared
    in one call each as soon as they are reported."""
    xs = [synth.stream(8100 + i, 24.0, word, gain=(1.5, 3.0), inserts_per_10s=(3, 3))[0] for i in range(3)]
    seen = {"gate": 0, "dense": 0}

    def on_chunk(f):
        d = f.ctx.dense_detect(None, 200, 0, 1, 20, 50)
        segs = [(int(r["stream"]), int(r["seg_start"]), int(r["seg_len"])) for r in d]
        if segs:
            f.check(segs, where="device", gap=1)
            seen["dense"] += len(segs)
        segs = [(int(e["stream"]), int(e["seg_start"]), int(e["seg_len"])) for e in f.events[-1] if e["kind"] == 2]
        if segs:
            f.check(segs, where="host")
            seen["gate"] += len(segs)

    f = Fed(fmt, to_ring(xs, fmt), templates=[word], ring=160000, on_chunk=on_chunk)
    try:
        assert seen["gate"] >= 3 and seen["dense"] >= 3, seen
    finally:
        f.close()


@pytest.mark.gpu
def test_errors_leave_the_output_untouched(fed):
    from easywakeword_b200 import _lib
    import torch
    w, Pp = fed.written, fed.P
    good = (0, w - 1000, 500)
    cases = {
        "not pushed yet": ([good, (1, w - 10, 11)], _lib.EWK_ERR_STATE),
        "overwritten": ([good, (2, w - Pp - 1, 100)], _lib.EWK_ERR_STATE),
        "len < 1": ([good, (1, w - 100, 0)], _lib.EWK_ERR_ARG),
        "len > P": ([(1, w - Pp - 1, Pp + 1)], _lib.EWK_ERR_ARG),
        "negative start": ([good, (1, -1, 10)], _lib.EWK_ERR_ARG),
        "stream out of range": ([good, (3, w - 100, 10)], _lib.EWK_ERR_ARG),
    }
    for name, (segs, rc_want) in cases.items():
        lens = [l for _, _, l in segs]
        offs = np.concatenate([[0], np.cumsum(np.maximum(lens, 1))[:-1]]).astype(np.int64)
        n = int(offs[-1] + max(lens[-1], 1))
        for where in ("host", "device"):
            buf = np.full(n, SENTINEL, np.uint32)
            if where == "host":
                rc = fed.raw(*zip(*segs), offs, buf.ctypes.data, n, _lib.HOST)
                after = buf
            else:
                t = torch.from_numpy(buf.copy().view(np.int32)).cuda()
                torch.cuda.synchronize()
                rc = fed.raw(*zip(*segs), offs, t.data_ptr(), n, _lib.DEVICE)
                after = t.cpu().numpy().view(np.uint32)
            assert rc == rc_want, (name, where, rc)
            assert np.all(after == SENTINEL), (name, where)
    # out_offsets out of range: negative, and one past out_len
    for offs, n in (([-1], 500), ([1], 500)):
        buf = np.full(n, SENTINEL, np.uint32)
        rc = fed.raw([0], [w - 1000], [500], np.asarray(offs, np.int64), buf.ctypes.data, n, _lib.HOST)
        assert rc == _lib.EWK_ERR_ARG and np.all(buf == SENTINEL), offs
    # a failed call leaves the context usable
    fed.check([good])
