"""GPU: frame alignment (include/ewk.h: ewk_get_template_frames, ewk_align_segments, ewk_align_buffers; K11).

The template frame store equals ewk_extract_mfcc's frames of each slot's audio bit for bit, from every writer; every
distance equals oracle/align_model.py bit for bit, computed from ctx.extract_mfcc frames of the same audio; the ring
form equals the buffer form of read_segment's audio; outputs agree across host / device, batched / per row, and
best_slot / best_dist are the argmin; errors write nothing; poison mode changes no byte."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

from easywakeword_b200 import _lib, synth
from easywakeword_b200.bank import WakeWordBank
from oracle import align_model as A

pytestmark = pytest.mark.gpu

SR = 16000
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MARGIN = 0.10                      # tests/test_align_model.py: order impostors vs perturbations on the bundled word
CFGS = [{}, {"n_mfcc": 13, "preemphasis": 0.97}]
CFG_IDS = ["default", "mfcc13_pre097"]


def _word():
    g = np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))
    return g["pcm_i16"].astype(np.float32) / np.float32(32768)


def ctx_(n=0, slots=80, fmt=_lib.PCM_I16, ring=4 * SR, frames=True, **kw):
    return _lib.Context(device=0, n_streams=n, ring_samples=ring, slack_samples=SR, pcm_format=fmt, max_templates=slots,
                        max_events=8192, template_frames=frames, **kw)


def audios(lens, seed):
    """word-like float32 audio of these lengths at random gains over a little noise"""
    rng = np.random.default_rng(seed)
    base = np.concatenate([synth.synthetic_word(seed=seed + i, duration=0.6 + 0.1 * i) for i in range(6)])
    out = []
    for L in lens:
        o = int(rng.integers(0, max(1, len(base) - L))) if L < len(base) else 0
        w = np.resize(base[o:], L)
        out.append((w * np.float32(rng.uniform(0.5, 3.0)) +
                    rng.standard_normal(L).astype(np.float32) * np.float32(0.003)).astype(np.float32))
    return out


def C_of(ctx):
    return int(ctx.cfg.n_mfcc) or 20


class Model:
    """oracle distances from the device's own frames: ctx.extract_mfcc of the segment, the slot's stored frames"""

    def __init__(self, ctx):
        self.ctx, self.C, self.t = ctx, C_of(ctx), {}

    def tmpl(self, k):
        if k not in self.t:
            self.t[k] = (self.ctx.template_frames(k), self.ctx.get_template(k)[0])
        return self.t[k]

    def row(self, x, first, count):
        mean, _, f = self.ctx.extract_mfcc(x, want_frames=True)
        return np.array([A.distance(f, mean, *self.tmpl(k), self.C) for k in range(first, first + count)], np.float32)


def check_best(dist, slot, best, first):
    for i, d in enumerate(dist):
        k = int(np.argmin(d))                                 # numpy: the first minimum, i.e. the lowest slot
        assert slot[i] == first[i] + k and best[i].tobytes() == d[k].tobytes(), (i, d, slot[i], best[i])


# ---------------------------------------------------------------------------------------------------- template store
@pytest.mark.parametrize("fmt", [_lib.PCM_I16, _lib.PCM_F32], ids=["i16", "f32"])
@pytest.mark.parametrize("cfg", CFGS, ids=CFG_IDS)
def test_store_equals_extract_mfcc(fmt, cfg):
    rng = np.random.default_rng(1)
    au = audios([1, 159, 160, 161, 640, 16000, 48000, 20000], 3)
    ctx = ctx_(2, slots=16, fmt=fmt, **cfg)
    ctx.set_template(0, au[5])
    ctx.set_templates([1, 2, 3, 4, 5, 6, 7], au[:7])
    x = (rng.standard_normal((2, 5 * SR)) * 0.1).astype(np.float32)
    x[:, SR:2 * SR] += np.stack([au[5], au[7][:SR]])
    ctx.set_stream_params(-1, live=1)
    for a in range(0, 5 * SR, SR):
        blk = np.ascontiguousarray(x[:, a:a + SR])
        ctx.push(synth.to_int16(blk) if fmt == _lib.PCM_I16 else blk)
    rows = [(0, 1000, 16000), (1, 3 * SR + 7, 161), (0, 4 * SR, 1)]
    ctx.set_templates_from_streams([8, 9, 10], *zip(*rows))
    want = {0: au[5], **{k + 1: a for k, a in enumerate(au[:7])}}
    want.update({8 + i: ctx.read_segment(*r) for i, r in enumerate(rows)})
    for k, a in want.items():
        f = ctx.template_frames(k)
        ref = ctx.extract_mfcc(a, want_frames=True)[2]
        assert f.shape == ref.shape and f.tobytes() == ref.tobytes(), k
    # no frames: features only, over 301 frames, cleared (empty)
    m, s, _ = ctx.get_template(3)
    ctx.set_template_features(3, m, s, 640)
    assert ctx.template_frames(3).shape == (0, 20)
    ctx.set_template(11, audios([48001], 5)[0])
    assert ctx.template_frames(11).shape == (0, 20) and ctx.get_template(11)[2] == 48001
    ctx.set_templates([12], audios([48001], 6))
    assert ctx.template_frames(12).shape == (0, 20)
    ctx.clear_template(4)
    with pytest.raises(ValueError, match="empty"):
        ctx.template_frames(4)
    ctx.close()


def test_store_off_and_launch_counts():
    au = audios([640, 16000, 48000, 48001], 9)
    counts = []
    for frames in (False, True):
        ctx = ctx_(1, slots=8, frames=frames)
        ctx.set_stream_params(-1, live=1)
        ctx.push(synth.to_int16(np.resize(au[1], (1, 3 * SR))))
        n0 = ctx.launch_count()
        ctx.set_template(0, au[0])
        ctx.set_templates([1, 2, 3, 4], au)
        ctx.set_templates([1, 2], au[:2], want_vad=True)
        ctx.set_templates_from_streams([5, 6], [0, 0], [0, 100], [16000, 333], want_vad=True)
        counts.append(ctx.launch_count() - n0)
        if not frames:
            with pytest.raises(_lib.EwkError, match="template_frames"):
                ctx.template_frames(0)
        ctx.close()
    assert counts[0] == counts[1]


# ---------------------------------------------------------------------------------------------------- exactness
def _bank_of_templates(ctx, seed):
    """slots 0..69: lengths 1..48000 (1 to 301 frames); slot 71 holds slot 70's audio (a tie)"""
    rng = np.random.default_rng(seed)
    lens = [1, 159, 160, 161, 640, 4000, 16000, 30000, 47999, 48000] + [int(v) for v in rng.integers(1, 48001, 61)]
    au = audios(lens, seed)
    ctx.set_templates(list(range(71)), au)
    ctx.set_template(71, au[70])
    return au


@pytest.mark.parametrize("cfg", CFGS, ids=CFG_IDS)
def test_buffers_exact(cfg):
    rng = np.random.default_rng(21)
    ctx = ctx_(0, slots=80, **cfg)
    tau = _bank_of_templates(ctx, 30)
    seg_lens = [1, 159, 160, 161, 640, 48000, 16000, 9000] + [int(v) for v in rng.integers(1, 48001, 8)]
    segs = audios(seg_lens, 77)
    segs[6] = np.zeros(16000, np.float32)                      # all-zero segment: cost 1 everywhere
    segs[7] = tau[70]                                          # against 70 and 71: distance 0 twice, slot 70 wins
    first = [0, 7, 0, 63, 10, 8, 3, 70] + [int(v) for v in rng.integers(0, 40, 8)]
    count = [64, 1, 1, 8, 2, 64, 5, 2] + [int(v) for v in rng.integers(1, 31, 8)]
    lens = np.array([len(s) for s in segs], np.int64)
    offs = np.concatenate([[5], 5 + np.cumsum(lens + 3)[:-1]]).astype(np.int64)
    pcm = np.zeros(int(offs[-1] + lens[-1] + 9), np.float32)
    for o, s in zip(offs, segs):
        pcm[o:o + len(s)] = s
    n0 = ctx.launch_count()
    dist, slot, best = ctx.align_buffers(pcm, offs, lens, first, count)
    assert ctx.launch_count() - n0 == 2                        # one K3 + one K11
    model = Model(ctx)
    for i, s in enumerate(segs):
        want = model.row(s, first[i], count[i])
        assert dist[i].tobytes() == want.tobytes(), (i, dist[i], want)
    mean, _, f = ctx.extract_mfcc(segs[6], want_frames=True)
    C = C_of(ctx)
    if np.all(f[:, :C] == mean[:C]):                           # constant frames: u = 0, every cost is 1
        n_f = len(f)
        assert np.all(np.abs(dist[6] - np.float32([max(n_f, 1 + len(tau[k]) // 160) / (n_f + 1 + len(tau[k]) // 160)
                                                  for k in range(3, 8)])) < 1e-6)
    assert dist[7][0] == 0 == dist[7][1] or dist[7][0] == dist[7][1]
    check_best(dist, slot, best, first)
    assert slot[7] == 70
    # per row == batched; int16 input == its float32 conversion
    for i in range(0, len(segs), 5):
        d1, s1, b1 = ctx.align_buffers(segs[i], [0], [len(segs[i])], first[i], count[i])
        assert d1[0].tobytes() == dist[i].tobytes() and s1[0] == slot[i] and b1[0] == best[i]
    q = synth.to_int16(segs[3])
    dq = ctx.align_buffers(q, [0], [len(q)], 0, 9)[0][0]
    assert dq.tobytes() == Model(ctx).row(synth.from_int16(q), 0, 9).tobytes()
    ctx.close()


def _ring_ctx(fmt, cfg, seed):
    """3 streams, 4 s ring + 1 s slack (80 000 samples), 8 s pushed in 1 s blocks: the ring has wrapped"""
    ctx = ctx_(3, slots=80, fmt=fmt, **cfg)
    tau = _bank_of_templates(ctx, seed)
    rng = np.random.default_rng(seed)
    base = np.concatenate(audios([SR] * 8, seed + 1))
    x = np.stack([np.roll(base, 3000 * s) for s in range(3)]) + (rng.standard_normal((3, 8 * SR)) * 0.01).astype(np.float32)
    x = x.astype(np.float32)
    ctx.set_stream_params(0, live=1, template_first=0, template_count=64)
    ctx.set_stream_params(1, live=1, template_first=64, template_count=8)
    ctx.set_stream_params(2, live=1, template_first=5, template_count=1)
    for a in range(0, 8 * SR, SR):
        blk = np.ascontiguousarray(x[:, a:a + SR])
        ctx.push(synth.to_int16(blk) if fmt == _lib.PCM_I16 else blk)
    return ctx, tau


RING_ROWS = [(0, 5 * SR, 16000), (1, 70000, 16000), (2, 79999, 2), (1, 4 * SR, 48000), (0, 8 * SR - 1, 1),
             (2, 6 * SR + 3, 159), (0, 75000, 9000), (0, 7 * SR, 640)]        # 70000 / 79999 / 75000: across the ring end


@pytest.mark.parametrize("fmt", [_lib.PCM_I16, _lib.PCM_F32], ids=["i16", "f32"])
@pytest.mark.parametrize("cfg", CFGS, ids=CFG_IDS)
def test_segments_exact(fmt, cfg):
    ctx, _ = _ring_ctx(fmt, cfg, 40)
    st, a0, ln = (list(v) for v in zip(*RING_ROWS))
    own = {0: (0, 64), 1: (64, 8), 2: (5, 1)}
    ctx.synchronize()                                          # lands the last push (K1), so that only the call counts
    n0 = ctx.launch_count()
    dist, slot, best = ctx.align_segments(st, a0, ln)            # each stream's own range
    assert ctx.launch_count() - n0 == 2
    first = [own[s][0] for s in st]
    model = Model(ctx)
    audio = [ctx.read_segment(s, a, n) for s, a, n in RING_ROWS]
    for i, (s, a, n) in enumerate(RING_ROWS):
        assert len(dist[i]) == own[s][1]
        assert dist[i].tobytes() == model.row(audio[i], *own[s]).tobytes(), i
    check_best(dist, slot, best, first)
    # explicit sets, mixed, against the buffer form of read_segment's audio
    f2 = [3, 0, 40, 70, 0, 11, 60, 1]
    c2 = [1, 64, 24, 2, 17, 33, 4, 8]
    d2, s2, b2 = ctx.align_segments(st, a0, ln, f2, c2)
    lens = np.array(ln, np.int64)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
    d3, s3, b3 = ctx.align_buffers(np.concatenate(audio), offs, lens, f2, c2)
    for i in range(len(st)):
        assert d2[i].tobytes() == d3[i].tobytes()
    assert s2.tobytes() == s3.tobytes() and b2.tobytes() == b3.tobytes()
    check_best(d2, s2, b2, f2)
    ctx.close()


def test_segments_device_outputs_and_repeats():
    import torch
    ctx, _ = _ring_ctx(_lib.PCM_I16, {}, 50)
    rows = RING_ROWS + RING_ROWS[:3]                               # repeated streams and ranges
    st, a0, ln = (list(v) for v in zip(*rows))
    dist, slot, best = ctx.align_segments(st, a0, ln)
    total = sum(len(d) for d in dist)
    dd = torch.full((total + 16,), -7.0, dtype=torch.float32, device="cuda:0")
    ds = torch.full((len(rows) + 4,), -9, dtype=torch.int32, device="cuda:0")
    db = torch.full((len(rows) + 4,), -7.0, dtype=torch.float32, device="cuda:0")
    assert ctx.align_segments(st, a0, ln, out_device_ptrs=(dd.data_ptr(), ds.data_ptr(), db.data_ptr()),
                              dist_cap=total + 16) is None
    torch.cuda.synchronize()
    assert dd[:total].cpu().numpy().tobytes() == np.concatenate(dist).tobytes()
    assert np.all(dd[total:].cpu().numpy() == -7.0) and np.all(ds[len(rows):].cpu().numpy() == -9)
    assert ds[:len(rows)].cpu().numpy().tobytes() == slot.tobytes()
    assert db[:len(rows)].cpu().numpy().tobytes() == best.tobytes()
    for i in range(len(RING_ROWS), len(rows)):
        j = i - len(RING_ROWS)
        assert dist[i].tobytes() == dist[j].tobytes() and slot[i] == slot[j]
    ctx.close()


# ---------------------------------------------------------------------------------------------------- end to end
def test_bank_verify_separates_reversed_word():
    w = _word()
    P = dict(speech_duration_min=0.69, speech_duration_max=1.38, timeout=30.0)
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((2, 20 * SR)) * 0.0005).astype(np.float32)
    x[0, 13 * SR:13 * SR + len(w)] += w * np.float32(2.0)
    x[1, 13 * SR:13 * SR + len(w)] += w[::-1] * np.float32(2.0)
    q = synth.to_int16(x)
    bank = WakeWordBank(2, [w], alignment=True, **P)
    seen = []
    ev = bank.run([np.ascontiguousarray(q[:, a:a + SR]) for a in range(0, q.shape[1], SR)],
                  on_match=lambda s, t, sc, txt: seen.append(s))
    hits = [e for e in ev if e["kind"] == 2 and e["matched"]]
    assert sorted(int(e["stream"]) for e in hits) == [0, 1] and sorted(seen) == [0, 1]
    assert all(float(e["score"]) >= 99.0 for e in hits), [float(e["score"]) for e in hits]
    rec, dist = bank.verify(hits)
    d = {int(r["stream"]): float(r["distance"]) for r in rec}
    assert d[1] - d[0] >= MARGIN, d
    assert list(rec["best_slot"]) == [0, 0] and [len(v) for v in dist] == [1, 1]
    # max_distance drops the reversed word before on_match; the same feed on a fresh bank
    bank2 = WakeWordBank(2, [w], alignment=True, **P)
    seen2 = []
    bank2.run([np.ascontiguousarray(q[:, a:a + SR]) for a in range(0, q.shape[1], SR)],
              on_match=lambda s, t, sc, txt: seen2.append(s), max_distance=(d[0] + d[1]) / 2)
    assert seen2 == [0]
    bank.close()
    bank2.close()
    # a dense detection goes through verify as it is, as the detections arrive (their audio is still in the rings)
    bank3 = WakeWordBank(2, [w], alignment=True, **P)
    n_det = 0
    for a in range(0, q.shape[1], SR):
        bank3.step(np.ascontiguousarray(q[:, a:a + SR]))
        det = bank3.dense_detect(own_templates=True)
        if len(det):
            rec2, _ = bank3.verify(det)
            assert list(rec2["seg_start"]) == list(det["seg_start"]) and list(rec2["seg_len"]) == list(det["seg_len"])
            ref = bank3.ctx.align_segments(det["stream"], det["seg_start"], det["seg_len"], 0, 1)
            assert rec2["distance"].tobytes() == ref[2].tobytes()
            n_det += len(det)
    assert n_det
    bank3.close()


# ---------------------------------------------------------------------------------------------------- errors
def _call_seg(ctx, st, a0, ln, first, count, cap=None, where=_lib.HOST):
    n = len(st)
    st = np.ascontiguousarray(st, np.int32)
    a0 = np.ascontiguousarray(a0, np.int64)
    ln = np.ascontiguousarray(ln, np.int64)
    tf = None if first is None else np.ascontiguousarray(first, np.int32)
    tc = None if count is None else np.ascontiguousarray(count, np.int32)
    dist = np.full(200, -3.0, np.float32)
    bs = np.full(n + 2, -5, np.int32)
    bd = np.full(n + 2, -3.0, np.float32)
    P32 = C.POINTER(C.c_int32)
    rc = ctx.lib.ewk_align_segments(ctx.h, n, st.ctypes.data_as(P32), _lib.i64ptr(a0), _lib.i64ptr(ln),
                                    None if tf is None else tf.ctypes.data_as(P32),
                                    None if tc is None else tc.ctypes.data_as(P32), _lib.f32ptr(dist),
                                    200 if cap is None else cap, bs.ctypes.data_as(P32), _lib.f32ptr(bd), where)
    assert np.all(dist == -3.0) and np.all(bs == -5) and np.all(bd == -3.0)
    return rc, ctx.lib.ewk_last_error(ctx.h).decode()


def _call_buf(ctx, lens, first, count, cap=200):
    n = len(lens)
    ln = np.ascontiguousarray(lens, np.int64)
    off = np.zeros(n, np.int64)
    pcm = np.zeros(max(1, int(max(lens, default=1))), np.float32)
    P32 = C.POINTER(C.c_int32)
    tf = None if first is None else np.ascontiguousarray(first, np.int32)
    tc = None if count is None else np.ascontiguousarray(count, np.int32)
    dist = np.full(200, -3.0, np.float32)
    rc = ctx.lib.ewk_align_buffers(ctx.h, n, pcm.ctypes.data, _lib.PCM_F32, _lib.HOST, _lib.i64ptr(off), _lib.i64ptr(ln),
                                   None if tf is None else tf.ctypes.data_as(P32),
                                   None if tc is None else tc.ctypes.data_as(P32), _lib.f32ptr(dist), cap, None, None,
                                   _lib.HOST)
    assert np.all(dist == -3.0)
    return rc, ctx.lib.ewk_last_error(ctx.h).decode()


def test_errors_write_nothing():
    ARG, NOT, STATE = _lib.EWK_ERR_ARG, _lib.EWK_ERR_NO_TEMPLATE, _lib.EWK_ERR_STATE
    ctx, _ = _ring_ctx(_lib.PCM_I16, {}, 60)
    m, s, _ = ctx.get_template(0)
    ctx.set_template_features(72, m, s, 640)                   # features only
    ctx.set_template(73, audios([48001], 2)[0])                # over 301 frames
    ok = ([0, 1], [5 * SR, 5 * SR], [16000, 16000])
    cases = [
        (([0, 3], *ok[1:], [0, 0], [1, 1]), ARG, "row 1 (stream 3)"),
        (([0, -1], *ok[1:], [0, 0], [1, 1]), ARG, "row 1 (stream -1)"),
        ((*ok[:2], [16000, 0], [0, 0], [1, 1]), ARG, "row 1 (stream 1)"),
        ((*ok[:2], [16000, 48001], [0, 0], [1, 1]), ARG, "row 1"),
        ((*ok, [0, 0], [1, 0]), ARG, "row 1 (stream 1)"),
        ((*ok, [0, 0], [1, 65]), ARG, "row 1 (stream 1)"),
        ((*ok, [0, 79], [1, 2]), ARG, "row 1 (stream 1)"),
        ((*ok, [0, -1], [1, 1]), ARG, "row 1"),
        ((*ok, [0, 0], None), ARG, "both"),
        ((*ok, [0, 72], [1, 1]), ARG, "slot 72 has no frames"),
        ((*ok, [0, 70], [1, 4]), ARG, "slot 72 has no frames"),
        ((*ok, [0, 73], [1, 1]), ARG, "slot 73 has no frames"),
        ((*ok, [0, 74], [1, 1]), NOT, "slot 74 is empty"),
        (([0, 1], [5 * SR, 8 * SR - 100], [16000, 101], [0, 0], [1, 1]), STATE, "row 1 (stream 1): segment not pushed"),
        (([0, 1], [5 * SR, 8 * SR - 80001], [16000, 16000], [0, 0], [1, 1]), STATE, "row 1 (stream 1): segment already"),
    ]
    for args, code, msg in cases:
        rc, err = _call_seg(ctx, *args)
        assert rc == code and msg in err, (args, rc, err)
    rc, err = _call_seg(ctx, *ok, [0, 0], [3, 3], cap=5)
    assert rc == ARG and "dist_cap" in err
    for lens, f, c, code, msg in [([16000, 0], [0, 0], [1, 1], ARG, "row 1"), ([16000, 48001], [0, 0], [1, 1], ARG, "row 1"),
                                  ([1, 1], None, None, ARG, "template_first"), ([1, 1], [0, 0], [1, 65], ARG, "row 1"),
                                  ([1, 1], [0, 72], [1, 1], ARG, "no frames"), ([1, 1], [0, 74], [1, 1], NOT, "empty")]:
        rc, err = _call_buf(ctx, lens, f, c)
        assert rc == code and msg in err, (lens, rc, err)
    assert ctx.align_segments([], [], [], [], [])[0] == []                  # n = 0
    ctx.close()
    off = ctx_(1, slots=4, frames=False)
    off.set_template(0, audios([640], 1)[0])
    off.set_stream_params(-1, live=1)
    off.push(np.zeros((1, SR), np.int16))
    rc, err = _call_seg(off, [0], [0], [640], [0], [1])
    assert rc == STATE and "template_frames" in err
    rc, err = _call_buf(off, [640], [0], [1])
    assert rc == STATE
    off.close()
    nostream = ctx_(0, slots=4)
    nostream.set_template(0, audios([640], 1)[0])
    rc, err = _call_seg(nostream, [0], [0], [640], [0], [1])
    assert rc == STATE and "n_streams = 0" in err
    nostream.close()


# ---------------------------------------------------------------------------------------------------- poison mode
@contextlib.contextmanager
def _env(v):
    old = os.environ.get("EWK_POISON")
    try:
        if v is None:
            os.environ.pop("EWK_POISON", None)
        else:
            os.environ["EWK_POISON"] = v
        yield
    finally:
        if old is None:
            os.environ.pop("EWK_POISON", None)
        else:
            os.environ["EWK_POISON"] = old


def _align_workload():
    """template store writers, both alignment forms (host and device outputs), template_frames reads: K3, K6, K11,
    the enrol kernels, ring gather"""
    import torch
    out = []
    ctx, tau = _ring_ctx(_lib.PCM_F32, {"n_mfcc": 13, "preemphasis": 0.97}, 70)
    ctx.set_templates_from_streams([74, 75], [0, 2], [5 * SR, 75000], [9000, 12000], want_vad=True)
    for k in (0, 9, 70, 74, 75):
        out.append(ctx.template_frames(k).tobytes())
    st, a0, ln = (list(v) for v in zip(*RING_ROWS))
    d, s, b = ctx.align_segments(st, a0, ln)
    out += [np.concatenate(d).tobytes(), s.tobytes(), b.tobytes()]
    d, s, b = ctx.align_segments(st, a0, ln, [74] * len(st), [2] * len(st))
    out += [np.concatenate(d).tobytes(), s.tobytes(), b.tobytes()]
    pcm = np.concatenate(tau[:6])
    lens = np.array([len(t) for t in tau[:6]], np.int64)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
    d, s, b = ctx.align_buffers(pcm, offs, lens, list(range(6)), [3] * 6)
    out += [np.concatenate(d).tobytes(), s.tobytes(), b.tobytes()]
    dd = torch.zeros(64, dtype=torch.float32, device="cuda:0")
    ctx.align_segments(st[:2], a0[:2], ln[:2], [0, 1], [4, 4], out_device_ptrs=(dd.data_ptr(), None, None))
    torch.cuda.synchronize()
    out.append(dd.cpu().numpy().tobytes())
    out.append(ctx.launch_count())
    return ctx, out


@pytest.mark.parametrize("pattern", ["0xff", "0x3c"])
def test_poison_patterns_agree(pattern):
    with _env(None):
        c0, base = _align_workload()
    c0.close()
    with _env(pattern):
        c1, got = _align_workload()
        c1.debug_check()
    c1.close()
    assert len(got) == len(base)
    for i, (a, b) in enumerate(zip(base, got)):
        assert a == b, f"output {i} differs with EWK_POISON={pattern}"
