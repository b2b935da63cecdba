"""GPU: batched template enrolment (ewk_set_templates, ewk_set_templates_from_streams) and 4096 template slots.
Every comparison is exact (byte equality / np.array_equal): a batch equals ewk_set_template of each template alone in
every field (K3's mean / std, the dense features through dense scores, n_samples) and ewk_analyze_templates; ring
enrolment equals ewk_set_template of ewk_read_segment; 4096 personal words score and detect on their own slots; errors
change no slot and no cached dense set; one call's launches do not grow with n; migration onto an enrolled slot."""
import numpy as np
import pytest

from easywakeword_b200 import _lib, synth

pytestmark = pytest.mark.gpu

SR = 16000


def ctx_(n=0, slots=64, fmt=_lib.PCM_I16, ring=SR * 10, **kw):
    return _lib.Context(device=0, n_streams=n, ring_samples=ring, slack_samples=SR, pcm_format=fmt,
                        max_templates=slots, max_events=8192, **kw)


def tmpl(ctx, slot):
    m, s, n = ctx.get_template(slot)
    return m.tobytes() + s.tobytes() + int(n).to_bytes(8, "little")


def words(n_words, seed):
    return [synth.synthetic_word(seed=seed + i, duration=0.6 + 0.4 * ((i * 7) % 10) / 9) for i in range(n_words)]


def audios_of(lens, seed):
    """float32 templates of these lengths: word-like audio over noise, at random gains"""
    rng = np.random.default_rng(seed)
    base = np.concatenate(words(6, seed))
    out = []
    for L in lens:
        o = int(rng.integers(0, max(1, len(base) - L))) if L <= len(base) else 0
        w = np.resize(base[o:], L) if L > len(base) - o else base[o:o + L]
        out.append((w * np.float32(rng.uniform(0.5, 3.0)) +
                    rng.standard_normal(L).astype(np.float32) * np.float32(0.003)).astype(np.float32))
    return out


def feed_blocks(word, n, seconds, seed, fmt):
    xs = [synth.stream(seed + i, seconds, word, gain=(1.5, 3.0), inserts_per_10s=(3, 4))[0] for i in range(n)]
    x = np.stack(xs)
    return synth.to_int16(x) if fmt == _lib.PCM_I16 else x.astype(np.float32)


def run_gate(ctx, x):
    """push 1 s blocks, tick what they pay for; all events"""
    ev = []
    for a in range(0, x.shape[1], SR):
        ctx.push(np.ascontiguousarray(x[:, a:a + SR]))
        ctx.tick(SR // 1600)
        ev.append(ctx.poll())
    return np.concatenate(ev)


BATCH_LENS = [1, 159, 160, 640, 16000, 48000, 60000]


@pytest.mark.parametrize("where", ["host", "device"])
@pytest.mark.parametrize("cfg", [{}, {"n_mfcc": 13}, {"preemphasis": 0.97}], ids=["default", "mfcc13", "preemph"])
def test_batch_equals_singles(where, cfg):
    rng = np.random.default_rng(40)
    lens = BATCH_LENS + [int(v) for v in rng.integers(1, 60001, 33)]
    au = audios_of(lens, 11)
    slots = rng.permutation(64)[:40].astype(np.int32)
    word = au[4]
    x = feed_blocks(word, 8, 30, 500, _lib.PCM_I16)          # gate events are sparse: 8 streams x 30 s
    A, B = ctx_(8, ring=3 * SR, **cfg), ctx_(8, ring=3 * SR, **cfg)
    if where == "host":
        vad = A.set_templates(slots, au, want_vad=True)
    else:
        import torch
        gap = 3                                              # unaligned offsets inside one device buffer
        offs = np.cumsum([0] + [L + gap for L in lens[:-1]]).astype(np.int64) + 1
        flat = np.zeros(int(offs[-1] + lens[-1]), np.float32)
        for o, a in zip(offs, au):
            flat[o:o + len(a)] = a
        dev = torch.from_numpy(flat).cuda()
        torch.cuda.synchronize()
        vad = A.set_templates(slots, (dev.data_ptr(), offs, np.array(lens, np.int64)), want_vad=True)
    for k, a in zip(slots, au):
        B.set_template(int(k), a)
    for k in range(64):
        if k in set(slots.tolist()):
            assert tmpl(A, k) == tmpl(B, k), k
        else:
            with pytest.raises(ValueError):
                A.get_template(k)
    assert vad.tobytes() == B.analyze_templates(au).tobytes()
    # dmean / dstd: dense scores of every slot dense scoring takes, and the gate over all 64 slots, on a shared feed
    for c in (A, B):
        c.set_stream_params(-1, frame_size=1600, template_first=0, template_count=64, similarity_threshold=60.0)
    ea, eb = run_gate(A, x), run_gate(B, x)
    assert len(ea) > 0 and ea.tobytes() == eb.tobytes()
    for k, L in zip(slots, lens):
        if 640 <= L <= 48000:
            sa = A.dense_scores(2920, 80, int(k), 1)         # windows still in the 64 000-sample ring
            sb = B.dense_scores(2920, 80, int(k), 1)
            assert np.array_equal(sa, sb, equal_nan=True), k
    A.close(), B.close()


@pytest.mark.parametrize("fmt", [_lib.PCM_I16, _lib.PCM_F32], ids=["i16", "f32"])
def test_from_rings(fmt):
    word = words(1, 70)[0]
    A, B = ctx_(8, fmt=fmt, ring=3 * SR), ctx_(0, 64)
    A.set_template(0, word)
    A.set_stream_params(-1, frame_size=1600, template_first=0, template_count=1, similarity_threshold=60.0)
    x = feed_blocks(word, 8, 30, 900, fmt)                   # 480 000 samples through a 64 000-sample physical ring
    P = (3 * SR + SR + 63) // 64 * 64
    rows, slots, vads, segs, src = [], [], [], [], {"gate": 0, "dense": 0}
    # enrol each block's new gate events and dense detections at once, while their audio is in the ring
    for a in range(0, x.shape[1], SR):
        A.push(np.ascontiguousarray(x[:, a:a + SR]))
        A.tick(SR // 1600)
        ev = A.poll()
        new = [(int(e["stream"]), int(e["seg_start"]), int(e["seg_len"]), "gate") for e in ev if e["kind"] == _lib.EV_SCORED]
        while True:
            d, (_, nh) = A.dense_detect(None, 200, 0, 1, 20, 50, hops=True)
            new += [(int(r["stream"]), int(r["seg_start"]), int(r["seg_len"]), "dense") for r in d]
            if nh.max() < 200:
                break
        new = new[:max(0, 60 - len(rows))]
        if not new:
            continue
        k = np.arange(len(rows), len(rows) + len(new), dtype=np.int32)
        vads.append(A.set_templates_from_streams(k, *(np.array(c, np.int64) for c in list(zip(*new))[:3]), want_vad=True))
        segs += [A.read_segment(s_, a_, L_) for s_, a_, L_, _ in new]
        for r in new:
            src[r[3]] += 1
        rows += new
        slots += k.tolist()
    assert src["gate"] > 0 and src["dense"] > 0, src
    W = x.shape[1]
    b = W // P * P
    wrap = [(1, b - 5000, 9000), (2, b - 100, 3000), (3, W - 400, 400), (0, W - P, P)]     # across the ring end
    assert all(a_ % P + L_ > P for _, a_, L_ in wrap[:2] + wrap[3:])
    k = np.arange(60, 64, dtype=np.int32)[::-1].copy()
    vads.append(A.set_templates_from_streams(k, *(np.array(c, np.int64) for c in zip(*wrap)), want_vad=True))
    segs += [A.read_segment(*r) for r in wrap]
    slots += k.tolist()
    for k_, sg in zip(slots, segs):
        B.set_template(int(k_), sg)
    for k_ in slots:
        assert tmpl(A, int(k_)) == tmpl(B, int(k_)), k_
    assert np.concatenate(vads).tobytes() == B.analyze_templates(segs).tobytes()
    written = W
    # state errors, naming the row and the stream
    with pytest.raises(_lib.EwkError, match=r"row 1 \(stream 2\).*overwritten"):
        A.set_templates_from_streams([60, 61], [0, 2], [written - 100, 0], [100, 100])
    with pytest.raises(_lib.EwkError, match=r"row 0 \(stream 3\).*not pushed"):
        A.set_templates_from_streams([60], [3], [written - 50], [100])
    with pytest.raises(ValueError, match=r"row 0 \(stream 8\)"):
        A.set_templates_from_streams([60], [8], [0], [100])
    # a pending pinned push lands before the gather reads it
    pin = _lib.PinnedArray((8, SR), np.int16 if fmt == _lib.PCM_I16 else np.float32)
    pin.array[...] = feed_blocks(word, 8, 1, 77, fmt)
    A.push(pin.array)
    A.set_templates_from_streams([62, 63], [1, 1], [written + 100, written], [12000, SR])
    got = [A.read_segment(1, written + 100, 12000), A.read_segment(1, written, SR)]
    pin.free()
    B.set_template(62, got[0]), B.set_template(63, got[1])
    assert tmpl(A, 62) == tmpl(B, 62) and tmpl(A, 63) == tmpl(B, 63)
    A.close(), B.close()


def test_4096_personal_words():
    from easywakeword_b200.bank import WakeWordBank
    N, T = 4096, 12
    bases = words(64, 3000)
    rng = np.random.default_rng(4096)
    wl = rng.integers(int(0.6 * SR), SR + 1, N)
    wo = rng.integers(0, 2000, N)
    gain = rng.uniform(1.5, 2.5, N).astype(np.float32)
    mine = [(np.resize(bases[s % 64], wo[s] + wl[s])[wo[s]:] * gain[s]).astype(np.float32) for s in range(N)]
    at = [SR, 5 * SR, 8 * SR, int(10.5 * SR)]                    # each stream says its word at these samples

    def block(t):
        b = np.random.default_rng(t).standard_normal((N, SR)).astype(np.float32) * np.float32(0.002)
        for s in range(N):
            for a in at:
                lo, hi = max(a, t * SR), min(a + wl[s], (t + 1) * SR)
                if lo < hi:
                    b[s, lo - t * SR:hi - t * SR] += mine[s][lo - a:hi - a]
        return synth.to_int16(b)

    bank = WakeWordBank(N, [bases[0]], buffer_seconds=3, template_slots=N, speech_duration_min=0.3,
                        speech_duration_max=2.0)
    sample = np.unique(np.concatenate([[0, 1, 63, 64, 4095], rng.choice(N, 59, replace=False)]))[:64]
    ref = ctx_(len(sample), N, ring=3 * SR)
    ref.set_stream_params(-1, frame_size=1600, live=1)
    blocks = [block(t) for t in range(2)]
    for b in blocks:
        bank.step(b)
        ref.push(np.ascontiguousarray(b[sample]))
    bank.poll()
    assert bank.enroll((np.arange(N), np.full(N, at[0]), wl), np.arange(N, dtype=np.int32), set_durations=False) is None
    for j, s in enumerate(sample):
        ref.set_template(int(s), bank.ctx.read_segment(int(s), at[0], int(wl[s])))     # the ring's int16 audio
        assert tmpl(ref, int(s)) == tmpl(bank.ctx, int(s)), s
    events, det, rdet = [], [], [[] for _ in sample]
    for t in range(2, T):
        b = block(t)
        bank.step(b)
        ref.push(np.ascontiguousarray(b[sample]))
        ev = bank.poll()
        ev = ev[(ev["kind"] == _lib.EV_SCORED) & (ev["stream"] > 63)]
        events.append(ev)
        for e in ev[:: max(1, len(ev) // 20)]:              # the gate's score == the batch matcher on that slot
            seg = bank.read_segment(e)
            sc, _ = bank.ctx.similarity_batch(int(e["stream"]), seg, [0], [len(seg)])
            assert sc.tobytes() == np.float32(e["score"]).tobytes(), e
        det.append(bank.dense_detect(own_templates=True))
        for j, s in enumerate(sample):
            while True:
                d, (_, nh) = ref.dense_detect([j], 500, int(s), 1, 20, 50, hops=True)
                rdet[j].append(d)
                if nh.max() < 500:
                    break
    det = np.concatenate(det)
    for j, s in enumerate(sample):
        mine_d = det[det["stream"] == s]
        r = np.concatenate(rdet[j])
        r["stream"] = s
        assert mine_d.tobytes() == r.tobytes(), s
    assert (det["template_slot"] == det["stream"]).all() and (det["stream"] > 63).sum() > 0
    ev = np.concatenate(events)
    assert len(ev) > 0 and (ev["template_slot"] == ev["stream"]).all()
    bank.close(), ref.close()


def test_limits():
    with pytest.raises(ValueError):
        ctx_(0, 4097)
    c = ctx_(8, 4096, ring=3 * SR)
    with pytest.raises(ValueError, match="EWK_MAX_STREAM_TEMPLATES"):
        c.set_stream_params(0, template_first=0, template_count=65)
    word = words(1, 5)[0]
    au = audios_of([len(word)] * 63, 6) + [word]
    c.set_templates(np.arange(4032, 4096, dtype=np.int32), au)
    c.set_stream_params(-1, frame_size=1600, template_first=4032, template_count=64, similarity_threshold=60.0)
    ev = run_gate(c, feed_blocks(word, 8, 30, 40, _lib.PCM_I16))
    ev = ev[ev["kind"] == _lib.EV_SCORED]
    assert len(ev) > 0
    for e in ev[-4:]:
        seg = c.read_segment(int(e["stream"]), int(e["seg_start"]), int(e["seg_len"]))
        sc = np.array([c.similarity_batch(k, seg, [0], [len(seg)])[0][0] for k in range(4032, 4096)], np.float32)
        best = int(np.nanargmax(sc))
        assert e["template_slot"] == 4032 + best and sc[best].tobytes() == np.float32(e["score"]).tobytes()
    c.close()


def test_errors_leave_nothing_behind():
    word = words(1, 8)[0]
    c = ctx_(4, 64)
    au = audios_of([12000, 16000, 9000, 20000], 9)
    c.set_templates(np.arange(4, dtype=np.int32), au)
    x = feed_blocks(word, 4, 13, 60, _lib.PCM_I16)            # 13 s through an 11 s physical ring
    c.set_stream_params(-1, frame_size=1600, live=1)
    for a in range(0, x.shape[1], SR):
        c.push(np.ascontiguousarray(x[:, a:a + SR]))
    sets = dict(template_first=[0, 1, 2, 0], template_count=[2, 3, 1, 4])
    args = ([0, 1, 2, 3], [1000] * 4, [200] * 4)
    before = c.dense_scores_sets(*args, **sets)               # builds and caches the four sets
    snap = [tmpl(c, k) for k in range(64) if k < 4]
    with pytest.raises(ValueError, match="entry 2.*listed twice"):
        c.set_templates([5, 1, 5], au[:3])
    with pytest.raises(ValueError, match="entry 1.*out of range"):
        c.set_templates([2, 64], au[:2])
    with pytest.raises(ValueError, match="entry 1"):
        c.set_templates([0, 1], [au[0], np.zeros(0, np.float32)])
    W = x.shape[1]
    with pytest.raises(_lib.EwkError, match=r"row 1 \(stream 1\).*overwritten"):
        c.set_templates_from_streams([0, 1, 2], [0, 1, 2], [W - 9000, 0, W - 9000], [8000] * 3)
    assert c.lib.ewk_set_templates(c.h, None, 1, None, 0, None, None, None) == _lib.EWK_ERR_ARG
    assert [tmpl(c, k) for k in range(4)] == snap
    for k in range(4, 64):
        with pytest.raises(ValueError):
            c.get_template(k)
    again = c.dense_scores_sets(*args, **sets)
    assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(before, again))
    c.close()


def test_reenrol_invalidates_cached_sets():
    word = words(1, 12)[0]
    au = audios_of([12000, 16000, 9000, 20000, 11000], 13)
    x = feed_blocks(word, 4, 6, 70, _lib.PCM_I16)
    c, fresh = ctx_(4, 64), ctx_(4, 64)
    c.set_templates(np.arange(4, dtype=np.int32), au[:4])
    fresh.set_templates(np.arange(4, dtype=np.int32), [au[0], au[4], au[2], au[3]])
    for k in (c, fresh):
        k.set_stream_params(-1, frame_size=1600, live=1)
        for a in range(0, x.shape[1], SR):
            k.push(np.ascontiguousarray(x[:, a:a + SR]))
    sets = dict(template_first=[0, 1, 0, 1], template_count=[2, 1, 4, 3])
    args = ([0, 1, 2, 3], [150] * 4, [300] * 4)
    c.dense_scores_sets(*args, **sets)                        # caches sets covering slot 1
    # slot 1 <- au[4], enrolled from the ring of a stream that holds it
    c.push_streams([3], [synth.to_int16(au[4])])
    c.set_templates_from_streams([1], [3], [6 * SR], [len(au[4])])
    fresh.set_template(1, c.read_segment(3, 6 * SR, len(au[4])))
    fresh.push_streams([3], [synth.to_int16(au[4])])
    got, want = c.dense_scores_sets(*args, **sets), fresh.dense_scores_sets(*args, **sets)
    assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(got, want))
    c.close(), fresh.close()


def test_launches_do_not_grow_with_n():
    c = ctx_(0, 4096)
    rng = np.random.default_rng(7)
    au = audios_of([int(v) for v in rng.integers(int(0.6 * SR), int(1.5 * SR), 4096)], 14)
    for vad in (False, True):
        d = []
        for n in (1, 4096):
            l0 = c.launch_count()
            c.set_templates(np.arange(n, dtype=np.int32), au[:n], want_vad=vad)
            d.append(c.launch_count() - l0)
        assert d[0] == d[1] == (3 if vad else 2), d
    c.close()


def test_migration_onto_enrolled_slot():
    word = words(1, 30)[0]
    w3000 = audios_of([14000], 31)[0]
    x = feed_blocks(w3000, 4, 30, 80, _lib.PCM_I16)

    def make(audio_3000):
        k = ctx_(4, 4096, ring=3 * SR)
        k.set_template(0, word)
        k.set_stream_params(-1, frame_size=1600, template_first=0, template_count=1, similarity_threshold=60.0)
        if audio_3000 is not None:
            k.set_templates([3000], [audio_3000])
        return k

    A = make(None)
    A.set_template(3000, w3000)
    A.set_stream_params(1, frame_size=1600, template_first=3000, template_count=1, similarity_threshold=60.0)
    half = 10 * SR
    for a in range(0, half, SR):
        A.push_streams([0, 1, 2, 3], list(x[:, a:a + SR]))
        A.tick_ready(4096)
    A.poll()
    blob = A.export_streams([1])
    B, C = make(w3000), make(audios_of([14000], 32)[0])
    with pytest.raises(_lib.EwkError, match="slot 3000"):
        C.import_streams([2], blob)
    B.import_streams([2], blob)
    ea, eb = [], []
    for a in range(half, x.shape[1], SR):
        A.push_streams([1], [x[1, a:a + SR]])
        A.tick_ready(4096)
        B.push_streams([2], [x[1, a:a + SR]])
        B.tick_ready(4096)
        ea.append(A.poll()), eb.append(B.poll())
    ea, eb = np.concatenate(ea), np.concatenate(eb)
    ea = ea[ea["stream"] == 1]
    eb["stream"] = 1
    assert len(ea) > 0 and ea.tobytes() == eb.tobytes()
    assert (ea["template_slot"][ea["kind"] == _lib.EV_SCORED] == 3000).all()
    A.close(), B.close(), C.close()
