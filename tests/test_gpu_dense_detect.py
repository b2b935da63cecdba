"""GPU: the dense detector (ewk_dense_detect, K4D).  Every detection record is compared field for field
(np.array_equal on the structured arrays) with oracle/dense_detect.py run over the same call's returned scores, and over
oracle/dense_model.py's exact scores: synthetic feeds with inserts, zero gaps and an all-zero stream, one template, the
4-template set and a duplicated template, per-stream thresholds (one equal to a score that occurs), several hold and
refractory values; split invariance under ragged pushes and calls; independence from the score-only entry points; reset;
every output form; level 3; and every error, each of which must leave cursors and detector state alone."""
import numpy as np
import pytest

from easywakeword_b200 import synth
from oracle import dense_detect as M
from test_gpu_dense_ragged import PACED, Want, four_templates, k3_frames, make_ctx, ring_values

pytestmark = pytest.mark.gpu


def set_thr(ctx, thr, live=True):
    for s, t in enumerate(thr):
        ctx.set_stream_params(s, frame_size=1600, template_count=1, live=1 if live else 0, similarity_threshold=float(t))


def feeds_of(seed, secs, word):
    kinds = [lambda s, i: synth.stream(seed + i, s, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4))[0],
             lambda s, i: synth.stream(seed + i, s, word, gain=(1.5, 3.0), zero_gaps=4, noise_sigma=0.0005)[0],
             lambda s, i: np.zeros(int(s * 16000), np.float32)]
    return [kinds[i % 3](sec, i) if sec else np.zeros(0, np.float32) for i, sec in enumerate(secs)]


def tone_bursts(seconds, on_hops=200, off_hops=30):
    """100 Hz bursts (period 160 samples: every window inside a burst is the same audio, so its scores tie exactly)
    separated by digital silence"""
    n = int(seconds * 16000)
    x = (0.3 * np.sin(2 * np.pi * 100.0 * np.arange(n) / 16000)).astype(np.float32)
    x[(np.arange(n) // 160) % (on_hops + off_hops) >= on_hops] = 0.0
    return x


def detect_all(ctx, streams, max_hops, tf, T, hold, refr, rng=None):
    """dense_detect until nothing is due -> (records, per-stream concatenated scores, per-stream call hop0 list)"""
    N = ctx.cfg.n_streams
    recs, sc, starts = [], [[] for _ in range(N)], [[] for _ in range(N)]
    while True:
        mh = max_hops if rng is None else int(rng.choice([1, 2, 5, 17, 64, 150]))
        d, (h0, rows) = ctx.dense_detect(streams, mh, tf, T, hold, refr, scores=True)
        lst = range(N) if streams is None else streams
        for s, a, r in zip(lst, h0, rows):
            sc[s].append(r)
            if len(r):
                starts[s].append(int(a))
        recs.append(d)
        if max((len(r) for r in rows), default=0) < mh:
            break
    return recs, [np.concatenate(c) if c else np.zeros((0, T), np.float32) for c in sc], starts


def model_records(scores_by_stream, thr, hold, refr, tf, lens, states=None):
    out, st_out = [], []
    for s, x in enumerate(scores_by_stream):
        ev, st = M.detect(x, 1, None if states is None else states[s], thr[s], hold, refr, tf, lens, stream=s)
        out.append(ev)
        st_out.append(st)
    return out, st_out


def by_stream(recs, N):
    d = np.concatenate(recs) if len(recs) else np.zeros(0, M.DETECTION_DTYPE)
    return [d[d["stream"] == s] for s in range(N)]


def assert_records(got, want, what):
    assert got.dtype == want.dtype, what
    if not np.array_equal(got, want):
        raise AssertionError(f"{what}: device {got[:4]} ({len(got)}) vs model {want[:4]} ({len(want)})")


CASES = {
    "T1_hold1_refr0": ("one", 1, 0),
    "T4_hold3_refr7": ("four", 3, 7),
    "dup_hold50_refr200": ("dup", 50, 200),
    "T4_hold50_refr0": ("four", 50, 0),
    "T1_hold3_refr200": ("one", 3, 200),
}


@pytest.mark.parametrize("case", list(CASES))
def test_model_equality(case, word):
    kind, hold, refr = CASES[case]
    tpls = {"one": [word], "four": four_templates(word), "dup": [word, word.copy()]}[kind]
    T = len(tpls)
    lens = [len(t) for t in tpls]
    xs = feeds_of(6000, [6.0, 5.0, 4.0, 5.5, 4.5, 3.0], word) + [tone_bursts(9.0)]
    ring, push = zip(*(ring_values(x, "i16") for x in xs))
    N = len(xs)
    ctx = make_ctx(N, "i16", tpls, live=True)
    ctx.push_streams(range(N), list(push))
    want = Want(ring, tpls, k3_frames(ctx))
    # thresholds: one per stream; stream 3's equals a score that occurs there
    pre = ctx.dense_scores_streams([3], [1], [len(push[3]) // 160], 0, T)[0]
    b = np.nanmax(np.where(np.isnan(pre), -np.inf, pre), axis=1)
    occurs = float(np.sort(b[np.isfinite(b)])[-40])
    # stream 6: its steady in-burst score, reached by long runs of exact ties; a run outlives hold, ends, and the next
    # burst comes back within 200 hops
    pre6 = ctx.dense_scores_streams([6], [1], [len(push[6]) // 160], 0, T)[0]
    b6 = np.max(np.where(np.isnan(pre6), -np.inf, pre6), axis=1)
    vals, cnt = np.unique(b6[np.isfinite(b6)], return_counts=True)
    steady = float(vals[np.argmax(cnt)])
    assert cnt.max() >= 50
    thr = [55.0, 50.0, 60.0, occurs, 65.0, 40.0, steady]
    set_thr(ctx, thr)
    recs, sc, _ = detect_all(ctx, None, 137, 0, T, hold, refr)
    got = by_stream(recs, N)
    m_own, _ = model_records(sc, thr, hold, refr, 0, lens)
    m_exact, _ = model_records([want(s, 1, len(push[s]) // 160) for s in range(N)], thr, hold, refr, 0, lens)
    n_det = 0
    for s in range(N):
        assert_records(got[s], m_own[s], f"{case} stream {s} vs model over returned scores")
        assert_records(got[s], m_exact[s], f"{case} stream {s} vs model over dense_model scores")
        n_det += len(got[s])
    assert len(got[3]) > 0 and len(got[2]) == 0 and len(got[6]) > 0 and n_det > 3
    assert np.any(b == np.float32(occurs))
    if kind == "dup":
        assert set(np.concatenate(got)["template_slot"].tolist()) == {0}
    print(f"{case}: {n_det} detections equal the model")
    ctx.close()


@pytest.mark.parametrize("variant", list(PACED))
def test_split_invariance(variant, word):
    """random ragged pushes to random subsets (lengths 0 included), dense_detect at random max_hops (1 included) after
    each push, against a one-piece feed; at least one run is ARMED across a call boundary"""
    cfg = dict(PACED[variant])
    fmt, ring_s, slack = cfg.pop("fmt"), cfg.pop("ring"), cfg.pop("slack")
    tpls = [word, synth.synthetic_word(seed=4, duration=1.0)[:16000]]
    lens = [len(t) for t in tpls]
    N, secs = 5, [5.0, 3.7, 4.4, 0.0, 2.9]
    xs = [synth.stream(6100 + i, sec, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4), zero_gaps=2 * (i % 2),
                       noise_sigma=0.0005)[0] if sec else np.zeros(0, np.float32) for i, sec in enumerate(secs)]
    ring, push = zip(*(ring_values(x, fmt) for x in xs))
    thr = [45.0, 50.0, 45.0, 50.0, 40.0]
    hold, refr = 3, 7
    rng = np.random.default_rng(21 + list(PACED).index(variant))
    ctx = make_ctx(N, fmt, tpls, ring=ring_s, slack=slack, live=True, **cfg)
    set_thr(ctx, thr)
    pos = [0] * N
    recs, starts = [], [[] for _ in range(N)]
    sc = [[] for _ in range(N)]
    while any(pos[s] < len(push[s]) for s in range(N)):
        streams = [int(s) for s in rng.choice(N, int(rng.integers(1, N + 1)), replace=False)]
        rows = []
        for s in streams:
            n = min(int(rng.integers(0, 9000)), len(push[s]) - pos[s])
            rows.append(push[s][pos[s]:pos[s] + n])
            pos[s] += n
        ctx.push_streams(streams, rows)
        r, c, st = detect_all(ctx, list(range(N)) if rng.random() < 0.5 else None, 0, 0, 2, hold, refr, rng)
        recs += r
        for s in range(N):
            sc[s].append(c[s])
            starts[s] += st[s]
    one = make_ctx(N, fmt, tpls, ring=max(ring_s, 6 * 16000), slack=slack, live=True, **cfg)
    set_thr(one, thr)
    one.push_streams([0, 1, 2, 4], [push[s] for s in (0, 1, 2, 4)])
    r1, _, _ = detect_all(one, None, 100000, 0, 2, hold, refr)
    got, ref = by_stream(recs, N), by_stream(r1, N)
    want = Want(ring, tpls, k3_frames(ctx), n_mfcc=cfg.get("n_mfcc", 20), preemphasis=cfg.get("preemphasis", 0.0))
    m, _ = model_records([want(s, 1, len(push[s]) // 160) for s in range(N)], thr, hold, refr, 0, lens)
    crossed = 0
    for s in range(N):
        assert_records(got[s], ref[s], f"{variant} stream {s}: ragged vs one piece")
        assert_records(got[s], m[s], f"{variant} stream {s}: vs model")
        for e in got[s]:                                      # emitted by a later call than the one its run started in
            crossed += any(e["run_start"] < a <= e["emit_hop"] for a in starts[s])
    assert crossed > 0 and sum(len(g) for g in got) > 0
    print(f"{variant}: {sum(len(g) for g in got)} detections, {crossed} across call boundaries")
    ctx.close()
    one.close()


def test_independence(word):
    """dense_ready / dense_scores / dense_scores_streams between detect calls change no detection, and dense_detect
    moves neither their cursor nor is moved by them"""
    tpls = [word]
    xs = feeds_of(6200, [4.0, 3.0, 3.5], word)
    _, push = zip(*(ring_values(x, "i16") for x in xs))
    N = 3
    a = make_ctx(N, "i16", tpls, live=True)
    b = make_ctx(N, "i16", tpls, live=True)
    for c in (a, b):
        set_thr(c, [50.0] * N)
    ra, rb = [], []
    ready_next = np.ones(N, np.int64)
    for p in range(0, 64000, 9000):
        for c in (a, b):
            c.push_streams(range(N), [q[p:p + 9000] for q in push])
        h0, rows = a.dense_ready(None, 60, 0, 1)
        assert np.array_equal(h0, ready_next)
        ready_next += [len(r) for r in rows]
        top = min(p + 9000, min(len(q) for q in push)) // 160
        if top > 1:
            a.dense_scores(1, top - 1, 0, 1)
        a.dense_scores_streams([1], [2], [20], 0, 1)
        ra.append(a.dense_detect(None, 45, 0, 1, 3, 7))
        rb.append(b.dense_detect(None, 45, 0, 1, 3, 7))
    while True:
        da, (_, na) = a.dense_detect(None, 45, 0, 1, 3, 7, hops=True)
        db = b.dense_detect(None, 45, 0, 1, 3, 7)
        ra.append(da)
        rb.append(db)
        if na.max() < 45:
            break
    assert_records(np.concatenate(ra), np.concatenate(rb), "with interleaved score calls")
    assert len(np.concatenate(ra)) > 0
    h0, _ = a.dense_ready(None, 1, 0, 1)
    assert np.array_equal(h0, ready_next)
    a.close()
    b.close()


def test_reset_while_armed(word):
    """stream 1 is reset while ARMED; afterwards it equals stream 1 of a new context fed the same audio, and the other
    streams equal a run without the reset"""
    tpls = [word]
    xs = feeds_of(6300, [4.0, 4.0, 4.0], word)
    xs[1] = synth.stream(6390, 4.0, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4))[0]
    new1 = synth.stream(6391, 3.0, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4))[0]
    ring, push = zip(*(ring_values(x, "i16") for x in xs))
    _, push_new = ring_values(new1, "i16")
    N, thr, hold, refr = 3, [50.0] * 3, 50, 7
    ctx, plain, fresh = (make_ctx(N, "i16", tpls, live=True) for _ in range(3))
    for c in (ctx, plain, fresh):
        set_thr(c, thr)
    want = Want(ring, tpls, k3_frames(ctx))
    b1 = want(1, 1, len(push[1]) // 160)[:, 0]
    h_star = int(np.argmax(b1 >= 50.0)) + 1
    assert b1[h_star - 1] >= 50.0
    for c in (ctx, plain):
        c.push_streams(range(N), list(push))
    d0 = ctx.dense_detect(None, h_star, 0, 1, hold, refr)
    p0 = plain.dense_detect(None, h_star, 0, 1, hold, refr)
    _, st = M.detect(want(1, 1, h_star), 1, None, 50.0, hold, refr, 0, [len(word)])
    assert st["mode"] == M.ARMED
    ctx.reset_streams([1])
    ctx.push_streams([1], [push_new])
    fresh.push_streams([1], [push_new])
    r_ctx, _, _ = detect_all(ctx, None, 200, 0, 1, hold, refr)
    r_plain, _, _ = detect_all(plain, None, 200, 0, 1, hold, refr)
    r_fresh, _, _ = detect_all(fresh, [1], 200, 0, 1, hold, refr)
    g, p = by_stream([d0] + r_ctx, N), by_stream([p0] + r_plain, N)
    assert_records(g[1], np.concatenate(r_fresh), "reset stream vs a new context")
    assert len(g[1]) > 0
    for s in (0, 2):
        assert_records(g[s], p[s], f"stream {s} untouched by the reset")
    for c in (ctx, plain, fresh):
        c.close()


@pytest.mark.parametrize("path", ["outputs", "pending", "overlap"])
def test_outputs(path, word):
    """host scores, device scores and no scores give the same detections; streams = NULL; empty rows; n = 0; det_cap
    exactly sum ceil(n_i / 2); a pending pinned push; overlap mode"""
    import torch
    from easywakeword_b200 import _lib
    tpls = [word]
    N = 4
    xs = feeds_of(6400, [3.0, 3.0, 3.0, 0.0], word)
    _, push = zip(*(ring_values(x, "i16") for x in xs))
    ctxs = [make_ctx(N, "i16", tpls, live=path != "overlap") for _ in range(3)]
    for c in ctxs:
        set_thr(c, [45.0] * N, live=path != "overlap")
    got = [[] for _ in ctxs]
    if path == "outputs":
        for c in ctxs:
            c.push_streams(range(3), list(push[:3]))
        assert len(ctxs[0].dense_detect([], 10)) == 0
        for rnd in range(4):
            lst = None if rnd % 2 else [3, 2, 0, 1]
            n = N if lst is None else len(lst)
            d0, (h0, rows) = ctxs[0].dense_detect(lst, 100, 0, 1, 3, 7, scores=True)
            dev = torch.full((n * 100 + 3,), -1.0, dtype=torch.float32, device="cuda:0")
            d1, (h1, n1) = ctxs[1].dense_detect(lst, 100, 0, 1, 3, 7, out_device_ptr=dev.data_ptr())
            torch.cuda.synchronize()
            need = int(sum((len(r) + 1) // 2 for r in rows))
            d2 = ctxs[2].dense_detect(lst, 100, 0, 1, 3, 7, det_cap=need)
            packed = np.concatenate([r.reshape(-1) for r in rows])
            d = dev.cpu().numpy()
            assert np.array_equal(d[:len(packed)], packed, equal_nan=True) and (d[len(packed):] == -1.0).all()
            assert np.array_equal(h0, h1) and [len(r) for r in rows] == n1.tolist()
            assert len(rows[lst.index(3) if lst else 3]) == 0
            for k, x in enumerate((d0, d1, d2)):
                got[k].append(x)
    elif path == "pending":
        pin = _lib.PinnedArray((N * 48000,), np.int16)
        pin.array[...] = np.concatenate([q if len(q) else np.zeros(48000, np.int16) for q in push])
        offs, lens = np.arange(N) * 48000, np.array([24000, 24000, 24000, 0])
        for c in ctxs[:2]:
            c.push_streams(range(N), (pin.ptr.value, offs, lens, N * 48000, np.int16))
            c.push_streams(range(N), (pin.ptr.value, offs + 24000, lens, N * 48000, np.int16))   # still in flight
        for k, c in enumerate(ctxs[:2]):
            while True:
                d, (_, nh) = c.dense_detect(None, 64, 0, 1, 3, 7, hops=True)
                got[k].append(d)
                if nh.max() < 64:
                    break
            assert c.status(0).written == 48000
        pin.free()
        ctxs[2].push_streams(range(N), list(push))
        got[2] += detect_all(ctxs[2], None, 300, 0, 1, 3, 7)[0]
    else:
        for c in ctxs[:2]:
            c.set_overlap(True)
        for p in range(0, 48000, 8000):
            for k, c in enumerate(ctxs):
                c.push_streams(range(N), [q[p:p + 8000] for q in push])
                if k < 2:
                    c.tick_ready(64)                       # K3 in flight on the match stream
                got[k].append(c.dense_detect(None, 64 if k else 1000, 0, 1, 3, 7))
                if k < 2:
                    c.poll()
    for k in (1, 2):
        assert_records(np.concatenate(got[k]), np.concatenate(got[0]), f"{path}: form {k}")
    assert len(np.concatenate(got[0])) > 0
    for c in ctxs:
        c.close()


def test_level3(word):
    """prepare_for_transcription takes the bank's detections as they are: one segment of seg_len samples each"""
    from easywakeword_b200.bank import WakeWordBank
    bank = WakeWordBank(3, [word], similarity_threshold=50.0)
    bank.ctx.set_stream_params(-1, **dict(bank.params, live=1))       # no ticks here
    xs = [synth.to_int16(x) for x in feeds_of(6500, [5.0, 4.0, 3.0], word)]
    for p in range(0, 80000, 16000):
        bank.push_streams([0, 1, 2], [x[p:p + 16000] for x in xs])
    det = bank.dense_detect()
    assert len(det) > 0
    key = list(zip(det["emit_hop"].tolist(), det["stream"].tolist()))
    assert key == sorted(key)
    seg = bank.prepare_for_transcription(det)
    assert [len(a) for a in seg] == det["seg_len"].tolist()
    bank.close()


def test_errors(word):
    """every refusal changes no cursor and no detector state: the run continued after the errors equals an
    uninterrupted one"""
    from easywakeword_b200 import _lib
    N = 5
    xs = feeds_of(6600, [3.0, 3.0, 3.0, 3.0], word)
    _, push = zip(*(ring_values(x, "i16") for x in xs))
    ctx = make_ctx(N, "i16", [word], ring=32000, slack=16000, live=True)
    ref = make_ctx(N, "i16", [word], ring=32000, slack=16000, live=True)
    for c in (ctx, ref):
        set_thr(c, [45.0] * N)
        c.push_streams(range(4), [q[:20000] for q in push])
    for _ in range(4):
        ctx.push_streams([4], [np.full(30000, 100, np.int16)])      # past its ring: its early hops are gone
    g0 = ctx.dense_detect([0, 1, 2, 3], 60, 0, 1, 3, 7)
    r0 = ref.dense_detect([0, 1, 2, 3], 60, 0, 1, 3, 7)
    launches = ctx.launch_count()
    cases = [
        (lambda: ctx.dense_detect([0, 1], 10, hold_hops=0), ValueError, ["hold_hops"]),
        (lambda: ctx.dense_detect([0, 1], 10, refractory_hops=-1), ValueError, ["refractory_hops"]),
        (lambda: ctx.dense_detect([0, 1], 10, det_cap=9), ValueError, ["need 10"]),
        (lambda: ctx.dense_detect([0, 1], 11, det_cap=11), ValueError, ["need 12"]),
        (lambda: ctx.dense_detect([0, 2, 0], 10), ValueError, ["stream 0", "twice"]),
        (lambda: ctx.dense_detect([0, 7], 10), ValueError, ["stream 7"]),
        (lambda: ctx.dense_detect([0, 4], 10), _lib.EwkError, ["stream 4", "no longer holds"]),
        (lambda: ctx.dense_detect(None, 10), _lib.EwkError, ["stream 4"]),
        (lambda: ctx.dense_detect([0], 10, template_first=1), ValueError, ["reference word"]),
        (lambda: ctx.dense_detect([0], 10, template_first=7, template_count=2), ValueError, ["template"]),
        (lambda: ctx.dense_detect([0], 0), ValueError, ["max_hops"]),
        (lambda: ctx.dense_detect([0], (1 << 20) + 1, det_cap=1), ValueError, ["max_hops"]),
        (lambda: ctx.dense_detect([0, 1], 10, scores=True, out_cap=19), ValueError, ["need 20"]),
    ]
    for fn, exc, words in cases:
        with pytest.raises(exc) as e:
            fn()
        for w in words:
            assert w in str(e.value), str(e.value)
        assert ctx.launch_count() == launches
    for c in (ctx, ref):
        c.push_streams(range(4), [q[20000:] for q in push])
    g = [g0] + detect_all(ctx, [0, 1, 2, 3], 60, 0, 1, 3, 7)[0]
    r = [r0] + detect_all(ref, [0, 1, 2, 3], 60, 0, 1, 3, 7)[0]
    assert_records(np.concatenate(g), np.concatenate(r), "run continued after the errors")
    assert len(np.concatenate(g)) > 0
    ctx.reset_streams([4])
    assert ctx.dense_detect([4], 10, hops=True)[1][0].tolist() == [1]
    ctx.close()
    ref.close()
