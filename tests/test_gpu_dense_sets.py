"""GPU: per-row template sets in dense scoring and detection (ewk_dense_scores_sets, ewk_dense_ready_sets,
ewk_dense_detect_sets).  Every row equals, bit for bit (np.array_equal(equal_nan=True)), the single-set call of that row
alone with its set and the uniform ewk_dense_scores (K4's other instance), and on a subset oracle/dense_model.py; paced calls equal per-set grouped ewk_dense_ready /
ewk_dense_detect calls and oracle/dense_detect.py record for record; one K4 launch per geometry plus one K4D; resets,
migration, cache invalidation and every error."""
import ctypes

import numpy as np
import pytest

from easywakeword_b200 import synth
from helpers import dense_geometry_sets
from oracle import dense_detect as M
from oracle import dense_model as D

pytestmark = pytest.mark.gpu

NT = 64
REFUSED = [640, 700, 800, 900, 1000, 1100, 1200, 48000]     # fits shared memory in no geometry as a whole


def layout(word):
    """Template lengths of the 64 slots and the named sets: every reachable geometry's set, a range that does not fit,
    the wake word, and one-template slots of random lengths."""
    from easywakeword_b200 import _lib
    geo = dense_geometry_sets(_lib.dense_plan)
    lens, sets = [], []
    for lst in geo.values():
        sets.append((len(lens), len(lst)))
        lens += lst
    refused = (len(lens), len(REFUSED))
    lens += REFUSED
    word_slot = len(lens)
    lens.append(len(word))
    rng = np.random.default_rng(64)
    while len(lens) < NT:
        lens.append(int(rng.integers(640, 48001)))
    return lens, sets, refused, word_slot


def make_templates(word, lens):
    out = []
    for i, L in enumerate(lens):
        out.append(word.copy() if L == len(word) else synth.synthetic_word(seed=900 + i, duration=3.0)[:L].copy())
    return out


def make_ctx(n, fmt, tpls, ring=200000, **kw):
    from easywakeword_b200 import _lib
    ctx = _lib.Context(device=0, n_streams=n, ring_samples=ring, slack_samples=16000,
                       pcm_format=_lib.PCM_I16 if fmt == "i16" else _lib.PCM_F32, max_templates=NT, max_events=4096, **kw)
    for i, t in enumerate(tpls):
        ctx.set_template(i, t)
    ctx.set_stream_params(-1, frame_size=1600, template_first=0, template_count=1, live=1, similarity_threshold=62.0)
    return ctx


def feeds(word, n, seconds, seed):
    xs = []
    for i in range(n):
        x = synth.stream(seed + i, seconds, word, gain=(1.5, 3.0), inserts_per_10s=(4, 6),
                         zero_gaps=2 if i % 3 == 1 else 0)[0]
        xs.append(synth.from_int16(synth.to_int16(x)))
    return xs


def pushed(x, fmt):
    return synth.to_int16(x) if fmt == "i16" else np.asarray(x, np.float32)


def random_set(rng, lens, sets, word_slot):
    """A plannable (first, count): a geometry's set, a random range, one slot, or the word."""
    from easywakeword_b200 import _lib
    r = rng.random()
    if r < 0.3:
        return sets[int(rng.integers(len(sets)))]
    if r < 0.45:
        return word_slot, 1
    if r < 0.75:
        return int(rng.integers(0, NT)), 1
    while True:
        c = int(rng.integers(1, 9))
        f = int(rng.integers(0, NT - c + 1))
        try:
            _lib.dense_plan(lens[f:f + c])
            return f, c
        except ValueError:
            continue


def assert_rows(got, want, what):
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape, (what, i, g.shape, w.shape)
        if not np.array_equal(g, w, equal_nan=True):
            bad = int((~((g == w) | (np.isnan(g) & np.isnan(w)))).sum())
            raise AssertionError(f"{what}: row {i}: {bad} of {g.size} scores differ")


@pytest.mark.parametrize("fmt,kw", [("i16", {}), ("f32", {}), ("i16", {"preemphasis": 0.97, "n_mfcc": 13})],
                         ids=["i16", "f32", "i16-pre-mfcc13"])
def test_scores_sets_equal_single_set_rows(word, fmt, kw):
    """Random stream lists, each row with a random set (shared, overlapping, identical, disjoint; every geometry; one-
    template sets of all 64 slots): every row equals ewk_dense_scores_streams of that row alone with its set and the
    uniform ewk_dense_scores of its hops and set, host and device output, and the model on a subset.  Launches: one K4 per geometry among the non-empty rows."""
    import torch
    from easywakeword_b200 import _lib
    lens, sets, _, word_slot = layout(word)
    tpls = make_templates(word, lens)
    N = 12
    xs = feeds(word, N, 3.0, 5100)
    ctx = make_ctx(N, fmt, tpls, **kw)
    ctx.push(np.stack([pushed(x, fmt) for x in xs]))
    hops = [len(x) // 160 for x in xs]
    ctx.dense_scores_streams(list(range(N)), hops, [1] * N, 0, 1)     # lands the push: launch counts below are K4's alone
    rng = np.random.default_rng(7 if fmt == "i16" else 8)
    one_slot_sets = set()
    model_rows = 0
    frames = lambda pcm: ctx.extract_mfcc(pcm, want_frames=True)[2]

    def alone(s, a, n, f, c):
        """row s alone through ewk_dense_scores_streams, checked against the uniform instance (every stream has the same
        length, so every stream holds these hops)"""
        row = ctx.dense_scores_streams([s], [a], [n], f, c)[0]
        assert_rows([row], [ctx.dense_scores(a, n, f, c)[s] if n else np.zeros((0, c), np.float32)],
                    f"uniform stream {s} hops {a}+{n} set {f}+{c}")
        return row
    for call in range(10):
        k = int(rng.integers(1, N + 1))
        streams = [int(s) for s in rng.choice(N, k, replace=False)]
        fs, cs, h0, nh = [], [], [], []
        for i, s in enumerate(streams):
            if call == 0:
                f, c = sets[i % len(sets)]                     # every geometry in one call
            elif call == 1:
                f, c = (i * 5) % NT, 1
            else:
                f, c = random_set(rng, lens, sets, word_slot)
            fs.append(f); cs.append(c)
            a = int(rng.integers(0, hops[s] - 5))
            h0.append(a)
            nh.append(0 if rng.random() < 0.15 else int(rng.integers(1, min(hops[s] - a, 140) + 1)))
            if c == 1:
                one_slot_sets.add(f)
        n0 = ctx.launch_count()
        got = ctx.dense_scores_sets(streams, h0, nh, fs, cs)
        tlens = [[len(tpls[j]) for j in range(f, f + c)] for f, c in zip(fs, cs)]
        groups = _lib.sets_launches([tl for tl, n in zip(tlens, nh) if n > 0])
        assert ctx.launch_count() - n0 == len(groups), (call, ctx.launch_count() - n0, groups)
        if groups:
            assert ctx.dense_last_plan()[:3] == list(groups)[-1]
        want = [alone(s, a, n, f, c) for s, a, n, f, c in zip(streams, h0, nh, fs, cs)]
        assert_rows(got, want, f"call {call}")
        # device output, packed as the header says
        off, total = _lib.sets_offsets(nh, cs)
        dev = torch.full((total + 3,), -7.0, dtype=torch.float32, device="cuda:0")
        ctx.dense_scores_sets(streams, h0, nh, fs, cs, out_device_ptr=dev.data_ptr())
        torch.cuda.synchronize()
        d = dev.cpu().numpy()
        assert np.all(d[total:] == -7.0)
        assert_rows([d[o:o + n * c].reshape(n, c) for o, n, c in zip(off, nh, cs)], want, f"call {call} device")
        if call < 3 and not kw:
            for s, a, n, f, c, g in list(zip(streams, h0, nh, fs, cs, got))[:2]:
                m = D.DenseModel(xs[s], tpls[f:f + c], frames)
                assert_rows([g[:40]], [m.scores(np.arange(a, a + min(n, 40)))], f"model call {call} stream {s}")
                model_rows += 1
    if fmt == "i16" and not kw:
        # every slot as a one-template set, 64 distinct sets in one call of 12 rows at a time
        for base in range(0, NT, N):
            fs = [(base + i) % NT for i in range(N)]
            got = ctx.dense_scores_sets(list(range(N)), [10] * N, [30] * N, fs, [1] * N)
            want = [alone(s, 10, 30, f, 1) for s, f in zip(range(N), fs)]
            assert_rows(got, want, f"one-slot sets from {base}")
            one_slot_sets.update(fs)
        assert len(one_slot_sets) >= 64
        assert model_rows > 0
    # both arrays NULL: each stream's own range, as set_stream_params set it
    own = [random_set(rng, lens, sets, word_slot) for _ in range(N)]
    for s, (f, c) in enumerate(own):
        ctx.set_stream_params(s, frame_size=1600, template_first=f, template_count=c, live=1)
    got = ctx.dense_scores_sets(list(range(N)), [5] * N, [50] * N)
    want = [alone(s, 5, 50, f, c) for s, (f, c) in enumerate(own)]
    assert_rows(got, want, "own ranges")
    ctx.close()


def test_paced_detect_sets_equal_grouped_calls(word):
    """ready_sets / detect_sets under random ragged pushes and random max_hops against a twin context served by per-set
    grouped ewk_dense_ready / ewk_dense_detect calls: the same hops, scores and detections (and oracle/dense_detect.py
    record for record), runs left ARMED across calls, streams switching sets between calls, errors that move nothing,
    K4 + K4D launch counts, a template change (cache invalidation), a reset and a migration."""
    from easywakeword_b200 import _lib
    lens, sets, refused, word_slot = layout(word)
    tpls = make_templates(word, lens)
    N = 10
    xs = feeds(word, N, 12.0, 6100)
    A = make_ctx(N, "i16", tpls)
    B = make_ctx(N, "i16", tpls)
    q = [synth.to_int16(x) for x in xs]
    pos = [0] * N
    rng = np.random.default_rng(11)
    cur = [random_set(rng, lens, sets, word_slot) if s % 2 else (word_slot, 1) for s in range(N)]
    ost = [None] * N                                            # oracle detector state per stream
    hold, refr = 6, 9
    n_det = n_switch = armed_carry = 0
    all_scores = {s: [] for s in range(N)}

    def push_some():
        st = [s for s in range(N) if pos[s] < len(q[s]) and rng.random() < 0.8]
        blocks = []
        for s in st:
            n = int(rng.integers(0, 9000))
            blocks.append(q[s][pos[s]:pos[s] + n])
            pos[s] += len(blocks[-1])
        if st:
            A.push_streams(st, blocks)
            B.push_streams(st, blocks)

    def grouped(streams, mh, which):
        """B's answer: one single-set call per distinct set, results back in list order"""
        by = {}
        for i, s in enumerate(streams):
            by.setdefault(cur[s], []).append(i)
        h0 = np.zeros(len(streams), np.int64)
        rows = [None] * len(streams)
        dets = []
        for (f, c), idx in by.items():
            lst = [streams[i] for i in idx]
            if which == "ready":
                h, r = B.dense_ready(lst, mh, f, c)
            else:
                d, (h, r) = B.dense_detect(lst, mh, f, c, hold, refr, scores=True)
                dets.append(d)
            for j, i in enumerate(idx):
                h0[i], rows[i] = h[j], r[j]
        return h0, rows, dets

    for step in range(40):
        push_some()
        if step % 5 == 4:                                       # some streams switch sets
            for s in rng.choice(N, 3, replace=False):
                cur[int(s)] = random_set(rng, lens, sets, word_slot) if rng.random() < 0.6 else (word_slot, 1)
                n_switch += 1
        streams = [int(s) for s in rng.choice(N, int(rng.integers(1, N + 1)), replace=False)]
        mh = int(rng.integers(1, 120))
        fs = [cur[s][0] for s in streams]
        cs = [cur[s][1] for s in streams]
        h0, rows = A.dense_ready_sets(streams, mh, fs, cs)
        bh, brows, _ = grouped(streams, mh, "ready")
        assert np.array_equal(h0, bh)
        assert_rows(rows, brows, f"ready step {step}")
        n0 = A.launch_count()
        d, (dh, drows) = A.dense_detect_sets(streams, mh, fs, cs, hold, refr, scores=True)
        tl = [[len(tpls[j]) for j in range(f, f + c)] for f, c, r in zip(fs, cs, drows) if len(r)]
        if tl:
            assert A.launch_count() - n0 == len(_lib.sets_launches(tl)) + 1
        gh, grows, gd = grouped(streams, mh, "detect")
        assert np.array_equal(dh, gh)
        assert_rows(drows, grows, f"detect scores step {step}")
        gd = np.concatenate(gd) if gd else np.zeros(0, _lib.DETECTION_DTYPE)
        order = {s: i for i, s in enumerate(streams)}
        gd = gd[np.lexsort((gd["emit_hop"], [order[int(s)] for s in gd["stream"]]))] if len(gd) else gd
        assert d.tobytes() == gd.tobytes(), (step, d, gd)
        # the host model, chunk by chunk with each chunk's set
        want = []
        for s, h, r, f, c in zip(streams, dh, drows, fs, cs):
            ev, ost[s] = M.detect(r, int(h), ost[s], 62.0, hold, refr, f, [len(tpls[j]) for j in range(f, f + c)], stream=s)
            want += list(ev)
            armed_carry += ost[s]["mode"] == M.ARMED and len(r) > 0
        assert len(want) == len(d)
        for a, b in zip(d, want):
            assert tuple(a.tolist()) == tuple(np.asarray(b, _lib.DETECTION_DTYPE).tolist()), (step, a, b)
        n_det += len(d)
        if step == 12:
            # errors: nothing moves (the next calls still equal the twin's)
            bad = [([0], [0]), ([0], [9]), ([-1], [1]), ([NT - 1], [2]), ([refused[0]], [refused[1]])]
            for f, c in bad:
                with pytest.raises(ValueError, match=r"row 0 \(stream"):
                    A.dense_detect_sets([streams[0]], mh, f, c, hold, refr)
                with pytest.raises(ValueError, match=r"row 0 \(stream"):
                    A.dense_ready_sets([streams[0]], mh, f, c)
            i32p, i64p = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
            tf_only = np.zeros(N, np.int32)
            h_, n_ = np.zeros(N, np.int64), np.zeros(N, np.int32)
            assert A.lib.ewk_dense_ready_sets(A.h, None, 0, 10, tf_only.ctypes.data_as(i32p), None,
                                              h_.ctypes.data_as(i64p), n_.ctypes.data_as(i32p), None, 0,
                                              _lib.HOST) == _lib.EWK_ERR_ARG
        if step == 20:
            # a template change invalidates the cached sets covering the slot: both contexts get the same new template
            slot = int(rng.integers(24, NT))
            t = synth.synthetic_word(seed=77, duration=1.2)
            A.set_template(slot, t); B.set_template(slot, t)
            tpls[slot] = t
            lens[slot] = len(t)
            cur[streams[0]] = (slot, 1)
            A.clear_template(slot + 0)
            with pytest.raises(ValueError, match="empty"):
                A.dense_scores_sets([0], [1], [1], [slot], [1])
            A.set_template(slot, t)
    assert n_det > 0 and n_switch > 0 and armed_carry > 0, (n_det, n_switch, armed_carry)

    # reset: stream 0 of A equals stream 0 of a new context fed the same audio after the reset
    A.poll()
    A.reset_streams([0])
    C = make_ctx(1, "i16", tpls)
    y = q[3][:80000]
    A.push_streams([0], [y]); C.push_streams([0], [y])
    f, c = sets[-1]
    da, (ha, ra) = A.dense_detect_sets([0], 1000, [f], [c], hold, refr, scores=True)
    dc, (hc, rc_) = C.dense_detect_sets([0], 1000, [f], [c], hold, refr, scores=True)
    assert np.array_equal(ha, hc) and da.tobytes() == dc.tobytes()
    assert_rows(ra, rc_, "reset")
    # migration: streams exported from B and imported into a new context go on bit for bit under *_sets
    B.poll()
    blob = B.export_streams(list(range(N)))
    E = make_ctx(N, "i16", tpls)
    E.import_streams(list(range(N)), blob)
    for s in range(N):
        rest = q[s][pos[s]:pos[s] + 24000]
        if len(rest):
            B.push_streams([s], [rest]); E.push_streams([s], [rest])
    fs = [cur[s][0] for s in range(N)]
    cs = [cur[s][1] for s in range(N)]
    db, (hb, rb) = B.dense_detect_sets(None, 400, fs, cs, hold, refr, scores=True)
    de, (he, re_) = E.dense_detect_sets(None, 400, fs, cs, hold, refr, scores=True)
    assert np.array_equal(hb, he) and db.tobytes() == de.tobytes()
    assert_rows(re_, rb, "migrated")
    with pytest.raises(ValueError, match="imported"):
        E.dense_ready_sets(None, 10)                            # own ranges of imported streams: not known in Python
    for x in (A, B, C, E):
        x.close()
