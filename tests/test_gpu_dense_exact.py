"""GPU: K4 (dense per-hop scoring) equals, bit for bit, the exact integer model of oracle/dense_model.py over K3's own
frames of each window (the context's extract_mfcc(window, want_frames=True)), for every scored window:
np.array_equal(device, model, equal_nan=True).  Covers the three window classes (un-floored, floored in grid rows
only = a way window, floored in an edge frame = frame by frame), way exhaustion (more than 8 floors in one sub-chunk),
every launch geometry ewk_dense_plan can choose, the ways a request can be cut into calls, ring wrap with int16 and
f32 rings, pre-emphasis, n_mfcc < 20, template subsets, and rows beyond the +-2047 clamp."""
import numpy as np
import pytest

from easywakeword_b200 import synth
from helpers import dense_geometry_sets
from oracle import dense_model as D

pytestmark = pytest.mark.gpu


def make_ctx(n_streams, fmt, templates, ring=200000, slack=16000, **kw):
    from easywakeword_b200 import _lib
    ctx = _lib.Context(device=0, n_streams=n_streams, ring_samples=ring, slack_samples=slack,
                       pcm_format=_lib.PCM_I16 if fmt == "i16" else _lib.PCM_F32, max_templates=8, **kw)
    for i, t in enumerate(templates):
        ctx.set_template(i, t)
    ctx.set_stream_params(-1, frame_size=1600, template_count=1)
    return ctx


def k3_frames(ctx):
    return lambda pcm: ctx.extract_mfcc(pcm, want_frames=True)[2]


def ring_values(x, fmt):
    """What the ring holds for float input x (the samples K4 and the model read) and what to push."""
    if fmt == "i16":
        q = synth.to_int16(x)
        return synth.from_int16(q), q
    return np.asarray(x, np.float32), np.asarray(x, np.float32)


def assert_exact(got, want, what):
    same = np.array_equal(got, want, equal_nan=True)
    if not same:
        bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
        ex = [(tuple(int(v) for v in b), float(got[tuple(b)]), float(want[tuple(b)])) for b in bad[:6]]
        raise AssertionError(f"{what}: {len(bad)} of {got.size} scores differ from the model, e.g. {ex}")


def clicks(seconds, a0=0.9, r=0.995):
    """Digital silence with a one-sample click every 20 ms at strictly decreasing amplitude; 4 of every 20 clicks left
    out, so that every window holds silent (floored) grid frames and its loudest frame — the earliest click — leaves
    the window every 2 hops: a new floor every 2 hops, far more than 8 per sub-chunk."""
    n = int(seconds * 16000)
    y = np.zeros(n, np.float32)
    a = a0
    for m, p in enumerate(range(160, n, 320)):
        if m % 20 < 16:
            y[p] = a
            a *= r
    return y


def class_counts(model, hops, k):
    c, f = model.classes(hops, k)
    return np.bincount(c[c >= 0], minlength=3), c, f


def test_window_classes_and_call_cuts(word):
    """Speech, exact-zero gaps, decaying clicks and an all-zero stream; 4 templates (r = 1 and 2, right-edge frames
    shared by the 16000-, 8000- and 640-sample templates, the 15503-sample word alone); the same hops scored in one
    call, in forward pieces not a multiple of DH starting at hop 0, in overlapping calls, after a backwards jump, after
    a gap and for a template subset.  Every cut equals the model."""
    from easywakeword_b200 import _lib
    tpls = [word, synth.synthetic_word(seed=4, duration=1.0)[:16000], synth.synthetic_word(seed=5, duration=0.5),
            word[4000:4640].copy()]
    lens = [len(t) for t in tpls]
    assert [D.window_geometry(L)[3] for L in lens] == [1, 2, 2, 2]
    sec, H = 4.0, 400
    xs = [synth.stream(4100, sec, word, gain=(1.5, 3.0), inserts_per_10s=(3, 3))[0],
          synth.stream(4101, sec, word, gain=(1.5, 3.0), zero_gaps=4, noise_sigma=0.0005)[0],
          clicks(sec), np.zeros(int(sec * 16000), np.float32)]
    ring, push = zip(*(ring_values(x, "i16") for x in xs))
    ctx = make_ctx(4, "i16", tpls)
    ctx.push(np.stack(push))
    plan = _lib.dense_plan(lens)
    models = [D.DenseModel(r, tpls, k3_frames(ctx)) for r in ring]
    want = np.stack([m.scores(np.arange(H)) for m in models])              # [stream, hop, template]
    cuts = {"forward pieces from hop 0": [(0, 37), (37, 50), (87, 71), (158, 93), (251, 45), (296, 104)],
            "one call": [(0, H)], "overlapping": [(100, 150), (180, 120)], "backwards jump": [(300, 100), (120, 90)],
            "gap": [(50, 40), (200, 60)]}
    for name, calls in cuts.items():
        for h0, nh in calls:
            got = ctx.dense_scores(h0, nh, 0, 4)
            assert ctx.dense_last_plan() == plan
            assert_exact(got, want[:, h0:h0 + nh], f"{name} ({h0}, {nh})")
    got = ctx.dense_scores(150, 130, 1, 2)
    assert_exact(got, want[:, 150:280, 1:3], "templates 1..2")
    assert np.isnan(want[3]).all(), "all-zero stream: std 0, cosine 0 / 0"
    hops = np.arange(H)
    names = ["speech", "zero gaps", "clicks", "all zero"]
    for s, m in enumerate(models):
        cnt = sum(class_counts(m, hops, k)[0] for k in range(4))
        print(f"{names[s]}: windows per class " + ", ".join(f"{n} {c}" for n, c in zip(D.CLASS_NAMES, cnt)))
    assert class_counts(models[0], hops, 0)[0][D.UNFLOORED] > 0
    assert sum(class_counts(models[1], hops, k)[0][D.EDGE] for k in range(4)) > 0
    # way exhaustion: the floors the clicks' way windows need per sub-chunk of the one call from hop 0, all templates
    flat_h, flat_c, flat_f = [], [], []
    for k in range(4):
        _, c, f = class_counts(models[2], hops, k)
        flat_h.append(hops), flat_c.append(c), flat_f.append(f)
    per = D.distinct_way_floors(np.concatenate(flat_h), np.concatenate(flat_c), np.concatenate(flat_f), plan[0], 0)
    print(f"clicks: distinct way-window floors per sub-chunk of DH = {plan[0]}: {per}")
    assert max(per.values()) > 8
    ctx.close()


def test_every_launch_geometry(word):
    """One template set per geometry ewk_dense_plan can choose; the call runs the planned geometry and equals the model."""
    from easywakeword_b200 import _lib
    reach = dense_geometry_sets(_lib.dense_plan)
    assert len(reach) == 8
    pool = np.concatenate([word, synth.synthetic_word(seed=6, duration=1.2), word[::-1],
                           synth.synthetic_word(seed=7, duration=0.97)]).astype(np.float32)
    x, _ = synth.stream(4300, 6.0, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4), zero_gaps=3, noise_sigma=0.001)
    r, q = ring_values(x, "i16")
    for g, lens in sorted(reach.items()):
        tpls = [np.roll(pool, 2311 * k)[:L].copy() for k, L in enumerate(lens)]
        ctx = make_ctx(1, "i16", tpls)
        ctx.push(q.reshape(1, -1))
        m = D.DenseModel(r, tpls, k3_frames(ctx))
        want = m.scores(np.arange(280, 480))
        got = np.concatenate([ctx.dense_scores(280, 77, 0, len(lens)), ctx.dense_scores(357, 123, 0, len(lens))], axis=1)
        assert ctx.dense_last_plan() == _lib.dense_plan(lens)
        assert_exact(got[0], want, f"geometry {g}, lengths {lens}")
        cnt = sum(class_counts(m, np.arange(280, 480), k)[0] for k in range(len(lens)))
        print(f"geometry {g} ({lens}): {np.isfinite(want).sum()} windows equal the model; classes {cnt.tolist()}")
        ctx.close()


@pytest.mark.parametrize("fmt", ["i16", "f32"])
def test_ring_wrap(fmt, word):
    """A ring barely larger than 1 s pushes with a ~1 s template need: pushed 1 s at a time, each piece's hops scored,
    windows and edge frames straddle the ring end."""
    tpls = [word, synth.synthetic_word(seed=4, duration=1.0)[:16000]]
    xs = [synth.stream(4400 + i, 8.0, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4), zero_gaps=2 * i)[0] for i in range(2)]
    ring, push = zip(*(ring_values(x, fmt) for x in xs))
    ctx = make_ctx(2, fmt, tpls, ring=16000, slack=16128)
    P = ((16000 + 16128 + 63) // 64) * 64
    models = [D.DenseModel(r, tpls, k3_frames(ctx)) for r in ring]
    straddle = 0
    q = np.stack(push)
    for p in range(8):
        ctx.push(np.ascontiguousarray(q[:, 16000 * p:16000 * (p + 1)]))
        ctx.tick(10)                         # the gate consumes the piece: the next one may overwrite the ring
        h0 = 100 * p + 1
        got = ctx.dense_scores(h0, 100, 0, 2)
        want = np.stack([m.scores(np.arange(h0, h0 + 100)) for m in models])
        assert_exact(got, want, f"{fmt} piece {p}")
        for L in (len(t) for t in tpls):
            n = D.window_geometry(L)[0]
            st = 160 * (np.arange(h0, h0 + 100) - n)
            st = st[st >= 0]
            straddle += int((((st - 256) % P) + L + 512 > P).sum())
    print(f"{fmt} ring of {P} samples: {straddle} windows straddle the ring end (incl. edge-frame context)")
    assert straddle > 0
    ctx.close()


@pytest.mark.parametrize("variant", ["preemphasis", "n_mfcc13"])
def test_front_end_instantiations(variant, word):
    kw = dict(preemphasis=0.97) if variant == "preemphasis" else dict(n_mfcc=13)
    tpls = [word, word[2000:2640].copy(), synth.synthetic_word(seed=8, duration=0.6)]
    xs = [synth.stream(4500 + i, 4.0, word, gain=(1.5, 3.0), inserts_per_10s=(3, 3), zero_gaps=3 * i,
                       noise_sigma=0.0005)[0] for i in range(2)]
    fmt = "f32" if variant == "preemphasis" else "i16"
    ring, push = zip(*(ring_values(x, fmt) for x in xs))
    ctx = make_ctx(2, fmt, tpls, **kw)
    ctx.push(np.stack(push))
    models = [D.DenseModel(r, tpls, k3_frames(ctx), n_mfcc=kw.get("n_mfcc", 20), preemphasis=kw.get("preemphasis", 0.0))
              for r in ring]
    want = np.stack([m.scores(np.arange(400)) for m in models])
    got = np.concatenate([ctx.dense_scores(0, 150, 0, 3), ctx.dense_scores(150, 250, 0, 3)], axis=1)
    assert_exact(got, want, variant)
    assert_exact(ctx.dense_scores(120, 200, 1, 2), want[:, 120:320, 1:3], variant + " templates 1..2")
    cnt = sum(class_counts(models[1], np.arange(400), k)[0] for k in range(3))
    print(f"{variant}: {np.isfinite(want).sum()} windows equal the model; gap stream classes {cnt.tolist()}")
    ctx.close()


def test_rows_beyond_the_clamp(word):
    """An f32 stream at 1e11 full scale: c0 of its loud frames passes 2047, where K4 clamps its rows (and so departs from
    the reference, which does not); the model clamps alike."""
    x, _ = synth.stream(4600, 3.0, word, gain=(2.0, 4.0), inserts_per_10s=(3, 3))
    x = (x * 1e11).astype(np.float32)
    ctx = make_ctx(1, "f32", [word])
    ctx.push(x.reshape(1, -1))
    m = D.DenseModel(x, [word], k3_frames(ctx))
    want = m.scores(np.arange(300))
    assert_exact(ctx.dense_scores(0, 300, 0, 1)[0], want, "clamp")
    fr = k3_frames(ctx)(x)
    print(f"clamp: max |MFCC| of the stream's frames {np.abs(fr).max():.1f}")
    assert np.abs(fr).max() > D.CLAMP
    ctx.close()
