"""GPU: ragged dense scoring (ewk_dense_scores_streams) and dense scores paced by each stream's audio (ewk_dense_ready).
Every score is compared with np.array_equal(..., equal_nan=True) against the exact model of oracle/dense_model.py over
K3's own frames of each window, the model test_gpu_dense_exact.py pins ewk_dense_scores to: per-row hop ranges, random
stream subsets, empty rows, every launch geometry, pacing by random ragged pushes, recycled streams, pending pushes,
overlap mode, device output, and every error (which must leave the cursors alone)."""
import numpy as np
import pytest

from easywakeword_b200 import synth
from easywakeword_b200.resample import ULAW_TABLE, due_hops
from helpers import dense_geometry_sets
from oracle import dense_model as D

pytestmark = pytest.mark.gpu


def make_ctx(n_streams, fmt, templates, ring=200000, slack=16000, live=False, **kw):
    from easywakeword_b200 import _lib
    ctx = _lib.Context(device=0, n_streams=n_streams, ring_samples=ring, slack_samples=slack,
                       pcm_format=_lib.PCM_I16 if fmt == "i16" else _lib.PCM_F32, max_templates=8, **kw)
    for i, t in enumerate(templates):
        ctx.set_template(i, t)
    ctx.set_stream_params(-1, frame_size=1600, template_count=1, live=1 if live else 0)
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
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got, want, equal_nan=True):
        bad = np.argwhere(~((got == want) | (np.isnan(got) & np.isnan(want))))
        ex = [(tuple(int(v) for v in b), float(got[tuple(b)]), float(want[tuple(b)])) for b in bad[:6]]
        raise AssertionError(f"{what}: {len(bad)} of {got.size} scores differ from the model, e.g. {ex}")


def clicks(seconds, a0=0.9, r=0.995):
    """Digital silence with a decaying one-sample click every 20 ms (4 of 20 left out): a new floor every 2 hops."""
    n = int(seconds * 16000)
    y = np.zeros(n, np.float32)
    a = a0
    for m, p in enumerate(range(160, n, 320)):
        if m % 20 < 16:
            y[p] = a
            a *= r
    return y


class Want:
    """Model scores per stream, computed once per hop: want(s, h0, n) -> [n, T_all]."""

    def __init__(self, ring_rows, tpls, frames_fn, **kw):
        self.models = [D.DenseModel(r, tpls, frames_fn, **kw) for r in ring_rows]
        self.cache = [dict() for _ in ring_rows]
        self.T = len(tpls)

    def __call__(self, s, h0, n):
        c = self.cache[s]
        miss = [h for h in range(h0, h0 + n) if h not in c]
        if miss:
            for h, row in zip(miss, self.models[s].scores(np.array(miss))):
                c[h] = row
        return np.stack([c[h] for h in range(h0, h0 + n)]) if n else np.zeros((0, self.T), np.float32)


def four_templates(word):
    return [word, synth.synthetic_word(seed=4, duration=1.0)[:16000], synth.synthetic_word(seed=5, duration=0.5),
            word[4000:4640].copy()]


def test_explicit_ragged_rows(word):
    """Speech, zero gaps, decaying clicks and an all-zero stream (two of each kind), fed different amounts by
    push_streams; random subsets with rows of 0 hops and rows not a multiple of DH; per stream, overlapping, backwards and
    gapped rows across calls; template subsets.  Every row equals the model, and where a uniform call is possible the
    matching rows of ewk_dense_scores."""
    tpls = four_templates(word)
    secs = [4.0, 2.6, 3.3, 1.9, 3.1, 2.2, 4.0, 1.4]
    kinds = [lambda s, i: synth.stream(4700 + i, s, word, gain=(1.5, 3.0), inserts_per_10s=(3, 3))[0],
             lambda s, i: synth.stream(4710 + i, s, word, gain=(1.5, 3.0), zero_gaps=4, noise_sigma=0.0005)[0],
             lambda s, i: clicks(s), lambda s, i: np.zeros(int(s * 16000), np.float32)]
    xs = [kinds[i % 4](sec, i) for i, sec in enumerate(secs)]
    ring, push = zip(*(ring_values(x, "i16") for x in xs))
    N = len(xs)
    ctx = make_ctx(N, "i16", tpls)
    order = [5, 0, 7, 2, 6, 1, 3, 4]
    ctx.push_streams(order, [push[s][:len(push[s]) // 2] for s in order])
    ctx.push_streams(order[::-1], [push[s][len(push[s]) // 2:] for s in order[::-1]])
    hops = [len(x) // 160 for x in xs]                       # last hop with audio per stream
    want = Want(ring, tpls, k3_frames(ctx))
    rng = np.random.default_rng(47)
    n_rows = n_empty = 0
    for call in range(14):
        k = int(rng.integers(1, N + 1))
        streams = [int(s) for s in rng.choice(N, k, replace=False)]
        tf, T = (0, 4) if call % 3 else (int(rng.integers(0, 3)), int(rng.integers(1, 3)))
        T = min(T, 4 - tf)
        h0, nh = [], []
        for s in streams:
            a = int(rng.integers(0, hops[s] - 5))
            n = 0 if rng.random() < 0.2 else int(rng.integers(1, min(hops[s] - a, 150) + 1))
            h0.append(a)
            nh.append(n)
        got = ctx.dense_scores_streams(streams, h0, nh, tf, T)
        for s, a, n, g in zip(streams, h0, nh, got):
            assert_exact(g, want(s, a, n)[:, tf:tf + T], f"call {call} stream {s} hops [{a}, {a + n}) templates {tf}+{T}")
            n_rows += 1
            n_empty += n == 0
    # one stream, consecutive calls: forward pieces, overlap, backwards jump, gap (the carried rows must not leak)
    for a, n in [(0, 37), (37, 50), (87, 71), (120, 90), (30, 45), (300, 77), (230, 10)]:
        g, = ctx.dense_scores_streams([6], [a], [n], 0, 4)
        assert_exact(g, want(6, a, n), f"stream 6 hops [{a}, {a + n})")
    # where a uniform call is possible (every stream has the audio) the rows equal its slices
    top = min(hops)
    uni = ctx.dense_scores(40, top - 40, 0, 4)
    streams, h0, nh = [3, 6, 1, 0], [40, 60, 40, 75], [top - 40, top - 60, 0, 50]
    got = ctx.dense_scores_streams(streams, h0, nh, 0, 4)
    for s, g, a, n in zip(streams, got, h0, nh):
        assert len(g) == n
        assert_exact(g, uni[s, a - 40:a - 40 + n], f"uniform slice, stream {s}")
    assert ctx.dense_scores_streams([], [], []) == []
    print(f"{n_rows} ragged rows ({n_empty} empty) equal the model")
    ctx.close()


def test_every_launch_geometry(word):
    """One template set per geometry ewk_dense_plan can choose, through the ragged entry point: rows of different
    lengths on three streams fed different amounts; dense_last_plan reports the planned geometry."""
    from easywakeword_b200 import _lib
    reach = dense_geometry_sets(_lib.dense_plan)
    assert len(reach) == 8
    pool = np.concatenate([word, synth.synthetic_word(seed=6, duration=1.2), word[::-1],
                           synth.synthetic_word(seed=7, duration=0.97)]).astype(np.float32)
    xs = [synth.stream(4800 + i, sec, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4), zero_gaps=3, noise_sigma=0.001)[0]
          for i, sec in enumerate([6.0, 4.5, 5.2])]
    ring, push = zip(*(ring_values(x, "i16") for x in xs))
    for g, lens in sorted(reach.items()):
        tpls = [np.roll(pool, 2311 * k)[:L].copy() for k, L in enumerate(lens)]
        ctx = make_ctx(3, "i16", tpls)
        ctx.push_streams([0, 1, 2], list(push))
        want = Want(ring, tpls, k3_frames(ctx))
        rows = [(1, 250, 113), (0, 280, 200), (2, 300, 0)]
        got = ctx.dense_scores_streams(*zip(*rows), 0, len(lens))
        assert ctx.dense_last_plan() == _lib.dense_plan(lens)
        for (s, a, n), gr in zip(rows, got):
            assert_exact(gr, want(s, a, n), f"geometry {g}, lengths {lens}, stream {s}")
        ctx.close()


def paced_run(ctx, streams_all, feeds, max_hops, T):
    """Feed 16 kHz pieces [(streams, rows)] with push_streams, each followed by dense_ready until nothing is due; -> (next
    cursor, concatenated scores) per stream, checking that hop0 values chain and counts follow due_hops."""
    N = len(streams_all)
    nxt = np.ones(N, np.int64)
    written = np.zeros(N, np.int64)
    got = [[] for _ in range(N)]
    for streams, rows in feeds:
        ctx.push_streams(streams, rows)
        for s, r in zip(streams, rows):
            written[s] += len(r)
        while True:
            lst = streams_all if len(streams) % 2 else None      # explicit list and NULL (= every stream) alike
            h0, out = ctx.dense_ready(lst, max_hops, 0, T)
            n = np.array([len(o) for o in out])
            assert np.array_equal(h0, nxt), (h0, nxt)
            assert np.array_equal(n, due_hops(written, nxt, max_hops))
            for s, o in enumerate(out):
                got[s].append(o)
            nxt += n
            if n.max(initial=0) < max_hops:
                break
    return nxt, [np.concatenate(g) for g in got]


PACED = {
    "i16_ring_wrap": dict(fmt="i16", ring=16000, slack=16128),
    "f32_ring_wrap": dict(fmt="f32", ring=16000, slack=16128),
    "preemphasis": dict(fmt="f32", ring=48000, slack=16000, preemphasis=0.97),
    "n_mfcc13": dict(fmt="i16", ring=48000, slack=16000, n_mfcc=13),
}


@pytest.mark.parametrize("variant", list(PACED))
def test_paced_equals_uniform(variant, word):
    """The same audio fed in random ragged pieces to random subsets, dense_ready after every push with max_hops small
    enough to cut rows, and fed in one piece: per stream the concatenated paced scores equal the model over hops
    1 .. written / 160, hop0 values chain without gaps, a parked stream gets 0 hops."""
    cfg = dict(PACED[variant])
    fmt, ring_s, slack = cfg.pop("fmt"), cfg.pop("ring"), cfg.pop("slack")
    tpls = [word, synth.synthetic_word(seed=4, duration=1.0)[:16000]]
    N, secs = 5, [5.0, 3.7, 4.4, 0.0, 2.9]                  # stream 3 stays parked
    xs = [synth.stream(4900 + i, sec, word, gain=(1.5, 3.0), inserts_per_10s=(4, 4), zero_gaps=2 * (i % 2),
                       noise_sigma=0.0005)[0] if sec else np.zeros(0, np.float32) for i, sec in enumerate(secs)]
    ring, push = zip(*(ring_values(x, fmt) for x in xs))
    rng = np.random.default_rng(11 + list(PACED).index(variant))
    pos = [0] * N
    feeds = []
    while any(pos[s] < len(push[s]) for s in range(N)):
        live = [s for s in range(N) if pos[s] < len(push[s])]
        streams = [int(s) for s in rng.choice(live, int(rng.integers(1, len(live) + 1)), replace=False)]
        rows = []
        for s in streams:
            n = min(int(rng.integers(0, 9000)), len(push[s]) - pos[s])
            rows.append(push[s][pos[s]:pos[s] + n])
            pos[s] += n
        feeds.append((streams, rows))
    ctx = make_ctx(N, fmt, tpls, ring=ring_s, slack=slack, live=True, **cfg)
    nxt, got = paced_run(ctx, list(range(N)), feeds, 23, 2)
    one = make_ctx(N, fmt, tpls, ring=max(ring_s, 6 * 16000), slack=slack, live=True, **cfg)
    nxt1, got1 = paced_run(one, list(range(N)), [([0, 1, 2, 4], [push[s] for s in (0, 1, 2, 4)])], 23, 2)
    want = Want(ring, tpls, k3_frames(ctx), n_mfcc=cfg.get("n_mfcc", 20), preemphasis=cfg.get("preemphasis", 0.0))
    for s in range(N):
        H = len(push[s]) // 160
        assert nxt[s] == nxt1[s] == H + 1
        assert_exact(got[s], want(s, 1, H), f"{variant} paced stream {s}")
        assert_exact(got1[s], got[s], f"{variant} one piece stream {s}")
    assert len(got[3]) == 0
    print(f"{variant}: {len(feeds)} ragged pushes, {sum(len(g) for g in got)} paced hops equal the model")
    ctx.close()
    one.close()


def ulaw_encode(q):
    table = ULAW_TABLE.astype(np.int32)
    order = np.argsort(table, kind="stable")
    srt = table[order]
    i = np.clip(np.searchsorted(srt, q.astype(np.int32)), 1, 255)
    pick = np.where(np.abs(srt[i] - q) < np.abs(srt[i - 1] - q), i, i - 1)
    return order[pick].astype(np.uint8)


def test_reset_recycles_cursors(word):
    """Streams 1 and 3 are reset mid-run and re-fed with 8 kHz mu-law (K8).  Their paced scores after the reset start at
    hop 1 and equal those of the same streams in a new context fed the same codes; the other streams' scores equal the
    model of their whole audio, as in a run without the reset."""
    tpls = [word, synth.synthetic_word(seed=5, duration=0.5)]
    N = 4
    xs = [synth.stream(5000 + i, 4.0, word, gain=(1.5, 3.0), inserts_per_10s=(3, 3))[0] for i in range(N)]
    ring, push = zip(*(ring_values(x, "i16") for x in xs))
    codes = [ulaw_encode(synth.to_int16(synth.stream(5100 + i, 3.0, word, gain=(1.5, 3.0))[0][::2])) for i in range(2)]
    ctx = make_ctx(N, "i16", tpls, live=True)
    fresh = make_ctx(N, "i16", tpls, live=True)
    before = [[] for _ in range(N)]
    after = {1: [], 3: []}
    ref = {1: [], 3: []}
    cut = 16000 * 2
    for p in range(0, cut, 7000):                             # 16 kHz pieces for everyone
        ctx.push_streams(list(range(N)), [q[p:min(p + 7000, cut)] for q in push])
        h0, out = ctx.dense_ready(None, 37, 0, 2)
        for s in range(N):
            before[s].append(out[s])
    ctx.reset_streams([3, 1])
    h0, out = ctx.dense_ready([1, 3], 37, 0, 2)
    assert h0.tolist() == [1, 1] and [len(o) for o in out] == [0, 0]
    for p in range(0, 24000, 3100):                           # reset streams: 8 kHz mu-law; others: the rest at 16 kHz
        ctx.push_streams([1, 3], [c[p:p + 3100] for c in codes], sr_in=8000, fmt="ulaw")
        fresh.push_streams([1, 3], [c[p:p + 3100] for c in codes], sr_in=8000, fmt="ulaw")
        q = cut + 2 * p
        ctx.push_streams([0, 2], [push[0][q:q + 6200], push[2][q:q + 6200]])
        for s, o in zip([0, 1, 2, 3], ctx.dense_ready([0, 1, 2, 3], 1000, 0, 2)[1]):
            (after[s] if s in after else before[s]).append(o)
        for s, o in zip([1, 3], fresh.dense_ready([1, 3], 1000, 0, 2)[1]):
            ref[s].append(o)
    want = Want(ring, tpls, k3_frames(ctx))
    for s in (0, 2):
        g = np.concatenate(before[s])
        assert_exact(g, want(s, 1, len(g)), f"stream {s} (not reset)")
        assert len(g) == len(push[s]) // 160
    for s in (1, 3):
        g, r = np.concatenate(after[s]), np.concatenate(ref[s])
        assert len(g) == ctx.status(s).written // 160 > 0
        assert_exact(g, r, f"stream {s} after reset vs a new context")
    ctx.close()
    fresh.close()


@pytest.mark.parametrize("path", ["pending", "overlap", "device"])
def test_feeds(path, word):
    """pending: a pinned host push still in flight lands only when a row reaches into it (ring_push launches).
    overlap: K3 on its own stream beside the calls.  device: packed output in device memory equals the host output."""
    import torch
    from easywakeword_b200 import _lib
    tpls = [word]
    N = 3
    xs = [synth.stream(5200 + i, 3.0, word, gain=(1.5, 3.0), inserts_per_10s=(3, 3))[0] for i in range(N)]
    ring, push = zip(*(ring_values(x, "i16") for x in xs))
    ctx = make_ctx(N, "i16", tpls, live=path != "overlap")
    want = Want(ring, tpls, k3_frames(ctx))
    if path == "pending":
        ctx.profile(True)
        pin = _lib.PinnedArray((N * 48000,), np.int16)
        pin.array[...] = np.concatenate(push)
        offs, lens = np.arange(N) * 48000, np.full(N, 24000)
        ctx.push_streams(range(N), (pin.ptr.value, offs, lens, N * 48000, np.int16))
        ctx.push_streams(range(N), (pin.ptr.value, offs + 24000, lens, N * 48000, np.int16))   # lands the first block
        assert ctx.profile_read()["ring_push"]["launches"] == 1                                # (read resets the counts)
        got = ctx.dense_scores_streams([2, 0], [10, 1], [140, 149], 0, 1)                      # inside block 1
        assert ctx.profile_read()["ring_push"]["launches"] == 0
        assert_exact(got[0], want(2, 10, 140), "pending: stream 2")
        assert_exact(got[1], want(0, 1, 149), "pending: stream 0")
        got = ctx.dense_scores_streams([1], [100], [60], 0, 1)                                 # reaches into block 2
        assert ctx.profile_read()["ring_push"]["launches"] == 1
        assert_exact(got[0], want(1, 100, 60), "pending: stream 1 in block 2")
        pin.free()
    elif path == "overlap":
        ctx.set_overlap(True)
        for p in range(0, 48000, 8000):
            ctx.push_streams(range(N), [q[p:p + 8000] for q in push])
            ctx.tick_ready(64)                                 # K3 in flight on the match stream
            h0, out = ctx.dense_ready(None, 64, 0, 1)
            for s in range(N):
                assert_exact(out[s], want(s, int(h0[s]), len(out[s])), f"overlap stream {s} at {p}")
            ctx.poll()
    else:
        ctx.push_streams(range(N), list(push))
        rows = ([2, 0, 1], [5, 100, 40], [120, 0, 77])
        host = ctx.dense_scores_streams(*rows, 0, 1)
        dev = torch.full((197 + 5,), -1.0, dtype=torch.float32, device="cuda:0")
        ctx.dense_scores_streams(*rows, 0, 1, out_device_ptr=dev.data_ptr())
        torch.cuda.synchronize()
        d = dev.cpu().numpy()
        assert_exact(d[:197], np.concatenate(host).reshape(-1), "device output")
        assert (d[197:] == -1.0).all()
        dev2 = torch.full((N * 50,), -1.0, dtype=torch.float32, device="cuda:0")
        h0, nh = ctx.dense_ready(None, 50, 0, 1, out_device_ptr=dev2.data_ptr())
        torch.cuda.synchronize()
        assert h0.tolist() == [1] * N and nh.tolist() == [50] * N
        for s in range(N):
            assert_exact(dev2.cpu().numpy()[50 * s:50 * (s + 1)].reshape(50, 1), want(s, 1, 50), f"device ready {s}")
    ctx.close()


def _err(fn, exc, *words):
    with pytest.raises(exc) as e:
        fn()
    for w in words:
        assert w in str(e.value), str(e.value)


def test_errors(word):
    """Each refusal names the stream (where there is one) and changes no state: no launch, no cursor moves."""
    from easywakeword_b200 import _lib
    N = 6
    ctx = make_ctx(N, "i16", [word], ring=32000, slack=16000, live=True)
    ctx.push_streams([0, 1, 2, 3], [np.full(n, 100, np.int16) for n in (16000, 8000, 16000, 16000)])
    for _ in range(4):                                          # past its ring: early hops are gone
        ctx.push_streams([4], [np.full(30000, 100, np.int16)])
    ctx.dense_ready([0, 1], 10, 0, 1)                           # cursors 0, 1 at 11
    launches = ctx.launch_count()

    cases = [
        (lambda: ctx.dense_scores_streams([N], [1], [5]), ValueError, ["stream 6"]),
        (lambda: ctx.dense_scores_streams([-1], [1], [5]), ValueError, ["stream -1"]),
        (lambda: ctx.dense_scores_streams([2, 0, 2], [1, 1, 1], [5, 5, 5]), ValueError, ["stream 2", "twice"]),
        (lambda: ctx.dense_scores_streams([0, 3], [1, -1], [5, 5]), ValueError, ["stream 3"]),
        (lambda: ctx.dense_scores_streams([3, 0], [1, 1], [-5, 5]), ValueError, ["stream 3"]),
        (lambda: ctx.dense_scores_streams([0, 1], [1, 40], [5, 20]), _lib.EwkError, ["stream 1", "samples"]),
        (lambda: ctx.dense_scores_streams([4], [1], [5]), _lib.EwkError, ["stream 4", "no longer holds"]),
        (lambda: ctx.dense_scores_streams([0, 2], [1, 1], [5, 5], out_cap=9), ValueError, ["need 10"]),
        (lambda: ctx.dense_scores_streams([0], [1], [5], template_first=1), ValueError, ["reference word"]),
        (lambda: ctx.dense_scores_streams([0], [1], [5], template_first=7, template_count=2), ValueError, ["template"]),
        (lambda: ctx.dense_ready([0, 1, 2], 10, out_cap=29), ValueError, ["need 30"]),
        (lambda: ctx.dense_ready([0, 2, 0], 10), ValueError, ["stream 0", "twice"]),
        (lambda: ctx.dense_ready([0, 7], 10), ValueError, ["stream 7"]),
        (lambda: ctx.dense_ready([0, 4], 10), _lib.EwkError, ["stream 4", "no longer holds"]),
        (lambda: ctx.dense_ready(None, 10), _lib.EwkError, ["stream 4"]),
        (lambda: ctx.dense_ready([0], 10, template_first=1), ValueError, ["reference word"]),
        (lambda: ctx.dense_ready([0], 0), ValueError, ["max_hops"]),
        (lambda: ctx.dense_ready([0], (1 << 20) + 1), ValueError, ["max_hops"]),
    ]
    for fn, exc, words in cases:
        _err(fn, exc, *words)
        assert ctx.launch_count() == launches
    # no cursor moved: 0, 1 continue at 11, 2 and 3 at 1; stream 4 is refused until it is reset
    h0, out = ctx.dense_ready([0, 1, 2, 3], 1000, 0, 1)
    assert h0.tolist() == [11, 11, 1, 1] and [len(o) for o in out] == [90, 40, 100, 100]
    ctx.reset_streams([4])
    h0, out = ctx.dense_ready([4], 10, 0, 1)
    assert h0.tolist() == [1] and len(out[0]) == 0
    ctx.close()
