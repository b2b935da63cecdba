"""CPU: the exact model of K4's dense scores (oracle/dense_model.py) and K4's launch planner (ewk_dense_plan).

The model restates K4's integer window statistics and float score arithmetic; tests/test_gpu_dense_exact.py compares
the device with it bit for bit over K3's frames.  Here, over the float64 oracle's frames, it must agree with the
reference's own pooling (oracle.dense_scores) to the quantisation error, its exact double FMA must be the compiled
one, and faults that plausible K4 bugs would cause must move the score bits while mostly staying inside the 0.01
tolerance of the older dense tests (the count is printed: that is what those tests cannot see)."""
from fractions import Fraction

import numpy as np
import pytest
import scipy.fft

from easywakeword_b200 import synth
from helpers import dense_geometry_sets
from oracle import dense_model as D
from oracle import ewk_oracle as O
from oracle import librosa_restated as L

SCORE_ATOL = 0.01          # tests/test_gpu_dense.py's tolerance


@pytest.fixture(scope="module")
def plan():
    from easywakeword_b200 import _lib, build
    build.build()
    return _lib.dense_plan


def gap_stream(word, seed=3100, seconds=5.0):
    x, _ = synth.stream(seed, seconds, word, gain=(2.0, 4.0), zero_gaps=5, noise_sigma=0.0005)
    return synth.from_int16(synth.to_int16(x))


def test_model_on_oracle_frames_matches_oracle(word):
    """Model over the oracle's frames vs oracle.dense_scores (float32 pooling of the same frames), at hops whose windows
    are un-floored, way and edge-floored; DESIGN §4 puts the quantisation error at ~2.3e-5."""
    x = gap_stream(word)
    tpls = [word, synth.synthetic_word(seed=9, duration=0.5), word[:16000 - 160 * 10]]
    m = D.DenseModel(x, tpls, D.oracle_frames())
    hops = np.arange(0, len(x) // 160 + 1, 2)
    got = m.scores(hops)
    ref = O.dense_scores(x, tpls, hops)
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    d = np.abs(got[ok].astype(np.float64) - ref[ok])
    counts = np.zeros(3, int)
    for k in range(len(tpls)):
        c, _ = m.classes(hops, k)
        counts += np.bincount(c[c >= 0], minlength=3)
    i = int(np.argmax(d))
    print(f"model (oracle frames) vs oracle.dense_scores: worst {d.max():.2e} (model {got[ok][i]:.6f}, oracle "
          f"{ref[ok][i]:.6f}) over {ok.sum()} windows; classes " +
          ", ".join(f"{n} {c}" for n, c in zip(D.CLASS_NAMES, counts)))
    assert d.max() <= 1e-4
    assert (counts > 0).all(), counts


def test_fma64_is_exact_and_the_model_uses_the_contracted_form():
    rng = np.random.default_rng(11)
    for _ in range(3000):
        a, b, c = (float(v) for v in rng.standard_normal(3) * 10.0 ** rng.integers(-30, 30, 3))
        assert D.fma64(a, b, c) == float(Fraction(a) * Fraction(b) + Fraction(c))
    # statistics of real size: q ~ 2^27 over up to 301 frames, a coefficient that barely moves across the window (the
    # variance cancels).  Find sums where the DFMA K4 compiles to and the uncontracted s2 - fl(fl(s1 s1) invf) give
    # different std bits, and check which one dense_stats returns
    found = 0
    for _ in range(3000):
        F = int(rng.integers(5, 302))
        q = int(rng.integers(-2 ** 27, 2 ** 27)) + rng.integers(-2 ** 12, 2 ** 12, F) // int(rng.choice([1, 64, 4096]))
        S1, S2 = int(q.sum()), int((q * q).sum())
        invf = 1.0 / F
        s1, s2 = float(S1), float(S2)
        fused = D.fma64(-(s1 * s1), invf, s2)
        plain = s2 - (s1 * s1) * invf
        if fused == plain:
            continue
        _, sd = D.dense_stats(np.array([S1]), np.array([S2]), F)
        want_f = np.sqrt(np.maximum(np.float32((fused * invf) * 2.0 ** -32), np.float32(0)))
        want_p = np.sqrt(np.maximum(np.float32((plain * invf) * 2.0 ** -32), np.float32(0)))
        assert sd[0] == want_f
        found += want_f != want_p
    print(f"{found} random sums whose std bits differ between the contracted and the uncontracted variance")
    assert found > 0


def test_model_statistics_vs_float64(word):
    """mean / std from the integer sums vs float64 mean / std (ddof 0) of the same rows: within the quantisation
    error (2^-17 per value) and float32 rounding."""
    x = gap_stream(word, seconds=3.0)
    fn = D.oracle_frames()
    worst = 0.0
    for s in range(0, len(x) - len(word), 160 * 37):
        rows = fn(x[s:s + len(word)])
        m, sd = D.window_features(rows)
        r64 = rows.astype(np.float64)
        dm = np.abs(m - r64.mean(axis=0))
        ds = np.abs(sd - r64.std(axis=0))
        worst = max(worst, float(dm.max()), float(ds.max()))
        assert (dm <= 2.0 ** -17 + 1.2e-7 * np.abs(r64.mean(axis=0))).all()
        assert (ds <= 2e-5 + 1.2e-7 * r64.std(axis=0)).all()
    print(f"integer statistics vs float64 mean / std of the same rows: worst {worst:.2e}")


def test_plan_geometries(plan, word):
    reach = dense_geometry_sets(plan)
    print("reachable K4 geometries (DH, threads, CTAs/SM): " +
          "; ".join(f"{g} <- {lens}" for g, lens in sorted(reach.items())))
    assert set(reach) == {(dh, th, 2) for dh in (64, 32) for th in (512, 448)} | \
        {(dh, th, 1) for dh in (64, 32) for th in (1024, 512)}
    # fixed points: one ~1 s word; the 4-template sweep with the 2.1 s phrase (bench.py sweep_templates)
    assert plan([len(word)])[:3] == (64, 512, 2)
    assert plan([len(word), 2 * len(word) + 2400, 16000, 9600])[:3] == (32, 1024, 1)
    for bad in ([639], [48001], [640] * 9, []):
        with pytest.raises(ValueError):
            plan(bad)


# ------------------------------------------------------------------------------------------------ blindness
def logmel_unfloored(pcm):
    return L.power_to_db(L.melspectrogram(np.asarray(pcm, np.float32)), top_db=None)        # [128, F]


def rows_from_logmel(lm, floor):
    v = np.maximum(lm, floor) if floor is not None else lm
    return scipy.fft.dct(v, axis=0, type=2, norm="ortho")[:20].T.astype(np.float32)


def test_blindness_of_the_tolerance_tests(word):
    """Four plausible K4 faults applied to the model's inputs.  Every faulted score changes its bits (the exact device
    test sees each one); the printed count is how many stay within 0.01 of the oracle, i.e. would pass the older
    tolerance tests."""
    x = gap_stream(word, seed=3101, seconds=6.0)
    tpl = np.concatenate([word, np.zeros(16000 - len(word), np.float32)])      # L % 160 == 0: two right-edge frames
    n, F, t_hi, r = D.window_geometry(len(tpl))
    assert r == 2
    tm, ts = D.template_features(D.oracle_frames()(tpl))

    def score(rows):
        m, s = D.window_features(rows)
        return D.score_features(tm, ts, m[None], s[None])[0]

    def score_sums(rows, keep):
        S1, S2 = D.sums(rows[keep])
        m, s = D.dense_stats(S1, S2, F)                                # a dropped frame keeps 1 / F
        return D.score_features(tm, ts, m[None], s[None])[0]

    hops = np.arange(n, len(x) // 160 + 1)
    ref = O.dense_scores(x, [tpl], hops)[:, 0]
    edge = np.zeros(F, bool)
    edge[:2] = True
    edge[t_hi + 1:] = True
    stats = {k: [0, 0] for k in ("floored grid row read un-floored", "second right-edge frame dropped",
                                 "left-edge row of start j+1", "floor without the edge frames")}

    def record(name, good, bad, i):
        assert not np.array_equal(np.float32(bad), np.float32(good), equal_nan=True), (name, int(hops[i]))
        stats[name][0] += 1
        stats[name][1] += bool(abs(float(bad) - float(ref[i])) <= SCORE_ATOL)

    for i, h in enumerate(hops[::3]):
        i *= 3
        s = 160 * (int(h) - n)
        lm = logmel_unfloored(x[s:s + len(tpl)])
        floor = lm.max() - 80.0
        rows = rows_from_logmel(lm, floor)
        good = score(rows)
        below = lm.min(axis=0) < floor
        if below.any() and not (below & edge).any():                   # a way window
            t = int(np.flatnonzero(below)[0])
            bad_rows = rows.copy()
            bad_rows[t] = rows_from_logmel(lm, None)[t]
            record("floored grid row read un-floored", good, score(bad_rows), i)
        keep = np.ones(F, bool)
        keep[F - 1] = False
        record("second right-edge frame dropped", good, score_sums(rows, keep), i)
        s2 = s + 160
        if s2 + len(tpl) <= len(x):
            lm2 = logmel_unfloored(x[s2:s2 + len(tpl)])
            # the kernel's frames carry their own floor test; a start-(j+1) row under this window's floor
            le = rows_from_logmel(lm2, floor if (lm2[:, 0] < floor).any() else None)[0]
            if not np.array_equal(le, rows[0]):
                bad_rows = rows.copy()
                bad_rows[0] = le
                record("left-edge row of start j+1", good, score(bad_rows), i)
        floor_g = lm[:, ~edge].max() - 80.0
        if floor_g != floor and (lm.min(axis=0) < max(floor, floor_g)).any():
            record("floor without the edge frames", good, score(rows_from_logmel(lm, floor_g)), i)
    print("faults the 0.01 tests cannot see (faulted windows within 0.01 of the oracle / windows the fault changes):")
    for k, (nw, within) in stats.items():
        print(f"  {k}: {within} / {nw}")
    assert all(nw > 0 for nw, _ in stats.values()), stats
