"""CPU: the float32 frame-alignment model (oracle/align_model.py) that K11 is checked against bit for bit.

It equals a cell-by-cell float32 statement of the same operations, agrees with a float64 DTW, and on the bundled word
separates order impostors (the right sounds in another order, which level 2 scores ~100) from ordinary perturbations."""
import os

import numpy as np
import pytest

from oracle import align_model as A
from oracle import ewk_oracle as O

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def _rand(rng, n):
    x = rng.standard_normal((n, 20)).astype(F32) * F32(rng.uniform(0.1, 30))
    return x, x.mean(0, dtype=F32)


@pytest.mark.parametrize("C", [20, 13, 1])
def test_vectorised_equals_cell_loop(C):
    rng = np.random.default_rng(C)
    shapes = [(1, 1), (1, 9), (7, 1), (2, 2), (13, 29), (31, 17)]
    for n, m in shapes:
        a, ma = _rand(rng, n)
        b, mb = _rand(rng, m)
        if n == 13:
            a[:] = a[0]                                      # all-constant segment: u = 0, r = 0, cost 1 everywhere
            ma = a[0].copy()
        x = A.distance(a, ma, b, mb, C)
        y = A.distance_loop(a, ma, b, mb, C)
        assert x.dtype == np.float32 and x.tobytes() == y.tobytes(), (n, m, x, y)
        if n == 13:                                          # the cheapest path takes max(n, m) cells
            assert abs(float(x) - max(n, m) / (n + m)) < 1e-6, x


def test_agrees_with_float64():
    rng = np.random.default_rng(5)
    for n, m in [(1, 1), (40, 33), (101, 150), (301, 301)]:
        a, ma = _rand(rng, n)
        b, mb = _rand(rng, m)
        x = float(A.distance(a, ma, b, mb))
        z = A.distance_f64(a, ma, b, mb)
        assert abs(x - z) <= 1e-5, (n, m, x, z)


def _word():
    g = np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))
    return g["pcm_i16"].astype(F32) / F32(32768)


def _speed(x, f):
    t = np.arange(int(round(len(x) / f))) * f
    return np.interp(t, np.arange(len(x)), x).astype(F32)


def _cases(w):
    rng = np.random.default_rng(7)
    q = len(w) // 4
    quiet = lambda: rng.standard_normal(3200).astype(F32) * F32(1e-4)       # 0.2 s of near-silence
    perturb = {"gain 0.5": w * F32(0.5),
               "noise 0.003": w + rng.standard_normal(len(w)).astype(F32) * F32(0.003),
               "5 % faster": _speed(w, 1.05), "8 % slower": _speed(w, 1 / 1.08),
               "padded": np.concatenate([quiet(), w, quiet()])}
    order = {"reversed": w[::-1].copy(), "halves swapped": np.concatenate([w[len(w) // 2:], w[:len(w) // 2]]),
             "quarters shuffled": np.concatenate([w[2 * q:3 * q], w[:q], w[3 * q:], w[q:2 * q]])}
    return perturb, order


# the separation the model gives on the bundled word: lowest order impostor minus highest perturbation (0.110)
MARGIN = 0.10


def test_order_impostors_separated_on_bundled_word():
    w = _word()
    m = O.WordMatcherOracle()
    m.set_reference(w)
    f = O.mfcc_frames(w).T.astype(F32)
    mu = f.mean(0, dtype=F32)

    def dist(x):
        g = O.mfcc_frames(np.asarray(x, F32)).T.astype(F32)
        return float(A.distance(g, g.mean(0, dtype=F32), f, mu))

    assert dist(w) < 1e-6
    perturb, order = _cases(w)
    dp = {k: dist(x) for k, x in perturb.items()}
    do = {k: dist(x) for k, x in order.items()}
    for k, x in order.items():
        assert float(m.calculate_similarity(x)) >= 99.99, k          # level 2 cannot tell them from the word
    assert max(dp.values()) < 0.13 and min(do.values()) > 0.23, (dp, do)
    assert min(do.values()) - max(dp.values()) >= MARGIN, (dp, do)
