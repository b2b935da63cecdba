"""CPU: the host side of per-row template sets (ewk_dense_scores_sets, ewk_dense_ready_sets, ewk_dense_detect_sets) —
exported symbols, the packing offsets, the launch grouping by geometry over every reachable geometry, and the argument
errors of the Python layer (a cached set's invalidation and the library's error table need a device:
test_gpu_dense_sets.py)."""
import os
import re
import types

import numpy as np
import pytest

from helpers import dense_geometry_sets

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_symbols_exported():
    from easywakeword_b200 import _lib
    hdr = open(os.path.join(REPO, "include", "ewk.h")).read()
    lib = _lib.load()
    for name in ("ewk_dense_scores_sets", "ewk_dense_ready_sets", "ewk_dense_detect_sets"):
        assert re.search(r"\b" + name + r"\s*\(", hdr), name
        assert hasattr(lib, name) and name in lib._protos, name


def test_packing_offsets_brute_force():
    """row i starts at sum_{j < i} n_hops[j] T_j; rows of 0 hops take no room"""
    from easywakeword_b200 import _lib
    rng = np.random.default_rng(3)
    for _ in range(200):
        n = int(rng.integers(0, 40))
        nh = rng.integers(0, 300, n) * (rng.random(n) > 0.2)
        T = rng.integers(1, 9, n)
        off, total = _lib.sets_offsets(nh, T)
        o = 0
        for i in range(n):
            assert off[i] == o
            o += int(nh[i]) * int(T[i])
        assert total == o
        buf = np.arange(total, dtype=np.float32)
        rows = _lib._unpack_rows_sets(buf, nh, T)
        assert [r.shape for r in rows] == [(int(a), int(b)) for a, b in zip(nh, T)]
        assert all(r.size == 0 or r[0, 0] == off[i] for i, r in enumerate(rows))


def test_geometry_grouping():
    """one launch per distinct geometry among the rows' sets, whatever the number of sets; each row in the group of
    the geometry its set has alone"""
    from easywakeword_b200 import _lib
    geo = dense_geometry_sets(_lib.dense_plan)
    assert len(geo) >= 2
    keys, sets = list(geo), list(geo.values())
    g = _lib.sets_launches(sets)
    assert list(g) == keys and all(g[k] == [i] for i, k in enumerate(keys))
    rng = np.random.default_rng(5)
    for _ in range(30):
        pick = rng.integers(0, len(sets), int(rng.integers(1, 60)))
        rows = [sets[i] for i in pick]
        g = _lib.sets_launches(rows)
        assert len(g) == len(set(pick.tolist())) <= 8
        for k, idx in g.items():
            assert all(_lib.dense_plan(rows[i])[:3] == k for i in idx)
        assert sorted(i for idx in g.values() for i in idx) == list(range(len(rows)))
    # many distinct one-template sets of one geometry: one launch
    ones = [[int(L)] for L in rng.integers(640, 2000, 64)]
    assert len(_lib.sets_launches(ones)) == len({_lib.dense_plan(s)[:3] for s in ones})


def test_python_argument_errors():
    from easywakeword_b200 import _lib
    ctx = _lib.Context.__new__(_lib.Context)
    ctx.cfg = types.SimpleNamespace(n_streams=4)
    with pytest.raises(ValueError, match="both"):
        ctx._row_sets(None, 4, [0, 0, 0, 0], None)
    with pytest.raises(ValueError, match="both"):
        ctx._row_sets(None, 4, None, [1, 1, 1, 1])
    with pytest.raises(ValueError, match="stream 0"):
        ctx._row_sets(None, 4, None, None)                 # ranges never set through this Context
    ctx._template_ranges()[:] = [[0, 1], [1, 2], [3, 1], [0, 4]]
    tf, tc, T = ctx._row_sets(np.array([3, 1], np.int32), 2, None, None)
    assert tf is None and tc is None and T.tolist() == [4, 2]
    ctx._template_ranges()[1] = -1                         # an imported stream
    with pytest.raises(ValueError, match="stream 1"):
        ctx._row_sets(np.array([3, 1], np.int32), 2, None, None)
    tf, tc, T = ctx._row_sets(None, 4, 2, [1, 2, 3, 4])
    assert tf.tolist() == [2] * 4 and tc.tolist() == [1, 2, 3, 4] and T.tolist() == [1, 2, 3, 4]
