"""CPU: the host side of ragged dense scoring — exported symbols, the due rule of ewk_dense_ready against brute force,
the packing and unpacking in Context.dense_scores_streams / dense_ready, and ShardedBank.dense_ready routing."""
import ctypes as C
import os
import re

import numpy as np

from easywakeword_b200.resample import due_hops

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_symbols_exported():
    from easywakeword_b200 import _lib
    hdr = open(os.path.join(REPO, "include", "ewk.h")).read()
    lib = _lib.load()
    for name in ("ewk_dense_scores_streams", "ewk_dense_ready"):
        assert re.search(r"\b" + name + r"\s*\(", hdr), name
        assert hasattr(lib, name) and name in lib._protos, name


def test_due_hops_brute_force():
    """hop h is due once 160 h samples have landed: count them one by one from the cursor"""
    rng = np.random.default_rng(1)
    written = rng.integers(0, 60000, 400)
    nxt = rng.integers(1, 400, 400)
    for cap in (None, 1, 7, 64, 1 << 20):
        got = due_hops(written, nxt, cap)
        for w, h, g in zip(written, nxt, got):
            k, n = int(h), 0
            while 160 * k <= w and (cap is None or n < cap):
                k, n = k + 1, n + 1
            assert g == n


class _FakeLib:
    """Writes score i of row r as 1000 r + i, and for dense_ready gives row r (r + 2) % 3 hops from hop 10 r + 1."""

    def __init__(self):
        self.calls = []

    def ewk_dense_scores_streams(self, h, st, n, h0, nh, tf, T, out, cap, where):
        self.calls.append(dict(streams=[st[i] for i in range(n)], hop0=[h0[i] for i in range(n)],
                               n_hops=[nh[i] for i in range(n)], tf=tf, T=T, cap=cap, where=where, out=out))
        if where == 0 and out:
            buf = (C.c_float * cap).from_address(out)
            o = 0
            for r in range(n):
                for i in range(nh[r] * T):
                    buf[o] = 1000 * r + i
                    o += 1
        return 0

    def ewk_dense_ready(self, h, st, n, max_hops, tf, T, h0, nh, out, cap, where):
        self.calls.append(dict(streams=None if not st else [st[i] for i in range(n)], n=n, max_hops=max_hops, tf=tf, T=T,
                               cap=cap, where=where))
        buf = (C.c_float * cap).from_address(out) if out and where == 0 else None
        o = 0
        for r in range(n):
            h0[r], nh[r] = 10 * r + 1, min((r + 2) % 3, max_hops)
            for i in range(nh[r] * T):
                if buf is not None:
                    buf[o] = 1000 * r + i
                o += 1
        return 0


def _ctx(n_streams=5):
    from easywakeword_b200 import _lib
    ctx = object.__new__(_lib.Context)
    ctx.lib, ctx.h = _FakeLib(), None
    ctx.cfg = _lib.Config(n_streams, 16000, 1600, _lib.PCM_I16, 4, 16, 0.0, 20, 0, 0)
    return ctx


def test_dense_scores_streams_packing():
    """rows of any length, 0 included, come back as [n_i, T] arrays cut from one packed buffer in list order"""
    from easywakeword_b200 import _lib
    ctx = _ctx()
    rows = ctx.dense_scores_streams([4, 0, 2], [7, 1, 30], [3, 0, 2], 1, 2)
    c = ctx.lib.calls[-1]
    assert c["streams"] == [4, 0, 2] and c["hop0"] == [7, 1, 30] and c["n_hops"] == [3, 0, 2]
    assert c["tf"] == 1 and c["T"] == 2 and c["cap"] == 10 and c["where"] == _lib.HOST
    assert [r.shape for r in rows] == [(3, 2), (0, 2), (2, 2)]
    assert np.array_equal(rows[0].reshape(-1), np.arange(6)) and np.array_equal(rows[2].reshape(-1), 2000 + np.arange(4))
    assert [r.shape for r in ctx.dense_scores_streams([1], [0], [0])] == [(0, 1)]
    assert ctx.dense_scores_streams([3], [2], [4], out_device_ptr=1234) is None
    c = ctx.lib.calls[-1]
    assert c["where"] == _lib.DEVICE and c["out"].value == 1234 and c["cap"] == 4
    ctx.dense_scores_streams([3], [2], [4], out_device_ptr=1234, out_cap=99)
    assert ctx.lib.calls[-1]["cap"] == 99
    for bad in (lambda: ctx.dense_scores_streams([0, 1], [1], [1, 1]), lambda: ctx.dense_scores_streams([0], [1], [2**31])):
        try:
            bad()
            raise AssertionError("accepted")
        except ValueError:
            pass


def test_dense_ready_packing():
    """dense_ready sizes out as n * max_hops * T, and unpacks the rows the library reports"""
    from easywakeword_b200 import _lib
    ctx = _ctx(5)
    h0, rows = ctx.dense_ready(None, 4, 0, 3)
    c = ctx.lib.calls[-1]
    assert c["streams"] is None and c["n"] == 5 and c["cap"] == 5 * 4 * 3 and c["max_hops"] == 4
    assert h0.tolist() == [1, 11, 21, 31, 41] and [len(r) for r in rows] == [2, 0, 1, 2, 0]
    for r, a in enumerate(rows):
        assert a.shape == (len(a), 3) and np.array_equal(a.reshape(-1), 1000 * r + np.arange(a.size))
    h0, rows = ctx.dense_ready([3, 1], 1, 0, 1)
    assert ctx.lib.calls[-1]["streams"] == [3, 1] and [len(r) for r in rows] == [1, 0]
    h0, nh = ctx.dense_ready([2], 8, 0, 2, out_device_ptr=99)
    assert ctx.lib.calls[-1]["where"] == _lib.DEVICE and nh.tolist() == [2]


def test_sharded_dense_ready_routing():
    """every rank takes the whole list, scores its own streams with local ids and reports them by global id"""
    from easywakeword_b200.dist import ShardedBank, shard_range

    class _Bank:
        def dense_ready(self, streams, tf, tc):
            self.got = list(streams)
            return np.array([100 + s for s in streams]), [np.full((s, 1), s, np.float32) for s in streams]

    n_total, world = 10, 3
    g = [9, 0, 4, 3, 7, 1]
    seen = {}
    for rank in range(world):
        sb = object.__new__(ShardedBank)
        sb.n_total, sb.world, sb.rank, sb.bank = n_total, world, rank, _Bank()
        sb.first, sb.last = shard_range(n_total, world, rank)
        out = sb.dense_ready(g)
        for gid, (h0, r) in out.items():
            loc = gid - sb.first
            assert 0 <= loc < sb.last - sb.first and h0 == 100 + loc and r.shape == (loc, 1)
            seen[gid] = rank
    assert sorted(seen) == sorted(g)
