"""CPU: the host side of the dense detector (ewk_dense_detect) — the export and record layout, the host model
(oracle/dense_detect.py) on hand-made score arrays, its split invariance, the ceil(n / 2) bound, the Python packing in
Context.dense_detect / WakeWordBank.dense_detect against a fake library, and ShardedBank.dense_detect routing."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import dense_detect as M

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAN = float("nan")
LENS = [16000, 8000, 12345, 640]


def test_export_and_sizes():
    from easywakeword_b200 import _lib
    hdr = open(os.path.join(REPO, "include", "ewk.h")).read()
    lib = _lib.load()
    assert re.search(r"\bewk_dense_detect\s*\(", hdr) and hasattr(lib, "ewk_dense_detect")
    assert "ewk_dense_detect" in lib._protos
    assert re.search(r"typedef struct ewk_detection \{[^}]*\} ewk_detection;", hdr, re.S)
    dt = _lib.DETECTION_DTYPE
    assert dt.itemsize == 48 and dt == M.DETECTION_DTYPE
    assert [dt.fields[f][1] for f in dt.names] == [0, 4, 8, 16, 24, 32, 40, 44]


def run(rows, thr=50.0, hold=3, refractory=5, hop0=1, slot0=0, lens=LENS, state=None):
    return M.detect(np.array(rows, np.float32).reshape(len(rows), -1), hop0, state, thr, hold, refractory, slot0,
                    lens[:np.array(rows).reshape(len(rows), -1).shape[1]])


def fields(ev, *names):
    return [tuple(int(e[n]) if n != "score" else float(e[n]) for n in names) for e in ev]


def test_nan_and_threshold_equal():
    """a NaN hop is never above and ends a run; NaN beside a number is ignored; a score equal to thr is detected"""
    ev, st = run([[NAN, NAN], [50.0, NAN], [NAN, 49.0], [NAN, NAN], [10.0, 60.0]], hold=10, refractory=2)
    assert fields(ev, "hop", "run_start", "emit_hop", "template_slot", "score") == [(2, 2, 3, 0, 50.0)]
    assert st["mode"] == M.ARMED and st["peak"] == 5 and st["slot"] == 1
    ev, _ = run([[49.999996], [NAN]])
    assert len(ev) == 0


def test_ties_lowest_slot_and_first_maximum():
    """equal scores across templates: the lowest k wins; equal peaks within a run: the first one stays"""
    ev, _ = run([[70.0, 70.0, 70.0], [0.0, 0.0, 0.0]], slot0=2)
    assert fields(ev, "template_slot", "seg_len", "seg_start") == [(2, 16000, 160 * (1 - 100))]
    ev, _ = run([[60.0, 61.0], [61.0, 55.0], [61.0, 61.0], [0.0, 0.0]], hold=50)
    assert fields(ev, "hop", "template_slot", "score", "emit_hop", "seg_len") == [(1, 1, 61.0, 4, 8000)]
    ev, _ = run([[60.0], [60.5], [60.5], [61.0], [1.0]], hold=50)
    assert fields(ev, "hop", "score") == [(4, 61.0)]


def test_hold_and_refractory_edges():
    """a run longer than hold emits at peak + hold and goes SPENT; quiet_until = end + refractory holds exactly"""
    ev, st = run([[80.0]] * 10, hold=3)
    assert fields(ev, "hop", "run_start", "emit_hop") == [(1, 1, 4)] and st["mode"] == M.SPENT
    ev, st = run([[80.0], [81.0], [82.0], [82.0], [82.0], [82.0], [0.0]], hold=3)
    assert fields(ev, "hop", "emit_hop") == [(3, 6)]
    assert st["mode"] == M.IDLE and st["quiet_until"] == 7 + 5
    ev, _ = run([[80.0], [81.0], [81.0], [0.0]], hold=1)               # hold 1: a new peak is emitted one hop later
    assert fields(ev, "hop", "emit_hop") == [(2, 3)]
    # refractory 5 after the run ends at hop 3: hops 4..7 above are ignored, hop 8 arms
    rows = [[80.0], [80.0], [0.0], [70.0], [70.0], [70.0], [70.0], [70.0], [0.0]]
    ev, _ = run(rows, hold=50, refractory=5)
    assert fields(ev, "hop", "run_start", "emit_hop") == [(1, 1, 3), (8, 8, 9)]
    ev, _ = run(rows, hold=50, refractory=0)
    assert fields(ev, "hop", "run_start", "emit_hop") == [(1, 1, 3), (4, 4, 9)]
    ev, _ = run(rows, hold=50, refractory=6)
    assert fields(ev, "emit_hop") == [(3,)]
    # SPENT -> IDLE sets quiet_until too
    ev, st = run([[80.0]] * 5 + [[0.0]] + [[80.0], [0.0]] * 3, hold=2, refractory=4)
    assert fields(ev, "emit_hop") == [(3,), (12,)]           # not (3,), (8,)
    with pytest.raises(ValueError):
        run([[1.0]], hold=0)


def test_split_invariance():
    """random cuts of the hop sequence with the state carried across give the same events"""
    rng = np.random.default_rng(3)
    for trial in range(40):
        n, T = int(rng.integers(1, 400)), int(rng.integers(1, 5))
        x = np.round(rng.normal(60, 12, (n, T)), 1).astype(np.float32)
        x[rng.random((n, T)) < 0.05] = np.nan
        kw = dict(thr=float(rng.choice([55.0, 60.0, x[0, 0] if x[0, 0] == x[0, 0] else 60.0])),
                  hold=int(rng.choice([1, 3, 50])), refractory=int(rng.choice([0, 7, 200])))
        whole, st_w = M.detect(x, 1, None, slot0=0, tmpl_lens=LENS[:T], **kw)
        cuts = np.sort(rng.choice(np.arange(1, n), min(n - 1, int(rng.integers(0, 12))), replace=False)) if n > 1 else []
        st, parts, a = None, [], 0
        for b in list(cuts) + [n]:
            ev, st = M.detect(x[a:b], 1 + a, st, slot0=0, tmpl_lens=LENS[:T], **kw)
            parts.append(ev)
            a = b
        assert np.array_equal(np.concatenate(parts), whole) and st == st_w


def test_bound_reached():
    """a run ARMED from the previous call and alternating above / below reaches ceil(n / 2) emissions exactly"""
    _, st = run([[90.0]], hold=1, refractory=0)
    assert st["mode"] == M.ARMED
    for n in (1, 2, 7, 64, 101):
        rows = [[0.0] if i % 2 == 0 else [90.0] for i in range(n)]
        ev, _ = run(rows, hop0=2, hold=1, refractory=0, state=st)
        assert len(ev) == (n + 1) // 2
        assert np.all(np.diff(ev["emit_hop"]) >= 2)


class _FakeLib:
    """Row r gets (r + 2) % 3 hops from hop 10 r + 1 and one detection per hop it takes (stream = list entry)."""

    def __init__(self):
        self.calls = []

    def ewk_dense_detect(self, h, st, n, max_hops, tf, T, hold, refr, det, det_cap, h0, nh, out, cap, where):
        self.calls.append(dict(streams=None if not st else [st[i] for i in range(n)], n=n, max_hops=max_hops, tf=tf, T=T,
                               hold=hold, refr=refr, det_cap=det_cap, cap=cap, where=where, out=out))
        recs = np.ctypeslib.as_array((C.c_char * (48 * det_cap)).from_address(det)).view(M.DETECTION_DTYPE) \
            if det else None
        buf = (C.c_float * cap).from_address(out) if out and where == 0 else None
        o = k = 0
        for r in range(n):
            h0[r], nh[r] = 10 * r + 1, min((r + 2) % 3, max_hops)
            for i in range(nh[r]):
                recs[k] = (st[r] if st else r, tf, h0[r] + i, h0[r], h0[r] + i + 1, 160 * i, 640, 75.0)
                k += 1
            for i in range(nh[r] * T):
                if buf is not None:
                    buf[o] = 1000 * r + i
                o += 1
        return k


def _ctx(n_streams=5):
    from easywakeword_b200 import _lib
    ctx = object.__new__(_lib.Context)
    ctx.lib, ctx.h = _FakeLib(), None
    ctx.cfg = _lib.Config(n_streams, 16000, 1600, _lib.PCM_I16, 4, 16, 0.0, 20, 0, 0)
    return ctx


def test_context_packing():
    from easywakeword_b200 import _lib
    ctx = _ctx(5)
    d = ctx.dense_detect(None, 4, 0, 2, hold_hops=3, refractory_hops=9)
    c = ctx.lib.calls[-1]
    assert c["streams"] is None and c["n"] == 5 and c["det_cap"] == 5 * 2 and c["out"] is None and c["cap"] == 0
    assert c["hold"] == 3 and c["refr"] == 9 and c["where"] == _lib.HOST
    assert d.dtype == _lib.DETECTION_DTYPE and d["stream"].tolist() == [0, 0, 2, 3, 3]
    d, (h0, rows) = ctx.dense_detect([3, 1], 7, 1, 3, scores=True)
    c = ctx.lib.calls[-1]
    assert c["streams"] == [3, 1] and c["det_cap"] == 2 * 4 and c["cap"] == 2 * 7 * 3 and c["out"]
    assert h0.tolist() == [1, 11] and [r.shape for r in rows] == [(2, 3), (0, 3)]
    assert np.array_equal(rows[0].reshape(-1), np.arange(6)) and d["template_slot"].tolist() == [1, 1]
    d, (h0, nh) = ctx.dense_detect([2], 8, 0, 1, out_device_ptr=77)
    c = ctx.lib.calls[-1]
    assert c["where"] == _lib.DEVICE and c["out"].value == 77 and c["cap"] == 8 and nh.tolist() == [2]
    ctx.dense_detect([2], 8, det_cap=2)
    assert ctx.lib.calls[-1]["det_cap"] == 2


def test_bank_rounds_and_order():
    """WakeWordBank.dense_detect loops until a round leaves no due hop and sorts by (emit_hop, stream)"""
    from easywakeword_b200 import _lib, bank
    calls = []

    class _Ctx:
        def dense_detect(self, streams, max_hops, tf, T, hold, refr, hops=False):
            calls.append((streams, max_hops, tf, T, hold, refr))
            k = len(calls)
            d = np.zeros(3, _lib.DETECTION_DTYPE)
            d["stream"], d["emit_hop"] = [4, 1, 0], [5 * k, 2 * k, 5 * k]
            return d, (np.ones(3, np.int64), np.array([0, bank.DENSE_ROUND if k < 3 else 7, 1], np.int32))

    b = object.__new__(bank.WakeWordBank)
    b.ctx, b.templates = _Ctx(), [None, None, None]
    d = b.dense_detect([4, 1, 0], template_first=1, hold_hops=5, refractory_hops=6)
    assert calls == [([4, 1, 0], bank.DENSE_ROUND, 1, 2, 5, 6)] * 3
    assert list(zip(d["emit_hop"].tolist(), d["stream"].tolist())) == sorted(zip(d["emit_hop"].tolist(),
                                                                                   d["stream"].tolist()))
    assert len(d) == 9


def test_sharded_routing():
    """every rank takes the whole list, detects on its own streams with local ids and reports global ids"""
    from easywakeword_b200 import _lib
    from easywakeword_b200.dist import ShardedBank, shard_range

    class _Bank:
        def dense_detect(self, streams, tf, tc, hold, refr):
            self.got = list(streams)
            d = np.zeros(len(streams), _lib.DETECTION_DTYPE)
            d["stream"], d["hop"] = streams, streams
            return d

    n_total, world = 10, 3
    g = [9, 0, 4, 3, 7, 1]
    seen = []
    for rank in range(world):
        sb = object.__new__(ShardedBank)
        sb.n_total, sb.world, sb.rank, sb.bank = n_total, world, rank, _Bank()
        sb.first, sb.last = shard_range(n_total, world, rank)
        d = sb.dense_detect(g)
        assert d.dtype == _lib.DETECTION_DTYPE
        assert np.array_equal(d["stream"], d["hop"] + sb.first)
        assert all(sb.first <= s < sb.last for s in d["stream"])
        seen += d["stream"].tolist()
    assert sorted(seen) == sorted(g)
