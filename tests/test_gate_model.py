"""oracle/gate_model.py, the exact model of the level-1 gate (K2), against the reference restatement
(oracle.ewk_oracle.detect_stream) and the reference-generated goldens; its f32 sum order against per-lane restatements of
the kernels that sum a block; the percentile's edge classes; exact ties.  CPU only: the device is compared with the model
in test_gpu_gate_exact.py."""
import math

import numpy as np
import pytest

from helpers import detect_stream_for
from easywakeword_b200 import synth
from oracle import ewk_oracle as O
from oracle import gate_model as G


def _stream(seed, seconds, word, **kw):
    x, _ = synth.stream(seed, seconds, word, noise_sigma=kw.pop("noise", 0.01), gain=kw.pop("gain", (2.0, 5.0)), **kw)
    return synth.to_int16(x)


def _compare_to_reference(x16, R, block, fmt="i16", exact=True, **params):
    """model vs detect_stream on one stream pushed whole, ticks up to the reference's last; returns the model"""
    xf = synth.from_int16(x16) if fmt == "i16" else x16
    o = O.detect_stream(xf, None, block=block, fast=True, ring_samples=R, **params)
    m = G.GateModel(R, G.physical_ring(R, 16000), fmt, [dict(frame_size=block, **params)])
    m.push(0, x16 if fmt == "i16" else xf)
    _, tr = m.tick(o["ticks_run"])
    tt = o["trace_tick"]
    _, first = np.unique(tt, return_index=True)           # a restart samples its tick twice: the first is the tick's own
    cols = tt[first] - 1
    assert np.all(tr["state"][0, :o["full_tick"] - 1] == 255) and tr["state"][0, o["full_tick"] - 1] != 255
    assert np.array_equal(tr["silent"][0, cols].astype(bool), o["trace_silent"][first])
    assert np.array_equal(tr["state"][0, cols], o["trace_state"][first])
    for k in ("thr", "rms"):
        if exact:
            assert np.array_equal(tr[k][0, cols], o[f"trace_{k}"][first]), k
        else:
            np.testing.assert_allclose(tr[k][0, cols], o[f"trace_{k}"][first], rtol=1e-12, atol=0)
    ev = m.event_array()
    sc = ev[ev[:, 1] == G.EV_SCORED]
    assert [(e["tick"], e["seg_len"]) for e in o["events"]] == [(int(a), int(b)) for a, b in sc[:, [2, 4]]]
    # seg_start = V - n_back: the segment is the last n_back samples the tick saw
    for e, r in zip(o["events"], sc):
        V = min((e["tick"] * 1600 // block) * block, len(x16) // block * block)
        assert r[3] == V - min(e["n_back"], R)
    assert list(o["timeouts"]) == [int(t) for t in ev[ev[:, 1] == G.EV_TIMEOUT][:, 2]]
    st = m.status(0)
    assert st["tick"] == o["ticks_run"] and st["silence_threshold"] == o["trace_thr"][-1]
    return m, o


@pytest.mark.parametrize("block", [160, 333, 512, 1000, 1600, 4800])
def test_model_equals_reference_on_int16(block, word):
    x = _stream(100 + block, 24.0, word, zero_gaps=1, distractor_prob=0.3)
    m, o = _compare_to_reference(x, 48000, block, speech_duration_min=0.3, timeout=6.0)
    assert len(o["timeouts"]) >= 2


def test_model_equals_goldens(golden_detect, word):
    """the detect.npz goldens (the reference's own classes, run unmodified) on int16 rings, as test_gpu_detect checks
    the device: thresholds bit for bit, silent flags, event ticks and lengths, timeouts"""
    g, cases = golden_detect
    n_ev = 0
    for c in cases:
        if c.get("special") == "config1":
            continue
        n = c["name"]
        x16 = synth.to_int16(detect_stream_for(c, word))
        p = dict(c["params"])
        p.pop("similarity_threshold", None)
        m = G.GateModel(160000, G.physical_ring(160000, 48000), "i16", [dict(frame_size=c["block"], **p)])
        m.push(0, x16)
        ticks_run, full_tick = int(g[f"{n}_ticks_run"]), int(g[f"{n}_full_tick"])
        _, tr = m.tick(ticks_run)
        gt = g[f"{n}_trace_tick"]
        _, first = np.unique(gt, return_index=True)
        cols = gt[first] - 1
        assert cols[0] == full_tick - 1
        assert np.array_equal(tr["thr"][0, cols], g[f"{n}_trace_thr"][first]), n
        assert np.array_equal(tr["silent"][0, cols].astype(bool), g[f"{n}_trace_silent"][first]), n
        ev = m.event_array()
        sc = ev[ev[:, 1] == G.EV_SCORED]
        assert list(sc[:, 2]) == list(g[f"{n}_ev_tick"]) and list(sc[:, 4]) == list(g[f"{n}_ev_len"]), n
        assert list(ev[ev[:, 1] == G.EV_TIMEOUT][:, 2]) == list(g[f"{n}_timeouts"]), n
        n_ev += len(sc)
    assert n_ev >= 50


def old_alias_rms(R, ms, Vp, V, first_full):
    """The RMS K2 took before the fix for a frame-size-1600 tick from Vp to V, restated from its phase-0 plan: when the
    new samples touch exactly one chunk c, dv = 1600 and q0 = Vp % R is 1600-aligned, it used chunk c's mean square as
    the recent window's (None where it did not; the first full tick is recomputed whole and never took the shortcut)."""
    fs, n_chunks, dv, q0 = 1600, R // 1600, V - Vp, Vp % R
    if first_full or dv != 1600 or q0 % 1600:
        return None
    e = q0 + dv
    e1 = min(e, R)
    c1 = q0 // fs
    n1 = (e1 - 1) // fs - c1 + 1
    n2 = (e - R - 1) // fs + 1 if e > R else 0
    pcs = [c for c in [c1 + i for i in range(n1)] + list(range(n2)) if c < n_chunks]
    if len(pcs) != 1:
        return None
    return math.sqrt(ms[pcs[0]] * fs / 1600)


@pytest.mark.parametrize("R,bad", [(16800, (32,)), (20000, (38,)), (24800, (47,))])
def test_rings_of_partial_ticks_and_the_old_alias_rule(R, bad, word):
    """At R % 1600 != 0 the model equals the reference restatement, and the gate's old shortcut — recent window ==
    the one chunk the tick's samples touched — reads the wrong samples at the tick whose new samples start at
    floor(R / 1600) * 1600: they cover the tail, which is in no chunk, and the start of chunk 0."""
    x = _stream(R, 8.0, word, noise=0.02, zero_gaps=1)
    _compare_to_reference(x, R, 1600, timeout=30.0)
    m = G.GateModel(R, G.physical_ring(R, 800 if R == 20000 else 16000), "i16", [dict(frame_size=1600)])
    m.push(0, x)
    wrong = []
    for k in range(1, len(x) // 1600 + 1):
        full_before = m.s[0].ms is not None
        _, tr = m.tick(1)
        if not full_before and m.s[0].ms is None:
            continue
        old = old_alias_rms(R, m.s[0].ms, (k - 1) * 1600, k * 1600, not full_before)
        if old is not None and old != tr["rms"][0, 0]:
            wrong.append(k)
    assert set(bad) <= set(wrong), wrong
    # ... and only there: every 1600-aligned ring lap puts such a tick at the same phase
    period = R // math.gcd(R, 1600)
    assert all((k * 1600 - 1600) % R == (R // 1600) * 1600 for k in wrong), (wrong, period)
    for R_whole in (16000, 19200):
        m = G.GateModel(R_whole, G.physical_ring(R_whole, 16000), "i16", [dict(frame_size=1600)])
        m.push(0, x)
        for k in range(1, len(x) // 1600 + 1):
            full_before = m.s[0].ms is not None
            _, tr = m.tick(1)
            if full_before:
                old = old_alias_rms(R_whole, m.s[0].ms, (k - 1) * 1600, k * 1600, False)
                assert old is None or old == tr["rms"][0, 0], (R_whole, k)


@pytest.mark.parametrize("block", [512, 1600, 1000])
def test_model_f32_within_1e12_of_float64_reference(block, word):
    rng = np.random.default_rng(block)
    x = (synth.from_int16(_stream(7 + block, 16.0, word, zero_gaps=1)) + rng.standard_normal(16 * 16000).astype(np.float32)
         * np.float32(1e-4)).astype(np.float32)
    _compare_to_reference(x, 32000, block, fmt="f32", exact=False, timeout=30.0)


# ---- the f32 summation order
def _push_sums_kernel(x):
    """ring_push_sums_kernel<float>: q[u] = word lane + 32 u (u < PER = 13, zero past 400), u odd -> a1d"""
    sq = x.astype(np.float64) ** 2
    a0, a1 = np.zeros(32), np.zeros(32)
    for lane in range(32):
        for u in range(13):
            k = lane + 32 * u
            for c in range(4):
                v = sq[4 * k + c] if k < 400 else 0.0
                if u & 1:
                    a1[lane] = a1[lane] + v
                else:
                    a0[lane] = a0[lane] + v
    return G._xor_tree(a0 + a1)


def _smem_kernel(x):
    """warp_sumsq_smem (K2's staged ticks and ring_push_bulk_kernel): u < 13, k < 400, u odd -> a1"""
    sq = x.astype(np.float64) ** 2
    a0, a1 = np.zeros(32), np.zeros(32)
    for lane in range(32):
        for u in range(13):
            k = lane + 32 * u
            if k < 400:
                for c in range(4):
                    if u & 1:
                        a1[lane] += sq[4 * k + c]
                    else:
                        a0[lane] += sq[4 * k + c]
    return G._xor_tree(a0 + a1)


def _warp_sumsq_vector(x):
    """warp_sumsq's vector path for 1600 aligned samples: k0 in (0, 256), u < 8, even u -> acc, odd u -> a1"""
    sq = x.astype(np.float64) ** 2
    acc, a1 = np.zeros(32), np.zeros(32)
    for lane in range(32):
        for k0 in (0, 256):
            for u in range(8):
                k = k0 + lane + 32 * u
                for c in range(4):
                    v = sq[4 * k + c] if k < 400 else 0.0
                    if u & 1:
                        a1[lane] += v
                    else:
                        acc[lane] += v
    return G._xor_tree(acc + a1)


def test_f32_block_sum_is_the_same_for_every_source():
    rng = np.random.default_rng(5)
    differ = 0
    for t in range(24):
        # magnitudes over several decades, so that rounding depends on the order of the additions
        x = (rng.standard_normal(1600) * np.exp(3 * rng.standard_normal(1600)) * rng.choice([1e-3, 0.1])).astype(np.float32)
        if t == 0:
            x[::7] = 0.0
        ref = G.warp_sumsq_f32(x, 0, 64 * 1600)
        for f in (_push_sums_kernel, _smem_kernel, _warp_sumsq_vector, G.block_sumsq_f32):
            assert f(x) == ref, f.__name__
        differ += np.sum(x.astype(np.float64) ** 2) != ref
    assert differ >= 16                                  # numpy's pairwise order is another order: the test tells them apart


def test_f32_scalar_path_and_split_ranges():
    """odd physical starts and wrapping ranges take the scalar loop (element i -> lane i % 32), a different order from
    the vector path for the same samples"""
    rng = np.random.default_rng(6)
    x = (rng.standard_normal(1600) * np.exp(3 * rng.standard_normal(1600))).astype(np.float32)
    sq = x.astype(np.float64) ** 2
    acc = np.zeros(32)
    for i in range(1600):
        acc[i % 32] += sq[i]
    scalar = G._xor_tree(acc)
    assert G.warp_sumsq_f32(x, 3, 1 << 20) == scalar        # unaligned start
    assert G.warp_sumsq_f32(x, 1000, 2000) == scalar        # wraps the physical ring
    assert G.warp_sumsq_f32(x, 4, 1 << 20) != scalar        # aligned: vector order
    # a tail after the vector body (len % 4 != 0): body words first, then elements 4 nv.. to lanes 0..
    y = x[:1003]
    v = G.warp_sumsq_f32(y, 0, 1 << 20)
    acc0, acc1 = np.zeros(32), np.zeros(32)
    s2 = y.astype(np.float64) ** 2
    for w in range(250):
        lane, m = w % 32, w // 32
        for c in range(4):
            if m % 2 == 0:
                acc0[lane] += s2[4 * w + c]
            else:
                acc1[lane] += s2[4 * w + c]
    acc = acc0 + acc1
    for i in range(1000, 1003):
        acc[i - 1000] += s2[i]
    assert v == G._xor_tree(acc)


# ---- the percentile K2 forms from its sorted mean squares
def percentile25_rms_sorted(S):
    """K2's percentile25_rms_sorted, restated: numpy's 'linear' method and _lerp on sqrt of two order statistics"""
    n = len(S)
    vi = n * 0.25 - 0.25
    k_lo = math.floor(vi)
    k_hi = min(k_lo + 1, n - 1)
    a, b = math.sqrt(S[k_lo]), math.sqrt(S[k_hi])
    t = vi - k_lo
    diff = b - a
    r = a + diff * t
    if t >= 0.5:
        r = b - diff * (1.0 - t)
    return r


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 6, 7, 8, 10, 100, 128, 129, 200, 2048])
def test_percentile_formula_equals_numpy(n):
    """every fractional class t = 0, .25, .5, .75 of the virtual index (n = 1..5 cover them), and chunk counts on both
    sides of 128 (K2 replaces in place up to 128 chunks, through a second buffer above)"""
    rng = np.random.default_rng(n)
    for _ in range(200):
        ms = np.sort(rng.random(n) ** 3 * rng.choice([1e-6, 1e-2, 1.0]))
        assert percentile25_rms_sorted(ms) == np.percentile(np.sqrt(ms), 25)
    t = (n * 0.25 - 0.25) % 1
    assert t in (0.0, 0.25, 0.5, 0.75)


def test_dropping_the_upper_lerp_changes_the_percentile():
    """t >= 0.5 (n = 3, 4 mod 4) takes numpy's second form; the first form alone differs in the last bit somewhere"""
    rng = np.random.default_rng(9)
    hits = 0
    for _ in range(2000):
        ms = np.sort(rng.random(4))
        a, b = math.sqrt(ms[0]), math.sqrt(ms[1])
        hits += (a + (b - a) * 0.75) != np.percentile(np.sqrt(ms), 25)
    assert hits > 100


# ---- exact ties
def tie_feed(levels, R=16000):
    """int16 constant blocks: levels[i] for tick i + 1 (1600 samples each)"""
    return np.concatenate([np.full(1600, v, np.int16) for v in levels])


def test_rms_equals_threshold_is_not_silent():
    """chunks of constant 2 make the 25th percentile exactly 2/32768, the threshold 3/32768; a block of constant 3 has
    RMS 3/32768: equal, so not silent (rms < thr)"""
    lv = [2] * 10 + [3] + [2] * 4
    m = G.GateModel(16000, G.physical_ring(16000, 16000), "i16", [dict(frame_size=1600, min_threshold=0.0)])
    m.push(0, tie_feed(lv))
    _, tr = m.tick(len(lv))
    k = 10                                              # tick 11: the block of 3s, chunks 2 2 .. 2 3 (P25 from the 2s)
    assert tr["thr"][0, k] == 3 / 32768 and tr["rms"][0, k] == 3 / 32768 and tr["silent"][0, k] == 0
    assert tr["silent"][0, k + 1] == 1 and tr["rms"][0, k + 1] == 2 / 32768


def test_threshold_equal_to_min_threshold():
    lv = [2] * 12
    for mt, want in ((3 / 32768, 3 / 32768), (np.nextafter(3 / 32768, 1), np.nextafter(3 / 32768, 1))):
        m = G.GateModel(16000, G.physical_ring(16000, 16000), "i16", [dict(frame_size=1600, min_threshold=float(mt))])
        m.push(0, tie_feed(lv))
        _, tr = m.tick(12)
        assert tr["thr"][0, 11] == want
    m = G.GateModel(16000, G.physical_ring(16000, 16000), "i16", [dict(frame_size=1600, min_threshold=3 / 32768)])
    m.push(0, tie_feed(lv))
    m.tick(12)
    assert np.percentile(np.sqrt(m.s[0].ms), 25) * 1.5 == 3 / 32768     # 1.5 * P25 == min_threshold: a true tie


def duration_feed():
    """digital silence to tick 18, sound (1000) at ticks 19-23, silence again: at ring 16000 the first full tick is 10
    (silence from 1.0 s), sound from 1.9 s, its end at 2.4 s, the cut at 2.8 s with the edges below"""
    return [0] * 10 + [0] * 8 + [1000] * 5 + [0] * 12


DUR_EDGES = {   # parameter: the exact difference of two tick times it is compared with in the feed
    "pre_speech_silence": 19 * 0.1 - 10 * 0.1,
    "speech_duration_min": 24 * 0.1 - 19 * 0.1,
    "speech_duration_max": 24 * 0.1 - 19 * 0.1,
    "post_speech_silence": 28 * 0.1 - 24 * 0.1,
}


def duration_params(name, side):
    p = dict(frame_size=1600, pre_speech_silence=0.5, speech_duration_min=0.2, speech_duration_max=1.0,
             post_speech_silence=0.3, min_threshold=0.005)
    v = DUR_EDGES[name]
    p[name] = float(v if side == 0 else np.nextafter(v, np.inf if name != "speech_duration_max" else -np.inf))
    if name == "speech_duration_min":
        p["speech_duration_max"] = 2.0
    return p


@pytest.mark.parametrize("name", sorted(DUR_EDGES))
def test_duration_ties_go_both_ways(name):
    """a parameter equal to the tick-time difference it is compared with, and the next double past it: the two runs of
    the model differ (so each >= / <= of the timing machine is exercised at its edge)"""
    out = []
    for side in (0, 1):
        m = G.GateModel(16000, G.physical_ring(16000, 16000), "i16", [duration_params(name, side)])
        m.push(0, tie_feed(duration_feed()))
        _, tr = m.tick(len(duration_feed()))
        out.append((tr["state"].copy(), m.event_array()))
    # at the edge the candidate is cut at tick 28; past it there is none, or (post_speech_silence) it comes a tick later
    assert len(out[0][1]) == 1 and out[0][1][0, 2] == 28
    assert len(out[1][1]) == 0 or out[1][1][0, 2] == 29
    assert not np.array_equal(out[0][0], out[1][0])
