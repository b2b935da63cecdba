"""Shared test helpers (stream regeneration identical to oracle/gen_golden.py)."""
import hashlib

import numpy as np

from easywakeword_b200 import synth


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def detect_stream_for(case, word):
    if case.get("special") == "config1":     # SURVEY §8(d) config 1
        rng = np.random.default_rng(7)
        s = (rng.standard_normal(400000) * 0.002).astype(np.float32)
        s[224000:224000 + len(word)] += (3.0 * word).astype(np.float32)
        return s
    x, _ = synth.stream(case["seed"], case["seconds"], word, noise_sigma=case["noise"], gain=tuple(case["gain"]),
                        zero_gaps=case.get("zero_gaps", 0), distractor_prob=case.get("distractor_prob", 0.0),
                        inserts_per_10s=tuple(case.get("inserts", (1, 3))))
    return synth.from_int16(synth.to_int16(x))


def mfcc_rel_l2(a, b):
    """Per-frame relative L2 error of MFCC matrices [20, F] (SURVEY §7 'hard parts': the parity metric)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    num = np.linalg.norm(a - b, axis=0)
    den = np.linalg.norm(b, axis=0)
    return num / np.maximum(den, 1e-30)


def dense_geometry_sets(plan_fn):
    """Template-length sets (1-8 templates of 640 .. 48000 samples, remainders mod 160 on both sides of 96 so that
    windows have 1 and 2 right-edge frames) through K4's planner -> {(DH, threads, CTAs per SM): lengths}, one set per
    reachable geometry: the one with the fewest templates and samples, so that a device test of every geometry stays
    cheap.  plan_fn(lengths) -> (DH, threads, CTAs per SM, shared-memory bytes)."""
    grid = [640, 1001, 4097, 8000, 15503, 16000, 24013, 33406, 40111, 48000]
    sets = set()
    for T in range(1, 9):
        for a in grid:
            for b in grid:
                if a <= b:
                    sets.add(tuple(sorted([a] * (T - 1) + [b])))
        for i in range(len(grid)):
            sets.add(tuple(sorted((grid * 2)[i:i + T])))
    rng = np.random.default_rng(160)
    for _ in range(400):
        T = int(rng.integers(1, 9))
        sets.add(tuple(sorted(int(v) for v in rng.integers(640, 48001, T))))
    reach = {}
    for lens in sorted(sets, key=lambda s: (len(s), sum(s), s)):
        try:
            g = tuple(plan_fn(list(lens))[:3])
        except ValueError:                       # does not fit shared memory: ewk_dense_scores refuses it too
            continue
        reach.setdefault(g, list(lens))
    return reach
