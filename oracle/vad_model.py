"""ORACLE — TEST INFRASTRUCTURE ONLY.  An exact model of template analysis (WakeWord._analyze_reference_audio_duration,
wakeword.py:872-893, after librosa.load): what K6 (template_vad_kernel, easywakeword_b200/csrc/ewk_vad.cuh) and the
host rule (easywakeword_b200.wakeword.analyze_reference_audio_duration) must produce, bit for bit.

Frame RMS.  librosa.feature.rms(frame_length=400, hop_length=160, center=True, pad_mode='constant') pads 200 zeros on
each side, frames through a strided view whose frame-sample axis is contiguous, squares in float32 and takes np.mean
over that axis.  A contiguous float32 reduction of n = 400 elements is numpy's pairwise sum, whose shape for 400 is
fixed: the halves [0, 200) and [200, 400), each split again at 96 (n / 2 rounded down to a multiple of 8), giving the
blocks [0, 96), [96, 200), [200, 296), [296, 400).  A block (at most 128 elements) runs 8 sequential accumulators,
r_a = x[a]^2 + x[a + 8]^2 + ... (12 or 13 terms), combined as ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)); the
blocks are combined as (B0 + B1) + (B2 + B3).  np.mean then divides by the count (a float64 division rounded to float32,
which equals the float32 division: 53 >= 2 * 24 + 2) and np.sqrt rounds in float32.  `frame_rms` below runs those 32
chains with elementwise float32 operations, one frame per row; it does not call numpy's reductions.

The rule.  thr = float32(max rms) * float32(0.1) (NEP 50: a Python float does not promote a float32 scalar); a frame is
voiced when rms > thr; duration = (last - first) * 160 / 16000 in float64, reported as max(duration, 0.2); the frame count
is 1 + len // 160, and an empty template is one all-zero frame, not voiced.
"""
from __future__ import annotations

import numpy as np

FRAME = 400
HOP = 160
SR = 16000
VOICE_ACTIVITY_THRESHOLD = 0.1
MIN_DETECTED_DURATION = 0.2
BLOCKS = ((0, 96), (96, 200), (200, 296), (296, 400))


def frames(y):
    """[n_frames, 400] float32 copy of the zero-padded frames (row t = y[160 t - 200 : 160 t + 200])."""
    y = np.asarray(y, dtype=np.float32).reshape(-1)
    n_frames = 1 + len(y) // HOP
    ypad = np.zeros(len(y) + FRAME, np.float32)
    ypad[FRAME // 2:FRAME // 2 + len(y)] = y
    idx = HOP * np.arange(n_frames)[:, None] + np.arange(FRAME)[None, :]
    return ypad[idx]


def _chain_sums(sq):
    """numpy's pairwise float32 sum of 400 values per row, as 32 explicit chains (4 blocks x 8 accumulators)."""
    block = []
    for a, b in BLOCKS:
        r = [sq[:, a + k].copy() for k in range(8)]
        for i in range(a + 8, b, 8):
            for k in range(8):
                r[k] = r[k] + sq[:, i + k]
        block.append(((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7])))
    return (block[0] + block[1]) + (block[2] + block[3])


def frame_rms(y):
    """librosa.feature.rms(y, frame_length=400, hop_length=160)[0] for float32 y -> float32 [1 + len // 160]."""
    x = frames(y)
    with np.errstate(under="ignore"):
        s = _chain_sums(x * x)
    return np.sqrt(s / np.float32(FRAME)).astype(np.float32)


def analyze(y, rms=None):
    """-> dict with the fields of ewk_vad_result (duration_s, max_rms, threshold, first_frame, last_frame, n_frames,
    voiced) for float32 y.  `rms` replaces the frame RMS (to ask what another arithmetic would decide)."""
    if rms is None:
        rms = frame_rms(y)
    rms = np.asarray(rms, dtype=np.float32)
    mx = np.float32(rms.max())
    thr = np.float32(mx * np.float32(VOICE_ACTIVITY_THRESHOLD))
    v = np.flatnonzero(rms > thr)
    out = dict(max_rms=mx, threshold=thr, n_frames=len(rms), voiced=int(len(v) > 0),
               first_frame=int(v[0]) if len(v) else -1, last_frame=int(v[-1]) if len(v) else -1)
    out["duration_s"] = max(int(v[-1] - v[0]) * HOP / SR, MIN_DETECTED_DURATION) if len(v) else 0.0
    return out


def duration(y):
    """The reference's return value: the duration in seconds, or None when no frame is voiced."""
    r = analyze(y)
    return r["duration_s"] if r["voiced"] else None


def frame_rms_double(y):
    """Frame RMS accumulated in double and rounded once: lane l of a warp adds x[l]^2, x[l + 32]^2, ... in double, a
    xor butterfly (16, 8, 4, 2, 1) adds the 32 lanes, then float32(sum / 400) and a float32 sqrt.  This is the
    arithmetic K6 used before it followed librosa's; the tests keep it to show that the near-threshold templates
    separate the two."""
    x = frames(y).astype(np.float64)
    sq = x * x
    s = np.zeros((len(sq), 32))
    for k in range(0, FRAME, 32):
        n = min(32, FRAME - k)
        s[:, :n] = s[:, :n] + sq[:, k:k + n]
    lane = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        s = s + s[:, lane ^ o]
    return np.sqrt((s[:, 0] / float(FRAME)).astype(np.float32))


def near_threshold_templates(seed, n_pairs):
    """2 * n_pairs templates whose first voiced frame sits on the threshold under librosa's arithmetic.

    Each is a quiet noise burst, a gap of zeros, then a loud +-0.5 square wave.  The loud block's squares and sums are
    exact in any order, so max rms = 0.5 and the threshold is the same for every arithmetic.  The burst's gain is
    bisected (64 steps) onto the point where frame_rms puts the burst's loudest frame above the threshold; the pair is
    the template just below (burst not voiced) and just above (burst voiced).  There a frame RMS that differs by one
    float32 ulp moves the first voiced frame by the whole gap: the duration changes, not just a bit."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_pairs):
        lead, nb, gap, nl = (int(rng.integers(0, 500)), int(rng.integers(400, 3000)), int(rng.integers(400, 1200)),
                             int(rng.integers(4000, 9000)))
        noise = rng.standard_normal(nb).astype(np.float32)
        period, high = int(rng.integers(20, 90)), int(rng.integers(5, 15))
        loud = np.where(np.arange(nl) % period < high, np.float32(0.5), np.float32(-0.5)).astype(np.float32)

        def make(g):
            return np.concatenate([np.zeros(lead, np.float32), noise * np.float32(g), np.zeros(gap, np.float32), loud,
                                   np.zeros(300, np.float32)]).astype(np.float32)

        loud_first = analyze(make(0.0))["first_frame"]
        lo, hi = 0.0, 1.0
        for _ in range(64):
            m = 0.5 * (lo + hi)
            if analyze(make(m))["first_frame"] < loud_first:
                hi = m
            else:
                lo = m
        out += [make(lo), make(hi)]
    return out
