"""ORACLE — TEST INFRASTRUCTURE ONLY.  CPU statement of the sample-rate conversion for SURVEY §8(f) row N3.

PARITY UNPINNED against the reference.  The reference converts non-16 kHz audio with
``librosa.load(path, sr=16000)`` / ``librosa.resample`` (/root/reference/easywakeword/wakeword.py:588, 866-870;
examples/tune_threshold.py:33-47), i.e. librosa 0.11's default ``res_type='soxr_hq'`` = python-soxr / libsoxr
quality HQ.  Neither librosa nor soxr is installable here and the reference holds no test or golden vector for
a resampled signal, so nothing in this file is checked against soxr output.  What is restated is soxr HQ's
PUBLISHED SPECIFICATION (soxr.h quality table: linear phase, pass-band end 0.913 of the lower Nyquist, stop-band
begin 1.0, ~20-bit / 125 dB rejection) as a single-stage Kaiser-windowed-sinc polyphase interpolator, and
librosa.resample's framing around it: output length ceil(n * target / orig), output sample n at input time
n * orig / target, zeros outside the input, no gain rescale (scale=False).  Two band-limiting filters that meet
the same spec agree on pass-band content to their ripple (<1e-5 here); they differ in the 0.913..1.0 transition
band.  tests/test_oracle.py pins THIS arithmetic against scipy.signal.resample_poly run with the same prototype
filter and against closed-form tones; tests/test_gpu_resample.py compares the CUDA kernel with it.
"""
from __future__ import annotations

import math

import numpy as np

TARGET_SR = 16000
PASSBAND = 0.913          # of the lower Nyquist
ATTENUATION_DB = 125.0
MAX_PHASES = 4096


def design(sr_in: int, sr_out: int = TARGET_SR):
    """-> dict(L, M, Minv, W, fc, beta): out[n] sits at input time n*M/L; W = half-width in input samples."""
    if sr_in <= 0 or sr_out <= 0:
        raise ValueError("sample rates must be positive")
    g = math.gcd(sr_in, sr_out)
    L, M = sr_out // g, sr_in // g
    if L > MAX_PHASES:
        raise ValueError(f"{sr_in} -> {sr_out} Hz needs {L} filter phases (max {MAX_PHASES})")
    lower = min(sr_in, sr_out)
    f_pass, f_stop = PASSBAND * lower / 2.0, lower / 2.0
    beta = 0.1102 * (ATTENUATION_DB - 8.7)
    d_omega = 2.0 * math.pi * (f_stop - f_pass) / sr_in
    n_taps = int(math.ceil((ATTENUATION_DB - 8.0) / (2.285 * d_omega)))
    W = (n_taps + 1) // 2
    fc = 0.5 * (f_pass + f_stop) / sr_in                    # cycles per input sample
    Minv = pow(M, -1, L) if L > 1 else 0
    return dict(L=L, M=M, Minv=Minv, W=W, fc=fc, beta=beta)


def kernel(tau, d):
    """g(tau): 2 fc sinc(2 fc tau) * kaiser(tau / W), zero for |tau| >= W.  float64."""
    tau = np.asarray(tau, dtype=np.float64)
    u = tau / d["W"]
    inside = np.abs(u) < 1.0
    w = np.where(inside, np.i0(d["beta"] * np.sqrt(np.clip(1.0 - u * u, 0.0, None))) / np.i0(d["beta"]), 0.0)
    return 2.0 * d["fc"] * np.sinc(2.0 * d["fc"] * tau) * w


def phase_table(d):
    """H[j, p] = g(p/L + W - 1 - j), j < 2W: the tap of input sample k_c - W + 1 + j for phase p.  float64."""
    j = np.arange(2 * d["W"], dtype=np.float64)[:, None]
    p = np.arange(d["L"], dtype=np.float64)[None, :]
    return kernel(p / d["L"] + d["W"] - 1 - j, d)


def out_len(n_in: int, sr_in: int, sr_out: int = TARGET_SR) -> int:
    """librosa.resample: int(np.ceil(n * target / orig))."""
    return int(math.ceil(n_in * sr_out / sr_in))


def resample(y, sr_in: int, sr_out: int = TARGET_SR, *, in_first: int = 0, out_first: int = 0, n_out=None,
             table_dtype=np.float32):
    """float64 evaluation of out[n] = sum_k y_abs[k] g(n M / L - k) for n in [out_first, out_first + n_out);
    y_abs[k] = y[k - in_first] inside the given buffer, 0 outside.  The taps are rounded to `table_dtype` first
    (the device keeps a float32 table)."""
    y = np.asarray(y, dtype=np.float64)
    if sr_in == sr_out:
        return y.astype(np.float32)
    d = design(sr_in, sr_out)
    if n_out is None:
        n_out = out_len(len(y), sr_in, sr_out) - out_first
    H = phase_table(d).astype(table_dtype).astype(np.float64)
    W, L, M = d["W"], d["L"], d["M"]
    n = out_first + np.arange(n_out, dtype=np.int64)
    kc, p = (n * M) // L, (n * M) % L
    ypad = np.concatenate([np.zeros(2 * W), y, np.zeros(2 * W)])
    out = np.zeros(n_out, dtype=np.float64)
    base = kc - W + 1 - in_first + 2 * W                     # index into ypad of tap j = 0
    for j in range(2 * W):
        idx = base + j
        ok = (idx >= 0) & (idx < len(ypad))
        out += np.where(ok, ypad[np.clip(idx, 0, len(ypad) - 1)], 0.0) * H[j, p]
    return out.astype(np.float32)


# ------------------------------------------------------------------------------------------------ float32 chain
# The device (K8, easywakeword_b200/csrc/ewk_resample_push.cuh) evaluates each output as one sequential fmaf chain
# from +0 over taps j = 0 .. 2W-1 of the float32 table.  The functions below restate that arithmetic exactly, so a
# test can compare the device with it bit for bit instead of within a tolerance.

def fmaf32(a, b, c):
    """C's fmaf on float32 arrays: a * b + c rounded once to float32 (round to nearest, ties to even).

    The product of two float32 values is exact in float64; TwoSum gives the sum exactly as s + e.  Rounding s to
    float32 is then correct unless s lies exactly on a float32 midpoint while e != 0, where the exact sum lies off
    the midpoint on e's side (plain float32(float64(a * b) + c) rounds twice and gets such cases wrong)."""
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    c = np.asarray(c, np.float32)
    p = a.astype(np.float64) * b.astype(np.float64)
    cd = c.astype(np.float64)
    s = p + cd
    bb = s - p
    e = (p - (s - bb)) + (cd - bb)
    r = s.astype(np.float32)
    rd = r.astype(np.float64)
    away = np.nextafter(r, np.where(s > rd, np.float32(np.inf), np.float32(-np.inf)))
    ad = away.astype(np.float64)
    flip = (s != rd) & (s - rd == ad - s) & (e != 0) & (np.sign(e) == np.sign(ad - rd))
    return np.where(flip, away, r)


def chain_input(y, law=None):
    """The float32 values the device's FIR reads: float32 as is, int16 / 32768, G.711 codes (uint8, law "ulaw" or
    "alaw") through the ITU-T expansion table / 32768."""
    y = np.asarray(y)
    if law is not None:
        if y.dtype != np.uint8:
            raise TypeError("G.711 input is uint8 codes")
        from easywakeword_b200.resample import ALAW_TABLE, ULAW_TABLE
        table = {"ulaw": ULAW_TABLE, "alaw": ALAW_TABLE}[law]
        return table[y].astype(np.float32) / np.float32(32768.0)
    if y.dtype == np.int16:
        return y.astype(np.float32) / np.float32(32768.0)
    if y.dtype != np.float32:
        raise TypeError(f"the device reads float32, int16 or G.711 input, not {y.dtype}")
    return y


def resample_chain(y, sr_in: int, *, in_first: int = 0, out_first: int = 0, n_out=None, law=None):
    """float32 outputs [out_first, out_first + n_out) of the device's chain, with resample()'s framing: y ([n] or
    [rows, n]) holds absolute input samples [in_first, in_first + n), zeros elsewhere.  Output n of a row is
    acc = fmaf(H[j][p], x[k_c - W + 1 + j], acc) for j = 0 .. 2W-1 from acc = +0, k_c = floor(n M / L),
    p = n M mod L, H = phase_table(d) rounded to float32."""
    x = chain_input(y, law)
    one_d = x.ndim == 1
    x = x.reshape(1, -1) if one_d else x
    d = design(sr_in)
    W, L, M = d["W"], d["L"], d["M"]
    if n_out is None:
        n_out = out_len(x.shape[1], sr_in) - out_first
    n_out = max(int(n_out), 0)
    H = phase_table(d).astype(np.float32)
    n = out_first + np.arange(n_out, dtype=np.int64)
    kc, p = (n * M) // L, (n * M) % L
    acc = np.zeros((x.shape[0], n_out), np.float32)
    if n_out:
        # absolute inputs [lo, hi) cover every tap of every output: zero-padded copy, one gather per tap
        lo, hi = int(kc[0]) - W + 1, int(kc[-1]) + W + 1
        xp = np.zeros((x.shape[0], hi - lo), np.float32)
        a, b = max(lo, in_first), min(hi, in_first + x.shape[1])
        if a < b:
            xp[:, a - lo:b - lo] = x[:, a - in_first:b - in_first]
        base = kc - W + 1 - lo
        for j in range(2 * W):
            acc = fmaf32(xp[:, base + j], H[j, p], acc)
    return acc[0] if one_d else acc


def ring_quantize(y):
    """What an int16 ring stores for output y: clip(rint(y * 32768), -32768, 32767), ties to even.  Reading the ring
    back gives the stored value / 32768."""
    q = np.rint(np.asarray(y, np.float32).astype(np.float64) * 32768.0)
    return np.clip(q, -32768, 32767).astype(np.int16)
