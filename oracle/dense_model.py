"""ORACLE — TEST INFRASTRUCTURE ONLY.  Exact model of K4's per-hop scores (easywakeword_b200/csrc/ewk_dense.cuh).

K4 scores the window x[160 (h - n) : 160 (h - n) + L] of every hop h (ewk_oracle.dense_window) from exact integer
statistics of the window's MFCC rows: every row value is clamped to +-2047 and quantised once, q = rint(x 2^16), and
S1 = sum q, S2 = sum q^2 are 64-bit integers.  Integer sums do not depend on their order, so this model needs none of
the kernel's scans, sub-chunks, floor ways or call cuts: for any window it takes the rows from `frames_fn(window)`
(float32 [F, 20]), forms S1 / S2 and restates, operation for operation, the float arithmetic the kernel applies to
them (dense_stats, score_window, score_from_dots).  With frames_fn = K3's own frame pipeline (the context's
extract_mfcc(window, want_frames=True), the same warp_frame_mfcc on the same samples with the same window-local
padding and top_db floor) the kernel's output must equal this model bit for bit; with the oracle's float64 frames
(ewk_oracle.mfcc_frames(window).T) it approximates the reference.

The model also classifies each window the way the kernel routes it — un-floored, floored in stream-grid rows only
(a "way" window, summed over a floored copy of the grid rows), or floored in an edge frame (summed frame by frame) —
from the oracle's log-mel of the window; `distinct_way_floors` counts how many floors the way windows of each
sub-chunk need, which tells whether the kernel's 8 ways ran out.
"""
from __future__ import annotations

import numpy as np

from . import librosa_restated as L
from .ewk_oracle import dense_window
from .resample_restated import fmaf32

N_MFCC = 20
CLAMP = 2047.0              # rows are clamped here before quantisation (K4 departs from the reference beyond it)
UNFLOORED, WAY, EDGE = 0, 1, 2
CLASS_NAMES = ("un-floored", "way", "edge-floored")


def window_geometry(L_samples):
    """(n, F, t_hi, r) of a template of L samples: n hops back, F frames, grid frames t = 2 .. t_hi, r right-edge frames."""
    n = -(-int(L_samples) // 160)
    F = 1 + int(L_samples) // 160
    t_hi = (int(L_samples) - 256) // 160
    return n, F, t_hi, F - 1 - t_hi


# ------------------------------------------------------------------------------------------------ integer statistics
def quantize(rows):
    """[F, 20] float32 rows -> int64 q = rint(clamp(x, +-2047) * 2^16), ties to even (__float2int_rn)."""
    x = np.clip(np.asarray(rows, np.float32), np.float32(-CLAMP), np.float32(CLAMP))
    return np.rint(x.astype(np.float64) * 65536.0).astype(np.int64)


def sums(rows):
    """(S1, S2) int64 [20] over the frames of `rows`."""
    q = quantize(rows)
    return q.sum(axis=0), (q * q).sum(axis=0)


def fma64(a, b, c):
    """a * b + c for finite floats, rounded once to double (C's fma).  Python 3.12 has no math.fma: the exact value is
    a ratio of integers with a power-of-two denominator, and int / int rounds correctly."""
    na, da = float(a).as_integer_ratio()
    nb, db = float(b).as_integer_ratio()
    nc, dc = float(c).as_integer_ratio()
    return (na * nb * dc + nc * da * db) / (da * db * dc)


def dense_stats(S1, S2, F):
    """K4's dense_stats as nvcc compiles it for sm_100a -> (mean, sd) float32 arrays.
        invf = 1.0 / F                                   (double)
        mean = f32((s1 * invf) * 2^-16)
        var  = (fma(-fl(s1 * s1), invf, s2) * invf) * 2^-32     nvcc contracts s2 - s1 * s1 * invf into DMUL + DFMA
        sd   = sqrtf(max(f32(var), 0)),  or exactly 0 where F S2 == S1^2 (all rows equal: the residue is not kept)"""
    S1 = np.asarray(S1, np.int64)
    S2 = np.asarray(S2, np.int64)
    invf = 1.0 / float(F)
    s1 = S1.astype(np.float64)
    s2 = S2.astype(np.float64)
    mean = ((s1 * invf) * (1.0 / 65536.0)).astype(np.float32)
    p = s1 * s1
    d = np.array([fma64(-pp, invf, ss) for pp, ss in zip(p.ravel().tolist(), s2.ravel().tolist())],
                 np.float64).reshape(p.shape)
    var = (d * invf) * (1.0 / 4294967296.0)
    sd = np.sqrt(np.maximum(var.astype(np.float32), np.float32(0.0)))
    flat = np.array([a * a == F * b for a, b in zip(S1.ravel().tolist(), S2.ravel().tolist())]).reshape(sd.shape)
    sd[flat] = 0.0
    return mean, sd


def window_features(rows):
    """(mean, sd) float32 [20] of one window's rows [F, 20]."""
    S1, S2 = sums(rows)
    return dense_stats(S1, S2, len(rows))


def template_features(rows, n_mfcc=N_MFCC):
    """TemplateFeat.dmean / dstd: the same statistics over the template's own frames, zero at and above n_mfcc."""
    m, s = window_features(rows)
    m[n_mfcc:] = 0.0
    s[n_mfcc:] = 0.0
    return m, s


# ------------------------------------------------------------------------------------------------ score
def score_features(tm, ts, wm, ws, n_mfcc=N_MFCC):
    """score_window + score_from_dots for windows [N, 20] against one template -> float32 [N].
    Six serial fmaf chains over c = 0 .. n_mfcc - 1, then per pair q = f32((double) uv / sqrt((double) fl32(uu vv))),
    d = clamp(1 - q, 0, 2) (NaN kept), combined = (1 - dm) 0.7 + (1 - ds) 0.3, p = 100 combined, score = p sqrtf(p) / 10,
    every step in float32."""
    wm = np.atleast_2d(np.asarray(wm, np.float32))
    ws = np.atleast_2d(np.asarray(ws, np.float32))
    tm = np.asarray(tm, np.float32)
    ts = np.asarray(ts, np.float32)
    z = np.zeros(len(wm), np.float32)
    uvm, uum, vvm, uvs, uus, vvs = z.copy(), z.copy(), z.copy(), z.copy(), z.copy(), z.copy()
    for c in range(n_mfcc):
        a, b = np.full_like(z, tm[c]), np.full_like(z, ts[c])
        uvm = fmaf32(a, wm[:, c], uvm)
        uum = fmaf32(a, a, uum)
        vvm = fmaf32(wm[:, c], wm[:, c], vvm)
        uvs = fmaf32(b, ws[:, c], uvs)
        uus = fmaf32(b, b, uus)
        vvs = fmaf32(ws[:, c], ws[:, c], vvs)
    with np.errstate(all="ignore"):
        def dist(uv, uu, vv):
            q = (uv.astype(np.float64) / np.sqrt((uu * vv).astype(np.float64))).astype(np.float32)
            d = np.float32(1.0) - q
            d = np.where(d < 0, np.float32(0.0), np.where(d > 2, np.float32(2.0), d))
            return d.astype(np.float32)
        dm, ds = dist(uvm, uum, vvm), dist(uvs, uus, vvs)
        combined = (np.float32(1.0) - dm) * np.float32(0.7) + (np.float32(1.0) - ds) * np.float32(0.3)
        p = combined * np.float32(100.0)
        return ((p * np.sqrt(p)) / np.float32(10.0)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ classification
def _logmel_minmax(windows, preemphasis=0.0):
    """Un-floored log-mel (float64) of every frame of each window [N, L] -> (min, max) over bands, [N, F] each."""
    y = np.asarray(windows, np.float32)
    if preemphasis:
        y = L.preemphasis(y, coef=preemphasis)
    n, ln = y.shape
    F = 1 + ln // 160
    ypad = np.zeros((n, ln + 512), np.float64)
    ypad[:, 256:256 + ln] = y
    idx = np.arange(512)[None, :] + 160 * np.arange(F)[:, None]
    fr = ypad[:, idx] * L.hann_window()[None, None, :]
    S = np.abs(np.fft.rfft(fr, axis=-1)) ** 2
    mel = S @ L.mel_filterbank().astype(np.float64).T
    lm = 10.0 * np.log10(np.maximum(1e-10, mel))
    return lm.min(axis=-1), lm.max(axis=-1)


def classify_windows(stream, starts, L_samples, preemphasis=0.0, chunk=64):
    """Class (UNFLOORED / WAY / EDGE) and float32 floor (max - 80; NaN when un-floored) of the windows
    stream[s : s + L] for s in `starts`, the way K4 routes them: a window none of whose frames reaches below its floor
    is un-floored; one whose floored frames are all stream-grid frames t = 2 .. t_hi is a way window; one with a
    floored edge frame (t = 0, 1 or t > t_hi) is summed frame by frame."""
    stream = np.asarray(stream, np.float32)
    _, F, t_hi, _ = window_geometry(L_samples)
    edge = np.zeros(F, bool)
    edge[:2] = True
    edge[t_hi + 1:] = True
    starts = np.asarray(starts, np.int64)
    cls = np.zeros(len(starts), np.int8)
    floor = np.full(len(starts), np.nan, np.float32)
    for a in range(0, len(starts), chunk):
        st = starts[a:a + chunk]
        W = np.stack([stream[s:s + L_samples] for s in st])
        mn, mx = _logmel_minmax(W, preemphasis)
        fl = mx.max(axis=1) - 80.0
        below = mn < fl[:, None]
        c = np.where(below.any(axis=1), np.where((below & edge[None, :]).any(axis=1), EDGE, WAY), UNFLOORED)
        cls[a:a + chunk] = c
        f32 = np.float32(mx.max(axis=1).astype(np.float32) - np.float32(80.0))
        floor[a:a + chunk] = np.where(c != UNFLOORED, f32, np.float32(np.nan))
    return cls, floor


def distinct_way_floors(hops, cls, floor, DH, hop0):
    """Distinct floors among the way windows of each sub-chunk of a call that starts at hop0 ([len(hops)] per-window
    class and floor, any number of templates flattened together) -> {sub-chunk index: count}.  More than 8 in one
    sub-chunk means some way window found no free way and was summed frame by frame."""
    hops = np.asarray(hops, np.int64)
    out = {}
    sel = np.asarray(cls) == WAY
    for h, f in zip(hops[sel], np.asarray(floor)[sel]):
        out.setdefault(int((h - hop0) // DH), set()).add(np.float32(f).tobytes())
    return {k: len(v) for k, v in sorted(out.items())}


# ------------------------------------------------------------------------------------------------ the model
class DenseModel:
    """Exact K4 scores of `stream` (the float32 samples the ring holds, from sample 0) against templates.

    frames_fn(pcm float32 [n]) -> float32 [1 + n // 160, 20] rows.  Windows are cached by (start, length), so templates
    of equal length share them."""

    def __init__(self, stream, templates, frames_fn, n_mfcc=N_MFCC, preemphasis=0.0):
        self.stream = np.asarray(stream, np.float32)
        self.templates = [np.asarray(t, np.float32) for t in templates]
        self.frames_fn = frames_fn
        self.n_mfcc = n_mfcc
        self.preemphasis = preemphasis
        self.tfeat = [template_features(frames_fn(t), n_mfcc) for t in self.templates]
        self._win = {}
        self._cls = {}

    def window_start(self, h, k):
        n, _ = dense_window(len(self.templates[k]))
        return 160 * (int(h) - n)

    def features(self, start, L_samples):
        key = (int(start), int(L_samples))
        if key not in self._win:
            self._win[key] = window_features(self.frames_fn(self.stream[start:start + L_samples]))
        return self._win[key]

    def scores(self, hops):
        """float32 [len(hops), T]; NaN where the window starts before the stream."""
        hops = np.asarray(hops, np.int64)
        out = np.full((len(hops), len(self.templates)), np.nan, np.float32)
        for k, t in enumerate(self.templates):
            starts = [self.window_start(h, k) for h in hops]
            ok = [i for i, s in enumerate(starts) if s >= 0]
            if not ok:
                continue
            feats = [self.features(starts[i], len(t)) for i in ok]
            wm = np.stack([f[0] for f in feats])
            ws = np.stack([f[1] for f in feats])
            out[ok, k] = score_features(self.tfeat[k][0], self.tfeat[k][1], wm, ws, self.n_mfcc)
        return out

    def classes(self, hops, k):
        """(class [len(hops)] int8, -1 before the stream; floor [len(hops)] float32) of template k's windows."""
        hops = np.asarray(hops, np.int64)
        Ls = len(self.templates[k])
        starts = np.array([self.window_start(h, k) for h in hops], np.int64)
        todo = sorted({int(s) for s in starts if s >= 0 and (int(s), Ls) not in self._cls})
        if todo:
            c, f = classify_windows(self.stream, todo, Ls, self.preemphasis)
            for s, cc, ff in zip(todo, c, f):
                self._cls[(s, Ls)] = (int(cc), ff)
        cls = np.full(len(hops), -1, np.int8)
        floor = np.full(len(hops), np.nan, np.float32)
        for i, s in enumerate(starts):
            if s >= 0:
                cls[i], floor[i] = self._cls[(int(s), Ls)]
        return cls, floor


def oracle_frames(preemphasis=0.0, n_mfcc=N_MFCC):
    """frames_fn from the float64 oracle (ewk_oracle.mfcc_frames), rows beyond n_mfcc zero."""
    from .ewk_oracle import mfcc_frames

    def fn(pcm):
        m = mfcc_frames(np.asarray(pcm, np.float32), preemphasis, N_MFCC).T.astype(np.float32)
        m[:, n_mfcc:] = 0.0
        return m
    return fn
