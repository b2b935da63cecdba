"""ORACLE — TEST INFRASTRUCTURE ONLY.  Exact float32 model of K3 (easywakeword_b200/csrc/ewk_segment.cuh over
ewk_frame.cuh): the frame pipeline warp_frame_mfcc, the top_db floor, the pooling of segment_features / fq_finish and
the cosine scores, restated operation for operation so that a test can compare the device with it bit for bit.

Every "lane" operation of the warp is an elementwise numpy float32 operation on arrays shaped [frames, ...]: numpy
rounds each float32 add / sub / mul / div / sqrt once, to nearest, as the device does; fused multiply-adds go through
resample_restated.fmaf32.  The tables are the device's own float32 images (`Tables.from_image`, written by the test
probe tests/k3_probe.cu from build_tables + load_frame_tables), so the model shares no table arithmetic with the oracle.

FMA contraction.  -O3 lets nvcc / ptxas fuse a multiply into an add; which product is fused decides the bits.  The
sites below are read from the SASS of warp_frame_mfcc in the built library (cuobjdump -sass libewk.so, function body
between the two shared-memory transposes, convergent path; every FFMA / FFMA2 of the function is one of them):
  1. Hann window fused into the first radix-8 butterfly (4 FMUL2 + 8 FFMA2): with m_k = fl(x[k+4] h[k+4]),
     a_k = fma(x[k], h[k], m_k) and b_k = fma(x[k], h[k], -m_k) for k < 4; the products x[k] h[k] are never rounded.
  2. cmul, both twiddle stages (14 FFMA per stage): re = fma(a.x, b.x, -fl(a.y b.y)), im = fma(a.y, b.x, fl(a.x b.y)).
  3. Untangle (2 FFMA per bin pair): tr = fma(qr, w.x, -fl(qi w.y)), ti = fma(qi, w.x, fl(qr w.y)).
  4. Power (2 FFMA per bin pair): 0.25 fma(ar, ar, fl(ai ai)), 0.25 fma(br, br, fl(bi bi)); P[128] = fma(zr, zr, fl(zi zi)).
  5. Pooling, segment_features and fq_finish alike (FMUL, FMUL, FFMA, FADD per partial):
     M2 = fl(M2 + fma(fl(delta delta), fl(fl(n cw) / nn), M2_w)).
The mel taps, the DCT and the partial M2 are explicit fmaf calls in the source; the 0.7071 rotations of the radix-8
butterflies are an FADD followed by an FMUL (nothing to fuse).

The log.  out = TEN_LOG10_2 * __log2f(fmaxf(S, 1e-10f)) compiles to FMNMX, MUFU.LG2 (with its denormal prescale, never
taken here since S >= 1e-10) and FMUL.  PTX gives only an error bound for lg2.approx, so the model takes the log as a
function `log_fn(S)`: on the device the test probe's k3p_log_mel, which runs the same source expression; on a CPU the
stand-in `log_mel_standin` (float32(log2(float64(x))) times TEN_LOG10_2 in float32).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .resample_restated import fmaf32

N_FFT, HOP, N_BINS, N_MELS, N_MFCC = 512, 160, 257, 128, 20
SEG_WARPS = 14                        # partials of the pooling (SEG_THREADS / 32)
SEG_SMEM_FRAMES = 301                 # frames K3 keeps in shared memory; more spill to a global workspace
MEL_TAPS = (1, 2, 3, 6)
TEN_LOG10_2 = np.float32(3.01029995663981195)
R_SQRT2 = np.float32(0.70710678118654752440)
F32 = np.float32

# load_frame_pairs_raw's branches (ewk_segment.cuh), in the order the loader tries them
FAST, ODD, MASKED_RING, MASKED_LINEAR, SCALAR = range(5)
BRANCH_NAMES = ("fast even", "odd", "masked ring", "masked linear", "scalar")


# ------------------------------------------------------------------------------------------------ tables
def _f2(n):
    return (np.float32, (n, 2))


DEVICE_TABLES = np.dtype({
    "names": ["hann", "w256", "w512", "mel_start", "mel_len", "mel_off", "mel_w", "dct_t", "mel_pad", "mel_first"],
    "formats": [(np.float32, 512), _f2(256), _f2(256), (np.int32, 128), (np.int32, 128), (np.int32, 128),
                (np.float32, 512), (np.float32, 2560), _f2(12 * 32), (np.int32, 128)],
    "offsets": [0, 2048, 4096, 6144, 6656, 7168, 7680, 9728, 19968, 23040], "itemsize": 23552})
FRAME_TABLES = np.dtype({
    "names": ["hw", "tw1", "tw3", "tw2", "melp", "mfirst", "coef_of_lane", "dct", "preemph", "n_mfcc"],
    "formats": [_f2(256), _f2(256), _f2(128), _f2(32), _f2(12 * 32), (np.int32, 128), (np.int32, 32),
                (np.float32, 32 * 44), np.float32, np.int32],
    "offsets": [0, 2048, 4096, 5120, 5376, 8448, 8960, 9088, 14720, 14724], "itemsize": 14736})
FRAME_IMAGE_OFFSET = 23552            # (sizeof(DeviceTables) + 15) & ~15


@dataclass
class Tables:
    """The float32 tables K3 reads, as numpy arrays in the lane layout of FrameTables."""
    flat: np.ndarray                  # DeviceTables record
    ft: np.ndarray                    # FrameTables record

    @classmethod
    def from_image(cls, image):
        b = np.frombuffer(bytes(image), np.uint8)
        if len(b) != FRAME_IMAGE_OFFSET + FRAME_TABLES.itemsize:
            raise ValueError(f"table image of {len(b)} bytes, expected {FRAME_IMAGE_OFFSET + FRAME_TABLES.itemsize}")
        flat = b[:DEVICE_TABLES.itemsize].view(DEVICE_TABLES)[0]
        ft = b[FRAME_IMAGE_OFFSET:].view(FRAME_TABLES)[0]
        return cls(flat, ft)

    @property
    def hw(self):                     # [a, lane, 2]
        return self.ft["hw"].reshape(8, 32, 2)

    @property
    def tw1(self):                    # [k, lane, 2]
        return self.ft["tw1"].reshape(8, 32, 2)

    @property
    def tw2(self):                    # [k, c, 2]
        return self.ft["tw2"].reshape(8, 4, 2)

    @property
    def tw3(self):                    # [m, lane, 2]
        return self.ft["tw3"].reshape(4, 32, 2)

    @property
    def melp(self):                   # [tap, lane, 2]
        return self.ft["melp"].reshape(12, 32, 2)

    @property
    def mfirst(self):                 # [j, lane]
        return self.ft["mfirst"].reshape(4, 32)

    @property
    def dct(self):                    # [lane, 44]: [band slot s < 4][m < 10], 4 zero pads
        return self.ft["dct"].reshape(32, 44)

    def mel_dense(self):
        """The [128, 257] filterbank the row-compressed flat tables hold."""
        t = self.flat
        m = np.zeros((N_MELS, N_BINS), np.float32)
        for b in range(N_MELS):
            s, n, o = int(t["mel_start"][b]), int(t["mel_len"][b]), int(t["mel_off"][b])
            m[b, s:s + n] = t["mel_w"][o:o + n]
        return m


def log_mel_standin(S):
    """CPU stand-in for TEN_LOG10_2 * __log2f(fmaxf(S, 1e-10f)): the log2 correctly rounded to float32."""
    x = np.maximum(np.asarray(S, np.float32), F32(1e-10))
    return (TEN_LOG10_2 * np.log2(x.astype(np.float64)).astype(np.float32)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ loader
def segment_values(pcm, fmt):
    """The float32 samples K3 reads: float32 as is, int16 as q * (1 / 32768)."""
    pcm = np.asarray(pcm)
    if fmt == "i16" or pcm.dtype == np.int16:
        return (pcm.astype(np.float32) * F32(1.0 / 32768.0)).astype(np.float32)
    return np.asarray(pcm, np.float32)


def preemphasize(y, a):
    """preemph_pairs over the whole segment: out[0] = fl(fl(fl(2 y0) - y1) + y0) (y1 = 0 when len == 1),
    out[n] = fl(fl(-a y[n-1]) + y[n])."""
    y = np.asarray(y, np.float32)
    nb = F32(-F32(a))
    out = np.empty_like(y)
    if len(y) == 0:
        return out
    out[1:] = (nb * y[:-1]) + y[1:]
    y1 = y[1] if len(y) > 1 else F32(0.0)
    out[0] = ((F32(2.0) * y[0]) - y1) + y[0]
    return out


def frame_samples(y, preemphasis=0.0, frames=None):
    """Segment y (float32 as K3 reads it) -> [F, 512] frames: frame t covers segment samples 160 t - 256 .. + 511,
    zero outside the segment; pre-emphasis is applied before the padding.  `frames` selects a subset of t."""
    y = np.asarray(y, np.float32)
    if preemphasis:
        y = preemphasize(y, preemphasis)
    L = len(y)
    F = 1 + L // HOP
    t = np.arange(F) if frames is None else np.asarray(frames)
    pad = np.zeros(L + 2 * N_FFT, np.float32)
    pad[N_FFT:N_FFT + L] = y
    idx = (HOP * t - N_FFT // 2 + N_FFT)[:, None] + np.arange(N_FFT)[None, :]
    return pad[idx]


def loader_branch(start, length, ring, fmt, aligned, t):
    """Which branch of load_frame_pairs_raw frame(s) t of a segment take.  start: the segment's first sample in the
    buffer (the ring position seg_start % ring when ring > 0), ring: ring length (0: linear buffer), fmt "f32" / "i16",
    aligned: the buffer base is 4-byte (int16) / 8-byte (float32) aligned."""
    t = np.asarray(t, np.int64)
    f0 = HOP * t - N_FFT // 2
    q = fmt == "i16"
    inside = (f0 >= 0) & (f0 + N_FFT <= length)
    p = start + f0
    if ring:
        p = np.where(p >= ring, p - ring, p)
        inside = inside & (p + N_FFT <= ring)
    fast = inside & (p % 2 == 0) & aligned
    odd = inside & (p % 2 == 1)
    if q:
        odd = odd & aligned
        if not ring:
            odd = odd & (f0 + N_FFT + 1 <= length)
    p00 = start + f0
    even = (p00 % 2 == 0) & (ring % 2 == 0) & aligned
    out = np.full(t.shape, SCALAR, np.int8)
    out[even & (ring == 0)] = MASKED_LINEAR
    if ring:
        out[even] = MASKED_RING
    out[odd] = ODD
    out[fast] = FAST
    return out


# ------------------------------------------------------------------------------------------------ power spectrum
def _cmul(a, b):
    """(ar, ai) * (br, bi) as nvcc contracts cmul: re = fma(ar, br, -fl(ai bi)), im = fma(ai, br, fl(ar bi))."""
    (ar, ai), (br, bi) = a, b
    return fmaf32(ar, br, -(ai * bi)), fmaf32(ai, br, ar * bi)


def _add(a, b):
    return a[0] + b[0], a[1] + b[1]


def _sub(a, b):
    return a[0] - b[0], a[1] - b[1]


def _dft4(y0, y1, y2, y3):
    s0, s1, s2, d = _add(y0, y2), _sub(y0, y2), _add(y1, y3), _sub(y1, y3)
    s3 = (d[1], -d[0])
    return _add(s0, s2), _add(s1, s3), _sub(s0, s2), _sub(s1, s3)        # Y0, Y1, Y2, Y3


def _fft8_tail(a, b):
    """fft8 after its first butterfly a_k = v_k + v_(k+4), b_k = v_k - v_(k+4)."""
    b1, b2, b3 = b[1], b[2], b[3]
    b1 = ((b1[0] + b1[1]) * R_SQRT2, (b1[1] - b1[0]) * R_SQRT2)
    b2 = (b2[1], -b2[0])
    b3 = ((b3[1] - b3[0]) * R_SQRT2, (-b3[0] - b3[1]) * R_SQRT2)
    Y0, Y1, Y2, Y3 = _dft4(a[0], a[1], a[2], a[3])
    Z0, Z1, Z2, Z3 = _dft4(b[0], b1, b2, b3)
    return [Y0, Z0, Y1, Z1, Y2, Z2, Y3, Z3]


def _fft8(v):
    return _fft8_tail([_add(v[k], v[k + 4]) for k in range(4)], [_sub(v[k], v[k + 4]) for k in range(4)])


def power_spectrum(x, T):
    """warp_power_spectrum: frames [N, 512] float32 -> P [N, 257] float32."""
    x = np.asarray(x, np.float32).reshape(-1, 8, 32, 2)            # [N, a, lane, (2 lane + 64 a, +1)]
    hw = T.hw
    xs = [(x[:, a, :, 0], x[:, a, :, 1]) for a in range(8)]
    hs = [(hw[a, :, 0], hw[a, :, 1]) for a in range(8)]
    # radix 8 over a, the Hann products of x[4..7] rounded and fused into the first butterfly
    m = [(xs[k + 4][0] * hs[k + 4][0], xs[k + 4][1] * hs[k + 4][1]) for k in range(4)]
    a = [(fmaf32(xs[k][0], hs[k][0], m[k][0]), fmaf32(xs[k][1], hs[k][1], m[k][1])) for k in range(4)]
    b = [(fmaf32(xs[k][0], hs[k][0], -m[k][0]), fmaf32(xs[k][1], hs[k][1], -m[k][1])) for k in range(4)]
    v = _fft8_tail(a, b)
    tw1 = T.tw1
    v = [v[0]] + [_cmul(v[k], (tw1[k, :, 0], tw1[k, :, 1])) for k in range(1, 8)]
    V1 = np.stack([np.stack(c, -1) for c in v], 1)                  # [N, k, lane, 2]
    # radix 8 over b: thread (ka, c) = lane 4 ka + c reads V1[ka, 4 b + c]
    U = V1.reshape(-1, 8, 8, 4, 2)                                   # [N, ka, b, c, 2]
    v = [(U[:, :, bb, :, 0], U[:, :, bb, :, 1]) for bb in range(8)]  # each [N, ka, c]
    v = _fft8(v)
    tw2 = T.tw2
    v = [v[0]] + [_cmul(v[k], (tw2[k, :, 0], tw2[k, :, 1])) for k in range(1, 8)]
    Y2 = np.stack([np.stack(c, -1) for c in v], 1)                  # [N, kb, ka, c, 2]
    # radix 4 over c: thread (ka2, j) = lane ka2 + 8 j, e < 2, reads Y2[j + 4 e, ka2, c]; o[e + 2 kc] = Z[lane + 32 m]
    W = Y2.reshape(-1, 2, 4, 8, 4, 2)                                # [N, e, j, ka, c, 2]
    w = [(W[..., i, 0], W[..., i, 1]) for i in range(4)]
    R = _dft4(*w)                                                    # kc = 0..3, each [N, e, j, ka]
    R = np.stack([np.stack(c, -1) for c in R], -2)                   # [N, e, j, ka, kc, 2]
    o = R.transpose(0, 2, 3, 4, 1, 5).reshape(-1, 32, 8, 2)          # [N, lane, m, 2]
    # real-FFT untangle
    N = o.shape[0]
    P = np.zeros((N, 264), np.float32)
    lane = np.arange(32)
    pl = (32 - lane) & 31
    tw3 = T.tw3
    for mm in range(4):
        part = o[:, pl, 7 - mm].copy()
        part[:, 0] = o[:, 0, (8 - mm) & 7]
        pr, pi = part[..., 0], part[..., 1]
        ox, oy = o[:, :, mm, 0], o[:, :, mm, 1]
        er, ei = ox + pr, oy - pi
        qr, qi = oy + pi, pr - ox
        wx, wy = tw3[mm, :, 0], tw3[mm, :, 1]
        tr = fmaf32(qr, wx, -(qi * wy))
        ti = fmaf32(qi, wx, qr * wy)
        ar, ai, br, bi = er + tr, ei + ti, er - tr, ei - ti
        P[:, lane + 32 * mm] = F32(0.25) * fmaf32(ar, ar, ai * ai)
        P[:, (32 - lane) + 32 * (7 - mm)] = F32(0.25) * fmaf32(br, br, bi * bi)
    z = o[:, 0, 4]
    P[:, 128] = fmaf32(z[:, 0], z[:, 0], z[:, 1] * z[:, 1])
    return P[:, :N_BINS]


# ------------------------------------------------------------------------------------------------ mel, log, DCT
def mel_sums(P, T):
    """warp_log_mel before the log: S[N, 128] = rise part of band b (from the lane that owns interval b) + fall part."""
    P = np.asarray(P, np.float32)
    N = P.shape[0]
    Pp = np.zeros((N, 264), np.float32)
    Pp[:, :P.shape[1]] = P
    melp, mfirst = T.melp, T.mfirst
    fall = np.zeros((N, 4, 32), np.float32)
    rise = np.zeros((N, 4, 32), np.float32)
    tap0 = 0
    for j, nt in enumerate(MEL_TAPS):
        f = np.zeros((N, 32), np.float32)
        r = np.zeros((N, 32), np.float32)
        for i in range(nt):
            wt = melp[tap0 + i]
            v = Pp[:, mfirst[j] + i]
            f = fmaf32(wt[:, 0], v, f)
            r = fmaf32(wt[:, 1], v, r)
        fall[:, j], rise[:, j] = f, r
        tap0 += nt
    rr = np.zeros_like(rise)
    rr[:, :, 1:] = rise[:, :, :-1]
    rr[:, 1:, 0] = rise[:, :-1, 31]
    S = rr + fall                                                     # [N, j, lane] = band lane + 32 j
    return S.reshape(N, N_MELS)


def log_mel(P, T, log_fn=log_mel_standin):
    return np.asarray(log_fn(mel_sums(P, T)), np.float32)


def dct20(lm, T):
    """warp_dct20 over floored log-mel rows [N, 128] -> MFCC [N, 20]."""
    x = np.asarray(lm, np.float32).reshape(-1, 4, 32)                # [N, j, lane]
    N = x.shape[0]
    rev = 31 - np.arange(32)
    y3, y2 = x[:, 3, rev], x[:, 2, rev]
    s0, d0, s1, d1 = x[:, 0] + y3, x[:, 0] - y3, x[:, 1] + y2, x[:, 1] - y2
    half = np.arange(32) >= 16
    partner = np.arange(32) ^ 16
    v = [np.where(half, d0, s0), np.where(half, d1, s1),
         np.where(half, d0[:, partner], s0[:, partner]), np.where(half, d1[:, partner], s1[:, partner])]
    dd = T.dct
    acc = np.zeros((N, 32, 10), np.float32)
    for r in range(40):                                              # row[q] order: flat index r = 4 q + i
        m, sl = r % 10, r // 10
        acc[:, :, m] = fmaf32(dd[:, r], v[sl], acc[:, :, m])
    A = acc.reshape(N, 2, 16, 10)                                    # [N, half, lane & 15, m]
    A = A[:, :, :8] + A[:, :, 8:]                                    # halving butterfly over lane bits 3, 2, 1, 0
    A = A[:, :, :4] + A[:, :, 4:]
    A = A[:, :, :2] + A[:, :, 2:]
    A = A[:, :, 0] + A[:, :, 1]                                      # [N, half, m]
    out = np.empty((N, N_MFCC), np.float32)
    out[:, 0::2] = A[:, 0]
    out[:, 1::2] = A[:, 1]
    return out


# ------------------------------------------------------------------------------------------------ segment
def segment_frames(y, T, log_fn=log_mel_standin, preemphasis=0.0):
    """One segment (float32 samples as K3 reads them) -> (MFCC rows [F, 20] after the top_db floor, un-floored log-mel
    [F, 128], floor).  Frames are computed in chunks so that long segments stay within memory."""
    y = np.asarray(y, np.float32)
    F = 1 + len(y) // HOP
    lm = np.empty((F, N_MELS), np.float32)
    for c in range(0, F, 2048):
        t = np.arange(c, min(F, c + 2048))
        lm[t] = log_mel(power_spectrum(frame_samples(y, preemphasis, t), T), T, log_fn)
    floor = F32(lm.max()) - F32(80.0)
    return dct20(np.maximum(lm, floor), T), lm, floor


def pool(mf, n_mfcc=N_MFCC):
    """segment_features phase D (and fq_finish): 14 strided partials, each a frame-order sum, its mean, its M2 about that
    mean; the partials merged in order (Chan et al.) -> (mean[20], std[20]), zero at and above n_mfcc."""
    mf = np.asarray(mf, np.float32)
    F = mf.shape[0]
    n = F32(0.0)
    mean = np.zeros(N_MFCC, np.float32)
    M2 = np.zeros(N_MFCC, np.float32)
    for w in range(min(SEG_WARPS, F)):
        rows = mf[w::SEG_WARPS]
        s = np.zeros(N_MFCC, np.float32)
        for r in rows:
            s = s + r
        mu = s / F32(len(rows))
        m2 = np.zeros(N_MFCC, np.float32)
        for r in rows:
            d = r - mu
            m2 = fmaf32(d, d, m2)
        cw = F32((F - w + SEG_WARPS - 1) // SEG_WARPS)
        delta = mu - mean
        nn = F32(n + cw)
        mean = fmaf32(delta, F32(cw / nn), mean)
        M2 = M2 + fmaf32(delta * delta, F32(F32(n * cw) / nn), m2)
        n = nn
    std = np.sqrt(M2 / F32(F)).astype(np.float32)
    mean = np.asarray(mean, np.float32).copy()
    mean[n_mfcc:] = 0.0
    std[n_mfcc:] = 0.0
    return mean, std


def segment(y, T, log_fn=log_mel_standin, preemphasis=0.0, n_mfcc=N_MFCC):
    """-> dict(frames = floored MFCC rows [F, 20], lm = un-floored log-mel [F, 128], floor, mean, std)."""
    mf, lm, floor = segment_frames(y, T, log_fn, preemphasis)
    mean, std = pool(mf, n_mfcc)
    return dict(frames=mf, lm=lm, floor=floor, mean=mean, std=std)


def score(tm, ts, mean, std):
    """similarity_score: serial fmaf dots over all 20 components, per pair q = f32((double) uv / sqrt((double)
    fl(uu vv))), d = clip(1 - q, 0, 2) (NaN kept), (1 - dm) 0.7 + (1 - ds) 0.3, p = 100 c, p sqrtf(p) / 10."""
    from .dense_model import score_features
    return score_features(tm, ts, np.atleast_2d(mean), np.atleast_2d(std), N_MFCC)[0]


def best_template(scores, t0=0):
    """The queue forms' pick over a stream's template scores: NaN never wins, the first best wins -> (score, slot)."""
    best, arg = F32(np.nan), (t0 if len(scores) else -1)
    for k, s in enumerate(np.asarray(scores, np.float32)):
        if not np.isnan(s) and (np.isnan(best) or s > best):
            best, arg = s, t0 + k
    return best, arg
