// K4 — dense_score: the level-2 score of WordMatcher.calculate_similarity
// (/root/reference/easywakeword/wakeword.py:591-625) for a template-length window at EVERY 10 ms hop
// of every stream and for every template of a set (SURVEY §8(a) row A9; usage shape of
// examples/tune_threshold.py:86-116 at hop granularity; BASELINE configs[1], [4]).  One CTA per stream walks the
// requested hops in sub-chunks of DH hops and never writes an intermediate to global memory.
//
// Window at hop h for template k (L samples, n = ceil(L/160), F = 1 + L/160 frames):
//     x[160 (h - n) : 160 (h - n) + L]      — the latest template-length window that starts on the
// hop grid and is complete at hop h (oracle.ewk_oracle.dense_window).  Handing that window to librosa
// means window-local zero-pad centring and a window-local top_db floor, so per window:
//   * frames t = 2 .. t_hi lie fully inside the window: they are frames of the STREAM grid
//     (centre 160 g, g = j + t, j = h - n), shared by all windows and all templates          -> ring G[g];
//   * frames t = 0, 1 (left edge) see zeros before the window start.  They depend on the START j only, not on
//     the template: computed once per start and shared by every template                    -> rings LE0[j], LE1[j];
//   * frames t = t_hi+1 .. F-1 (right edge, 1 or 2) see zeros after the window end 160 h - delta, delta = 160 n - L:
//     stream-grid frame h - goff cut at the window end.  Templates with the same delta share them -> RE[u][hop];
//   * floor = (max log-mel over the window's frames) - 80 (librosa.power_to_db(top_db=80)).  Frames are computed
//     un-floored together with their log-mel min / max; a window none of whose frames reaches below its floor is
//     scored from the un-floored rows, the others take the floored paths below.
//
// Statistics.  mean / std over the F frames of a window are formed from EXACT integer sums: every MFCC value
// is quantised once to q = rint(x * 2^16) (|x| < 2^11: q fits 28 bits) and S1 = sum q, S2 = sum q^2 are 64-bit integers,
// so consecutive windows are related by S(h) = S(h-1) + q(new row) - q(old row) with no drift and no dependence on
// where a request is cut into calls or sub-chunks: the 32 hops of a half sub-chunk are the 32 lanes of a warp, which
// forms the first window's sums directly, the others by an inclusive scan of the row differences, one coefficient at
// a time.  mean = S1 / (F 2^16), var = (S2 - S1^2 / F) / (F 2^32) in double, rounded once to float32 (quantisation
// error <= 7.6e-6 absolute per value: below float32 resolution of the pooled statistics the reference forms).  The
// template's own features for this kernel (TemplateFeat.dmean / dstd) come from the same arithmetic on the template's
// frames, so a window that IS the template scores exactly 100.0.
//
// Floors.  Consecutive windows share their loudest frame, hence their floor, and so do windows of different templates
// that contain the same event: the distinct floor values alive in a stream are few.  Up to DENSE_WAYS of them own a
// "way": a copy G2[way] of the stream-grid rows that floor changes (each recomputed once, tagged with the floor), over
// which the same sliding sums run.  Windows whose EDGE frames are floored, or whose floor found no free way, are
// summed frame by frame by one warp each.
//
// Phases per sub-chunk (tasks are taken from shared-memory counters, one warp per task):
//   A   frames: new stream-grid rows, left-edge rows of new starts, right-edge rows of every (delta group, hop)  | barrier
//   B   per (template, half, quarter of the frame range): partial window max / min                    (B0)
//       per (template, half, coefficient): un-floored window sums -> (mean, std) for 32 hops          (B1)      | barrier
//   S   per (template, half): floor test, cosine score of the un-floored windows, way of the floored ones        | barrier
//   -- only when a window is floored --
//   C   stream-grid rows floored by each way's floor -> G2[way]                                                   | barrier
//   D   per (template, half, way, coefficient): window sums over G2[way] | G  -> (mean, std)          (D1)
//       frame-by-frame windows, one warp each                                                         (D slow)   | barrier
//   E   per (template, half): cosine score of the floored windows
#pragma once
#include <climits>

#include "ewk_segment.cuh"
#include "ewk_streams.cuh"

namespace ewk {

constexpr int DENSE_MAX_T = 8;         // templates per launch
constexpr int DENSE_MAX_RE = 2 * DENSE_MAX_T;   // distinct right-edge frames per hop
constexpr int DENSE_MIN_L = 640;       // shorter templates would make a frame both left- and right-masked
constexpr int DENSE_MAX_L = MAX_SEG;   // 3.0 s: the reference's own segment cap (wakeword.py:1114-1118)
constexpr int ROW = N_MFCC + 3;        // mfcc[20], log-mel min, log-mel max, pad: odd stride, lanes that walk rows hit 32 banks
constexpr int R_MIN = N_MFCC, R_MAX = N_MFCC + 1;
constexpr int DENSE_KEEP = 304;        // stream-grid rows carried from one call to the next (>= frames of the longest window)
constexpr int B0_PARTS = 4;            // the frame range of a window is scanned for its max / min in this many tasks
constexpr int DENSE_WAYS = 8;          // floor values with a cached copy of the rows they change
constexpr int TAG_NONE = 0x7fc00001;   // matches no floor
// control words: [0] phase-A tasks [1] phase-B tasks [2] phase-S tasks [3] frame-by-frame windows [4] phase-D tasks [5] way windows
// [6] phase-E tasks [7] (template, half, way) combinations with way windows; [8 + k] ring row of grid frame hs - n_k;
// [16 + k] LE slot of start hs - n_k; [24 + w] floor bits of way w; [32 + w] way used in this sub-chunk;
// [40 + 2 k + half] ways used by the windows of (template, half); [56 ...] the combinations: (k * 2 + half) * DENSE_WAYS + w
constexpr int DENSE_CTL = 56 + 2 * DENSE_MAX_T * DENSE_WAYS;

struct DenseTmplDev {
    int L, n, F, t_hi, r, slot;        // r = F - 1 - t_hi right-edge frames
    int re_u[2];                       // right-edge frame e of this template: row RE[re_u[e] * DH + hl]
    double inv_f;                      // 1 / F (IEEE double division: the same bits on host and device)
};

// One row of a ragged call (ewk_dense_scores_streams / ewk_dense_ready): CTA x scores stream `stream` at hops
// [hop0, hop0 + n_hops) into out[out, out + n_hops T), laid out [n_hops][T]
struct DenseRow {
    long long hop0, out;
    int stream, n_hops;
};

struct DenseArgs {
    long long hop0;                    // first hop scored (hop h <-> 160 h samples of the stream); uniform instance only
    int n_hops;
    int T;
    int DH;                            // hops per sub-chunk (32 or 64)
    int DG;                            // rows of the grid-frame ring (>= DH + n_max + 2)
    int DLE;                           // starts held by the left-edge rings (>= DH + n_max - n_min)
    int n_re_u;                        // distinct right-edge frames per hop
    int n_min, n_max;                  // shortest / longest window in hops
    int g_back;                        // min over templates of n - t_hi: the newest grid row a sub-chunk needs is hop - g_back
    int pad;
    // distinct right-edge frame u: stream-grid frame (hop - goff) with the samples from 160 hop - delta on zeroed; rep / rep_e:
    // a template and edge index that use it (window view of the generic loader); n_first: the shortest window using it
    int re_goff[DENSE_MAX_RE], re_delta[DENSE_MAX_RE], re_rep[DENSE_MAX_RE], re_rep_e[DENSE_MAX_RE], re_nfirst[DENSE_MAX_RE];
    DenseTmplDev t[DENSE_MAX_T];
    float* out;                        // uniform: [n_streams][n_hops][T]; rows: packed as their descriptors say
    const DenseRow* rows;              // ROWS instance: one descriptor per CTA
    float* g2;                         // [n_streams][DENSE_WAYS][DG][20]: grid rows floored with a way's floor (tags in shared memory)
    // carry-over between consecutive calls: the newest stream-grid rows of every stream (functions of the PCM only)
    float* keep_rows;                  // [n_streams][DENSE_KEEP][ROW], row of grid frame g at g % DENSE_KEEP
    long long* keep_end;               // [n_streams][2]: grid frames [keep_end[2s], keep_end[2s+1]) are stored (0, 0: nothing)
};

__host__ __device__ inline size_t dense_smem_bytes(int nwarps, int T, int DH, int DG, int DLE, int n_re_u) {
    const size_t words = (size_t)nwarps * SCR_WARP + (size_t)2 * T * N_MFCC * DH + (size_t)DG * ROW + (size_t)2 * DLE * ROW +
                         (size_t)n_re_u * DH * ROW + (size_t)2 * T * DH * B0_PARTS + (size_t)2 * T * DH + (size_t)nwarps * N_MFCC +
                         (size_t)DENSE_WAYS * DG + (size_t)2 * T * DH + DENSE_CTL;
    return sizeof(FrameTables) + 4 * words;
}

// ---- exact integer statistics -------------------------------------------------------------------------------
__device__ __forceinline__ int quant16(float x) {           // rint(x * 2^16) of a row value (|x| <= 2047: clamped where rows are written)
    return __float2int_rn(x * 65536.0f);
}

// (S1, S2) over F frames -> mean, std (ddof 0) as float32; the same function serves windows and templates.
// Rows that are all equal (digital silence, a constant signal) have variance exactly 0, but once S2 passes 2^53 the
// double formula leaves a rounding residue there: such a window would get a std, and a score, where the reference's
// std is 0 and its cosine 0 / 0 = NaN.  F S2 == S1^2 (exact in 128 bits) detects them.
__device__ __forceinline__ void dense_stats(long long S1, long long S2, int F, double invf, float& mean, float& sd) {
    const double s1 = (double)S1, s2 = (double)S2;
    mean = (float)(s1 * invf * (1.0 / 65536.0));
    const double var = (s2 - s1 * s1 * invf) * invf * (1.0 / 4294967296.0);
    const bool flat = (__int128)S1 * S1 == (__int128)F * S2;
    sd = flat ? 0.f : sqrtf(fmaxf((float)var, 0.f));
}

// Template features for this kernel: the integer statistics of the template's own MFCC frames (K3's frames_out).
__global__ void dense_template_features_kernel(const float* __restrict__ frames, int F, int n_mfcc, float* __restrict__ out40) {
    const int lane = threadIdx.x;
    long long S1 = 0, S2 = 0;
    if (lane < N_MFCC)
        for (int t = 0; t < F; t++) {
            const int q = quant16(fminf(fmaxf(frames[(size_t)t * N_MFCC + lane], -2047.f), 2047.f));   // K3's rows are not clamped
            S1 += q;
            S2 += (long long)q * q;
        }
    float mean, sd;
    dense_stats(S1, S2, F, 1.0 / (double)F, mean, sd);
    if (lane < N_MFCC) {
        out40[lane] = lane < n_mfcc ? mean : 0.f;
        out40[N_MFCC + lane] = lane < n_mfcc ? sd : 0.f;
    }
}

// ---- frame loaders for ring views (no pre-emphasis): frame sample m = 2 lane + 64 a, pairs from one aligned word -----
// p0: ring position of frame sample 0 (even; may be negative by less than P).  Samples m < LO and m >= hi are zero
// (window-local zero padding); LO is a compile-time multiple of 32 so that fully masked words are never loaded.
template <int LO, bool RIGHT>
__device__ __forceinline__ void dense_load_pairs(const void* ring_s, int fmt, int P, int p0, int hi, int lane, float2 (&x)[8]) {
    if (p0 < 0) p0 += P;
    const int w0 = (p0 >> 1) + lane, WP = P >> 1;
    const bool wrap = p0 + N_FFT > P;                           // warp-uniform
#pragma unroll
    for (int a = 0; a < 8; a++) {
        if (64 * a + 64 <= LO) { x[a] = make_float2(0.f, 0.f); continue; }
        int w = w0 + 32 * a;
        if (wrap && w >= WP) w -= WP;
        float2 v;
        if (fmt == 1) {
            const unsigned u = __ldg(reinterpret_cast<const unsigned*>(ring_s) + w);
            v = make_float2((float)(short)(u & 0xffff) * (1.0f / 32768.0f), (float)((int)u >> 16) * (1.0f / 32768.0f));
        } else v = __ldg(reinterpret_cast<const float2*>(ring_s) + w);
        const int m = 2 * lane + 64 * a;
        if (64 * a < LO && m < LO) v = make_float2(0.f, 0.f);   // LO is even: a pair is masked as a whole
        if (RIGHT) { if (m >= hi) v.x = 0.f; if (m + 1 >= hi) v.y = 0.f; }
        x[a] = v;
    }
}

enum : int { FR_GRID = 0, FR_LE0 = 1, FR_LE1 = 2, FR_RE = 3 };

// One frame of the dense kernel -> row (20 MFCCs [+ min, max when stats]).  `pos` is the ring position of the frame's
// sample 0 for grid frames, of the WINDOW's sample 0 for edge frames (t: frame index in the window, L: window length).
template <bool PRE>
__device__ __noinline__ void dense_frame(int kind, const void* ring_s, int fmt, int P, int pos, int t, int L, float pre,
                                         const FrameTables& ft, float* scr, int lane, float floor_db,
                                         float* __restrict__ row, bool stats) {
    float2 x[8];
    if (PRE) {
        // generic loader through a window view (pre-emphasis needs x[n-1] and the window's own initial state)
        PcmReader rd;
        rd.f = fmt == 0 ? (const float*)ring_s : nullptr;
        rd.q = fmt == 1 ? (const short*)ring_s : nullptr;
        rd.ring = P; rd.pre = pre;
        int f0;
        if (kind == FR_GRID) {                                   // view starts 2 samples early: no window starts there
            int p = pos - 2; if (p < 0) p += P;
            rd.start = p; rd.len = N_FFT + 2; f0 = 2;
        } else {
            rd.start = pos; rd.len = L; f0 = t * HOP - N_FFT / 2;
        }
        load_frame_pairs_at<true>(rd, f0, lane, x);
    } else {
        if (kind == FR_GRID) dense_load_pairs<0, false>(ring_s, fmt, P, pos, N_FFT, lane, x);
        else if (kind == FR_LE0) dense_load_pairs<256, false>(ring_s, fmt, P, pos - 256, N_FFT, lane, x);
        else if (kind == FR_LE1) dense_load_pairs<96, false>(ring_s, fmt, P, pos - 96, N_FFT, lane, x);
        else {
            int p = pos + t * HOP - N_FFT / 2; if (p >= P) p -= P;
            dense_load_pairs<0, true>(ring_s, fmt, P, p, L - (t * HOP - N_FFT / 2), lane, x);
        }
    }
    float mn, mx;
    warp_frame_mfcc(x, ft, scr, lane, floor_db, row, mn, mx);
    if (stats && lane == 0) { row[R_MIN] = mn; row[R_MAX] = mx; }
    // rows are clamped once here (|MFCC| < 2^11 holds for any audio below ~1e4 x full scale), so quant16 needs no clamp
    __syncwarp();
    if (lane < N_MFCC) row[lane] = fminf(fmaxf(row[lane], -2047.f), 2047.f);
}

__device__ __forceinline__ int next_task(int* counter, int lane) {
    int t = 0;
    if (lane == 0) t = atomicAdd(counter, 1);
    return __shfl_sync(FULL, t, 0);
}

__device__ __forceinline__ int wrap1(int r, int n) { return r >= n ? r - n : r; }

// ROWS = false: CTA s scores stream s at the call's hops [A.hop0, A.hop0 + A.n_hops).  ROWS = true: CTA x takes
// descriptor A.rows[x] (its stream, hop range and output block); the body is the same.
template <bool PRE, bool ROWS>
__global__ void __launch_bounds__(1024, 1)
dense_score_kernel(const DeviceTables* __restrict__ T, BankView B, const TemplateFeat* __restrict__ tmpl, DenseArgs A) {
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5, nthr = blockDim.x;
    const int DH = A.DH, DG = A.DG, DLE = A.DLE, NT = A.T;
    FrameTables* ft = reinterpret_cast<FrameTables*>(smem);
    float* scratch = smem + sizeof(FrameTables) / sizeof(float);
    float2* MS = reinterpret_cast<float2*>(scratch + (size_t)nwarps * SCR_WARP);   // [T][20][DH] (mean, std) of a coefficient
    float* G = reinterpret_cast<float*>(MS + (size_t)NT * N_MFCC * DH);            // [DG][ROW], grid frame g at g % DG
    float* LE0 = G + (size_t)DG * ROW;                           // [DLE][ROW], start j at j % DLE: frame t = 0
    float* LE1 = LE0 + (size_t)DLE * ROW;                        //                                  frame t = 1
    float* RE = LE1 + (size_t)DLE * ROW;                         // [n_re_u][DH][ROW]
    float* PM = RE + (size_t)A.n_re_u * DH * ROW;                // [T][B0_PARTS][2][DH] partial (max over all frames, min over grid frames)
    float* WFL = PM + (size_t)2 * NT * DH * B0_PARTS;            // [T][DH] floor of a floored window, +INF otherwise
    float* EMN = WFL + (size_t)NT * DH;                          // [T][DH] min over the window's edge frames
    float* patchb = EMN + (size_t)NT * DH;                       // [nwarps][20]
    int* g2tag = reinterpret_cast<int*>(patchb + (size_t)nwarps * N_MFCC);          // [DENSE_WAYS][DG] floor bits of the row's copy
    int* FLIST = g2tag + DENSE_WAYS * DG;                        // [T][DH] frame-by-frame windows: k * DH + hl
    int* WAY = FLIST + NT * DH;                                  // [T][DH] way of a floored window (-1: none)
    int* ctl = WAY + NT * DH;                                    // [DENSE_CTL]
    int* WAYF = ctl + 24;
    int* WAYU = ctl + 32;
    int* WAYMASK = ctl + 40;
    int* COMBO = ctl + 56;
    const int s = ROWS ? A.rows[blockIdx.x].stream : blockIdx.x;
    // the row's hops are re-read where they are used: values kept live across the kernel would cost registers
    auto hop0 = [&]() -> long long { return ROWS ? A.rows[blockIdx.x].hop0 : A.hop0; };
    auto n_hops = [&]() -> int { return ROWS ? A.rows[blockIdx.x].n_hops : A.n_hops; };
    // score of hop (hs + hl), template k
    auto out_at = [&](long long hs, int hl, int k) -> float* {
        if (ROWS) return A.out + A.rows[blockIdx.x].out + (size_t)(hs - hop0() + hl) * NT + k;
        return A.out + ((size_t)s * A.n_hops + (size_t)(hs - A.hop0 + hl)) * NT + k;
    };
    copy_frame_tables(*ft, T, tid, nthr);
    float* scr = scratch + warp * SCR_WARP;
    float* patch = patchb + warp * N_MFCC;
    for (int i = tid; i < DENSE_WAYS * DG; i += nthr) g2tag[i] = TAG_NONE;
    if (tid < DENSE_CTL) ctl[tid] = (tid >= 24 && tid < 24 + DENSE_WAYS) ? TAG_NONE : 0;

    const size_t esz = B.fmt == 1 ? 2 : 4;
    const void* ring_s = (const char*)B.ring + (size_t)s * B.P * esz;
    const int fmt = B.fmt, P = B.P;
    float* G2 = A.g2 + (size_t)s * DENSE_WAYS * DG * N_MFCC;
    __syncthreads();
    const float pre = PRE ? ft->preemph : 0.f;
    const int n_mfcc = ft->n_mfcc;

    long long g_done = LLONG_MIN, g_valid_lo = LLONG_MAX;        // ring G holds rows [max(g_valid_lo, g_done - DG), g_done)
    long long le_done = LLONG_MIN;                               // left-edge rows of starts < le_done are in the LE rings
    {
        // rows computed by the previous call are reused when this call continues where it stopped: the history of
        // the first window (up to n_max frames) is loaded instead of recomputed
        long long need_lo = hop0() - A.n_max + 1;
        if (need_lo < 2) need_lo = 2;
        const long long klo = A.keep_rows ? A.keep_end[2 * s] : 0, kend = A.keep_rows ? A.keep_end[2 * s + 1] : 0;
        if (klo <= need_lo && need_lo < kend && kend - need_lo <= DG) {
            const float* kr = A.keep_rows + (size_t)s * DENSE_KEEP * ROW;
            const int cnt = (int)(kend - need_lo);
            for (int i = tid; i < cnt * ROW; i += nthr) {
                const long long g = need_lo + i / ROW;
                G[(size_t)(g % DG) * ROW + i % ROW] = kr[(size_t)(g % DENSE_KEEP) * ROW + i % ROW];
            }
            g_done = kend;
            g_valid_lo = need_lo;
        }
        __syncthreads();
    }

    // value of ring row r, coefficient c, as way w's floor f sees it (the floored copy where the floor changes the row)
    auto way_value = [&](int w, float f, int r, int c) -> float {
        return G[r * ROW + R_MIN] < f ? __ldcg(G2 + ((size_t)w * DG + r) * N_MFCC + c) : G[r * ROW + c];
    };

    // (mean, std) of coefficient c for the 32 hops of half hh of template k from exact integer window sums over the
    // stream-grid rows as way w sees them (w < 0: un-floored) plus the window's un-floored edge rows; lanes = hops
    auto window_sums = [&](int k, int c, int hh, int nh, long long hs, int w, float f, bool& valid_o, float& mean_o, float& sd_o) {
        const DenseTmplDev& tp = A.t[k];
        const int hl = 32 * hh + lane;
        const bool valid = hl < nh && hs + hl - tp.n >= 0;
        valid_o = valid;
        mean_o = sd_o = 0.f;
        const unsigned vm = __ballot_sync(FULL, valid);
        if (vm == 0) return;
        const int l0 = __ffs(vm) - 1;                                   // first valid hop; valid hops are contiguous
        const int rb = ctl[8 + k] + 32 * hh;                            // ring row of "grid frame" j of lane 0 (< 2 DG)
        auto val = [&](int r) -> int { return quant16(w < 0 ? G[r * ROW + c] : way_value(w, f, r, c)); };
        // base: the first valid window's interior frames t = 2 .. t_hi, lanes = rows
        long long b1 = 0, b2 = 0;
        {
            int r = rb + l0 + 2 + lane;
            while (r >= DG) r -= DG;
            for (int t = 2 + lane; t <= tp.t_hi; t += 32) {
                const int v = val(r);
                b1 += v; b2 += (long long)v * v;
                r += 32; while (r >= DG) r -= DG;
            }
#pragma unroll
            for (int o = 16; o; o >>= 1) { b1 += __shfl_xor_sync(FULL, b1, o); b2 += __shfl_xor_sync(FULL, b2, o); }
        }
        // differences: window j (lane > l0) = window j - 1 + row (j + t_hi) - row (j + 1)
        long long d1 = 0, d2 = 0;
        if (valid && lane > l0) {
            int rin = rb + lane + tp.t_hi, rout = rb + lane + 1;
            while (rin >= DG) rin -= DG;
            while (rout >= DG) rout -= DG;
            const int vin = val(rin), vout = val(rout);
            d1 = (long long)vin - vout;
            d2 = (long long)vin * vin - (long long)vout * vout;
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long u1 = __shfl_up_sync(FULL, d1, o), u2 = __shfl_up_sync(FULL, d2, o);
            if (lane >= o) { d1 += u1; d2 += u2; }
        }
        if (valid) {
            long long S1 = b1 + d1, S2 = b2 + d2;
            const int sl = wrap1(ctl[16 + k] + hl, DLE);
            int v = quant16(LE0[sl * ROW + c]);  S1 += v; S2 += (long long)v * v;
            v = quant16(LE1[sl * ROW + c]);      S1 += v; S2 += (long long)v * v;
            for (int e = 0; e < tp.r; e++) {
                v = quant16(RE[(tp.re_u[e] * DH + hl) * ROW + c]);
                S1 += v; S2 += (long long)v * v;
            }
            dense_stats(S1, S2, tp.F, tp.inv_f, mean_o, sd_o);
        }
    };

    // scipy cosine of (template mean, window mean) and (template std, window std) from MS, serial float32 dot products
    auto score_window = [&](int k, int hl, const TemplateFeat& tf) -> float {
        float uvm = 0.f, uum = 0.f, vvm = 0.f, uvs = 0.f, uus = 0.f, vvs = 0.f;
        for (int c = 0; c < n_mfcc; c++) {
            const float2 ms = MS[((size_t)k * N_MFCC + c) * DH + hl];
            const float tm = tf.dmean[c], ts = tf.dstd[c];
            uvm = fmaf(tm, ms.x, uvm); uum = fmaf(tm, tm, uum); vvm = fmaf(ms.x, ms.x, vvm);
            uvs = fmaf(ts, ms.y, uvs); uus = fmaf(ts, ts, uus); vvs = fmaf(ms.y, ms.y, vvs);
        }
        return score_from_dots(uvm, uum, vvm, uvs, uus, vvs);
    };

    for (long long hs = hop0(); hs < hop0() + n_hops(); hs += DH) {
        const int nh = (int)min((long long)DH, hop0() + n_hops() - hs);
        const int n_half = (nh + 31) >> 5;
        // ================================================================ phase A: frames of this sub-chunk
        // stream-grid rows [g_from, g_hi]: every template's windows of these hops reach back to hs - n + 1 (the row a
        // sliding difference removes) and forward to hop - (n - t_hi)
        long long g_lo = hs - A.n_max + 1;
        if (g_lo < 2) g_lo = 2;                                   // grid frame g needs samples from 160 g - 256 >= 0
        const long long g_hi = hs + nh - 1 - A.g_back;
        const long long g_from = max(g_lo, g_done);
        if (g_valid_lo == LLONG_MAX) g_valid_lo = g_from;
        const int n_g = (int)max(0LL, g_hi - g_from + 1);
        // left-edge rows of the starts these hops use: [hs - n_max, hs + nh - n_min), those not yet in the rings
        long long le_lo = hs - A.n_max;
        if (le_lo < 0) le_lo = 0;
        const long long le_hi = hs + nh - A.n_min;               // exclusive
        const long long le_from = max(le_lo, le_done);
        const int n_le = (int)max(0LL, le_hi - le_from);
        const int n_re = A.n_re_u * nh;                          // enumerated as (distinct right-edge frame, hop slot)
        // 32-bit bases for this sub-chunk: ring position of sample 160 * hs, ring rows / slots of the first new frames
        const int hs_pos = (int)((160 * hs) % P);
        const int gfrom_row = n_g > 0 ? (int)(g_from % DG) : 0;
        const int gfrom_rel = (int)(g_from - hs), lefrom_rel = (int)(le_from - hs);
        const int lefrom_slot = n_le > 0 ? (int)(le_from % DLE) : 0;
        if (tid == 0) { ctl[1] = 0; ctl[2] = 0; ctl[3] = 0; ctl[4] = 0; ctl[5] = 0; ctl[6] = 0; ctl[7] = 0; }
        if (tid < NT) {
            // per template: ring row of grid frame (hs - n) and LE slot of start (hs - n), both possibly "negative" frames
            const long long j0 = hs - A.t[tid].n;
            ctl[8 + tid] = (int)(((j0 % DG) + DG) % DG);
            ctl[16 + tid] = (int)(((j0 % DLE) + DLE) % DLE);
            WAYMASK[2 * tid] = 0; WAYMASK[2 * tid + 1] = 0;
        }
        if (tid >= 64 && tid < 64 + DENSE_WAYS) {                 // a way nobody used in the previous sub-chunk is free again
            const int w = tid - 64;
            if (!WAYU[w]) WAYF[w] = TAG_NONE;
            WAYU[w] = 0;
        }
        const int n_tasks_a = n_g + 2 * n_le + n_re;
        for (int job = next_task(ctl + 0, lane); job < n_tasks_a; job = next_task(ctl + 0, lane)) {
            if (job < n_g) {
                int pos = hs_pos + 160 * (gfrom_rel + job) - N_FFT / 2;          // |offset| < P: one wrap
                if (pos < 0) pos += P; else if (pos >= P) pos -= P;
                const int r = wrap1(gfrom_row + job, DG);
                if (lane < DENSE_WAYS) g2tag[lane * DG + r] = TAG_NONE;
                dense_frame<PRE>(FR_GRID, ring_s, fmt, P, pos, 0, 0, pre, *ft, scr, lane, -INFINITY, G + r * ROW, true);
            } else if (job < n_g + 2 * n_le) {
                const int q = job - n_g, i = q >> 1, e = q & 1;
                int pos = hs_pos + 160 * (lefrom_rel + i);                      // window start
                if (pos < 0) pos += P; else if (pos >= P) pos -= P;
                const int sl = wrap1(lefrom_slot + i, DLE);
                // window length for the generic (pre-emphasis) view: any L >= 640 gives the same left-edge frames
                dense_frame<PRE>(e ? FR_LE1 : FR_LE0, ring_s, fmt, P, pos, e, DENSE_MIN_L, pre, *ft, scr, lane, -INFINITY,
                                 (e ? LE1 : LE0) + sl * ROW, true);
            } else {
                const int q = job - n_g - 2 * n_le;
                const int u = q / nh, hl = q - u * nh;
                if (hs + hl - A.re_nfirst[u] < 0) continue;                     // every window that uses it starts before the stream
                // through the window of a template that uses it (the frame itself depends on (goff, delta) only)
                const DenseTmplDev& tp = A.t[A.re_rep[u]];
                int pos = hs_pos + 160 * (hl - tp.n);
                if (pos < 0) pos += P; else if (pos >= P) pos -= P;
                dense_frame<PRE>(FR_RE, ring_s, fmt, P, pos, tp.t_hi + 1 + A.re_rep_e[u], tp.L, pre, *ft, scr, lane, -INFINITY,
                                 RE + (u * DH + hl) * ROW, true);
            }
        }
        g_done = g_hi + 1;
        le_done = le_hi;
        __syncthreads();

        // ================================================================ phase B: window max / min and un-floored window sums
        if (tid == 0) ctl[0] = 0;
        const int n_b0 = NT * n_half * B0_PARTS, n_b1 = NT * n_half * n_mfcc;
        for (int job = warp; job < n_b0 + n_b1; job += nwarps) {                      // uniform tasks: a static share
            if (job < n_b0) {
                // ---- B0: partial max / min over a quarter of the window's frames, lanes = hops
                const int p = job % B0_PARTS, kh = job / B0_PARTS, hh = kh % n_half, k = kh / n_half;
                const DenseTmplDev& tp = A.t[k];
                const int hl = 32 * hh + lane;
                const bool valid = hl < nh && hs + hl - tp.n >= 0;
                float wmax = -INFINITY, wmin = INFINITY;
                if (valid) {
                    const int cnt = tp.t_hi - 1;                                // grid frames t = 2 .. t_hi
                    const int ta = 2 + (cnt * p) / B0_PARTS, tb = 2 + (cnt * (p + 1)) / B0_PARTS;
                    int r = wrap1(ctl[8 + k] + hl + ta, DG);
                    for (int t = ta; t < tb; t++) {
                        wmax = fmaxf(wmax, G[r * ROW + R_MAX]);
                        wmin = fminf(wmin, G[r * ROW + R_MIN]);
                        if (++r == DG) r = 0;
                    }
                    if (p == 0) {
                        const int sl = wrap1(ctl[16 + k] + hl, DLE);
                        wmax = fmaxf(wmax, fmaxf(LE0[sl * ROW + R_MAX], LE1[sl * ROW + R_MAX]));
                        float emin = fminf(LE0[sl * ROW + R_MIN], LE1[sl * ROW + R_MIN]);
                        for (int e = 0; e < tp.r; e++) {
                            const float* re = RE + (tp.re_u[e] * DH + hl) * ROW;
                            wmax = fmaxf(wmax, re[R_MAX]);
                            emin = fminf(emin, re[R_MIN]);
                        }
                        EMN[k * DH + hl] = emin;
                    }
                }
                if (hl < DH) {
                    float* pm = PM + (size_t)((k * B0_PARTS + p) * 2) * DH + hl;
                    pm[0] = wmax; pm[DH] = wmin;
                }
            } else {
                // ---- B1: (mean, std) of one coefficient for the 32 hops of a half, un-floored rows
                const int q = job - n_b0;
                const int c = q % n_mfcc, kh = q / n_mfcc, hh = kh % n_half, k = kh / n_half;
                bool valid; float mean, sd;
                window_sums(k, c, hh, nh, hs, -1, 0.f, valid, mean, sd);
                if (32 * hh + lane < DH) MS[((size_t)k * N_MFCC + c) * DH + 32 * hh + lane] = make_float2(mean, sd);
            }
        }
        __syncthreads();

        // ================================================================ phase S: floors, scores of un-floored windows
        for (int job = warp; job < NT * n_half; job += nwarps) {
            const int hh = job % n_half, k = job / n_half;
            const DenseTmplDev& tp = A.t[k];
            const int hl = 32 * hh + lane;
            const TemplateFeat& tf = tmpl[tp.slot];
            if (hl >= nh) continue;
            float* outp = out_at(hs, hl, k);
            WAY[k * DH + hl] = -1;
            if (hs + hl - tp.n < 0 || !tf.valid) { *outp = __int_as_float(0x7fc00000); WFL[k * DH + hl] = INFINITY; continue; }
            float wmax = -INFINITY, wmin = INFINITY;
#pragma unroll
            for (int p = 0; p < B0_PARTS; p++) {
                const float* pm = PM + (size_t)((k * B0_PARTS + p) * 2) * DH + hl;
                wmax = fmaxf(wmax, pm[0]); wmin = fminf(wmin, pm[DH]);
            }
            const float floor_db = wmax - 80.0f;                                // librosa.power_to_db(top_db=80) on this window
            const float emin = EMN[k * DH + hl];
            if (fminf(wmin, emin) < floor_db) {                                 // some frame reaches below the floor
                WFL[k * DH + hl] = floor_db;
                // the way that holds this floor, or a free one: its copy serves the stream-grid rows the floor changes
                int way = -1;
                const int fb = __float_as_int(floor_db);
                for (int w = 0; w < DENSE_WAYS && way < 0; w++) {
                    int cur = *(volatile int*)(WAYF + w);
                    if (cur == TAG_NONE) cur = atomicCAS(WAYF + w, TAG_NONE, fb), cur = cur == TAG_NONE ? fb : cur;
                    if (cur == fb) way = w;
                }
                if (way >= 0) WAYU[way] = 1;
                if (way >= 0 && !(emin < floor_db)) {
                    // only stream-grid rows are floored: sliding sums over the way's copy
                    WAY[k * DH + hl] = way;
                    if (!((atomicOr(WAYMASK + 2 * k + hh, 1 << way) >> way) & 1))
                        COMBO[atomicAdd(ctl + 7, 1)] = (2 * k + hh) * DENSE_WAYS + way;
                    ctl[5] = 1;
                } else FLIST[atomicAdd(ctl + 3, 1)] = k * DH + hl;              // edge frames floored, or no way left: frame by frame
                continue;
            }
            WFL[k * DH + hl] = INFINITY;
            *outp = score_window(k, hl, tf);
        }
        __syncthreads();

        // ================================================================ floored windows
        const int n_slow = ctl[3];
        if (n_slow > 0 || ctl[5]) {
            // ---- C: stream-grid rows a way's floor changes, recomputed once into the way's copy (tagged with the floor)
            const long long span_lo = max(g_lo, g_valid_lo);
            const int span = (int)max(0LL, g_hi - span_lo + 1);
            const int row_lo = span > 0 ? (int)(span_lo % DG) : 0;
            const int lo_rel = (int)(span_lo - hs);
            for (int w = 0; w < DENSE_WAYS; w++) {
                if (!WAYU[w]) continue;
                const int fbits = WAYF[w];
                const float f = __int_as_float(fbits);
                for (int i = warp; i < span; i += nwarps) {
                    const int r = wrap1(row_lo + i, DG);
                    if (!(G[r * ROW + R_MIN] < f) || g2tag[w * DG + r] == fbits) continue;      // warp-uniform
                    int pos = hs_pos + 160 * (lo_rel + i) - N_FFT / 2;
                    if (pos < 0) pos += P; else if (pos >= P) pos -= P;
                    dense_frame<PRE>(FR_GRID, ring_s, fmt, P, pos, 0, 0, pre, *ft, scr, lane, f, patch, false);
                    __syncwarp();
                    if (lane < N_MFCC) __stcg(G2 + ((size_t)w * DG + r) * N_MFCC + lane, patch[lane]);
                    if (lane == 0) g2tag[w * DG + r] = fbits;
                    __syncwarp();
                }
            }
            __syncthreads();
            // ---- D: frame-by-frame windows first (long tasks), then the way windows' sums per (template, half, way, coefficient)
            const int n_d1 = ctl[7] * n_mfcc;
            for (int job = next_task(ctl + 4, lane); job < n_slow + n_d1; job = next_task(ctl + 4, lane)) {
                if (job >= n_slow) {
                    const int q = job - n_slow;
                    const int c = q % n_mfcc, cb = COMBO[q / n_mfcc], w = cb % DENSE_WAYS, kh = cb / DENSE_WAYS, hh = kh & 1, k = kh >> 1;
                    bool valid; float mean, sd;
                    window_sums(k, c, hh, nh, hs, w, __int_as_float(WAYF[w]), valid, mean, sd);
                    const int hl = 32 * hh + lane;
                    if (valid && WAY[k * DH + hl] == w) MS[((size_t)k * N_MFCC + c) * DH + hl] = make_float2(mean, sd);
                    continue;
                }
                const int e_ = FLIST[job], k = e_ / DH, hl = e_ - k * DH;
                const DenseTmplDev& tp = A.t[k];
                const float f = WFL[k * DH + hl];
                const int fb = __float_as_int(f);
                int way = -1;                                                   // the way that holds this floor, if any
                for (int w = 0; w < DENSE_WAYS; w++) if (WAYF[w] == fb) way = w;
                int wpos = hs_pos + 160 * (hl - tp.n);                          // ring position of the window's sample 0
                if (wpos < 0) wpos += P; else if (wpos >= P) wpos -= P;
                long long S1 = 0, S2 = 0;
                auto add = [&](float v) { const int q = quant16(v); S1 += q; S2 += (long long)q * q; };
                const int sl = wrap1(ctl[16 + k] + hl, DLE);
                for (int e = 0; e < 2; e++) {
                    const float* le = (e ? LE1 : LE0) + sl * ROW;
                    float v;
                    if (le[R_MIN] < f) {
                        dense_frame<PRE>(e ? FR_LE1 : FR_LE0, ring_s, fmt, P, wpos, e, tp.L, pre, *ft, scr, lane, f, patch, false);
                        __syncwarp();
                        v = lane < N_MFCC ? patch[lane] : 0.f;
                        __syncwarp();
                    } else v = lane < N_MFCC ? le[lane] : 0.f;
                    add(v);
                }
                // stream-grid frames t = 2 .. t_hi: their un-floored sums in a tight loop (lane = coefficient; lanes >= 20
                // carry don't-care values), then the floored rows — found 32 at a time with lanes = rows — replace their
                // un-floored contribution by the floored one
                const int r0 = wrap1(ctl[8 + k] + hl + 2, DG);
                {
                    const int cl = lane < N_MFCC ? lane : 0;
                    int r = r0;
                    for (int t = 2; t <= tp.t_hi; t++) {
                        const int q = quant16(G[r * ROW + cl]);
                        S1 += q; S2 += (long long)q * q;
                        if (++r == DG) r = 0;
                    }
                }
                for (int t0 = 2; t0 <= tp.t_hi; t0 += 32) {
                    int rl = r0 + (t0 - 2) + lane;
                    while (rl >= DG) rl -= DG;
                    unsigned m = __ballot_sync(FULL, t0 + lane <= tp.t_hi && G[rl * ROW + R_MIN] < f);
                    while (m) {
                        const int b_ = __ffs(m) - 1;
                        m &= m - 1;
                        const int t = t0 + b_;
                        int r = r0 + (t - 2);
                        while (r >= DG) r -= DG;
                        float v;
                        if (way >= 0 && g2tag[way * DG + r] == fb) v = lane < N_MFCC ? __ldcg(G2 + ((size_t)way * DG + r) * N_MFCC + lane) : 0.f;
                        else {
                            int pos = wpos + t * HOP - N_FFT / 2; if (pos >= P) pos -= P;
                            dense_frame<PRE>(FR_GRID, ring_s, fmt, P, pos, 0, 0, pre, *ft, scr, lane, f, patch, false);
                            __syncwarp();
                            v = lane < N_MFCC ? patch[lane] : 0.f;
                            __syncwarp();
                        }
                        const int qf = quant16(v), qu = quant16(G[r * ROW + (lane < N_MFCC ? lane : 0)]);
                        S1 += qf - qu;
                        S2 += (long long)qf * qf - (long long)qu * qu;
                    }
                }
                for (int e = 0; e < tp.r; e++) {
                    const float* re = RE + (tp.re_u[e] * DH + hl) * ROW;
                    float v;
                    if (re[R_MIN] < f) {
                        dense_frame<PRE>(FR_RE, ring_s, fmt, P, wpos, tp.t_hi + 1 + e, tp.L, pre, *ft, scr, lane, f, patch, false);
                        __syncwarp();
                        v = lane < N_MFCC ? patch[lane] : 0.f;
                        __syncwarp();
                    } else v = lane < N_MFCC ? re[lane] : 0.f;
                    add(v);
                }
                // the same exact sums as a way window's, so the same (mean, std) bits: phase E scores both alike
                float mean, sd;
                dense_stats(S1, S2, tp.F, tp.inv_f, mean, sd);
                if (lane < n_mfcc) MS[((size_t)k * N_MFCC + lane) * DH + hl] = make_float2(mean, sd);
                if (lane == 0) WAY[k * DH + hl] = DENSE_WAYS;
            }
            __syncthreads();
            // ---- E: scores of the floored windows (both kinds)
            for (int job = warp; job < NT * n_half; job += nwarps) {
                const int hh = job % n_half, k = job / n_half;
                const int hl = 32 * hh + lane;
                if (hl >= nh || WAY[k * DH + hl] < 0) continue;
                *out_at(hs, hl, k) = score_window(k, hl, tmpl[A.t[k].slot]);
            }
            __syncthreads();
        }
    }
    if (A.keep_rows && g_done > 2) {
        // keep the newest rows for the next call, as many as its first window reaches back
        float* kr = A.keep_rows + (size_t)s * DENSE_KEEP * ROW;
        const long long lo = max(g_valid_lo, g_done - min(min(DENSE_KEEP, DG), A.n_max + 1));
        const int cnt = (int)max(0LL, g_done - lo);
        for (int i = tid; i < cnt * ROW; i += nthr) {
            const long long g = lo + i / ROW;
            kr[(size_t)(g % DENSE_KEEP) * ROW + i % ROW] = G[(size_t)(g % DG) * ROW + i % ROW];
        }
        if (tid == 0) { A.keep_end[2 * s] = lo; A.keep_end[2 * s + 1] = g_done; }
    }
}

// ---- K4D — dense_detect: a per-stream peak picker over the scores K4 just wrote (ewk_dense_detect) -------------------
// Per hop h: b = max over the call's templates of score[h][k] ignoring NaN (NaN when all are), k* the lowest k reaching
// it, above = b >= the stream's similarity_threshold (NaN: never).  State machine per stream (DetState, carried between
// calls):
//   IDLE,  above, h >= quiet_until  -> ARMED, pending = peak h, run_start h, score b, slot, window of k*
//   ARMED, above                    -> peak fields replaced if b > pending score (first maximum wins); then, once
//                                      h - peak >= hold: emit at h -> SPENT
//   ARMED, not above                -> emit at h, quiet_until = h + refractory -> IDLE
//   SPENT, not above                -> quiet_until = h + refractory -> IDLE
// oracle/dense_detect.py is the same machine on the host.  Only comparisons and integer arithmetic: the result is exact.
constexpr int DETECT_WARPS = 4;        // rows (one warp each) per CTA

struct DetRecord {                     // mirrors ewk_detection (include/ewk.h)
    int stream, template_slot;
    long long hop, run_start, emit_hop, seg_start;
    int seg_len;
    float score;
};

// One non-empty row of a detect call: stream `stream`, hops [hop0, hop0 + n_hops), scores at `scores` ([n_hops][T]
// floats into the call's packed K4 output); its records go to rec[det, det + ceil(n_hops / 2)) and their count to
// counts[row] (row: the stream's index in the call's list)
struct DetRow {
    long long hop0, scores, det;
    int stream, n_hops, row, pad;
};

struct DetArgs {
    int T, slot0, hold, refractory;    // templates [slot0, slot0 + T) of the call
    int n[DENSE_MAX_T], L[DENSE_MAX_T]; // per template: window in hops (ceil(L / 160)) and samples
    const DetRow* rows;
    int n_rows;
    const float* scores;
    DetState* state;                   // [n_streams]
    DetRecord* rec;                    // host-mapped: only emitted records cross PCIe
    int* counts;                       // host-mapped [list length]
};

__global__ void __launch_bounds__(32 * DETECT_WARPS)
dense_detect_kernel(const StreamParams* __restrict__ prm, DetArgs A) {
    const int lane = threadIdx.x & 31, w = blockIdx.x * DETECT_WARPS + (threadIdx.x >> 5);
    if (w >= A.n_rows) return;
    const DetRow r = A.rows[w];
    const float thr = prm[r.stream].similarity_threshold;
    const float* __restrict__ sc = A.scores + r.scores;
    DetRecord* __restrict__ out = A.rec + r.det;
    DetState st = A.state[r.stream];
    int nd = 0;
    for (int base = 0; base < r.n_hops; base += 32) {
        // lane j: b and k* of hop base + j
        float b = __int_as_float(0x7fc00000);
        int kb = 0;
        if (base + lane < r.n_hops) {
            const float* row = sc + (size_t)(base + lane) * A.T;
            for (int k = 0; k < A.T; k++) {
                const float v = row[k];
                if (v > b || (b != b && v == v)) { b = v; kb = k; }
            }
        }
        const int cnt = min(32, r.n_hops - base);
        for (int i = 0; i < cnt; i++) {                      // the walk, in hop order (warp-uniform)
            const float bh = __shfl_sync(FULL, b, i);
            const int kh = __shfl_sync(FULL, kb, i);
            const long long h = r.hop0 + base + i;
            int nk = 0, Lk = 0;                                  // window of k* (selects: no local copy of A)
#pragma unroll
            for (int t = 0; t < DENSE_MAX_T; t++)
                if (t == kh) { nk = A.n[t]; Lk = A.L[t]; }
            const bool above = bh >= thr;
            bool emit = false;
            if (st.mode == DET_IDLE) {
                if (above && h >= st.quiet_until) {
                    st.mode = DET_ARMED; st.peak = h; st.run_start = h; st.score = bh; st.slot = A.slot0 + kh;
                    st.seg_start = 160LL * (h - nk); st.seg_len = Lk;
                }
            } else if (st.mode == DET_ARMED) {
                if (above) {
                    if (bh > st.score) {
                        st.peak = h; st.score = bh; st.slot = A.slot0 + kh;
                        st.seg_start = 160LL * (h - nk); st.seg_len = Lk;
                    }
                    if (h - st.peak >= A.hold) { emit = true; st.mode = DET_SPENT; }
                } else {
                    emit = true; st.quiet_until = h + A.refractory; st.mode = DET_IDLE;
                }
            } else if (!above) {
                st.quiet_until = h + A.refractory; st.mode = DET_IDLE;
            }
            if (emit) {
                if (lane == 0) {
                    DetRecord* o = out + nd;
                    o->stream = r.stream; o->template_slot = st.slot; o->hop = st.peak; o->run_start = st.run_start;
                    o->emit_hop = h; o->seg_start = st.seg_start; o->seg_len = st.seg_len; o->score = st.score;
                }
                nd++;
            }
        }
    }
    if (lane == 0) {
        A.state[r.stream] = st;
        A.counts[r.row] = nd;
    }
}

}  // namespace ewk
