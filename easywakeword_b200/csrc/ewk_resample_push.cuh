// K8 — resample_push_kernel: a native-rate feed (8 / 44.1 / 48 kHz ..., f32, int16 or G.711 codes) converted to 16 kHz
// and landed in the rings in one launch (ewk_push_resampled).  It evaluates the filter that ewk_resample.cuh designs and
// tabulates: output n of stream s is the sequential fmaf chain, from +0, over taps j = 0 .. 2W-1 of H[j][p] * x[k_c - W + 1 + j],
// k_c = floor(n M / L), p = n M mod L, x = 0 outside the input, so the
// ring holds, bit for bit, what a one-shot conversion of everything pushed so far gives.  ewk_resample runs the same
// kernel with RsPushArgs.out set (float32 rows, no ring, tail or commit): there is one FIR in the library.
//
// Streaming: after c input samples, outputs [0, ready(c)) are in the ring, ready(c) = max(0, ceil((c - W) L / M)), and
// the inputs later outputs still need, [t0(c), c) with t0(c) = max(0, floor(ready(c) M / L) - W + 1), at most 2W - 1 of
// them, sit in a per-stream tail (float32: the input value the FIR reads, so a stream may change input format between
// calls).  A call with n new inputs lands outputs [ready(c), ready(c + n)).  The host picks the tile so that only CTA 0
// of a stream reads the tail; CTA 0 copies it to shared memory and rewrites it in place after a barrier.
//
// Work mapping.  CTA = (output tile, stream), or flat tile x of a list of per-row descriptors (RsPushArgs.rows); the tile's input span, the 256-entry G.711 expansion table and (when small)
// the filter table are staged in shared memory as float32.
//   fast path (L in {1, 2, 4, 8}, M in {1, 2, 3}: 8, 12, 24, 32, 48 kHz): warp-uniform phase, each thread holds K
//     outputs of that phase in consecutive groups, n_q = (g + q) L + r.  Their tap-j inputs are x[b + q M + j], so tap
//     j + M of output q reads what tap j of output q + 1 read: M rotating register windows of K inputs take one new
//     shared-memory load per tap, and every tap costs one table broadcast + one input load for K FMAs.
//   generic path (every other rate, e.g. 44.1 kHz with M = 441: same-phase outputs share no inputs): one output per
//     thread and step, input and table loads per FMA.
#pragma once
#include <cuda_runtime.h>

#include "ewk_streams.cuh"

namespace ewk {

constexpr int RSP_THREADS = 256;
// same-phase outputs per thread on the fast path: odd, so that the window loads of a warp (K M words apart) hit 32
// different banks when M is odd, and small enough for M = 3 that M K window registers + K accumulators fit 2 CTAs per SM
__host__ __device__ constexpr int rsp_k(int m) { return m == 3 ? 11 : 15; }
constexpr int RSP_TABLE_SMEM = 8192;      // filter tables up to this many floats are staged in shared memory
constexpr int RSP_GENERIC_TILE = 2048;    // outputs per CTA on the generic path (at least; see rsp_plan)

enum : int { RSP_IN_F32 = 0, RSP_IN_I16 = 1, RSP_IN_ULAW = 2, RSP_IN_ALAW = 3 };

struct RsPushArgs {
    const void* in;             // [n_streams][in_stride] new input samples of the call (format in_fmt)
    long long in_stride, n_in;
    float* tail;                // [bank streams][tail_cap] input samples [t0_old, c) of each stream
    const float* H;             // [2W][L]
    long long c, o0, o1;        // inputs before the call, outputs landed before / after it (uniform over the call's streams)
    long long t0_old, t0_new;   // first input sample kept in the tail before / after the call
    int tail_cap, in_fmt, L, M, W, stream0, frame_latch, tile, table_smem, span;   // span: staged input floats per CTA
    float* out;                 // non-null: ewk_resample — outputs [o0, o1) of row y go to out + y * out_stride as float32;
    long long out_stride;       //   the input holds absolute samples [c, c + n_in) (c = t0_old, no tail); no ring, no commit
    const RowDesc* rows;        // non-null: per-row descriptors [n_rows] (ewk_push_streams, ewk_push_resampled_each): CTA x
    int n_rows;                 //   is flat output tile x; its row's stream, input, position and frame latch come from the
                                //   descriptor, and c, o0, o1, t0_old, t0_new follow from them (rsp_row)
};

// outputs whose W inputs of look-ahead have arrived after c inputs, and the first input any later output reads (the
// host's rs_ready / rs_tail_start)
__device__ __forceinline__ long long rsp_ready(long long c, const RsPushArgs& A) {
    const long long a = c - A.W;
    return a <= 0 ? 0 : (a * A.L + A.M - 1) / A.M;
}
__device__ __forceinline__ long long rsp_tail_start(long long c, const RsPushArgs& A) {
    const long long t = rsp_ready(c, A) * A.M / A.L - A.W + 1;
    return t > 0 ? t : 0;
}

// row y of the call: per-row (EACH: descriptor A.rows[y]) or the call's uniform values (row y = stream stream0 + y at
// in + y in_stride).  The uniform instance reads n_in and the latch from the parameter bank (rsp_n_in, rsp_latch),
// which leaves its register count (and occupancy) as it was
struct RsRow { long long c, n_in, o0, o1, t0_old, t0_new; int latch; };
template <bool EACH> __device__ __forceinline__ long long rsp_n_in(const RsPushArgs& A, const RsRow& R) { return EACH ? R.n_in : A.n_in; }
template <bool EACH> __device__ __forceinline__ int rsp_latch(const RsPushArgs& A, const RsRow& R) { return EACH ? R.latch : A.frame_latch; }
template <bool EACH>
__device__ __forceinline__ RsRow rsp_row(const RsPushArgs& A, int y) {
    if (!EACH) return RsRow{A.c, A.n_in, A.o0, A.o1, A.t0_old, A.t0_new, A.frame_latch};
    const RowDesc d = A.rows[y];
    const long long c = d.pos;
    return RsRow{c, d.len, rsp_ready(c, A), rsp_ready(c + d.len, A), rsp_tail_start(c, A), rsp_tail_start(c + d.len, A),
                 d.latch};
}

__device__ __forceinline__ float g711_value(int code, int alaw) {
    int v;
    if (alaw) {
        const int a = code ^ 0x55, e = (a >> 4) & 7, m = a & 0x0F;
        v = e == 0 ? (m << 4) + 8 : ((m << 4) + 0x108) << (e - 1);
        v = (a & 0x80) ? v : -v;
    } else {
        const int u = ~code & 0xFF;
        v = ((((u & 0x0F) << 3) + 0x84) << ((u >> 4) & 7)) - 0x84;
        v = (u & 0x80) ? -v : v;
    }
    return (float)v * (1.0f / 32768.0f);
}

// input sample i of the call's new chunk (0 <= i < n_in), as the float the FIR reads
__device__ __forceinline__ float rsp_chunk(const RsPushArgs& A, const void* row, long long i, const float* lut) {
    switch (A.in_fmt) {
        case RSP_IN_F32: return __ldg(reinterpret_cast<const float*>(row) + i);
        case RSP_IN_I16: return (float)__ldg(reinterpret_cast<const short*>(row) + i) * (1.0f / 32768.0f);
        default: return lut[__ldg(reinterpret_cast<const unsigned char*>(row) + i)];
    }
}

// absolute input sample k of the stream: zeros before 0 and beyond what has arrived.  Below t0_old (> 0 once the stream
// is under way) only outputs before o0 read, which this call computes on the fast path but does not store.
template <bool EACH>
__device__ __forceinline__ float rsp_input(const RsPushArgs& A, const RsRow& R, const float* tail, const void* row,
                                           long long k, const float* lut) {
    if (k < R.t0_old) return 0.f;
    if (k < R.c) return tail[k - R.t0_old];
    if (k < R.c + rsp_n_in<EACH>(A, R)) return rsp_chunk(A, row, k - R.c, lut);
    return 0.f;
}

__device__ __forceinline__ void rsp_store(void* ring, int ring_fmt, long long idx, float y) {
    if (ring_fmt == 1) {
        int q = __float2int_rn(y * 32768.0f);                   // rint(y * 32768), ties to even (synth.to_int16)
        q = q < -32768 ? -32768 : (q > 32767 ? 32767 : q);
        reinterpret_cast<short*>(ring)[idx] = (short)q;
    } else {
        reinterpret_cast<float*>(ring)[idx] = y;
    }
}

// fast path: thread (r, t) computes outputs (g0 + q) L + r, q < K; xs = staged inputs, b = smem index of tap 0 of q = 0
template <int M, int RSP_K = rsp_k(M)>
__device__ __forceinline__ void rsp_fir_windows(const float* __restrict__ xs, int b, const float* __restrict__ h, int L,
                                                int taps, float (&acc)[RSP_K]) {
    float win[M][RSP_K];                                        // win[r][m % K] = x[b + m M + r]
#pragma unroll
    for (int r = 0; r < M; r++)
#pragma unroll
        for (int m = 0; m < RSP_K; m++) win[r][m] = xs[b + m * M + r];
#pragma unroll
    for (int q = 0; q < RSP_K; q++) acc[q] = 0.f;
    const int blocks = taps / (M * RSP_K);
    int j = 0;
    for (int blk = 0; blk < blocks; blk++) {
#pragma unroll
        for (int u = 0; u < RSP_K; u++) {                       // tap step jj = blk K + u: taps j = jj M + r
#pragma unroll
            for (int r = 0; r < M; r++) {
                const float hv = h[(j + r) * L];
#pragma unroll
                for (int q = 0; q < RSP_K; q++) acc[q] = fmaf(win[r][(u + q) % RSP_K], hv, acc[q]);
                // x[b + (jj + K) M + r] replaces x[b + jj M + r], which no output needs any more
                win[r][u] = xs[b + (blk * RSP_K + u + RSP_K) * M + r];
            }
            j += M;
        }
    }
    for (; j < taps; j++) {                                     // remaining taps, same order
        const float hv = h[j * L];
#pragma unroll
        for (int q = 0; q < RSP_K; q++) acc[q] = fmaf(xs[b + q * M + j], hv, acc[q]);
    }
}

template <int M, bool EACH>
__global__ void __launch_bounds__(RSP_THREADS, 2) resample_push_kernel(BankView B, RsPushArgs A) {
    extern __shared__ float smem[];
    float* lut = smem;                                          // [256]
    float* tail_s = lut + 256;                                  // [tail_cap] CTA 0's copy of the stream's tail
    float* hs = tail_s + A.tail_cap;                            // [2W L] when A.table_smem
    float* xs = hs + (A.table_smem ? 2 * A.W * A.L : 0);        // [span]
    // the CTA's row and output tile: the grid's (tile, row), or flat tile x of the descriptors' list.  The uniform
    // instance reads blockIdx where it needs them (held in registers across the FIR, they cost it 5 registers at M = 3)
    const unsigned y_each = EACH ? (unsigned)row_of_item(A.rows, A.n_rows, blockIdx.x) : 0u;
    const unsigned tile_each = EACH ? blockIdx.x - (unsigned)A.rows[y_each].item0 : 0u;
    auto row_y = [&] { return EACH ? y_each : blockIdx.y; };
    auto tile_x = [&] { return EACH ? tile_each : blockIdx.x; };
    const int s = EACH ? A.rows[y_each].stream : A.stream0 + (int)blockIdx.y;
    const void* row = reinterpret_cast<const char*>(A.in) + (EACH ? (size_t)A.rows[y_each].off : (size_t)blockIdx.y * A.in_stride) *
                      (A.in_fmt == RSP_IN_F32 ? 4 : A.in_fmt == RSP_IN_I16 ? 2 : 1);
    float* tail = A.out ? nullptr : A.tail + (size_t)s * A.tail_cap;
    const int tid = threadIdx.x;
    if (A.in_fmt >= RSP_IN_ULAW) lut[tid] = g711_value(tid, A.in_fmt == RSP_IN_ALAW);
    __syncthreads();
    const int taps = 2 * A.W;
    if (A.table_smem)
        for (int i = tid; i < taps * A.L; i += RSP_THREADS) hs[i] = __ldg(A.H + i);
    const float* h = A.table_smem ? hs : A.H;

    // the CTA's outputs [n0, n0 + tile) and the input span they read, from absolute sample s0
    const RsRow R = rsp_row<EACH>(A, row_y());
    const bool fast = M > 0;
    long long n0, s0;
    if (fast) {
        n0 = (R.o0 / A.L) * A.L + (long long)tile_x() * A.tile;
        s0 = (n0 / A.L) * M - A.W + 1;
    } else {
        n0 = R.o0 + (long long)tile_x() * A.tile;
        s0 = n0 * A.M / A.L - A.W + 1;
    }
    // tile 0 always runs (tail, commit)
    if (tile_x() > 0 && n0 >= R.o1) return;
    for (int i = tid; i < A.span; i += RSP_THREADS) xs[i] = rsp_input<EACH>(A, R, tail, row, s0 + i, lut);
    if (tile_x() == 0)
        for (int i = tid; i < (int)(R.c - R.t0_old); i += RSP_THREADS) tail_s[i] = tail[i];
    __syncthreads();

    void* ring = A.out ? nullptr : reinterpret_cast<char*>(B.ring) + (size_t)s * B.P * (B.fmt == 1 ? 2 : 4);
    float* out = A.out ? A.out + (size_t)row_y() * A.out_stride - R.o0 : nullptr;
    const int p_n0 = A.out ? 0 : (int)(n0 % B.P);               // ring position of n0: one 64-bit modulo per CTA
    auto store = [&](long long n, float y) {
        if (out) { out[n] = y; return; }
        int i = p_n0 + (int)(n - n0);                           // n - n0 < tile
        while (i >= B.P) i -= B.P;
        rsp_store(ring, B.fmt, i, y);
    };
    const long long lo = R.o0 > n0 ? R.o0 : n0, hi = R.o1 < n0 + A.tile ? R.o1 : n0 + A.tile;
    if (fast) {
        constexpr int MM = M > 0 ? M : 1, RSP_K = rsp_k(MM);
        const int tp = RSP_THREADS / A.L;                       // threads per phase (a multiple of 32)
        const int r = tid / tp, t = tid - r * tp;
        const long long g0 = n0 / A.L + (long long)t * RSP_K;
        const int p = (r * MM) % A.L;
        const int b = (int)(g0 * MM + (r * MM) / A.L - A.W + 1 - s0);
        if (g0 * A.L + r < hi) {
            float acc[RSP_K];
            rsp_fir_windows<MM>(xs, b, hs + p, A.L, taps, acc);    // the host takes this path only with the table staged
#pragma unroll
            for (int q = 0; q < RSP_K; q++) {
                const long long n = (g0 + q) * A.L + r;
                if (n >= lo && n < hi) store(n, acc[q]);
            }
        }
    } else {
        for (long long n = n0 + tid; n < hi; n += RSP_THREADS) {
            if (n < lo) continue;
            const long long kc = n * A.M / A.L;
            const int p = (int)(n * A.M - kc * A.L);
            const float* x = xs + (kc - A.W + 1 - s0);
            const float* hp = h + p;
            float acc = 0.f;
            for (int j = 0; j < taps; j++) acc = fmaf(x[j], hp[(size_t)j * A.L], acc);
            store(n, acc);
        }
    }

    if (tile_x() == 0 && !A.out) {
        // the tail for the next call: inputs [t0_new, c + n_in), from the old tail's copy or the new chunk
        const int keep = (int)(R.c + rsp_n_in<EACH>(A, R) - R.t0_new);
        for (int i = tid; i < keep; i += RSP_THREADS) {
            const long long k = R.t0_new + i;
            tail[i] = k < R.c ? tail_s[k - R.t0_old] : rsp_chunk(A, row, k - R.c, lut);
        }
        if (tid == 0) {                                         // commit: what ring_commit_kernel does for an unsummed push
            StreamState& st = B.st[s];
            if (st.frame_size == 0) {
                const int fs = B.prm[s].frame_size;
                st.frame_size = fs > 0 ? fs : rsp_latch<EACH>(A, R);
            }
            st.written = R.o1;
            st.ss_from = R.o1;
        }
    }
}

}  // namespace ewk
