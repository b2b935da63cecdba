// K11 — segment_align: dynamic time warping of segments' MFCC frames against each row's templates (second-stage check
// of level-2 candidates: pooled mean / std cannot see the order of the frames, an alignment can).
//
// One CTA per row, one thread per segment frame i (the row's normalised frame u_i and its inverse norm r_i stay in that
// thread's registers).  The CTA loops over the row's template slots in slot order: the template's normalised frames v_j
// and inverse norms s_j go to shared memory, then the DP runs as an anti-diagonal wavefront over three rotating
// diagonals (cell (i, d - i) of diagonal d by thread i), one barrier per diagonal.
//
// The arithmetic is pinned (oracle/align_model.py states it in float32 and matches it bit for bit): every operation is an
// explicitly rounded intrinsic, so nvcc contracts nothing.
//   u_i[c] = f_i[c] - mean[c]                       c < C (the context's n_mfcc)
//   uu_i   = serial fma chain of u_i[c]^2 from +0;  r_i = uu_i > 0 ? 1 / sqrt(uu_i) : 0     (template: v_j, s_j alike)
//   cost   = 1 - (dot_ij * r_i) * s_j,  dot_ij the serial fma chain of u_i[c] v_j[c] from +0
//   D_00 = cost_00;  D_i0 = D_{i-1,0} + cost_i0;  D_0j = D_{0,j-1} + cost_0j;
//   D_ij = cost_ij + fminf(fminf(D_{i-1,j-1}, D_{i-1,j}), D_{i,j-1});   distance = D_{n-1,m-1} / (n + m)
#pragma once
#include "ewk_segment.cuh"

namespace ewk {

constexpr int ALIGN_MAX_FRAMES = SEG_SMEM_FRAMES;      // 301: segments and stored templates of at most 48 000 samples
constexpr int ALIGN_MAX_SAMPLES = (ALIGN_MAX_FRAMES - 1) * HOP;
constexpr int ALIGN_THREADS = 320;                     // >= ALIGN_MAX_FRAMES: one thread per segment frame
constexpr int ALIGN_STRIDE = N_MFCC + 1;               // odd row stride of the template frames: thread i reads row d - i
constexpr int ALIGN_MAX_T = 64;                        // templates per row (EWK_MAX_STREAM_TEMPLATES)

struct AlignRow {
    long long frames_off;  // first frame of the segment in K3's frames_out
    long long dist_off;    // first distance of the row in the packed output
    int n;                 // segment frames, 1 .. ALIGN_MAX_FRAMES
    int first, count;      // template slots [first, first + count), each with stored frames
    int pad;
};

// tfr: the context's template frame store [max_templates][ALIGN_MAX_FRAMES][N_MFCC]; a slot's frame count is
// 1 + n_samples / HOP (the host checks that the slot holds frames).  feat: K3's [rows][FEAT] (mean first).
// dist / best_dist / best_slot may be null.
__global__ void __launch_bounds__(ALIGN_THREADS, 3)
segment_align_kernel(const AlignRow* __restrict__ rows, const float* __restrict__ seg_frames,
                     const float* __restrict__ feat, const float* __restrict__ tfr, const TemplateFeat* __restrict__ tmpl,
                     int C, float* __restrict__ dist, float* __restrict__ best_dist, int* __restrict__ best_slot)
{
    __shared__ float v[ALIGN_MAX_FRAMES * ALIGN_STRIDE];
    __shared__ float s[ALIGN_MAX_FRAMES];
    __shared__ float diag[3][ALIGN_MAX_FRAMES];
    __shared__ float tmean[N_MFCC];
    const AlignRow r = rows[blockIdx.x];
    const int i = threadIdx.x;
    const bool own = i < r.n;
    float u[N_MFCC];
    float ri;
    {
        const float* f = seg_frames + (size_t)(r.frames_off + (own ? i : 0)) * N_MFCC;
        const float* mean = feat + (size_t)blockIdx.x * FEAT;
        float uu = 0.f;
#pragma unroll
        for (int c = 0; c < N_MFCC; c++) {
            u[c] = 0.f;
            if (own && c < C) {
                u[c] = __fsub_rn(f[c], mean[c]);
                uu = __fmaf_rn(u[c], u[c], uu);
            }
        }
        ri = uu > 0.f ? __fdiv_rn(1.0f, __fsqrt_rn(uu)) : 0.f;
    }
    float best = 0.f;
    int best_k = -1;
    for (int k = r.first; k < r.first + r.count; k++) {
        const int m = 1 + (int)(tmpl[k].n_samples / HOP);
        __syncthreads();                                         // the previous template's DP is done with v, s, diag
        if (i < N_MFCC) tmean[i] = tmpl[k].mean[i];
        __syncthreads();
        const float* g = tfr + (size_t)k * ALIGN_MAX_FRAMES * N_MFCC;
        for (int e = i; e < m * C; e += ALIGN_THREADS) {
            const int j = e / C, c = e - j * C;
            v[j * ALIGN_STRIDE + c] = __fsub_rn(g[(size_t)j * N_MFCC + c], tmean[c]);
        }
        __syncthreads();
        if (i < m) {
            float vv = 0.f;
            for (int c = 0; c < C; c++) vv = __fmaf_rn(v[i * ALIGN_STRIDE + c], v[i * ALIGN_STRIDE + c], vv);
            s[i] = vv > 0.f ? __fdiv_rn(1.0f, __fsqrt_rn(vv)) : 0.f;
        }
        __syncthreads();
        float* dm2 = diag[0];
        float* dm1 = diag[1];
        float* dc = diag[2];
        for (int d = 0; d < r.n + m - 1; d++) {
            const int j = d - i;
            if (own && j >= 0 && j < m) {
                const float* vj = v + j * ALIGN_STRIDE;
                float dot = 0.f;
#pragma unroll
                for (int c = 0; c < N_MFCC; c++)
                    if (c < C) dot = __fmaf_rn(u[c], vj[c], dot);
                const float cost = __fsub_rn(1.0f, __fmul_rn(__fmul_rn(dot, ri), s[j]));
                float acc;
                if (i == 0 && j == 0) acc = cost;
                else if (i == 0) acc = __fadd_rn(dm1[0], cost);                  // D_{0,j-1}
                else if (j == 0) acc = __fadd_rn(dm1[i - 1], cost);              // D_{i-1,0}
                else acc = __fadd_rn(cost, fminf(fminf(dm2[i - 1], dm1[i - 1]), dm1[i]));
                dc[i] = acc;
            }
            __syncthreads();
            float* t = dm2; dm2 = dm1; dm1 = dc; dc = t;
        }
        if (i == r.n - 1) {                                      // D_{n-1,m-1} is on the last diagonal
            const float dd = __fdiv_rn(dm1[i], (float)(r.n + m));
            if (dist) dist[r.dist_off + (k - r.first)] = dd;
            if (best_k < 0 || dd < best) { best = dd; best_k = k; }   // slot order: the lowest slot wins ties
        }
    }
    if (i == r.n - 1) {
        if (best_dist) best_dist[blockIdx.x] = best;
        if (best_slot) best_slot[blockIdx.x] = best_k;
    }
}

}  // namespace ewk
