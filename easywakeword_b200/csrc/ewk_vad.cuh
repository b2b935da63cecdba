// K6 — template_vad: WakeWord._analyze_reference_audio_duration (/root/reference/easywakeword/wakeword.py:872-893)
// for a batch of templates (SURVEY §8(f) row N2).  One CTA per template:
//   rms[t] = sqrt(mean(x[160 t - 200 : 160 t + 200]^2)), zeros outside the template
//            (librosa.feature.rms(frame_length=400, hop_length=160, center=True, pad_mode='constant'))
//   threshold = max(rms) * 0.1 (float32), voiced = rms > threshold, duration = (last - first) * 160 / 16000,
//   returned as max(duration, 0.2); "not voiced" (all-zero input) is reported through `voiced = 0`.
// The frame RMS is librosa's float32 arithmetic bit for bit (oracle/vad_model.py): its np.mean over a contiguous frame
// is numpy's pairwise sum, which for 400 samples is four blocks [0,96) [96,200) [200,296) [296,400) of 8 sequential
// accumulators each, combined ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) per block and (B0+B1)+(B2+B3) across blocks, then
// a float32 divide by 400 and a float32 sqrt.  One warp per frame: lane l runs block l/8's accumulator l%8 (12 or 13
// squares), and a xor butterfly over offsets 1, 2, 4, 8, 16 is exactly that grouping (float addition commutes).  The
// _rn intrinsics keep every square and sum a separate rounding: nothing contracts into an FMA.
#pragma once
#include <cuda_runtime.h>

namespace ewk {

constexpr int VAD_THREADS = 256;
constexpr int VAD_FRAME = 400;      // int(0.025 * 16000)
constexpr int VAD_HOP = 160;        // int(0.010 * 16000)

struct VadDesc {
    const float* base;      // device PCM (float32)
    long long start;        // first sample
    long long len;          // samples (>= 0)
    long long rms_off;      // frame offset into the rms workspace
};

struct VadResult {          // mirrors ewk_vad_result
    double duration_s;
    float max_rms, threshold;
    int first_frame, last_frame, n_frames, voiced;
};

__global__ void __launch_bounds__(VAD_THREADS)
template_vad_kernel(const VadDesc* __restrict__ descs, VadResult* __restrict__ out, float* __restrict__ rms_ws) {
    const VadDesc d = descs[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = VAD_THREADS / 32;
    const long long F = 1 + d.len / VAD_HOP;
    const float* x = d.base + d.start;
    float* rms = rms_ws + d.rms_off;
    __shared__ float red_f[NW];
    __shared__ long long red_lo[NW], red_hi[NW];
    // frame RMS, one warp per frame: lane = (block, accumulator) of numpy's pairwise float32 sum
    const int blk = lane >> 3, acc = lane & 7;
    const int b0 = blk == 0 ? 0 : blk == 1 ? 96 : blk == 2 ? 200 : 296;
    const int nterm = (blk & 1) ? 13 : 12;                   // blocks of 96 and 104 samples
    float vmax = 0.f;
    for (long long t = warp; t < F; t += NW) {
        const long long i0 = t * VAD_HOP - VAD_FRAME / 2 + b0 + acc;
        float r = 0.f;
        for (int k = 0; k < nterm; k++) {
            const long long p = i0 + 8 * k;
            const float v = (p >= 0 && p < d.len) ? __ldg(x + p) : 0.f;
            const float sq = __fmul_rn(v, v);
            r = k ? __fadd_rn(r, sq) : sq;
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) r = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, o));
        r = __fsqrt_rn(__fdiv_rn(r, (float)VAD_FRAME));
        if (lane == 0) rms[t] = r;
        vmax = fmaxf(vmax, r);
    }
    if (lane == 0) red_f[warp] = vmax;
    __syncthreads();
    vmax = red_f[0];
#pragma unroll
    for (int w = 1; w < NW; w++) vmax = fmaxf(vmax, red_f[w]);
    const float thr = __fmul_rn(vmax, 0.1f);                 // np.float32 * python float -> float32 (NEP 50)
    long long lo = F, hi = -1;
    for (long long t = tid; t < F; t += VAD_THREADS)
        if (rms[t] > thr) { lo = lo < t ? lo : t; hi = hi > t ? hi : t; }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        const long long l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
        lo = lo < l2 ? lo : l2;
        hi = hi > h2 ? hi : h2;
    }
    if (lane == 0) { red_lo[warp] = lo; red_hi[warp] = hi; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < NW; w++) { lo = lo < red_lo[w] ? lo : red_lo[w]; hi = hi > red_hi[w] ? hi : red_hi[w]; }
        VadResult r;
        r.max_rms = vmax; r.threshold = thr; r.n_frames = (int)F;
        r.voiced = hi >= 0 ? 1 : 0;
        r.first_frame = hi >= 0 ? (int)lo : -1;
        r.last_frame = (int)hi;
        const double dur = (double)((hi - lo) * VAD_HOP) / 16000.0;
        r.duration_s = hi >= 0 ? (dur > 0.2 ? dur : 0.2) : 0.0;
        out[blockIdx.x] = r;
    }
}

}  // namespace ewk
