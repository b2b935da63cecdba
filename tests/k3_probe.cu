// Test-only probe of K3's frame pipeline (built by tests/test_frame_model.py and tests/test_gpu_k3_exact.py into a
// temporary directory with the library's nvcc flags, loaded with ctypes).  It includes the library's own headers and
// restates no arithmetic: each entry point runs one stage of ewk_frame.cuh as the kernels do, so that a difference
// between the device and oracle/frame_model.py can be pinned to a stage.  Every device buffer is freed before return.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <vector>

#include "ewk_frame.cuh"
#include "ewk_tables.hpp"

using namespace ewk;

namespace {

// the library's table image: DeviceTables, then the FrameTables image at FRAME_IMAGE_OFFSET (as ewk_ctx::init)
std::vector<unsigned char> table_image() {
    std::vector<unsigned char> img(FRAME_IMAGE_OFFSET + sizeof(FrameTables), 0);
    DeviceTables* T = new DeviceTables();
    build_tables(*T);
    FrameTables* ft = new FrameTables();
    std::memset(ft, 0, sizeof(FrameTables));
    load_frame_tables(*ft, T, 0, 1);
    ft->preemph = 0.f;
    ft->n_mfcc = N_MFCC;
    std::memcpy(img.data(), T, sizeof(DeviceTables));
    std::memcpy(img.data() + FRAME_IMAGE_OFFSET, ft, sizeof(FrameTables));
    delete ft;
    delete T;
    return img;
}

__global__ void log_mel_kernel(const float* __restrict__ S, float* __restrict__ out, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = TEN_LOG10_2 * __log2f(fmaxf(S[i], 1e-10f));      // warp_log_mel's expression
}

// one warp per frame; x: [n][512] samples already loaded (lane holds pairs 2 lane + 64 a, +1, as load_frame_pairs)
__global__ void frames_kernel(const DeviceTables* __restrict__ T, const float* __restrict__ x, float floor_db,
                              float* __restrict__ mfcc, float* __restrict__ lm, float* __restrict__ power) {
    extern __shared__ __align__(16) float smem[];
    FrameTables* ft = reinterpret_cast<FrameTables*>(smem);
    float* scr = smem + sizeof(FrameTables) / sizeof(float);
    const int lane = threadIdx.x;
    copy_frame_tables(*ft, T, lane, 32);
    __syncthreads();
    const float2* fx = reinterpret_cast<const float2*>(x + (size_t)blockIdx.x * N_FFT);
    float2 v[8];
#pragma unroll
    for (int a = 0; a < 8; a++) v[a] = fx[lane + 32 * a];
    if (power) {
        warp_power_spectrum(v, *ft, scr, lane);
        for (int k = lane; k < N_BINS; k += 32) power[(size_t)blockIdx.x * N_BINS + k] = scr[k];
        return;
    }
    float mn, mx;
    warp_frame_mfcc(v, *ft, scr, lane, floor_db, mfcc + (size_t)blockIdx.x * N_MFCC, mn, mx,
                    lm + (size_t)blockIdx.x * N_MELS);
}

int run_frames(const float* x, int n, float floor_db, float* mfcc_out, float* lm_out, float* power_out) {
    if (!x || n < 1) return 1;
    const std::vector<unsigned char> img = table_image();
    void *dT = nullptr, *dx = nullptr, *dm = nullptr, *dl = nullptr, *dp = nullptr;
    int rc = 0;
    const size_t smem = sizeof(FrameTables) + sizeof(float) * SCR_WARP;
    if (cudaMalloc(&dT, img.size()) || cudaMalloc(&dx, sizeof(float) * N_FFT * (size_t)n) ||
        cudaMalloc(&dm, sizeof(float) * N_MFCC * (size_t)n) || cudaMalloc(&dl, sizeof(float) * N_MELS * (size_t)n) ||
        cudaMalloc(&dp, sizeof(float) * N_BINS * (size_t)n))
        rc = 2;
    if (!rc && (cudaMemcpy(dT, img.data(), img.size(), cudaMemcpyHostToDevice) ||
                cudaMemcpy(dx, x, sizeof(float) * N_FFT * (size_t)n, cudaMemcpyHostToDevice)))
        rc = 3;
    if (!rc) {
        frames_kernel<<<n, 32, smem>>>((const DeviceTables*)dT, (const float*)dx, floor_db, (float*)dm, (float*)dl,
                                       power_out ? (float*)dp : nullptr);
        if (cudaGetLastError() || cudaDeviceSynchronize()) rc = 4;
    }
    if (!rc && power_out && cudaMemcpy(power_out, dp, sizeof(float) * N_BINS * (size_t)n, cudaMemcpyDeviceToHost)) rc = 5;
    if (!rc && mfcc_out && cudaMemcpy(mfcc_out, dm, sizeof(float) * N_MFCC * (size_t)n, cudaMemcpyDeviceToHost)) rc = 5;
    if (!rc && lm_out && cudaMemcpy(lm_out, dl, sizeof(float) * N_MELS * (size_t)n, cudaMemcpyDeviceToHost)) rc = 5;
    for (void* p : {dT, dx, dm, dl, dp}) if (p) cudaFree(p);
    return rc;
}

}  // namespace

// Host only: the DeviceTables image followed (at FRAME_IMAGE_OFFSET) by the FrameTables image, as the library uploads
// them (front-end parameters at their defaults: no pre-emphasis, 20 coefficients).  Returns the image size in bytes;
// writes nothing when cap is smaller.  sizes (nullable): sizeof(DeviceTables), FRAME_IMAGE_OFFSET, sizeof(FrameTables).
extern "C" long long k3p_tables(unsigned char* out, long long cap, long long* sizes) {
    const std::vector<unsigned char> img = table_image();
    if (sizes) { sizes[0] = (long long)sizeof(DeviceTables); sizes[1] = (long long)FRAME_IMAGE_OFFSET; sizes[2] = (long long)sizeof(FrameTables); }
    if (out && cap >= (long long)img.size()) std::memcpy(out, img.data(), img.size());
    return (long long)img.size();
}

// out[i] = TEN_LOG10_2 * __log2f(fmaxf(S[i], 1e-10f)) on the device.  Returns 0 on success.
extern "C" int k3p_log_mel(const float* S, float* out, long long n) {
    if (!S || !out || n < 1) return 1;
    void *dS = nullptr, *dO = nullptr;
    int rc = 0;
    if (cudaMalloc(&dS, sizeof(float) * (size_t)n) || cudaMalloc(&dO, sizeof(float) * (size_t)n)) rc = 2;
    if (!rc && cudaMemcpy(dS, S, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice)) rc = 3;
    if (!rc) {
        log_mel_kernel<<<(unsigned)((n + 255) / 256), 256>>>((const float*)dS, (float*)dO, n);
        if (cudaGetLastError() || cudaDeviceSynchronize()) rc = 4;
    }
    if (!rc && cudaMemcpy(out, dO, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost)) rc = 5;
    if (dS) cudaFree(dS);
    if (dO) cudaFree(dO);
    return rc;
}

// warp_frame_mfcc on n already-loaded frames x[n][512] under floor_db: mfcc_out[n][20], un-floored log-mel lm_out[n][128].
extern "C" int k3p_frames(const float* x, int n_frames, float floor_db, float* mfcc_out, float* lm_out) {
    if (!mfcc_out || !lm_out) return 1;
    return run_frames(x, n_frames, floor_db, mfcc_out, lm_out, nullptr);
}

// warp_power_spectrum alone: power_out[n][257].
extern "C" int k3p_power(const float* x, int n_frames, float* power_out) {
    if (!power_out) return 1;
    return run_frames(x, n_frames, 0.f, nullptr, nullptr, power_out);
}
