// libewk: C ABI (include/ewk.h) over the sm_100a kernels.  No torch types, no CPU fallback.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/ewk.h"
#include "ewk_ctx.hpp"

using namespace ewk;

static thread_local std::string g_create_error = "";

void ewk_ctx::fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    err = buf;
}

extern "C" int ewk_abi_version(void) { return EWK_ABI_VERSION; }

extern "C" const char* ewk_last_error(const ewk_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int ewk_host_table(int which, float* out, int cap) {
    static DeviceTables T;
    static std::vector<float> mel;
    static bool built = false;
    if (!built) { build_tables(T); build_mel_dense(mel); built = true; }
    if (which == 0) {
        if (out && cap >= N_FFT) std::memcpy(out, T.hann, sizeof(float) * N_FFT);
        return N_FFT;
    }
    if (which == 1) {
        if (out && cap >= N_MELS * N_BINS) std::memcpy(out, mel.data(), sizeof(float) * N_MELS * N_BINS);
        return N_MELS * N_BINS;
    }
    if (which == 2) {
        if (out && cap >= N_MFCC * N_MELS)
            for (int k = 0; k < N_MFCC; k++)
                for (int b = 0; b < N_MELS; b++) out[k * N_MELS + b] = T.dct_t[b * N_MFCC + k];
        return N_MFCC * N_MELS;
    }
    return EWK_ERR_ARG;
}

#define CK(call)                                                                                    \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess) {                                                                    \
            ctx->fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__);  \
            return EWK_ERR_CUDA;                                                                    \
        }                                                                                           \
    } while (0)

// ------------------------------------------------------------------------------------------
// Pool (ewk_ctx.hpp): every allocation of a context; poison mode fills, guards and checks them.
cudaError_t Pool::fill(void* p, size_t bytes, bool host) {
    cudaError_t e = cudaDeviceSynchronize();             // nothing in flight still reads or writes the block
    if (e != cudaSuccess) return e;
    if (host) { std::memset(p, poison, bytes); return cudaSuccess; }
    if (!stream && (e = cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(p, poison, bytes, stream)) != cudaSuccess) return e;
    return cudaStreamSynchronize(stream);
}

cudaError_t Pool::alloc(void** p, size_t bytes, const char* name) {
    if (poison < 0) return cudaMalloc(p, bytes);
    cudaError_t e = cudaMalloc(p, bytes + GUARD);
    if (e != cudaSuccess) return e;
    blocks[*p] = Block{name, bytes, false};
    return fill(*p, bytes + GUARD, false);
}

cudaError_t Pool::alloc_host(void** p, size_t bytes, unsigned flags, const char* name) {
    if (poison < 0) return cudaHostAlloc(p, bytes, flags);
    cudaError_t e = cudaHostAlloc(p, bytes + GUARD, flags);
    if (e != cudaSuccess) return e;
    blocks[*p] = Block{name, bytes, true};
    return fill(*p, bytes + GUARD, true);
}

cudaError_t Pool::refill(void* p) {
    auto it = blocks.find(p);
    return it == blocks.end() ? cudaSuccess : fill(p, it->second.bytes, it->second.host);
}

cudaError_t Pool::check_block(void* p, const Block& b, std::string* report) {
    unsigned char g[GUARD];
    const unsigned char* q = (const unsigned char*)p + b.bytes;
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return e;
    if (b.host) {
        std::memcpy(g, q, GUARD);
    } else {
        if ((e = cudaMemcpyAsync(g, q, GUARD, cudaMemcpyDeviceToHost, stream)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(stream)) != cudaSuccess) return e;
    }
    for (size_t i = 0; i < GUARD; i++)
        if (g[i] != (unsigned char)poison) {
            char buf[256];
            snprintf(buf, sizeof(buf), "%s%s (%zu bytes): guard damaged from byte %zu", report->empty() ? "" : "; ", b.name,
                     b.bytes, b.bytes + i);
            *report += buf;
            break;
        }
    return cudaSuccess;
}

cudaError_t Pool::free(void* p, bool host) {
    cudaError_t e = cudaSuccess;
    auto it = blocks.find(p);
    if (it != blocks.end()) {
        e = check_block(p, it->second, &damage);
        blocks.erase(it);
    }
    const cudaError_t f = host ? cudaFreeHost(p) : cudaFree(p);    // freed even when the guard could not be read
    return e != cudaSuccess ? e : f;
}

cudaError_t Pool::check(std::string* report) {
    *report = damage;
    for (auto& kv : blocks) {
        cudaError_t e = check_block(kv.first, kv.second, report);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

extern "C" int ewk_debug_check(ewk_ctx* ctx) {
    if (!ctx) return EWK_ERR_ARG;
    if (ctx->pool.poison < 0) {
        ctx->fail("ewk_debug_check: poison mode is off (set EWK_POISON before ewk_create)");
        return EWK_ERR_STATE;
    }
    CK(cudaSetDevice(ctx->device));
    std::string report;
    CK(ctx->pool.check(&report));
    if (!report.empty()) { ctx->fail("ewk_debug_check: %s", report.c_str()); return EWK_ERR_STATE; }
    return EWK_OK;
}

extern "C" int ewk_create(int device, const ewk_config* cfg, ewk_ctx** out) {
    if (!cfg || !out) { g_create_error = "ewk_create: null argument"; return EWK_ERR_ARG; }
    *out = nullptr;
    if (cfg->n_streams < 0 || cfg->max_templates < 1 || cfg->max_templates > EWK_MAX_TEMPLATE_SLOTS ||
        (cfg->pcm_format != EWK_PCM_F32 && cfg->pcm_format != EWK_PCM_I16) ||
        (cfg->n_streams > 0 && (cfg->ring_samples < EWK_TICK_SAMPLES || cfg->slack_samples < 0))) {
        g_create_error = "ewk_create: invalid ewk_config";
        return EWK_ERR_ARG;
    }
    if (!(cfg->preemphasis >= 0.f && cfg->preemphasis < 1.f)) {
        g_create_error = "ewk_create: preemphasis must be in [0, 1)";
        return EWK_ERR_ARG;
    }
    if (cfg->n_mfcc < 0 || cfg->n_mfcc > EWK_N_MFCC || (cfg->template_frames != 0 && cfg->template_frames != 1) ||
        cfg->reserved1 != 0) {
        g_create_error = "ewk_create: n_mfcc must be 0 (= 20) or in [1, 20], template_frames 0 or 1; reserved1 must be 0";
        return EWK_ERR_ARG;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("ewk_create: no CUDA device (") + cudaGetErrorString(e) +
                         "); libewk has no CPU fallback";
        return EWK_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) { g_create_error = "ewk_create: device index out of range"; return EWK_ERR_ARG; }
    ewk_ctx* ctx = new ewk_ctx();
    ctx->device = device;
    ctx->cfg = *cfg;
    int rc = ctx->init();
    if (rc != EWK_OK) {
        g_create_error = ctx->err;
        ctx->release();
        delete ctx;
        return rc;
    }
    *out = ctx;
    return EWK_OK;
}

extern "C" int ewk_destroy(ewk_ctx* ctx) {
    if (!ctx) return EWK_ERR_ARG;
    cudaSetDevice(ctx->device);
    ctx->release();
    delete ctx;
    return EWK_OK;
}

extern "C" int ewk_set_cuda_stream(ewk_ctx* ctx, void* s) {
    if (!ctx) return EWK_ERR_ARG;
    if (ctx->match_inflight) {                       // results of the old stream's ticks stay ordered before the switch
        CK(cudaSetDevice(ctx->device));
        CK(cudaStreamSynchronize(ctx->match_stream));
        ctx->match_inflight = false;
    }
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return EWK_OK;
}

extern "C" int ewk_synchronize(ewk_ctx* ctx) {
    if (!ctx) return EWK_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (ctx->bank.n_streams) { int rc = ctx->flush_pending(); if (rc) return rc; }
    int jr = ctx->join_match();
    if (jr) return jr;
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->pub_stream) CK(cudaStreamSynchronize(ctx->pub_stream));
    return EWK_OK;
}

int ewk_ctx::init() {
    ewk_ctx* ctx = this;
    CK(cudaSetDevice(device));
    if (const char* e = getenv("EWK_POISON"); e && *e) {     // test mode (ewk::Pool): the fill byte, decimal or 0x..
        char* end = nullptr;
        const long v = strtol(e, &end, 0);
        if (*end || v < 0 || v > 255) { fail("ewk_create: EWK_POISON=%s is not a byte (0..255)", e); return EWK_ERR_ARG; }
        pool.poison = (int)v;
    }
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    sm_count = prop.multiProcessorCount;
    if (const char* e = getenv("EWK_SEG_LM")) use_lm = atoi(e) != 0;       // 0: recompute floored frames from the PCM
    if (prop.major < 10) {
        fail("ewk_create: device %d is sm_%d%d; libewk is built for sm_100a only", device, prop.major, prop.minor);
        return EWK_ERR_CUDA;
    }
    CK(cudaStreamCreateWithFlags(&own_stream, cudaStreamNonBlocking));
    stream = own_stream;
    CK(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) {
        CK(cudaEventCreateWithFlags(&ev_ready[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ev_free[i], cudaEventDisableTiming));
    }
    DeviceTables* h = new DeviceTables();
    int nnz = build_tables(*h);
    if (nnz < 0) { delete h; fail("mel table overflow"); return EWK_ERR_STATE; }
    // flat tables, then the per-CTA layout of them (FrameTables image) that K3 / K4 copy into shared memory
    FrameTables* img = new FrameTables();
    load_frame_tables(*img, h, 0, 1);
    img->preemph = cfg.preemphasis;
    img->n_mfcc = cfg.n_mfcc > 0 ? cfg.n_mfcc : N_MFCC;
    img->pad_[0] = img->pad_[1] = 0;
    CK(pool.alloc(&d_tables, FRAME_IMAGE_OFFSET + sizeof(FrameTables), "d_tables"));
    CK(cudaMemcpy(d_tables, h, sizeof(DeviceTables), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(reinterpret_cast<char*>(d_tables) + FRAME_IMAGE_OFFSET, img, sizeof(FrameTables), cudaMemcpyHostToDevice));
    delete img;
    delete h;
    h_tmpl.assign(cfg.max_templates, TemplateFeat{});
    CK(pool.alloc(&d_tmpl, sizeof(TemplateFeat) * cfg.max_templates, "d_tmpl"));
    CK(cudaMemset(d_tmpl, 0, sizeof(TemplateFeat) * cfg.max_templates));
    h_tfr_n.assign(cfg.max_templates, 0);
    if (cfg.template_frames)      // written per slot by the template writers; K11 reads only a slot's stored frames
        CK(pool.alloc(&d_tfr, sizeof(float) * ALIGN_MAX_FRAMES * N_MFCC * (size_t)cfg.max_templates, "d_tfr"));
    CK(cudaFuncSetAttribute(segment_mfcc_match_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)seg_smem_bytes(SEG_SMEM_FRAMES)));
    CK(cudaFuncSetAttribute(segment_mfcc_match_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)seg_smem_bytes(SEG_SMEM_FRAMES)));
    int rc = init_streams();
    if (rc != EWK_OK) return rc;
    return EWK_OK;
}

void ewk_ctx::release() {
    cudaSetDevice(device);
    if (own_stream) cudaStreamSynchronize(own_stream);
    release_streams();
    for (DevBuf* b : {&b_pcm, &b_desc, &b_ws, &b_lm, &b_feat, &b_scores, &b_matched, &b_frames, &b_off}) b->free();
    for (auto& kv : rs_tables) if (kv.second.H) pool.free(kv.second.H);
    rs_tables.clear();
    b_rs_in.free(); b_rs_out.free();
    if (d_wait_flag) { pool.free(d_wait_flag); d_wait_flag = nullptr; }
    if (pub_stream) { cudaStreamSynchronize(pub_stream); cudaStreamDestroy(pub_stream); pub_stream = nullptr; }
    if (ev_k3) { cudaEventDestroy(ev_k3); ev_k3 = nullptr; }
    for (int i = 0; i < 2; i++) if (ev_pub[i]) { cudaEventDestroy(ev_pub[i]); ev_pub[i] = nullptr; }
    if (d_pub_snap) { pool.free(d_pub_snap); d_pub_snap = nullptr; }
    if (d_tables) pool.free(d_tables);
    if (d_tmpl) pool.free(d_tmpl);
    if (d_tfr) pool.free(d_tfr);
    d_tfr = nullptr;
    if (copy_stream) { cudaStreamSynchronize(copy_stream); cudaStreamDestroy(copy_stream); }
    if (match_stream) { cudaStreamSynchronize(match_stream); cudaStreamDestroy(match_stream); match_stream = nullptr; }
    if (ev_gate) { cudaEventDestroy(ev_gate); ev_gate = nullptr; }
    if (ev_match) { cudaEventDestroy(ev_match); ev_match = nullptr; }
    for (int i = 0; i < 2; i++) {
        if (ev_ready[i]) cudaEventDestroy(ev_ready[i]);
        if (ev_free[i]) cudaEventDestroy(ev_free[i]);
        ev_ready[i] = ev_free[i] = nullptr;
        b_stage2[i].free();
        b_raw[i].free();
        if (ev_pos[i]) cudaEventDestroy(ev_pos[i]);
        if (h_pos[i]) pool.free(h_pos[i], true);
        ev_pos[i] = nullptr; h_pos[i] = nullptr;
        b_pos[i].free();
    }
    dset_stage.free(); drows.free(); ddets.free(); b_dset.free();
    h_dset.clear();
    if (h_det_map) pool.free(h_det_map, true);
    h_det_map = nullptr; det_map_cap = 0;
    b_reset.free();
    b_blob.free();
    b_mig.free();
    if (own_stream) cudaStreamDestroy(own_stream);
    if (pool.stream) cudaStreamDestroy(pool.stream);
    pool.stream = nullptr;
    d_tables = nullptr; d_tmpl = nullptr; own_stream = nullptr; copy_stream = nullptr;
}

// ------------------------------------------------------------------------------------------
// Launch K3 over `n_seg` descriptors already on the device.
int ewk_ctx::launch_segments(const SegDesc* d_segs, int n_seg, int max_frames, long long spill_frames,
                             long long lm_frames, int n_tmpl, int tmpl_first, float threshold, float* d_feat,
                             float* d_frames, float* d_scores, unsigned char* d_matched) {
    ewk_ctx* ctx = this;
    const int cap = std::min(max_frames, SEG_SMEM_FRAMES);
    float* ws = nullptr;
    if (spill_frames > 0) {
        CK(b_ws.ensure(sizeof(float) * (size_t)spill_frames * FR_STRIDE));
        ws = (float*)b_ws.p;
    }
    // log-mel rows of every frame (512 B each), so that the top_db floor costs one DCT per floored frame; beyond
    // LM_WS_MAX_BYTES the kernel recomputes floored frames from the PCM instead
    float* lm = nullptr;
    if (use_lm && lm_frames > 0 && sizeof(float) * (size_t)lm_frames * LM_ROW <= LM_WS_MAX_BYTES) {
        CK(b_lm.ensure(sizeof(float) * (size_t)lm_frames * LM_ROW));
        lm = (float*)b_lm.p;
    }
    cudaEvent_t pe = prof_begin(3);
    auto k3 = cfg.preemphasis != 0.f ? segment_mfcc_match_kernel<true> : segment_mfcc_match_kernel<false>;
    k3<<<n_seg, SEG_THREADS, seg_smem_bytes(cap), stream>>>(
        d_tables, d_segs, cap, ws, lm, d_tmpl, n_tmpl, tmpl_first, threshold, d_feat, d_frames, d_scores, d_matched);
    prof_end(pe, 3);
    CK(cudaGetLastError());
    launches++;
    return EWK_OK;
}

// WordMatcher.extract_mfcc on one buffer; dense40 (nullable): the same features from K4's integer statistics of the frames.
static int extract_impl(ewk_ctx* ctx, const float* pcm, int64_t n, int where, float* mean20, float* std20,
                        float* frames, int64_t frames_cap, float* dense40) {
    if (!pcm || n < 1 || n > (int64_t)1 << 30 || !mean20 || !std20) {
        ctx->fail("ewk_extract_mfcc: need pcm, 1 <= n < 2^30, mean20, std20 (n=%lld)", (long long)n);
        return EWK_ERR_ARG;
    }
    const int64_t F = 1 + n / HOP;
    if (frames && frames_cap < F) { ctx->fail("ewk_extract_mfcc: frames_cap %lld < %lld frames", (long long)frames_cap, (long long)F); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    const float* d_pcm = pcm;
    if (where == EWK_HOST) {
        CK(ctx->b_pcm.ensure(sizeof(float) * (size_t)n));
        CK(cudaMemcpyAsync(ctx->b_pcm.p, pcm, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
        d_pcm = (const float*)ctx->b_pcm.p;
    }
    SegDesc sd{};
    sd.base = d_pcm; sd.start = 0; sd.ring = 0; sd.len = (int)n; sd.fmt = 0; sd.ws_frame_off = 0; sd.frames_off = 0;
    sd.lm_off = 0;
    CK(ctx->b_desc.ensure(sizeof(SegDesc)));
    CK(cudaMemcpyAsync(ctx->b_desc.p, &sd, sizeof(sd), cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx->b_feat.ensure(sizeof(float) * 2 * FEAT));
    float* d_frames = nullptr;
    if (frames || dense40) { CK(ctx->b_frames.ensure(sizeof(float) * (size_t)F * N_MFCC)); d_frames = (float*)ctx->b_frames.p; }
    int rc = ctx->launch_segments((const SegDesc*)ctx->b_desc.p, 1, (int)F, F > SEG_SMEM_FRAMES ? F : 0, F, 0, 0, 0.f,
                                  (float*)ctx->b_feat.p, d_frames, nullptr, nullptr);
    if (rc != EWK_OK) return rc;
    if (dense40) {
        dense_template_features_kernel<<<1, 32, 0, ctx->stream>>>(d_frames, (int)F, ctx->cfg.n_mfcc > 0 ? ctx->cfg.n_mfcc : N_MFCC,
                                                                  (float*)ctx->b_feat.p + FEAT);
        CK(cudaGetLastError());
        ctx->launches++;
    }
    float feat[2 * FEAT];
    CK(cudaMemcpyAsync(feat, ctx->b_feat.p, sizeof(float) * (dense40 ? 2 * FEAT : FEAT), cudaMemcpyDeviceToHost, ctx->stream));
    if (frames) CK(cudaMemcpyAsync(frames, d_frames, sizeof(float) * (size_t)F * N_MFCC, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    std::memcpy(mean20, feat, sizeof(float) * N_MFCC);
    std::memcpy(std20, feat + N_MFCC, sizeof(float) * N_MFCC);
    if (dense40) std::memcpy(dense40, feat + FEAT, sizeof(float) * FEAT);
    return EWK_OK;
}

extern "C" int ewk_extract_mfcc(ewk_ctx* ctx, const float* pcm, int64_t n, int where, float* mean20, float* std20,
                                float* frames, int64_t frames_cap) {
    if (!ctx) return EWK_ERR_ARG;
    return extract_impl(ctx, pcm, n, where, mean20, std20, frames, frames_cap, nullptr);
}

static int check_slot(ewk_ctx* ctx, int slot, const char* who) {
    if (slot < 0 || slot >= ctx->cfg.max_templates) {
        ctx->fail("%s: template slot %d out of range [0, %d)", who, slot, ctx->cfg.max_templates);
        return EWK_ERR_ARG;
    }
    return EWK_OK;
}

static int install_template(ewk_ctx* ctx, int slot, const float* mean20, const float* std20, const float* dense40, int64_t n_samples) {
    CK(cudaSetDevice(ctx->device));
    TemplateFeat tf{};
    std::memcpy(tf.mean, mean20, sizeof(tf.mean));
    std::memcpy(tf.std, std20, sizeof(tf.std));
    // features for the dense kernel: its own integer statistics of the template's frames when the audio is known,
    // the given features otherwise
    std::memcpy(tf.dmean, dense40 ? dense40 : mean20, sizeof(tf.dmean));
    std::memcpy(tf.dstd, dense40 ? dense40 + N_MFCC : std20, sizeof(tf.dstd));
    tf.n_samples = n_samples;
    tf.valid = 1;
    ctx->h_tmpl[slot] = tf;
    ctx->dense_sets_forget(slot);
    CK(cudaMemcpyAsync(ctx->d_tmpl + slot, &ctx->h_tmpl[slot], sizeof(tf), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

// Template frame store: slot <- the 1 + n / HOP frames of a template of n samples, K3's frames_out at d_src (device), on
// the context's stream; a template over ALIGN_MAX_SAMPLES samples (the segments K11 takes) keeps none.
void ewk_ctx::store_frames(int slot, const float* d_src, long long n) {
    h_tfr_n[slot] = 0;
    if (!d_tfr || n > ALIGN_MAX_SAMPLES) return;
    const long long F = 1 + n / HOP;
    h_tfr_n[slot] = (int)F;
    cudaMemcpyAsync(d_tfr + (size_t)slot * ALIGN_MAX_FRAMES * N_MFCC, d_src, sizeof(float) * N_MFCC * (size_t)F,
                    cudaMemcpyDeviceToDevice, stream);
}

extern "C" int ewk_set_template_features(ewk_ctx* ctx, int slot, const float* mean20, const float* std20, int64_t n_samples) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = check_slot(ctx, slot, "ewk_set_template_features");
    if (rc) return rc;
    if (!mean20 || !std20 || n_samples < 1) { ctx->fail("ewk_set_template_features: null features or n_samples < 1"); return EWK_ERR_ARG; }
    ctx->h_tfr_n[slot] = 0;                                  // features without audio: no frames to align against
    return install_template(ctx, slot, mean20, std20, nullptr, n_samples);
}

extern "C" int ewk_set_template(ewk_ctx* ctx, int slot, const float* pcm, int64_t n) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = check_slot(ctx, slot, "ewk_set_template");
    if (rc) return rc;
    float mean[N_MFCC], sd[N_MFCC], dense[FEAT];
    rc = extract_impl(ctx, pcm, n, EWK_HOST, mean, sd, nullptr, 0, dense);
    if (rc) return rc;
    ctx->store_frames(slot, (const float*)ctx->b_frames.p, n);             // extract_impl left the frames there
    CK(cudaGetLastError());
    return install_template(ctx, slot, mean, sd, dense, n);
}

extern "C" int ewk_get_template(ewk_ctx* ctx, int slot, float* mean20, float* std20, int64_t* n_samples) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = check_slot(ctx, slot, "ewk_get_template");
    if (rc) return rc;
    const TemplateFeat& tf = ctx->h_tmpl[slot];
    if (!tf.valid) { ctx->fail("No reference word set. Call set_reference() first."); return EWK_ERR_NO_TEMPLATE; }
    if (mean20) std::memcpy(mean20, tf.mean, sizeof(tf.mean));
    if (std20) std::memcpy(std20, tf.std, sizeof(tf.std));
    if (n_samples) *n_samples = tf.n_samples;
    return EWK_OK;
}

extern "C" int ewk_clear_template(ewk_ctx* ctx, int slot) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = check_slot(ctx, slot, "ewk_clear_template");
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    ctx->h_tmpl[slot] = TemplateFeat{};
    ctx->h_tfr_n[slot] = 0;
    ctx->dense_sets_forget(slot);
    CK(cudaMemcpyAsync(ctx->d_tmpl + slot, &ctx->h_tmpl[slot], sizeof(TemplateFeat), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

extern "C" int ewk_similarity_batch(ewk_ctx* ctx, int slot, const void* pcm, int pcm_format, int where,
                                    const int64_t* offsets, const int64_t* lens, int n_seg, float threshold,
                                    float* scores, uint8_t* matched, float* features) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = check_slot(ctx, slot, "ewk_similarity_batch");
    if (rc) return rc;
    if (!ctx->h_tmpl[slot].valid) { ctx->fail("No reference word set. Call set_reference() first."); return EWK_ERR_NO_TEMPLATE; }
    if (n_seg == 0) return EWK_OK;
    if (!pcm || !offsets || !lens || n_seg < 0 || !scores || (pcm_format != EWK_PCM_F32 && pcm_format != EWK_PCM_I16)) {
        ctx->fail("ewk_similarity_batch: bad arguments");
        return EWK_ERR_ARG;
    }
    const size_t esz = pcm_format == EWK_PCM_I16 ? 2 : 4;
    int64_t extent = 0, spill = 0, lm_frames = 0;
    int max_frames = 1;
    std::vector<SegDesc> sd(n_seg);
    for (int i = 0; i < n_seg; i++) {
        if (offsets[i] < 0 || lens[i] < 1 || lens[i] > (int64_t)1 << 30) {
            ctx->fail("ewk_similarity_batch: segment %d has offset %lld len %lld", i, (long long)offsets[i], (long long)lens[i]);
            return EWK_ERR_ARG;
        }
        extent = std::max(extent, offsets[i] + lens[i]);
        const int F = 1 + (int)(lens[i] / HOP);
        max_frames = std::max(max_frames, F);
        sd[i] = SegDesc{};
        sd[i].start = offsets[i]; sd[i].ring = 0; sd[i].len = (int)lens[i]; sd[i].fmt = pcm_format == EWK_PCM_I16 ? 1 : 0;
        sd[i].ws_frame_off = (int)spill;
        if (F > SEG_SMEM_FRAMES) spill += F;
        sd[i].lm_off = lm_frames;
        lm_frames += F;
    }
    CK(cudaSetDevice(ctx->device));
    const void* d_pcm = pcm;
    if (where == EWK_HOST) {
        CK(ctx->b_pcm.ensure(esz * (size_t)extent));
        CK(cudaMemcpyAsync(ctx->b_pcm.p, pcm, esz * (size_t)extent, cudaMemcpyHostToDevice, ctx->stream));
        d_pcm = ctx->b_pcm.p;
    }
    for (int i = 0; i < n_seg; i++) sd[i].base = d_pcm;
    CK(ctx->b_desc.ensure(sizeof(SegDesc) * (size_t)n_seg));
    CK(cudaMemcpyAsync(ctx->b_desc.p, sd.data(), sizeof(SegDesc) * (size_t)n_seg, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx->b_feat.ensure(sizeof(float) * FEAT * (size_t)n_seg));
    CK(ctx->b_scores.ensure(sizeof(float) * (size_t)n_seg));
    CK(ctx->b_matched.ensure((size_t)n_seg));
    rc = ctx->launch_segments((const SegDesc*)ctx->b_desc.p, n_seg, max_frames, spill, lm_frames, 1, slot, threshold,
                              (float*)ctx->b_feat.p, nullptr, (float*)ctx->b_scores.p, (unsigned char*)ctx->b_matched.p);
    if (rc != EWK_OK) return rc;
    CK(cudaMemcpyAsync(scores, ctx->b_scores.p, sizeof(float) * (size_t)n_seg, cudaMemcpyDeviceToHost, ctx->stream));
    if (matched) CK(cudaMemcpyAsync(matched, ctx->b_matched.p, (size_t)n_seg, cudaMemcpyDeviceToHost, ctx->stream));
    if (features) CK(cudaMemcpyAsync(features, ctx->b_feat.p, sizeof(float) * FEAT * (size_t)n_seg, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

extern "C" int ewk_analyze_templates(ewk_ctx* ctx, const float* pcm, int where, const int64_t* offsets,
                                     const int64_t* lens, int n, ewk_vad_result* out, float* rms_out, int64_t rms_cap) {
    static_assert(sizeof(ewk_vad_result) == sizeof(VadResult) && sizeof(VadResult) == 32, "ewk_vad_result layout");
    if (!ctx) return EWK_ERR_ARG;
    if (n == 0) return EWK_OK;
    if (!pcm || !offsets || !lens || n < 0 || !out) { ctx->fail("ewk_analyze_templates: bad arguments"); return EWK_ERR_ARG; }
    int64_t extent = 0, frames = 0;
    std::vector<VadDesc> vd(n);
    for (int i = 0; i < n; i++) {
        if (offsets[i] < 0 || lens[i] < 0 || lens[i] > (int64_t)1 << 32) {
            ctx->fail("ewk_analyze_templates: template %d has offset %lld len %lld", i, (long long)offsets[i], (long long)lens[i]);
            return EWK_ERR_ARG;
        }
        extent = std::max(extent, offsets[i] + lens[i]);
        vd[i].start = offsets[i]; vd[i].len = lens[i]; vd[i].rms_off = frames;
        frames += 1 + lens[i] / VAD_HOP;
    }
    if (rms_out && rms_cap < frames) { ctx->fail("ewk_analyze_templates: rms_cap %lld < %lld frames", (long long)rms_cap, (long long)frames); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    const float* d_pcm = pcm;
    if (where == EWK_HOST) {
        CK(ctx->b_pcm.ensure(sizeof(float) * (size_t)std::max<int64_t>(extent, 1)));
        CK(cudaMemcpyAsync(ctx->b_pcm.p, pcm, sizeof(float) * (size_t)extent, cudaMemcpyHostToDevice, ctx->stream));
        d_pcm = (const float*)ctx->b_pcm.p;
    }
    for (int i = 0; i < n; i++) vd[i].base = d_pcm;
    CK(ctx->b_desc.ensure(sizeof(VadDesc) * (size_t)n));
    CK(cudaMemcpyAsync(ctx->b_desc.p, vd.data(), sizeof(VadDesc) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx->b_feat.ensure(sizeof(VadResult) * (size_t)n));
    CK(ctx->b_frames.ensure(sizeof(float) * (size_t)frames));
    cudaEvent_t pe = ctx->prof_begin(3);
    template_vad_kernel<<<n, VAD_THREADS, 0, ctx->stream>>>((const VadDesc*)ctx->b_desc.p, (VadResult*)ctx->b_feat.p,
                                                            (float*)ctx->b_frames.p);
    ctx->prof_end(pe, 3);
    CK(cudaGetLastError());
    ctx->launches++;
    CK(cudaMemcpyAsync(out, ctx->b_feat.p, sizeof(VadResult) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    if (rms_out) CK(cudaMemcpyAsync(rms_out, ctx->b_frames.p, sizeof(float) * (size_t)frames, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

// ---- batched enrolment: ewk_set_templates, ewk_set_templates_from_streams ----------------------------------------------
// The checks both entry points share; entry i is template i (rows of the ring form).
static int check_enrol(ewk_ctx* ctx, const char* who, const int32_t* slots, int n, const int64_t* offsets,
                       const int64_t* lens) {
    if (n < 0 || (n > 0 && (!slots || !offsets || !lens))) {
        ctx->fail("%s: bad arguments (n=%d, slots, offsets / starts and lens must not be NULL)", who, n);
        return EWK_ERR_ARG;
    }
    std::vector<char> seen((size_t)ctx->cfg.max_templates, 0);
    for (int i = 0; i < n; i++) {
        if (slots[i] < 0 || slots[i] >= ctx->cfg.max_templates) {
            ctx->fail("%s: entry %d: template slot %d out of range [0, %d)", who, i, slots[i], ctx->cfg.max_templates);
            return EWK_ERR_ARG;
        }
        if (seen[slots[i]]) { ctx->fail("%s: entry %d: template slot %d is listed twice", who, i, slots[i]); return EWK_ERR_ARG; }
        seen[slots[i]] = 1;
        if (offsets[i] < 0 || lens[i] < 1 || lens[i] > (int64_t)1 << 30) {
            ctx->fail("%s: entry %d (slot %d): offset %lld len %lld (need offset >= 0, 1 <= len <= 2^30)", who, i, slots[i],
                      (long long)offsets[i], (long long)lens[i]);
            return EWK_ERR_ARG;
        }
    }
    return EWK_OK;
}

// Where the templates' float32 audio comes from: host memory (copied to b_pcm first), device memory, or the rings
// (gather rows, packed into b_pcm by one gather launch; offsets are then the packed offsets).
struct EnrolSource { const float* pcm; int where; const std::vector<PrepDesc>* gather; };

// Templates slots[i] <- audio [offsets[i], offsets[i] + lens[i]) of the source, after check_enrol.  Launches: the gather
// (ring source), one K3 over all templates, one dense_template_install_kernel, one K6 when vad is given; one upload of
// every descriptor, one copy back of the features (and VAD results), one synchronisation.
static int enrol_impl(ewk_ctx* ctx, const char* who, const int32_t* slots, int n, const EnrolSource& src,
                      const int64_t* offsets, const int64_t* lens, ewk_vad_result* vad) {
    int64_t extent = 0, spill = 0, frames = 0;
    int max_frames = 1;
    for (int i = 0; i < n; i++) {
        extent = std::max(extent, offsets[i] + lens[i]);
        const int64_t F = 1 + lens[i] / HOP;
        max_frames = (int)std::max<int64_t>(max_frames, F);
        if (F > SEG_SMEM_FRAMES) spill += F;
        frames += F;
    }
    // K3 keeps every frame's log-mel row (the top_db floor's input) only up to LM_WS_MAX_BYTES; ewk_set_template always
    // does for one template, so a batch beyond it would take the other path
    if (ctx->use_lm && sizeof(float) * (size_t)frames * LM_ROW > ewk_ctx::LM_WS_MAX_BYTES) {
        ctx->fail("%s: the templates hold %lld frames together; one call takes at most %lld (split the batch)", who,
                  (long long)frames, (long long)(ewk_ctx::LM_WS_MAX_BYTES / (sizeof(float) * LM_ROW)));
        return EWK_ERR_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    int rc = ctx->join_match();                              // overlap mode: K3 of the last tick still reads the table
    if (rc) return rc;
    const float* d_pcm = src.pcm;
    if (src.where == EWK_HOST || src.gather) {
        CK(ctx->b_pcm.ensure(sizeof(float) * (size_t)extent));
        if (!src.gather) CK(cudaMemcpyAsync(ctx->b_pcm.p, src.pcm, sizeof(float) * (size_t)extent, cudaMemcpyHostToDevice, ctx->stream));
        d_pcm = (const float*)ctx->b_pcm.p;
    }
    // descriptors, one upload: SegDesc [n] | VadDesc [n] | int32 slots [n] | PrepDesc [gather rows]
    const size_t o_vad = sizeof(SegDesc) * (size_t)n, o_slot = o_vad + sizeof(VadDesc) * (size_t)n;
    const size_t o_gat = (o_slot + sizeof(int32_t) * (size_t)n + 15) & ~(size_t)15;
    const size_t n_gat = src.gather ? src.gather->size() : 0;
    std::vector<char> desc(o_gat + sizeof(PrepDesc) * n_gat);
    SegDesc* sd = reinterpret_cast<SegDesc*>(desc.data());
    VadDesc* vd = reinterpret_cast<VadDesc*>(desc.data() + o_vad);
    int64_t ws_off = 0, f_off = 0;
    for (int i = 0; i < n; i++) {
        const int64_t F = 1 + lens[i] / HOP;
        sd[i] = SegDesc{};
        sd[i].base = d_pcm; sd[i].start = offsets[i]; sd[i].ring = 0; sd[i].len = (int)lens[i]; sd[i].fmt = 0;
        sd[i].ws_frame_off = (int)ws_off; sd[i].frames_off = f_off; sd[i].lm_off = f_off;
        if (F > SEG_SMEM_FRAMES) ws_off += F;
        vd[i] = VadDesc{d_pcm, offsets[i], lens[i], f_off};
        f_off += F;
    }
    std::memcpy(desc.data() + o_slot, slots, sizeof(int32_t) * (size_t)n);
    if (n_gat) std::memcpy(desc.data() + o_gat, src.gather->data(), sizeof(PrepDesc) * n_gat);
    CK(ctx->b_desc.ensure(desc.size()));
    char* d_desc = (char*)ctx->b_desc.p;
    CK(cudaMemcpyAsync(d_desc, desc.data(), desc.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (n_gat) {
        int64_t longest = 0;
        for (const PrepDesc& g : *src.gather) longest = std::max<int64_t>(longest, g.len);
        const dim3 grid((unsigned)std::min<int64_t>(64, (longest + 1023) / 1024), (unsigned)n_gat);
        ring_gather_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->bank, (const PrepDesc*)(d_desc + o_gat), (float*)ctx->b_pcm.p);
        CK(cudaGetLastError());
        ctx->launches++;
    }
    // b_feat: K3 features [n][40] | dense features [n][40] | VadResult [n], copied back in one piece
    const size_t feat_bytes = sizeof(float) * 2 * FEAT * (size_t)n, back = feat_bytes + (vad ? sizeof(VadResult) * (size_t)n : 0);
    CK(ctx->b_feat.ensure(feat_bytes + sizeof(VadResult) * (size_t)n));
    CK(ctx->b_frames.ensure(sizeof(float) * (size_t)frames * N_MFCC));
    float* d_feat = (float*)ctx->b_feat.p;
    rc = ctx->launch_segments((const SegDesc*)d_desc, n, max_frames, spill, frames, 0, 0, 0.f, d_feat,
                              (float*)ctx->b_frames.p, nullptr, nullptr);
    if (rc != EWK_OK) return rc;
    dense_template_install_kernel<<<(n + ENROL_WARPS - 1) / ENROL_WARPS, ENROL_WARPS * 32, 0, ctx->stream>>>(
        (const SegDesc*)d_desc, (const int*)(d_desc + o_slot), n, ctx->cfg.n_mfcc > 0 ? ctx->cfg.n_mfcc : N_MFCC, (const float*)ctx->b_frames.p, d_feat,
        d_feat + (size_t)FEAT * n, ctx->d_tmpl);
    CK(cudaGetLastError());
    ctx->launches++;
    if (vad) {
        CK(ctx->b_scores.ensure(sizeof(float) * (size_t)frames));      // K6's frame RMS workspace
        cudaEvent_t pe = ctx->prof_begin(3);
        template_vad_kernel<<<n, VAD_THREADS, 0, ctx->stream>>>((const VadDesc*)(d_desc + o_vad),
                                                                (VadResult*)((char*)d_feat + feat_bytes), (float*)ctx->b_scores.p);
        ctx->prof_end(pe, 3);
        CK(cudaGetLastError());
        ctx->launches++;
    }
    // the template frame store: one device-to-device copy per template (no launch)
    for (int i = 0; i < n; i++) ctx->store_frames(slots[i], (const float*)ctx->b_frames.p + (size_t)sd[i].frames_off * N_MFCC,
                                                  lens[i]);
    CK(cudaGetLastError());
    std::vector<char> h(back);
    CK(cudaMemcpyAsync(h.data(), d_feat, back, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // the host mirror of what the install kernel wrote (install_template's fields)
    const float* hf = reinterpret_cast<const float*>(h.data());
    for (int i = 0; i < n; i++) {
        TemplateFeat tf{};
        std::memcpy(tf.mean, hf + (size_t)i * FEAT, sizeof(tf.mean));
        std::memcpy(tf.std, hf + (size_t)i * FEAT + N_MFCC, sizeof(tf.std));
        std::memcpy(tf.dmean, hf + (size_t)(n + i) * FEAT, sizeof(tf.dmean));
        std::memcpy(tf.dstd, hf + (size_t)(n + i) * FEAT + N_MFCC, sizeof(tf.dstd));
        tf.n_samples = lens[i];
        tf.valid = 1;
        ctx->h_tmpl[slots[i]] = tf;
        ctx->dense_sets_forget(slots[i]);
    }
    if (vad) std::memcpy(vad, h.data() + feat_bytes, sizeof(VadResult) * (size_t)n);
    return EWK_OK;
}

extern "C" int ewk_set_templates(ewk_ctx* ctx, const int32_t* slots, int n, const float* pcm, int where,
                                 const int64_t* offsets, const int64_t* lens, ewk_vad_result* vad) {
    if (!ctx) return EWK_ERR_ARG;
    const char* who = "ewk_set_templates";
    int rc = check_enrol(ctx, who, slots, n, offsets, lens);
    if (rc) return rc;
    if (n == 0) return EWK_OK;
    if (!pcm || (where != EWK_HOST && where != EWK_DEVICE)) {
        ctx->fail("%s: pcm must not be NULL and where must be EWK_HOST or EWK_DEVICE", who);
        return EWK_ERR_ARG;
    }
    return enrol_impl(ctx, who, slots, n, EnrolSource{pcm, where, nullptr}, offsets, lens, vad);
}

// ------------------------------------------------------------------------------------------ K7 resampling
extern "C" int ewk_resample_info(int sr_in, int32_t* half_width, int32_t* up, int32_t* down) {
    ResampleDesign d;
    if (sr_in < 1000 || sr_in > 768000 || !rs_design(sr_in, d)) return EWK_ERR_ARG;
    if (half_width) *half_width = d.W;
    if (up) *up = d.L;
    if (down) *down = d.M;
    return EWK_OK;
}

extern "C" int64_t ewk_resample_out_len(int64_t n_in, int sr_in) {
    if (n_in <= 0 || sr_in <= 0) return 0;
    return (int64_t)std::ceil((double)n_in * RS_TARGET / (double)sr_in);     // librosa.resample: int(np.ceil(n * ratio))
}

int ewk_ctx::resample_table(int sr_in, const ResampleTable** out) {
    ewk_ctx* ctx = this;
    auto it = rs_tables.find(sr_in);
    if (it == rs_tables.end()) {
        ResampleTable t;
        if (sr_in < 1000 || sr_in > 768000 || !rs_design(sr_in, t.d)) {
            fail("ewk_resample: %d Hz -> 16000 Hz is not supported (needs more than %d filter phases)", sr_in, RS_MAX_PHASES);
            return EWK_ERR_ARG;
        }
        std::vector<float> H;
        rs_build_table(t.d, H);
        CK(pool.alloc(&t.H, sizeof(float) * H.size(), "rs_table"));
        CK(cudaMemcpyAsync(t.H, H.data(), sizeof(float) * H.size(), cudaMemcpyHostToDevice, stream));
        CK(cudaStreamSynchronize(stream));
        it = rs_tables.emplace(sr_in, t).first;
    }
    *out = &it->second;
    return EWK_OK;
}

extern "C" int ewk_resample(ewk_ctx* ctx, const void* in, int pcm_format, int where_in, int n_rows, int64_t n_in,
                            int64_t in_stride, int sr_in, int64_t in_first, int64_t out_first, int64_t n_out, float* out,
                            int64_t out_stride, int where_out) {
    if (!ctx) return EWK_ERR_ARG;
    if (n_rows == 0 || n_out == 0) return EWK_OK;
    if (!in || !out || n_rows < 0 || n_in < 0 || n_out < 0 || in_stride < n_in || out_stride < n_out || out_first < 0 ||
        (pcm_format != EWK_PCM_F32 && pcm_format != EWK_PCM_I16) || n_in > (int64_t)1 << 34 || n_out > (int64_t)1 << 34) {
        ctx->fail("ewk_resample: bad arguments");
        return EWK_ERR_ARG;
    }
    if (sr_in == RS_TARGET) { ctx->fail("ewk_resample: input is already at 16000 Hz"); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    const ewk_ctx::ResampleTable* t = nullptr;
    int rc = ctx->resample_table(sr_in, &t);
    if (rc) return rc;
    const size_t esz = pcm_format == EWK_PCM_I16 ? 2 : 4;
    if (n_rows > 65535) { ctx->fail("ewk_resample: at most 65535 rows per call"); return EWK_ERR_ARG; }
    RsPushArgs A{};
    A.in = in; A.in_stride = in_stride;
    if (where_in == EWK_HOST) {
        CK(ctx->b_rs_in.ensure(esz * (size_t)n_rows * (size_t)std::max<int64_t>(n_in, 1)));
        if (n_in > 0)
            CK(cudaMemcpy2DAsync(ctx->b_rs_in.p, esz * (size_t)n_in, in, esz * (size_t)in_stride, esz * (size_t)n_in,
                                 (size_t)n_rows, cudaMemcpyHostToDevice, ctx->stream));
        A.in = ctx->b_rs_in.p; A.in_stride = n_in;
    }
    A.out = out; A.out_stride = out_stride;
    if (where_out == EWK_HOST) {
        CK(ctx->b_rs_out.ensure(sizeof(float) * (size_t)n_rows * (size_t)n_out));
        A.out = (float*)ctx->b_rs_out.p; A.out_stride = n_out;
    }
    // the input buffer is absolute samples [in_first, in_first + n_in), zeros elsewhere: no tail
    A.n_in = n_in; A.c = A.t0_old = A.t0_new = in_first; A.o0 = out_first; A.o1 = out_first + n_out;
    A.in_fmt = pcm_format; A.H = t->H; A.L = t->d.L; A.M = t->d.M; A.W = t->d.W;
    rc = ctx->launch_fir(*t, A, n_rows, 3, "ewk_resample");
    if (rc) return rc;
    if (where_out == EWK_HOST) {
        CK(cudaMemcpy2DAsync(out, sizeof(float) * (size_t)out_stride, ctx->b_rs_out.p, sizeof(float) * (size_t)n_out,
                             sizeof(float) * (size_t)n_out, (size_t)n_rows, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return EWK_OK;
}

// ==========================================================================================
// stream bank
// ==========================================================================================
static_assert(sizeof(StreamParams) == sizeof(ewk_stream_params), "ewk_stream_params layout");
static_assert(sizeof(EventRec) == sizeof(ewk_event), "ewk_event layout");
static_assert(sizeof(StreamResult) == sizeof(ewk_stream_result), "ewk_stream_result layout");
constexpr int MIN_FRAME_SIZE = 160;
constexpr int GATE_SMEM_CHUNKS = 2048;   // storage-order chunks a warp of K2 can hold in shared memory (3 arrays x 4 warps)

extern "C" int ewk_default_stream_params(ewk_stream_params* p) {
    if (!p) return EWK_ERR_ARG;
    std::memset(p, 0, sizeof(*p));
    p->similarity_threshold = 75.0f;
    p->frame_size = 0;
    p->pre_speech_silence = 0.8;
    p->speech_duration_min = 0.3;
    p->speech_duration_max = 2.0;
    p->post_speech_silence = 0.4;
    p->timeout = 30.0;
    p->min_threshold = 0.005;
    p->template_first = 0;
    p->template_count = 1;
    p->live = 0;
    return EWK_OK;
}

int ewk_ctx::init_streams() {
    ewk_ctx* ctx = this;
    const int n = cfg.n_streams;
    if (n == 0) return EWK_OK;
    const size_t esz = cfg.pcm_format == EWK_PCM_I16 ? 2 : 4;
    bank.n_streams = n;
    bank.R = cfg.ring_samples;
    bank.P = ((cfg.ring_samples + cfg.slack_samples + 63) / 64) * 64;
    bank.fmt = cfg.pcm_format == EWK_PCM_I16 ? 1 : 0;
    chunk_cap = std::max(1, cfg.ring_samples / MIN_FRAME_SIZE);
    bank.chunk_cap = chunk_cap;
    bank.max_events = std::max(16, cfg.max_events);
    CK(pool.alloc(&bank.ring, esz * (size_t)n * bank.P, "bank.ring"));
    CK(cudaMemsetAsync(bank.ring, 0, esz * (size_t)n * bank.P, stream));          // np.zeros   wakeword.py:428
    CK(pool.alloc(&bank.st, sizeof(StreamState) * (size_t)n, "bank.st"));
    CK(pool.alloc(&bank.prm, sizeof(StreamParams) * (size_t)n, "bank.prm"));
    CK(pool.alloc(&bank.chunk_ms, sizeof(double) * (size_t)n * 2 * chunk_cap, "bank.chunk_ms"));   // per stream: ms[cap] ++ sorted[cap]
    // K2 reads only chunks below chunks_valid, but K10 copies whole rows into blobs: zeros keep a blob's bytes a function of
    // the stream's history
    CK(cudaMemsetAsync(bank.chunk_ms, 0, sizeof(double) * (size_t)n * 2 * chunk_cap, stream));
    CK(pool.alloc(&bank.events, sizeof(EventRec) * (size_t)bank.max_events, "bank.events"));
    CK(pool.alloc(&bank.ev_count, sizeof(int) * 8, "bank.ev_count"));
    CK(cudaMemsetAsync(bank.ev_count, 0, sizeof(int) * 8, stream));
    CK(pool.alloc(&bank.bk_count, sizeof(int) * SEG_NB, "bank.bk_count"));
    CK(cudaMemsetAsync(bank.bk_count, 0, sizeof(int) * SEG_NB, stream));
    CK(pool.alloc(&bank.bk_list, sizeof(int) * (size_t)SEG_NB * bank.max_events, "bank.bk_list"));
#ifdef EWK_K3_TRACE
    if (getenv("EWK_K3_TRACE")) {
        CK(pool.alloc(&bank.k3_trace, sizeof(long long) * K3_TRACE_WORDS * (size_t)queue_grid(), "bank.k3_trace"));
        CK(cudaMemsetAsync(bank.k3_trace, 0, sizeof(long long) * K3_TRACE_WORDS * (size_t)queue_grid(), stream));
    }
#endif

    bank.NB = bank.P / TICK;
    CK(pool.alloc(&bank.block_ss, sizeof(double) * (size_t)n * std::max(1, bank.NB), "bank.block_ss"));
    CK(cudaMemsetAsync(bank.block_ss, 0, sizeof(double) * (size_t)n * std::max(1, bank.NB), stream));   // as chunk_ms
    CK(pool.alloc(&own_results, sizeof(StreamResult) * (size_t)n, "own_results"));
    bank.results = (StreamResult*)own_results;
    if (const char* e = getenv("EWK_K3")) k3_frames = atoi(e) == 2;      // EWK_K3=2: the frame-parallel form (measured, not the default)
    if (!k3_frames) {
        if (use_lm) CK(pool.alloc(&bank.lm_ws, sizeof(float) * (size_t)queue_grid() * SEG_SMEM_FRAMES * LM_ROW, "bank.lm_ws"));
    } else {
        // frame-parallel K3: a frame table for the candidates of ONE ewk_tick call (it restarts after every K3 launch)
        const size_t cap = std::min<size_t>((size_t)bank.max_events * SEG_SMEM_FRAMES, ((size_t)2 << 30) / (FROW * sizeof(float)));
        bank.frow_cap = (int)cap;
        CK(pool.alloc(&bank.frow, sizeof(float) * FROW * cap, "bank.frow"));
        CK(pool.alloc(&bank.frame_ev, sizeof(int) * cap, "bank.frame_ev"));
        CK(pool.alloc(&bank.ev_done, sizeof(int) * (size_t)bank.max_events, "bank.ev_done"));
    }
    std::vector<StreamState> st(n);
    std::memset(st.data(), 0, sizeof(StreamState) * n);
    for (auto& x : st) { x.thr = 0.01; x.last_ev = -1; }                            // wakeword.py:431
    CK(cudaMemcpyAsync(bank.st, st.data(), sizeof(StreamState) * n, cudaMemcpyHostToDevice, stream));
    ewk_stream_params dp;
    ewk_default_stream_params(&dp);
    StreamParams sp;
    std::memcpy(&sp, &dp, sizeof(sp));
    h_prm.assign(n, sp);
    max_post = sp.post_speech_silence;
    CK(cudaMemcpyAsync(bank.prm, h_prm.data(), sizeof(StreamParams) * n, cudaMemcpyHostToDevice, stream));
    std::vector<StreamResult> rs(n);
    for (auto& r : rs) { r.score = std::nanf(""); r.flags = 0; }
    CK(cudaMemcpyAsync(bank.results, rs.data(), sizeof(StreamResult) * n, cudaMemcpyHostToDevice, stream));
    CK(cudaStreamSynchronize(stream));
    h_written.assign(n, 0);
    h_visible_lb.assign(n, 0);
    h_tick.assign(n, 0);
    h_dense_next.assign(n, 1);
    h_det_next.assign(n, 1);
    h_frame_size.assign(n, 0);
    h_rate.assign(n, 0);
    h_inputs.assign(n, 0);
    CK(cudaFuncSetAttribute(segment_queue_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)seg_smem_bytes(SEG_SMEM_FRAMES)));
    CK(cudaFuncSetAttribute(segment_queue_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)seg_smem_bytes(SEG_SMEM_FRAMES)));
    CK(cudaFuncSetAttribute(segment_frames_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fq_smem_bytes()));
    CK(cudaFuncSetAttribute(segment_frames_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fq_smem_bytes()));
    CK(cudaFuncSetAttribute(ring_push_bulk_kernel<short>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    CK(cudaFuncSetAttribute(ring_push_bulk_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    {
        const size_t big = sizeof(double) * 3 * (size_t)(std::min(chunk_cap, GATE_SMEM_CHUNKS) + 1) * GATE_WARPS;
        const size_t staged = sizeof(double) * 3 * (size_t)130 * GATE_WARPS + (size_t)2 * TICK * 4 * GATE_WARPS;
        CK(cudaFuncSetAttribute(tick_gate_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(big, staged)));
        CK(cudaFuncSetAttribute(tick_gate_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max(big, staged)));
    }
    return EWK_OK;
}

void ewk_ctx::release_streams() {
#ifdef EWK_K3_TRACE
    if (bank.k3_trace) {                          // the last launch's timeline -> $EWK_K3_TRACE (raw int64 [CTAs][K3_TRACE_WORDS])
        cudaDeviceSynchronize();
        std::vector<long long> h((size_t)K3_TRACE_WORDS * queue_grid());
        cudaMemcpy(h.data(), bank.k3_trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        if (FILE* f = fopen(getenv("EWK_K3_TRACE"), "wb")) { fwrite(h.data(), sizeof(long long), h.size(), f); fclose(f); }
        pool.free(bank.k3_trace);
    }
#endif
    if (d_rs_tail) { pool.free(d_rs_tail); d_rs_tail = nullptr; rs_tail_cap = 0; }
    for (void* p : {bank.ring, (void*)bank.st, (void*)bank.prm, (void*)bank.chunk_ms, (void*)bank.events,
                    (void*)bank.ev_count, (void*)bank.block_ss, (void*)bank.lm_ws, own_results, (void*)bank.frow,
                    (void*)bank.frame_ev, (void*)bank.ev_done, (void*)bank.bk_count, (void*)bank.bk_list})
        if (p) pool.free(p);
    bank = BankView{};
    own_results = nullptr;
    b_trace.free(); b_read.free(); b_dense.free(); b_keep_rows.free(); b_keep_end.free(); b_g2.free(); b_det_state.free();
    for (auto& p : prof_pairs) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    for (auto e : prof_free) cudaEventDestroy(e);
    prof_pairs.clear(); prof_free.clear();
}

int ewk_ctx::gate_chunks() const {
    int m = 1;
    for (int s = 0; s < bank.n_streams; s++) {
        const int fs = h_frame_size[s] > 0 ? h_frame_size[s] : h_prm[s].frame_size;
        if (fs > 0) m = std::max(m, std::min(bank.chunk_cap, bank.R / fs));
    }
    return m;
}

// Makes the context's stream wait for a K3 launch that is still running on the match stream (overlap mode).
int ewk_ctx::join_match() {
    ewk_ctx* ctx = this;
    if (!match_inflight) return EWK_OK;
    match_inflight = false;
    CK(cudaStreamWaitEvent(stream, ev_match, 0));
    return EWK_OK;
}

// Every stream-bank entry point starts here.  All of them except ewk_push order themselves after an in-flight K3.
static int need_streams(ewk_ctx* ctx, const char* who, bool join = true) {
    if (ctx->bank.n_streams == 0) { ctx->fail("%s: context was created with n_streams = 0", who); return EWK_ERR_STATE; }
    if (join) return ctx->join_match();
    return EWK_OK;
}

extern "C" int ewk_set_overlap(ewk_ctx* ctx, int enable) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_set_overlap");
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    if (enable && !ctx->match_stream) {
        CK(cudaStreamCreateWithFlags(&ctx->match_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->ev_gate, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ctx->ev_match, cudaEventDisableTiming));
    }
    ctx->overlap = enable != 0;
    return EWK_OK;
}

extern "C" int ewk_join(ewk_ctx* ctx) {
    if (!ctx) return EWK_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    return ctx->join_match();
}

extern "C" int64_t ewk_launch_count(const ewk_ctx* ctx) { return ctx ? ctx->launches : 0; }

extern "C" int ewk_set_stream_params(ewk_ctx* ctx, int stream, const ewk_stream_params* p) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_set_stream_params");
    if (rc) return rc;
    const int n = ctx->bank.n_streams;
    if (!p || stream < -1 || stream >= n) { ctx->fail("ewk_set_stream_params: bad stream %d", stream); return EWK_ERR_ARG; }
    // the reference's constructor checks (wakeword.py:752-763), same messages
    if (!(p->pre_speech_silence > 0)) { ctx->fail("pre_speech_silence must be positive"); return EWK_ERR_ARG; }
    if (!(p->speech_duration_min > 0)) { ctx->fail("speech_duration_min must be positive"); return EWK_ERR_ARG; }
    if (!(p->speech_duration_max > 0)) { ctx->fail("speech_duration_max must be positive"); return EWK_ERR_ARG; }
    if (p->speech_duration_min > p->speech_duration_max) { ctx->fail("speech_duration_min must be <= speech_duration_max"); return EWK_ERR_ARG; }
    if (!(p->post_speech_silence > 0)) { ctx->fail("post_speech_silence must be positive"); return EWK_ERR_ARG; }
    if (p->frame_size != 0 && (p->frame_size < MIN_FRAME_SIZE || p->frame_size > ctx->bank.R)) {
        ctx->fail("frame_size must be 0 or in [%d, %d]", MIN_FRAME_SIZE, ctx->bank.R);
        return EWK_ERR_ARG;
    }
    if (p->template_first < 0 || p->template_count < 0 || p->template_first + p->template_count > ctx->cfg.max_templates) {
        ctx->fail("template range [%d, %d) outside [0, %d)", p->template_first, p->template_first + p->template_count, ctx->cfg.max_templates);
        return EWK_ERR_ARG;
    }
    if (p->template_count > EWK_MAX_STREAM_TEMPLATES) {
        ctx->fail("template_count %d above EWK_MAX_STREAM_TEMPLATES (%d): a stream is scored against at most %d slots",
                  p->template_count, EWK_MAX_STREAM_TEMPLATES, EWK_MAX_STREAM_TEMPLATES);
        return EWK_ERR_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    StreamParams sp;
    std::memcpy(&sp, p, sizeof(sp));
    const int a = stream < 0 ? 0 : stream, b = stream < 0 ? n : stream + 1;
    for (int s = a; s < b; s++) ctx->h_prm[s] = sp;
    ctx->max_post = 0.0;
    for (int s = 0; s < n; s++) ctx->max_post = std::max(ctx->max_post, ctx->h_prm[s].post_speech_silence);
    CK(cudaMemcpyAsync(ctx->bank.prm + a, ctx->h_prm.data() + a, sizeof(StreamParams) * (size_t)(b - a),
                       cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

// K1 on device-resident PCM (caller's buffer or a staging slot): rings <- src, per-block sums, bookkeeping.
int ewk_ctx::land(int stream0, int n_streams, const void* d_src, long long d_stride, long long n, int stage_slot) {
    ewk_ctx* ctx = this;
    BankView& B = bank;
    const size_t esz = B.fmt == 1 ? 2 : 4;
    int with_sums = 0;
    // fused copy + per-block sums when every stream of the push sits on a 0.1 s block boundary
    bool aligned = (n % TICK) == 0 && (B.P % TICK) == 0 && B.NB > 0 && ((size_t)d_src & 15) == 0 && ((d_stride * esz) & 15) == 0;
    for (int s = stream0; aligned && s < stream0 + n_streams; s++) aligned = (h_written[s] % TICK) == 0;
    if (stage_slot >= 0) CK(cudaStreamWaitEvent(stream, ev_ready[stage_slot], 0));
    cudaEvent_t pe = prof_begin(0);
    static const int bulk_env = [] { const char* e = getenv("EWK_PUSH_BULK"); return e ? atoi(e) : 1; }();
    if (aligned && bulk_env && match_inflight && (long long)n_streams * (n / TICK) >= 4LL * sm_count * PUSH_BULK_WARPS) {
        // TMA form while K3 is running on the match stream: persistent CTAs of two warps whose bytes in flight sit in
        // shared-memory stages, small enough (2.5 k registers, 26 KB) to share the SMs with K3's CTAs.  Alone, the
        // register-staged kernel below is faster (47 vs 60 us at 4096 x 1.0 s), so it keeps the sequential case.
        static const int env_stages = [] { const char* e = getenv("EWK_PUSH_STAGES"); return e ? atoi(e) : 0; }();
        static const int env_grid = [] { const char* e = getenv("EWK_PUSH_GRID"); return e ? atoi(e) : 0; }();
        const int stages = env_stages > 0 ? env_stages : (B.fmt == 1 ? 4 : 2);
        const size_t smem = (size_t)PUSH_BULK_WARPS * stages * TICK * esz + sizeof(unsigned long long) * PUSH_BULK_WARPS * stages;
        const int grid = (env_grid > 0 ? env_grid : 2) * sm_count;
        if (B.fmt == 1) ring_push_bulk_kernel<short><<<grid, PUSH_BULK_WARPS * 32, smem, stream>>>(B, stream0, n_streams, (const short*)d_src, d_stride, (int)n, stages);
        else ring_push_bulk_kernel<float><<<grid, PUSH_BULK_WARPS * 32, smem, stream>>>(B, stream0, n_streams, (const float*)d_src, d_stride, (int)n, stages);
        with_sums = 1;
    } else if (aligned) {
        dim3 grid((unsigned)((n / TICK + 3) / 4), (unsigned)n_streams);
        if (B.fmt == 1) ring_push_sums_kernel<short><<<grid, 128, 0, stream>>>(B, stream0, (const short*)d_src, d_stride, (int)n);
        else ring_push_sums_kernel<float><<<grid, 128, 0, stream>>>(B, stream0, (const float*)d_src, d_stride, (int)n);
        with_sums = 1;
    } else {
        const int per = esz == 2 ? 8 : 4;
        dim3 grid((unsigned)std::max<long long>(1, std::min<long long>(64, (n / per + 255) / 256)), (unsigned)n_streams);
        if (B.fmt == 1) ring_push_kernel<short><<<grid, 256, 0, stream>>>(B, stream0, (const short*)d_src, d_stride, (int)n);
        else ring_push_kernel<float><<<grid, 256, 0, stream>>>(B, stream0, (const float*)d_src, d_stride, (int)n);
    }
    prof_end(pe, 0);
    CK(cudaGetLastError());
    launches++;
    if (stage_slot >= 0) {
        CK(cudaEventRecord(ev_free[stage_slot], stream));
        ev_free_valid[stage_slot] = true;
    }
    ring_commit_kernel<<<(n_streams + 255) / 256, 256, 0, stream>>>(B, stream0, n_streams, (int)n, with_sums);
    CK(cudaGetLastError());
    launches++;
    // do the per-block sums of K1 cover everything pushed since the last tick, for every stream?
    if (!with_sums) all_presummed = false;
    else if (stream0 == 0 && n_streams == B.n_streams && pushes_since_tick == 0) all_presummed = true;
    pushes_since_tick++;
    for (int s = stream0; s < stream0 + n_streams; s++) {
        h_written[s] += n;
        if (h_frame_size[s] == 0) h_frame_size[s] = h_prm[s].frame_size > 0 ? h_prm[s].frame_size : (int)n;
    }
    return EWK_OK;
}

// A host push whose H2D copy is in flight on the copy stream lands (K1) only when something needs its samples:
// the next push, a tick that reaches into it, or any read of stream state.  That keeps K1(i+1) — which must wait
// for its copy — out of the way of the kernels of step i on the compute stream, so copy and compute overlap.
int ewk_ctx::flush_pending() {
    if (!pending.valid) return EWK_OK;
    pending.valid = false;
    if (pending.rs_rate) {
        const bool each = pending.rows_slot >= 0;
        return land_resampled(pending.stream0, pending.n_streams, b_raw[pending.slot].p, pending.rs_n_in, pending.rs_fmt,
                              pending.rs_n_in, pending.rs_rate, pending.rs_c, each ? pending.rows.data() : nullptr,
                              pending.rows_slot, pending.n_items, pending.slot);
    }
    if (pending.rows_slot >= 0)
        return land_list(pending.rows, pending.rows_slot, pending.n_items, b_raw[pending.slot].p, pending.rs_fmt, pending.slot);
    return land(pending.stream0, pending.n_streams, b_stage2[pending.slot].p, pending.n, pending.n, pending.slot);
}

// A stream's input rate is fixed by its first push: 16 kHz pushes (ewk_push, ewk_push_g711) refuse a native-rate stream.
static int check_16k(ewk_ctx* ctx, const char* who, int stream0, int n_streams) {
    for (int s = stream0; s < stream0 + n_streams; s++)
        if (ctx->h_rate[s] != 0 && ctx->h_rate[s] != RS_TARGET) {
            ctx->fail("%s: stream %d takes %d Hz input through ewk_push_resampled", who, s, ctx->h_rate[s]);
            return EWK_ERR_STATE;
        }
    return EWK_OK;
}

static void latch_16k(ewk_ctx* ctx, int stream0, int n_streams, long long n) {
    for (int s = stream0; s < stream0 + n_streams; s++) { ctx->h_rate[s] = RS_TARGET; ctx->h_inputs[s] += n; }
}

extern "C" int ewk_push(ewk_ctx* ctx, int stream0, int n_streams, const void* pcm, int64_t n, int64_t stride, int where) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_push", false);        // a push does not wait for the matching of the previous ticks
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (!pcm || n_streams < 1 || stream0 < 0 || stream0 + n_streams > B.n_streams || n < 1 || stride < n) {
        ctx->fail("ewk_push: bad arguments (stream0=%d n_streams=%d n=%lld stride=%lld)", stream0, n_streams, (long long)n, (long long)stride);
        return EWK_ERR_ARG;
    }
    if (n > B.P - B.R && n > B.R) { ctx->fail("ewk_push: %lld samples exceed the ring (%d)", (long long)n, B.R); return EWK_ERR_ARG; }
    rc = check_16k(ctx, "ewk_push", stream0, n_streams);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();
    if (rc) return rc;
    // audio-clock streams: the push may not overwrite samples a pending tick still has to see
    for (int s = stream0; s < stream0 + n_streams; s++) {
        if (ctx->h_prm[s].live) continue;
        const long long ahead = ctx->h_written[s] + n - ctx->h_visible_lb[s];
        if (ctx->h_visible_lb[s] >= B.R && ahead > (long long)(B.P - B.R)) {
            ctx->fail("ewk_push: stream %d would hold %lld un-gated samples, more than slack_samples=%d; call ewk_tick first",
                      s, ahead, B.P - B.R);
            return EWK_ERR_STATE;
        }
        // before the first full tick every sample from 0 upward is still needed (the first-full tick forms all chunks
        // from samples): nothing may wrap onto them
        if (ctx->h_visible_lb[s] < B.R && ctx->h_written[s] + n > (long long)B.P) {
            ctx->fail("ewk_push: stream %d would hold %lld samples before its first full tick, more than the physical ring "
                      "(%d); call ewk_tick first", s, ctx->h_written[s] + n, B.P);
            return EWK_ERR_STATE;
        }
    }
    const size_t esz = B.fmt == 1 ? 2 : 4;
    latch_16k(ctx, stream0, n_streams, n);
    if (where != EWK_HOST) return ctx->land(stream0, n_streams, pcm, stride, n, -1);
    // Host PCM: H2D on a dedicated copy stream into one of two staging buffers.  Contiguous sources
    // ([n_streams][n]) go as ONE linear copy (55 GB/s over PCIe 5 vs 47 GB/s pitched).
    const int b = ctx->stage_idx;
    ctx->stage_idx ^= 1;
    CK(ctx->b_stage2[b].ensure(esz * (size_t)n * n_streams));
    if (ctx->ev_free_valid[b]) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_free[b], 0));
    if (stride == n)
        CK(cudaMemcpyAsync(ctx->b_stage2[b].p, pcm, esz * (size_t)n * n_streams, cudaMemcpyHostToDevice, ctx->copy_stream));
    else
        CK(cudaMemcpy2DAsync(ctx->b_stage2[b].p, (size_t)n * esz, pcm, (size_t)stride * esz, (size_t)n * esz, n_streams,
                             cudaMemcpyHostToDevice, ctx->copy_stream));
    CK(cudaEventRecord(ctx->ev_ready[b], ctx->copy_stream));
    ctx->pending = ewk_ctx::Pending{};
    ctx->pending.valid = true; ctx->pending.slot = b; ctx->pending.stream0 = stream0; ctx->pending.n_streams = n_streams;
    ctx->pending.n = n;
    return EWK_OK;
}

// G.711 feed: 8-bit mu-law (law 0) / A-law (law 1) codes, expanded on the device to the 16-bit samples of the standard
// and pushed like PCM16.  Host codes cross PCIe at one byte per sample; the expansion (K0) runs on the copy stream right
// behind the copy, into the same double-buffered staging the PCM path uses, and lands lazily like any host push.
extern "C" int ewk_push_g711(ewk_ctx* ctx, int stream0, int n_streams, const uint8_t* codes, int64_t n, int64_t stride, int where, int law) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_push_g711", false);
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (B.fmt != 1) { ctx->fail("ewk_push_g711: the context's rings must be int16 (pcm_format EWK_PCM_I16)"); return EWK_ERR_STATE; }
    if (!codes || n_streams < 1 || stream0 < 0 || stream0 + n_streams > B.n_streams || n < 1 || stride < n || law < 0 || law > 1) {
        ctx->fail("ewk_push_g711: bad arguments (stream0=%d n_streams=%d n=%lld stride=%lld law=%d)", stream0, n_streams,
                  (long long)n, (long long)stride, law);
        return EWK_ERR_ARG;
    }
    if (n > B.P - B.R && n > B.R) { ctx->fail("ewk_push_g711: %lld samples exceed the ring (%d)", (long long)n, B.R); return EWK_ERR_ARG; }
    rc = check_16k(ctx, "ewk_push_g711", stream0, n_streams);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();
    if (rc) return rc;
    for (int s = stream0; s < stream0 + n_streams; s++) {     // same guard as ewk_push
        if (ctx->h_prm[s].live) continue;
        const long long ahead = ctx->h_written[s] + n - ctx->h_visible_lb[s];
        if (ctx->h_visible_lb[s] >= B.R && ahead > (long long)(B.P - B.R)) {
            ctx->fail("ewk_push_g711: stream %d would hold %lld un-gated samples, more than slack_samples=%d; call ewk_tick first",
                      s, ahead, B.P - B.R);
            return EWK_ERR_STATE;
        }
        // before the first full tick every sample from 0 upward is still needed (the first-full tick forms all chunks
        // from samples): nothing may wrap onto them
        if (ctx->h_visible_lb[s] < B.R && ctx->h_written[s] + n > (long long)B.P) {
            ctx->fail("ewk_push_g711: stream %d would hold %lld samples before its first full tick, more than the physical ring "
                      "(%d); call ewk_tick first", s, ctx->h_written[s] + n, B.P);
            return EWK_ERR_STATE;
        }
    }
    latch_16k(ctx, stream0, n_streams, n);
    const int b = ctx->stage_idx;
    ctx->stage_idx ^= 1;
    CK(ctx->b_stage2[b].ensure(sizeof(short) * (size_t)n * n_streams));
    if (ctx->ev_free_valid[b]) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_free[b], 0));
    const unsigned char* d_codes = codes;
    long long d_stride = stride;
    if (where == EWK_HOST) {
        CK(ctx->b_raw[b].ensure((size_t)n * n_streams));
        if (stride == n)
            CK(cudaMemcpyAsync(ctx->b_raw[b].p, codes, (size_t)n * n_streams, cudaMemcpyHostToDevice, ctx->copy_stream));
        else
            CK(cudaMemcpy2DAsync(ctx->b_raw[b].p, (size_t)n, codes, (size_t)stride, (size_t)n, n_streams, cudaMemcpyHostToDevice, ctx->copy_stream));
        d_codes = (const unsigned char*)ctx->b_raw[b].p;
        d_stride = n;
    } else {
        // device-resident codes were produced on the context's stream: the copy stream starts behind it
        CK(cudaEventRecord(ctx->ev_ready[b], ctx->stream));
        CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_ready[b], 0));
    }
    const long long work = (long long)n * n_streams / 16 + 1;
    const int grid = (int)std::min<long long>((work + 255) / 256, 8LL * ctx->sm_count);
    g711_decode_kernel<<<grid, 256, 0, ctx->copy_stream>>>(d_codes, (short*)ctx->b_stage2[b].p, n_streams, (long long)n, d_stride, law);
    CK(cudaGetLastError());
    ctx->launches++;
    CK(cudaEventRecord(ctx->ev_ready[b], ctx->copy_stream));
    ctx->pending = ewk_ctx::Pending{};
    ctx->pending.valid = true; ctx->pending.slot = b; ctx->pending.stream0 = stream0; ctx->pending.n_streams = n_streams;
    ctx->pending.n = n;
    return EWK_OK;
}

// ------------------------------------------------------------------------------------------ K8 native-rate push
// outputs whose W inputs of look-ahead have arrived after c inputs (StreamResampler.push's rule)
static long long rs_ready(long long c, const ResampleDesign& d) {
    const long long a = c - d.W;
    return a <= 0 ? 0 : (a * d.L + d.M - 1) / d.M;
}
// first input sample any output from ready(c) on reads
static long long rs_tail_start(long long c, const ResampleDesign& d) {
    return std::max(0LL, rs_ready(c, d) * d.M / d.L - d.W + 1);
}
static size_t rs_in_size(int in_fmt) { return in_fmt == EWK_PCM_F32 ? 4 : in_fmt == EWK_PCM_I16 ? 2 : 1; }

// K8's work mapping for a rate: fast or generic path, outputs per tile, staged input span
struct FirPlan { int fast_m, tile, span, table_smem; };
static FirPlan fir_plan(const ResampleDesign& d) {
    FirPlan f{};
    const int taps = 2 * d.W;
    f.table_smem = (long long)taps * d.L <= RSP_TABLE_SMEM;
    // fast path: warp-uniform phases and register windows; its tile must leave the tail (if any) to CTA 0 alone
    if ((d.L == 1 || d.L == 2 || d.L == 4 || d.L == 8) && d.M <= 3 && f.table_smem &&
        (RSP_THREADS / d.L) * rsp_k(d.M) * d.M >= taps + d.M)
        f.fast_m = d.M;
    if (f.fast_m) {
        f.tile = RSP_THREADS * rsp_k(d.M);
        f.span = (RSP_THREADS / d.L) * rsp_k(d.M) * d.M + taps + d.M + 1;
    } else {
        auto span = [&](long long tile) { return (tile * d.M + d.L - 1) / d.L + taps + 1; };
        long long tile = RSP_GENERIC_TILE;
        while (tile > RSP_THREADS && span(tile) > 24576) tile /= 2;
        const long long need = ((long long)taps * d.L + d.M - 1) / d.M;      // tile M / L >= 2W: CTAs >= 1 start past the tail
        tile = std::max(tile, (need + RSP_THREADS - 1) / RSP_THREADS * RSP_THREADS);
        f.tile = (int)tile;
        f.span = (int)span(tile);
    }
    return f;
}
// output tiles of a row: its outputs [o0, o1) from the first tile start (fast path: o0 rounded down to a phase group)
static long long fir_tiles(const FirPlan& f, const ResampleDesign& d, long long o0, long long o1) {
    const long long first = f.fast_m ? (o0 / d.L) * d.L : o0;
    return std::max<long long>(1, (o1 - first + f.tile - 1) / f.tile);
}

// The FIR (K8) over rows [0, n_rows) of A: plans the work mapping and launches.
int ewk_ctx::launch_fir(const ResampleTable& t, RsPushArgs& A, int n_rows, int prof_cls, const char* who,
                        long long n_items) {
    ewk_ctx* ctx = this;
    const ResampleDesign& d = t.d;
    const int taps = 2 * d.W;
    const FirPlan f = fir_plan(d);
    const int fast_m = f.fast_m;
    A.table_smem = f.table_smem; A.tile = f.tile; A.span = f.span;
    const size_t smem = sizeof(float) * ((size_t)256 + A.tail_cap + (A.table_smem ? (size_t)taps * d.L : 0) + A.span);
    if (smem > (size_t)200 * 1024) { fail("%s: %d Hz needs %zu bytes of shared memory", who, d.sr_in, smem); return EWK_ERR_ARG; }
    // per-row descriptors: one flat list of every row's tiles, so that rows of very different lengths leave no CTA idle
    const dim3 grid = A.rows ? dim3((unsigned)n_items, 1) : dim3((unsigned)fir_tiles(f, d, A.o0, A.o1), (unsigned)n_rows);
    auto pick = [&](auto each) {
        constexpr bool E = decltype(each)::value;
        return fast_m == 1 ? resample_push_kernel<1, E> : fast_m == 2 ? resample_push_kernel<2, E>
             : fast_m == 3 ? resample_push_kernel<3, E> : resample_push_kernel<0, E>;
    };
    auto k8 = A.rows ? pick(std::true_type{}) : pick(std::false_type{});
    CK(cudaFuncSetAttribute(k8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEvent_t pe = prof_begin(prof_cls);
    k8<<<grid, RSP_THREADS, smem, stream>>>(bank, A);
    prof_end(pe, prof_cls);
    CK(cudaGetLastError());
    launches++;
    return EWK_OK;
}

// K8 on device-resident input (the caller's buffer or a staging slot): uniform rows from position c, or per-row
// descriptors (see ewk_ctx.hpp)
int ewk_ctx::land_resampled(int stream0, int n_streams, const void* d_src, long long d_stride, int in_fmt, long long n_in,
                            int sr_in, long long c, const RowDesc* rows, int rows_slot, long long n_items, int stage_slot) {
    ewk_ctx* ctx = this;
    const ResampleTable* t = nullptr;
    int rc = resample_table(sr_in, &t);
    if (rc) return rc;
    const ResampleDesign& d = t->d;
    RsPushArgs A{};
    A.in = d_src; A.in_stride = d_stride; A.n_in = n_in; A.in_fmt = in_fmt;
    A.tail = d_rs_tail; A.tail_cap = rs_tail_cap; A.H = t->H;
    A.L = d.L; A.M = d.M; A.W = d.W; A.stream0 = stream0;
    A.c = c; A.o0 = rs_ready(c, d); A.o1 = rs_ready(c + n_in, d);
    A.t0_old = rs_tail_start(c, d); A.t0_new = rs_tail_start(c + n_in, d);
    A.frame_latch = (int)ewk_resample_out_len(n_in, sr_in);
    if (rows_slot >= 0) { A.rows = (const RowDesc*)b_pos[rows_slot].p; A.n_rows = n_streams; }
    if (stage_slot >= 0) CK(cudaStreamWaitEvent(stream, ev_ready[stage_slot], 0));
    rc = launch_fir(*t, A, n_streams, 7, "ewk_push_resampled", n_items);
    if (rc) return rc;
    if (stage_slot >= 0) {
        CK(cudaEventRecord(ev_free[stage_slot], stream));
        ev_free_valid[stage_slot] = true;
    }
    if (rows_slot >= 0) {                   // the descriptors' slot is free once this K8 has read them
        CK(cudaEventRecord(ev_pos[rows_slot], stream));
        ev_pos_valid[rows_slot] = true;
    }
    all_presummed = false;                  // K8 forms no block sums: K2 reads these samples
    pushes_since_tick++;
    for (int i = 0; i < n_streams; i++) {
        const int s = rows ? rows[i].stream : stream0 + i;
        h_written[s] = rows ? rs_ready(rows[i].pos + rows[i].len, d) : rs_ready(c + n_in, d);
        const int latch = rows ? rows[i].latch : A.frame_latch;
        if (h_frame_size[s] == 0) h_frame_size[s] = h_prm[s].frame_size > 0 ? h_prm[s].frame_size : latch;
    }
    return EWK_OK;
}

// descriptors (at most one per stream) -> the next of two pinned + device slots, copied on stream `on`; a slot is reused
// only once the kernel that read its previous contents has run (ev[k]).  *slot receives its index.
template <class D>
static int upload_slot(ewk_ctx* ctx, D* (&h)[2], DevBuf (&b)[2], cudaEvent_t (&ev)[2], const bool (&ev_valid)[2], int& idx,
                       const std::vector<D>& rows, cudaStream_t on, int* slot) {
    const int k = idx;
    idx ^= 1;
    const size_t bytes = sizeof(D) * (size_t)ctx->bank.n_streams;
    if (!h[k]) {
        CK(ctx->pool.alloc_host(&h[k], bytes, cudaHostAllocDefault, "upload_slot host"));
        CK(cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming));
    }
    CK(b[k].ensure(bytes));
    if (ev_valid[k]) CK(cudaEventSynchronize(ev[k]));
    std::memcpy(h[k], rows.data(), sizeof(D) * rows.size());
    CK(cudaMemcpyAsync(b[k].p, h[k], sizeof(D) * rows.size(), cudaMemcpyHostToDevice, on));
    *slot = k;
    return EWK_OK;
}

int ewk_ctx::upload_rows(const std::vector<RowDesc>& rows, cudaStream_t on, int* slot) {
    return upload_slot(this, h_pos, b_pos, ev_pos, ev_pos_valid, pos_idx, rows, on, slot);
}

// tails for the widest filter in use; rows of streams already running move with their content
int ewk_ctx::ensure_rs_tail(int cap) {
    ewk_ctx* ctx = this;
    if (rs_tail_cap >= cap) return EWK_OK;
    float* nt = nullptr;
    CK(pool.alloc(&nt, sizeof(float) * (size_t)bank.n_streams * cap, "d_rs_tail"));
    if (d_rs_tail) {
        CK(cudaMemcpy2DAsync(nt, sizeof(float) * cap, d_rs_tail, sizeof(float) * rs_tail_cap, sizeof(float) * rs_tail_cap,
                             bank.n_streams, cudaMemcpyDeviceToDevice, stream));
        CK(cudaStreamSynchronize(stream));
        CK(pool.free(d_rs_tail));
    }
    d_rs_tail = nt;
    rs_tail_cap = cap;
    return EWK_OK;
}

// K1L on device-resident input (the caller's buffer or a staging slot)
int ewk_ctx::land_list(const std::vector<RowDesc>& rows, int rows_slot, long long n_items, const void* d_src, int in_fmt,
                       int stage_slot) {
    ewk_ctx* ctx = this;
    if (stage_slot >= 0) CK(cudaStreamWaitEvent(stream, ev_ready[stage_slot], 0));
    const RowDesc* d_rows = (const RowDesc*)b_pos[rows_slot].p;
    cudaEvent_t pe = prof_begin(0);
    if (bank.fmt == 1) ring_push_list_kernel<short><<<(unsigned)n_items, 256, 0, stream>>>(bank, d_src, in_fmt, d_rows, (int)rows.size());
    else ring_push_list_kernel<float><<<(unsigned)n_items, 256, 0, stream>>>(bank, d_src, in_fmt, d_rows, (int)rows.size());
    prof_end(pe, 0);
    CK(cudaGetLastError());
    launches++;
    if (stage_slot >= 0) {
        CK(cudaEventRecord(ev_free[stage_slot], stream));
        ev_free_valid[stage_slot] = true;
    }
    CK(cudaEventRecord(ev_pos[rows_slot], stream));
    ev_pos_valid[rows_slot] = true;
    all_presummed = false;                  // K1L forms no block sums: K2 reads these samples
    pushes_since_tick++;
    for (const RowDesc& r : rows) {
        h_written[r.stream] = r.pos + r.len;
        if (h_frame_size[r.stream] == 0) h_frame_size[r.stream] = h_prm[r.stream].frame_size > 0 ? h_prm[r.stream].frame_size : r.latch;
    }
    return EWK_OK;
}

// ewk_push_resampled (each = false: every stream of the call at the same input position, returns the landed count) and
// ewk_push_resampled_each (streams at their own positions, landed counts into landed[])
static int push_resampled_impl(ewk_ctx* ctx, const char* who, int stream0, int n_streams, const void* in, int in_format,
                               int64_t n_in, int64_t stride, int where, int sr_in, bool each, int64_t* landed) {
    int rc = need_streams(ctx, who, false);
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (!in || n_streams < 1 || stream0 < 0 || stream0 + n_streams > B.n_streams || n_in < 1 || stride < n_in ||
        in_format < EWK_PCM_F32 || in_format > EWK_IN_ALAW || n_in > (int64_t)1 << 34 || (each && !landed)) {
        ctx->fail("%s: bad arguments (stream0=%d n_streams=%d n_in=%lld stride=%lld in_format=%d%s)", who, stream0,
                  n_streams, (long long)n_in, (long long)stride, in_format, each && !landed ? ", landed is NULL" : "");
        return EWK_ERR_ARG;
    }
    ResampleDesign d;
    if (sr_in == RS_TARGET || sr_in < 1000 || sr_in > 768000 || !rs_design(sr_in, d)) {
        ctx->fail("%s: %d Hz is not a supported input rate (16000 Hz input goes through ewk_push)", who, sr_in);
        return EWK_ERR_ARG;
    }
    const long long c = ctx->h_inputs[stream0];
    bool uniform = true;
    for (int s = stream0; s < stream0 + n_streams; s++) {
        if (ctx->h_rate[s] != 0 && ctx->h_rate[s] != sr_in) {
            ctx->fail("%s: stream %d already takes %d Hz input", who, s, ctx->h_rate[s]);
            return EWK_ERR_STATE;
        }
        if (ctx->h_inputs[s] != c) {
            if (!each) {
                ctx->fail("%s: streams %d and %d have received %lld and %lld input samples; one call takes streams "
                          "at the same position", who, stream0, s, c, ctx->h_inputs[s]);
                return EWK_ERR_STATE;
            }
            uniform = false;
        }
    }
    for (int s = stream0; s < stream0 + n_streams; s++) {
        const long long n = rs_ready(ctx->h_inputs[s] + n_in, d) - rs_ready(ctx->h_inputs[s], d);   // samples it lands
        if (n > B.P - B.R && n > B.R) { ctx->fail("%s: %lld samples exceed the ring (%d)", who, n, B.R); return EWK_ERR_ARG; }
    }
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();
    if (rc) return rc;
    for (int s = stream0; s < stream0 + n_streams; s++) {     // same guard as ewk_push, on the stream's landed count
        if (ctx->h_prm[s].live) continue;
        const long long n = rs_ready(ctx->h_inputs[s] + n_in, d) - rs_ready(ctx->h_inputs[s], d);
        const long long ahead = ctx->h_written[s] + n - ctx->h_visible_lb[s];
        if (ctx->h_visible_lb[s] >= B.R && ahead > (long long)(B.P - B.R)) {
            ctx->fail("%s: stream %d would hold %lld un-gated samples, more than slack_samples=%d; call "
                      "ewk_tick first", who, s, ahead, B.P - B.R);
            return EWK_ERR_STATE;
        }
        if (ctx->h_visible_lb[s] < B.R && ctx->h_written[s] + n > (long long)B.P) {
            ctx->fail("%s: stream %d would hold %lld samples before its first full tick, more than the physical "
                      "ring (%d); call ewk_tick first", who, s, ctx->h_written[s] + n, B.P);
            return EWK_ERR_STATE;
        }
    }
    const ewk_ctx::ResampleTable* t = nullptr;
    rc = ctx->resample_table(sr_in, &t);
    if (rc) return rc;
    rc = ctx->ensure_rs_tail(2 * d.W);
    if (rc) return rc;
    // streams at different positions: per-row descriptors (identity streams, equal lengths) in a slot of their own,
    // which a later push reuses only after the K8 that reads them has run
    std::vector<RowDesc> rows;
    long long n_items = 0;
    const FirPlan f = fir_plan(d);
    const int latch = (int)ewk_resample_out_len(n_in, sr_in);
    for (int i = 0; i < n_streams; i++) {
        const int s = stream0 + i;
        const long long p = ctx->h_inputs[s];
        if (landed) landed[i] = rs_ready(p + n_in, d) - rs_ready(p, d);
        if (!uniform) {
            rows.push_back(RowDesc{(where == EWK_HOST ? n_in : stride) * i, n_in, p, s, (int)n_items, latch, 0});
            n_items += fir_tiles(f, d, rs_ready(p, d), rs_ready(p + n_in, d));
        }
        ctx->h_rate[s] = sr_in;
        ctx->h_inputs[s] = p + n_in;
    }
    const int n_ret = (int)(rs_ready(c + n_in, d) - rs_ready(c, d));
    int k = -1;
    // host input: on the copy stream ahead of the input's copy, so the K8 that waits for that copy finds them
    if (!uniform) {
        rc = ctx->upload_rows(rows, where == EWK_HOST ? ctx->copy_stream : ctx->stream, &k);
        if (rc) return rc;
    }
    if (where != EWK_HOST) {
        rc = ctx->land_resampled(stream0, n_streams, in, stride, in_format, n_in, sr_in, c, k >= 0 ? rows.data() : nullptr,
                                 k, n_items, -1);
        return rc ? rc : (each ? EWK_OK : n_ret);
    }
    // host input: its compact bytes cross PCIe on the copy stream and land lazily, as with ewk_push
    const size_t esz = rs_in_size(in_format);
    const int b = ctx->stage_idx;
    ctx->stage_idx ^= 1;
    CK(ctx->b_raw[b].ensure(esz * (size_t)n_in * n_streams));
    if (ctx->ev_free_valid[b]) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_free[b], 0));
    if (stride == n_in)
        CK(cudaMemcpyAsync(ctx->b_raw[b].p, in, esz * (size_t)n_in * n_streams, cudaMemcpyHostToDevice, ctx->copy_stream));
    else
        CK(cudaMemcpy2DAsync(ctx->b_raw[b].p, esz * (size_t)n_in, in, esz * (size_t)stride, esz * (size_t)n_in, n_streams,
                             cudaMemcpyHostToDevice, ctx->copy_stream));
    CK(cudaEventRecord(ctx->ev_ready[b], ctx->copy_stream));
    ctx->pending = ewk_ctx::Pending{};
    ctx->pending.valid = true; ctx->pending.slot = b; ctx->pending.stream0 = stream0; ctx->pending.n_streams = n_streams;
    ctx->pending.n = n_ret;
    ctx->pending.rs_rate = sr_in; ctx->pending.rs_fmt = in_format; ctx->pending.rs_n_in = n_in; ctx->pending.rs_c = c;
    if (k >= 0) { ctx->pending.rows_slot = k; ctx->pending.n_items = n_items; ctx->pending.rows = std::move(rows); }
    return each ? EWK_OK : n_ret;
}

extern "C" int ewk_push_resampled(ewk_ctx* ctx, int stream0, int n_streams, const void* in, int in_format, int64_t n_in,
                                  int64_t stride, int where, int sr_in) {
    if (!ctx) return EWK_ERR_ARG;
    return push_resampled_impl(ctx, "ewk_push_resampled", stream0, n_streams, in, in_format, n_in, stride, where, sr_in,
                               false, nullptr);
}

extern "C" int ewk_push_resampled_each(ewk_ctx* ctx, int stream0, int n_streams, const void* in, int in_format,
                                       int64_t n_in, int64_t stride, int where, int sr_in, int64_t* landed) {
    if (!ctx) return EWK_ERR_ARG;
    return push_resampled_impl(ctx, "ewk_push_resampled_each", stream0, n_streams, in, in_format, n_in, stride, where,
                               sr_in, true, landed);
}

extern "C" int ewk_stream_input(ewk_ctx* ctx, int stream, int32_t* sr_in, int64_t* n_in) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_stream_input", false);
    if (rc) return rc;
    if (stream < 0 || stream >= ctx->bank.n_streams) { ctx->fail("ewk_stream_input: bad stream %d", stream); return EWK_ERR_ARG; }
    if (sr_in) *sr_in = ctx->h_rate[stream];
    if (n_in) *n_in = ctx->h_inputs[stream];
    return EWK_OK;
}

// Ragged push to a list of streams: row i = in[offsets[i], offsets[i] + lens[i]) goes to stream streams[i].  Every rule
// is the one of pushing the row alone with ewk_push / ewk_push_g711 (16 kHz) or ewk_push_resampled (other rates).
extern "C" int ewk_push_streams(ewk_ctx* ctx, const int32_t* streams, int n, const void* in, int in_format,
                                const int64_t* offsets, const int64_t* lens, int64_t in_len, int where, int sr_in,
                                int64_t* landed) {
    static const char* who = "ewk_push_streams";
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, who, false);
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (n == 0) return EWK_OK;
    if (n < 0 || !streams || !offsets || !lens || (!in && in_len > 0) || in_len < 0 || in_format < EWK_PCM_F32 ||
        in_format > EWK_IN_ALAW || !landed) {
        ctx->fail("%s: bad arguments (n=%d in_len=%lld in_format=%d%s)", who, n, (long long)in_len, in_format,
                  landed ? "" : ", landed is NULL");
        return EWK_ERR_ARG;
    }
    const bool direct = sr_in == RS_TARGET;
    ResampleDesign d;
    if (!direct && (sr_in < 1000 || sr_in > 768000 || !rs_design(sr_in, d))) {
        ctx->fail("%s: %d Hz is not a supported input rate", who, sr_in);
        return EWK_ERR_ARG;
    }
    if (direct && in_format >= EWK_IN_ULAW && B.fmt != 1) {
        ctx->fail("%s: G.711 at 16000 Hz needs int16 rings (pcm_format EWK_PCM_I16)", who);
        return EWK_ERR_ARG;
    }
    if (direct && in_format < EWK_IN_ULAW && in_format != B.fmt) {
        ctx->fail("%s: in_format %d at 16000 Hz must be the rings' pcm_format (%d) or G.711", who, in_format, B.fmt);
        return EWK_ERR_ARG;
    }
    // samples row i lands: its own length at 16 kHz, else ready(c + len) - ready(c) from the stream's input position
    auto lands = [&](int i) {
        const long long c = ctx->h_inputs[streams[i]];
        return direct ? (long long)lens[i] : rs_ready(c + lens[i], d) - rs_ready(c, d);
    };
    std::vector<char> seen((size_t)B.n_streams, 0);
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        if (s < 0 || s >= B.n_streams) { ctx->fail("%s: bad stream %d (context has %d)", who, s, B.n_streams); return EWK_ERR_ARG; }
        if (seen[s]) { ctx->fail("%s: stream %d is listed twice", who, s); return EWK_ERR_ARG; }
        seen[s] = 1;
        if (lens[i] < 0 || offsets[i] < 0 || offsets[i] > in_len - lens[i] || lens[i] > (int64_t)1 << 34) {
            ctx->fail("%s: row %d of stream %d, [%lld, %lld + %lld), lies outside the input [0, %lld)", who, i, s,
                      (long long)offsets[i], (long long)offsets[i], (long long)lens[i], (long long)in_len);
            return EWK_ERR_ARG;
        }
        const long long m = lands(i);
        if (m > B.P - B.R && m > B.R) {
            ctx->fail("%s: stream %d: %lld samples exceed the ring (%d)", who, s, m, B.R);
            return EWK_ERR_ARG;
        }
    }
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        if (lens[i] == 0) continue;
        if (direct && ctx->h_rate[s] != 0 && ctx->h_rate[s] != RS_TARGET) {
            ctx->fail("%s: stream %d takes %d Hz input through ewk_push_resampled", who, s, ctx->h_rate[s]);
            return EWK_ERR_STATE;
        }
        if (!direct && ctx->h_rate[s] != 0 && ctx->h_rate[s] != sr_in) {
            ctx->fail("%s: stream %d already takes %d Hz input", who, s, ctx->h_rate[s]);
            return EWK_ERR_STATE;
        }
    }
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();
    if (rc) return rc;
    for (int i = 0; i < n; i++) {             // the guards of ewk_push, per stream on its landed count
        const int s = streams[i];
        if (lens[i] == 0 || ctx->h_prm[s].live) continue;
        const long long m = lands(i);
        const long long ahead = ctx->h_written[s] + m - ctx->h_visible_lb[s];
        if (ctx->h_visible_lb[s] >= B.R && ahead > (long long)(B.P - B.R)) {
            ctx->fail("%s: stream %d would hold %lld un-gated samples, more than slack_samples=%d; call ewk_tick first",
                      who, s, ahead, B.P - B.R);
            return EWK_ERR_STATE;
        }
        if (ctx->h_visible_lb[s] < B.R && ctx->h_written[s] + m > (long long)B.P) {
            ctx->fail("%s: stream %d would hold %lld samples before its first full tick, more than the physical ring "
                      "(%d); call ewk_tick first", who, s, ctx->h_written[s] + m, B.P);
            return EWK_ERR_STATE;
        }
    }
    const ewk_ctx::ResampleTable* t = nullptr;
    if (!direct) {
        rc = ctx->resample_table(sr_in, &t);
        if (rc) return rc;
        rc = ctx->ensure_rs_tail(2 * d.W);
        if (rc) return rc;
    }
    // descriptors of the non-empty rows, and the flat work list: LIST_CHUNK-sample chunks (K1L) or output tiles (K8)
    std::vector<RowDesc> rows;
    long long n_items = 0;
    const FirPlan f = direct ? FirPlan{} : fir_plan(d);
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        landed[i] = lands(i);
        if (lens[i] == 0) continue;
        const long long c = ctx->h_inputs[s];
        RowDesc r{offsets[i], lens[i], direct ? ctx->h_written[s] : c, s, (int)n_items,
                  direct ? (int)lens[i] : (int)ewk_resample_out_len(lens[i], sr_in), 0};
        n_items += direct ? (lens[i] + LIST_CHUNK - 1) / LIST_CHUNK : fir_tiles(f, d, rs_ready(c, d), rs_ready(c + lens[i], d));
        if (n_items > INT_MAX) { ctx->fail("%s: too much input for one call", who); return EWK_ERR_ARG; }
        rows.push_back(r);
        ctx->h_rate[s] = direct ? RS_TARGET : sr_in;
        ctx->h_inputs[s] = c + lens[i];
    }
    if (rows.empty()) return EWK_OK;
    int k = -1;
    rc = ctx->upload_rows(rows, where == EWK_HOST ? ctx->copy_stream : ctx->stream, &k);
    if (rc) return rc;
    if (where != EWK_HOST)
        return direct ? ctx->land_list(rows, k, n_items, in, in_format, -1)
                      : ctx->land_resampled(0, (int)rows.size(), in, 0, in_format, 0, sr_in, 0, rows.data(), k, n_items, -1);
    // host input: [0, in_len) crosses PCIe as one copy on the copy stream and lands lazily, as with ewk_push
    const size_t esz = rs_in_size(in_format);
    const int b = ctx->stage_idx;
    ctx->stage_idx ^= 1;
    CK(ctx->b_raw[b].ensure(esz * (size_t)in_len));
    if (ctx->ev_free_valid[b]) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_free[b], 0));
    CK(cudaMemcpyAsync(ctx->b_raw[b].p, in, esz * (size_t)in_len, cudaMemcpyHostToDevice, ctx->copy_stream));
    CK(cudaEventRecord(ctx->ev_ready[b], ctx->copy_stream));
    ctx->pending = ewk_ctx::Pending{};
    ctx->pending.valid = true; ctx->pending.slot = b; ctx->pending.n_streams = (int)rows.size();
    ctx->pending.rs_rate = direct ? 0 : sr_in; ctx->pending.rs_fmt = in_format;
    ctx->pending.rows_slot = k; ctx->pending.n_items = n_items; ctx->pending.rows = std::move(rows);
    return EWK_OK;
}

// K9: streams back to the state ewk_create gives them, in one launch; host mirrors with them.  all_presummed may stay
// set: K2 takes a stream's block sums only for ticks at or past its ss_from (reset to 0, as in a new context), a stream
// with nothing written reads no samples at all, and the next push of the stream restarts its sums or clears the flag.
extern "C" int ewk_reset_streams(ewk_ctx* ctx, const int32_t* streams, int n) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_reset_streams");       // overlap mode: K3 still reads the rings
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (n < 0 || (n > 0 && !streams)) { ctx->fail("ewk_reset_streams: bad stream list (n=%d)", n); return EWK_ERR_ARG; }
    for (int i = 0; i < n; i++)
        if (streams[i] < 0 || streams[i] >= B.n_streams) {
            ctx->fail("ewk_reset_streams: bad stream %d (context has %d)", streams[i], B.n_streams);
            return EWK_ERR_ARG;
        }
    if (n == 0) return EWK_OK;
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();                              // a pending host push belongs to the old sessions
    if (rc) return rc;
    // events carry no session: one polled after its stream restarted would point at the new session's audio
    int cnt[2] = {0, 0};
    CK(cudaMemcpyAsync(cnt, B.ev_count, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (cnt[0] != 0 || cnt[1] != 0) {
        ctx->fail("ewk_reset_streams: %d events are queued; poll first", cnt[0]);
        return EWK_ERR_STATE;
    }
    CK(ctx->b_reset.ensure(sizeof(int32_t) * (size_t)n));
    CK(cudaMemcpyAsync(ctx->b_reset.p, streams, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
    const size_t row_bytes = (size_t)B.P * (B.fmt == 1 ? 2 : 4);
    const dim3 grid((unsigned)((row_bytes + RESET_SLICE - 1) / RESET_SLICE), (unsigned)std::min(n, 65535));
    stream_reset_kernel<<<grid, RESET_THREADS, 0, ctx->stream>>>(B, (const int*)ctx->b_reset.p, n,
                                                                 (long long*)ctx->b_keep_end.p,
                                                                 (DetState*)ctx->b_det_state.p);
    CK(cudaGetLastError());
    ctx->launches++;
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        ctx->h_written[s] = 0; ctx->h_visible_lb[s] = 0; ctx->h_tick[s] = 0; ctx->h_dense_next[s] = 1; ctx->h_det_next[s] = 1;
        ctx->h_frame_size[s] = 0; ctx->h_rate[s] = 0; ctx->h_inputs[s] = 0;
    }
    return EWK_OK;
}

// ------------------------------------------------------------------------------------------ K10 (stream migration)
// Blob version 1: header (ewk_stream_blob) | int32 source ids [n] | StreamMeta [n] | BlobTemplate [n_templates] | bulk
// rows [n] (MigrateGeom), each section 16-byte aligned.  The layout follows from the fingerprint and three counts, so
// an importer recomputes it and takes no offset on trust.
struct BlobTemplate {       // a template slot a stream of the blob is scored against, as the source context holds it
    int32_t slot, valid;
    int64_t n_samples;
    float mean[N_MFCC], std[N_MFCC];
};
static_assert(sizeof(BlobTemplate) == 176 && sizeof(ewk_stream_blob) == 96, "blob version 1 layout");

struct BlobLayout { long long ids, meta, tmpl, bulk, total; MigrateGeom g; };

static long long align16(long long v) { return (v + 15) & ~15LL; }

static BlobLayout blob_layout(const BankView& B, int n, int n_tmpl, int tail_floats) {
    BlobLayout L{};
    const long long esz = B.fmt == 1 ? 2 : 4;
    L.g.ss_off = (long long)B.P * esz;
    L.g.ms_off = L.g.ss_off + align16(8LL * B.NB);
    L.g.tail_off = L.g.ms_off + 16LL * B.chunk_cap;
    L.g.tail_floats = tail_floats;
    L.g.row_bytes = align16(L.g.tail_off + 4LL * tail_floats);
    L.ids = (long long)sizeof(ewk_stream_blob);
    L.meta = align16(L.ids + 4LL * n);
    L.tmpl = L.meta + (long long)sizeof(StreamMeta) * n;
    L.bulk = L.tmpl + (long long)sizeof(BlobTemplate) * n_tmpl;
    L.total = L.bulk + L.g.row_bytes * n;
    return L;
}

// live K8 input tail of a stream latched to `rate` after `inputs` input samples: inputs [rs_tail_start, inputs), the only
// part of its tail row a later push reads (0 at rate 0 or 16000: direct pushes keep none); -1 for a rate K8 rejects
static int tail_len_of(int rate, long long inputs) {
    if (rate == 0 || rate == RS_TARGET) return 0;
    ResampleDesign d;
    if (rate < 1000 || rate > 768000 || !rs_design(rate, d) || inputs < 0) return -1;
    return (int)(inputs - rs_tail_start(inputs, d));
}

static int round4(int v) { return (v + 3) & ~3; }

static int n_mfcc_of(const ewk_config& c) { return c.n_mfcc > 0 ? c.n_mfcc : N_MFCC; }

static uint32_t float_bits(float f) { uint32_t u; std::memcpy(&u, &f, 4); return u; }

static int check_stream_list(ewk_ctx* ctx, const char* who, const int32_t* streams, int n) {
    const int ns = ctx->bank.n_streams;
    if (n < 0 || (n > 0 && !streams)) { ctx->fail("%s: bad stream list (n=%d)", who, n); return EWK_ERR_ARG; }
    std::vector<char> seen((size_t)ns, 0);
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        if (s < 0 || s >= ns) { ctx->fail("%s: bad stream %d (context has %d)", who, s, ns); return EWK_ERR_ARG; }
        if (seen[s]) { ctx->fail("%s: stream %d is listed twice", who, s); return EWK_ERR_ARG; }
        seen[s] = 1;
    }
    return EWK_OK;
}

static int check_blob_ptr(ewk_ctx* ctx, const char* who, const void* blob, int where) {
    if (!blob) { ctx->fail("%s: blob is NULL", who); return EWK_ERR_ARG; }
    if (where == EWK_HOST) return EWK_OK;
    if (where != EWK_DEVICE) { ctx->fail("%s: where must be EWK_HOST or EWK_DEVICE", who); return EWK_ERR_ARG; }
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, blob) != cudaSuccess) {
        cudaGetLastError();
        ctx->fail("%s: the device blob is not CUDA memory", who);
        return EWK_ERR_ARG;
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != ctx->device) {
        ctx->fail("%s: the device blob is not memory of the context's device %d (copy it there first)", who, ctx->device);
        return EWK_ERR_ARG;
    }
    if ((uintptr_t)blob & 15) { ctx->fail("%s: the device blob must be 16-byte aligned", who); return EWK_ERR_ARG; }
    return EWK_OK;
}

static dim3 migrate_grid(const BankView& B, int n) {
    const size_t ring_bytes = (size_t)B.P * (B.fmt == 1 ? 2 : 4);
    return dim3((unsigned)((ring_bytes + RESET_SLICE - 1) / RESET_SLICE), (unsigned)std::min(n, 65535));
}

extern "C" int64_t ewk_stream_blob_bytes(const ewk_ctx* ctx, int n) {
    if (!ctx || n < 0) return EWK_ERR_ARG;
    if (ctx->bank.n_streams == 0) return EWK_ERR_STATE;
    return blob_layout(ctx->bank, n, ctx->cfg.max_templates, round4(ctx->rs_tail_cap)).total;
}

extern "C" int ewk_export_streams(ewk_ctx* ctx, const int32_t* streams, int n, void* blob, int64_t blob_cap, int where) {
    if (!ctx) return EWK_ERR_ARG;
    const char* who = "ewk_export_streams";
    int rc = need_streams(ctx, who);                          // overlap mode: K3 may still write the result records
    if (rc) return rc;
    BankView& B = ctx->bank;
    rc = check_stream_list(ctx, who, streams, n);
    if (rc) return rc;
    rc = check_blob_ptr(ctx, who, blob, where);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();                                // its samples belong to the streams
    if (rc) return rc;
    const int T = ctx->cfg.max_templates;
    std::vector<char> used((size_t)T, 0);
    int tail = 0;
    for (int i = 0; i < n; i++) {
        const StreamParams& p = ctx->h_prm[streams[i]];
        for (int k = p.template_first; k < p.template_first + p.template_count; k++) used[k] = 1;
        tail = std::max(tail, tail_len_of(ctx->h_rate[streams[i]], ctx->h_inputs[streams[i]]));
    }
    const int n_tmpl = (int)std::count(used.begin(), used.end(), 1);
    const BlobLayout L = blob_layout(B, n, n_tmpl, round4(tail));
    if (blob_cap < L.total) {
        ctx->fail("%s: blob_cap %lld is below the %lld bytes of this blob", who, (long long)blob_cap, L.total);
        return EWK_ERR_ARG;
    }
    // everything in front of the bulk rows is host knowledge; K10 adds each stream's device state to its meta record
    std::vector<char> pre((size_t)L.bulk, 0);
    ewk_stream_blob* h = reinterpret_cast<ewk_stream_blob*>(pre.data());
    h->magic = EWK_STREAM_BLOB_MAGIC; h->version = EWK_STREAM_BLOB_VERSION; h->n_streams = n;
    h->ring_samples = ctx->cfg.ring_samples; h->slack_samples = ctx->cfg.slack_samples; h->pcm_format = ctx->cfg.pcm_format;
    h->n_mfcc = n_mfcc_of(ctx->cfg); h->preemphasis_bits = float_bits(ctx->cfg.preemphasis);
    h->meta_bytes = (int32_t)sizeof(StreamMeta); h->n_templates = n_tmpl; h->tail_floats = L.g.tail_floats;
    h->ids_offset = L.ids; h->meta_offset = L.meta; h->template_offset = L.tmpl; h->bulk_offset = L.bulk;
    h->bulk_row_bytes = L.g.row_bytes; h->total_bytes = L.total;
    if (n > 0) std::memcpy(pre.data() + L.ids, streams, sizeof(int32_t) * (size_t)n);
    StreamMeta* meta = reinterpret_cast<StreamMeta*>(pre.data() + L.meta);
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        StreamMeta& m = meta[i];
        m.written = ctx->h_written[s]; m.visible_lb = ctx->h_visible_lb[s]; m.tick = ctx->h_tick[s];
        m.dense_next = ctx->h_dense_next[s]; m.det_next = ctx->h_det_next[s]; m.inputs = ctx->h_inputs[s];
        m.frame_size = ctx->h_frame_size[s]; m.rate = ctx->h_rate[s]; m.tail_len = tail_len_of(ctx->h_rate[s], ctx->h_inputs[s]);
        m.prm = ctx->h_prm[s];
    }
    BlobTemplate* tp = reinterpret_cast<BlobTemplate*>(pre.data() + L.tmpl);
    for (int k = 0, j = 0; k < T; k++) {
        if (!used[k]) continue;
        const TemplateFeat& tf = ctx->h_tmpl[k];
        tp[j].slot = k; tp[j].valid = tf.valid; tp[j].n_samples = tf.n_samples;
        std::memcpy(tp[j].mean, tf.mean, sizeof(tf.mean));
        std::memcpy(tp[j].std, tf.std, sizeof(tf.std));
        j++;
    }
    char* target = (char*)blob;
    if (where == EWK_HOST) {                                  // the blob forms in scratch and crosses PCIe in one copy
        CK(ctx->b_blob.ensure((size_t)L.total));
        target = (char*)ctx->b_blob.p;
    }
    CK(cudaMemcpyAsync(target, pre.data(), (size_t)L.bulk, cudaMemcpyHostToDevice, ctx->stream));
    if (n > 0) {
        stream_export_kernel<<<migrate_grid(B, n), RESET_THREADS, 0, ctx->stream>>>(
            B, (const int*)(target + L.ids), n, (const DetState*)ctx->b_det_state.p, ctx->d_rs_tail, ctx->rs_tail_cap,
            (StreamMeta*)(target + L.meta), target + L.bulk, L.g);
        CK(cudaGetLastError());
        ctx->launches++;
    }
    if (where == EWK_HOST) CK(cudaMemcpyAsync(blob, target, (size_t)L.total, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

// the name of the first field of a meta record that no sequence of calls produces in a context of this geometry
static const char* bad_meta_field(const ewk_ctx* ctx, const StreamMeta& m, int tail_floats) {
    const BankView& B = ctx->bank;
    auto frame_ok = [&](int fs) { return fs == 0 || (fs >= MIN_FRAME_SIZE && fs <= B.R); };
    if (m.written < 0 || m.st.written != m.written) return "written";
    if (m.st.ss_from < 0 || m.st.ss_from > m.written) return "ss_from";
    if (m.st.visible < 0 || m.st.visible > m.written || m.visible_lb < 0 || m.visible_lb > m.written) return "visible";
    if (m.tick < 0 || m.st.tick < 0) return "tick";
    if (!frame_ok(m.frame_size) || !frame_ok(m.st.frame_size)) return "frame_size";
    if (m.st.state < ST_WAITING || m.st.state > ST_AFTER_SOUND) return "state";
    const long long last_hop = m.written / HOP + 1;
    if (m.dense_next < 1 || m.dense_next > last_hop) return "dense cursor";
    if (m.det_next < 1 || m.det_next > last_hop) return "detect cursor";
    const int tl = tail_len_of(m.rate, m.inputs);
    if (tl < 0) return m.inputs < 0 ? "inputs" : "rate";
    if (m.rate == 0 ? (m.inputs != 0 || m.written != 0) : m.rate == RS_TARGET ? m.inputs != m.written : false) return "inputs";
    if (m.rate != 0 && m.rate != RS_TARGET) {
        ResampleDesign d;
        rs_design(m.rate, d);
        if (m.inputs < 0 || rs_ready(m.inputs, d) != m.written) return "inputs";
    }
    if (m.tail_len != tl || tl > tail_floats) return "tail_len";
    if (m.det.mode < DET_IDLE || m.det.mode > DET_SPENT) return "detector mode";
    const StreamParams& p = m.prm;
    if (!(p.pre_speech_silence > 0) || !(p.speech_duration_min > 0) || !(p.speech_duration_max > 0) ||
        !(p.speech_duration_min <= p.speech_duration_max) || !(p.post_speech_silence > 0) || !frame_ok(p.frame_size))
        return "stream parameters";
    if (p.template_first < 0 || p.template_count < 0 || p.template_count > EWK_MAX_STREAM_TEMPLATES ||
        p.template_first + p.template_count > ctx->cfg.max_templates)
        return "template range";
    return nullptr;
}

extern "C" int ewk_import_streams(ewk_ctx* ctx, const int32_t* streams, int n, const void* blob, int64_t blob_len,
                                  int where) {
    if (!ctx) return EWK_ERR_ARG;
    const char* who = "ewk_import_streams";
    int rc = need_streams(ctx, who);                          // overlap mode: K3 still reads the rings
    if (rc) return rc;
    BankView& B = ctx->bank;
    rc = check_stream_list(ctx, who, streams, n);
    if (rc) return rc;
    rc = check_blob_ptr(ctx, who, blob, where);
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    ewk_stream_blob h;
    if (blob_len < (int64_t)sizeof(h)) { ctx->fail("%s: blob_len %lld holds no blob header", who, (long long)blob_len); return EWK_ERR_ARG; }
    if (where == EWK_HOST) std::memcpy(&h, blob, sizeof(h));
    else {
        CK(cudaMemcpyAsync(&h, blob, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    if (h.magic != EWK_STREAM_BLOB_MAGIC || h.version != EWK_STREAM_BLOB_VERSION) {
        ctx->fail("%s: not a stream blob of version %d (magic 0x%08x, version %u)", who, EWK_STREAM_BLOB_VERSION, h.magic, h.version);
        return EWK_ERR_ARG;
    }
    if (h.n_streams != n) { ctx->fail("%s: the blob holds %d streams, the list %d", who, h.n_streams, n); return EWK_ERR_ARG; }
    const struct { const char* name; long long blob, mine; } fp[] = {
        {"ring_samples", h.ring_samples, ctx->cfg.ring_samples}, {"slack_samples", h.slack_samples, ctx->cfg.slack_samples},
        {"pcm_format", h.pcm_format, ctx->cfg.pcm_format}, {"n_mfcc", h.n_mfcc, n_mfcc_of(ctx->cfg)},
        {"preemphasis", h.preemphasis_bits, float_bits(ctx->cfg.preemphasis)}};
    for (const auto& f : fp)
        if (f.blob != f.mine) {
            ctx->fail("%s: the blob's %s (%lld) differs from the context's (%lld)", who, f.name, f.blob, f.mine);
            return EWK_ERR_ARG;
        }
    if (h.meta_bytes != (int32_t)sizeof(StreamMeta) || h.n_templates < 0 || h.n_templates > EWK_MAX_TEMPLATE_SLOTS ||
        h.tail_floats < 0 || (h.tail_floats & 3) || h.tail_floats > 1 << 20) {
        ctx->fail("%s: bad blob header (meta_bytes %d, n_templates %d, tail_floats %d)", who, h.meta_bytes, h.n_templates,
                  h.tail_floats);
        return EWK_ERR_ARG;
    }
    const BlobLayout L = blob_layout(B, n, h.n_templates, h.tail_floats);
    if (h.ids_offset != L.ids || h.meta_offset != L.meta || h.template_offset != L.tmpl || h.bulk_offset != L.bulk ||
        h.bulk_row_bytes != L.g.row_bytes || h.total_bytes != L.total) {
        ctx->fail("%s: the blob's section offsets are not those of its header's counts", who);
        return EWK_ERR_ARG;
    }
    if (blob_len < L.total) {
        ctx->fail("%s: blob_len %lld is below the blob's %lld bytes", who, (long long)blob_len, L.total);
        return EWK_ERR_ARG;
    }
    std::vector<char> dev_pre;
    const char* pre = (const char*)blob;
    if (where == EWK_DEVICE) {
        dev_pre.resize((size_t)L.bulk);
        CK(cudaMemcpyAsync(dev_pre.data(), blob, (size_t)L.bulk, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        pre = dev_pre.data();
    }
    // a private copy of the meta records: what is checked is what the kernel gets
    std::vector<StreamMeta> meta((size_t)n);
    if (n > 0) std::memcpy(meta.data(), pre + L.meta, sizeof(StreamMeta) * (size_t)n);
    const BlobTemplate* tp = reinterpret_cast<const BlobTemplate*>(pre + L.tmpl);
    std::vector<int> tmpl_of((size_t)ctx->cfg.max_templates, -1);       // slot -> its record
    for (int j = 0; j < h.n_templates; j++) {
        if (tp[j].slot < 0 || tp[j].slot >= ctx->cfg.max_templates || tmpl_of[tp[j].slot] >= 0) {
            ctx->fail("%s: template record %d names slot %d (the context has %d slots)", who, j, tp[j].slot, ctx->cfg.max_templates);
            return EWK_ERR_ARG;
        }
        tmpl_of[tp[j].slot] = j;
    }
    bool need_det = false;
    int need_tail = 0;
    for (int i = 0; i < n; i++) {
        const StreamMeta& m = meta[i];
        if (const char* f = bad_meta_field(ctx, m, h.tail_floats)) {
            ctx->fail("%s: blob stream %d: %s is outside what the entry points produce", who, i, f);
            return EWK_ERR_ARG;
        }
        for (int k = m.prm.template_first; k < m.prm.template_first + m.prm.template_count; k++)
            if (tmpl_of[k] < 0) { ctx->fail("%s: blob stream %d: template slot %d has no record", who, i, k); return EWK_ERR_ARG; }
        const DetState z{};
        need_det |= std::memcmp(&m.det, &z, sizeof(z)) != 0;
        need_tail = std::max(need_tail, m.tail_len);
    }
    for (int i = 0; i < n; i++) {
        const StreamParams& p = meta[i].prm;
        for (int k = p.template_first; k < p.template_first + p.template_count; k++) {
            const BlobTemplate& t = tp[tmpl_of[k]];
            const TemplateFeat& mine = ctx->h_tmpl[k];
            if (t.valid != mine.valid || t.n_samples != mine.n_samples || std::memcmp(t.mean, mine.mean, sizeof(t.mean)) ||
                std::memcmp(t.std, mine.std, sizeof(t.std))) {
                ctx->fail("%s: blob stream %d (source stream %d) is scored against template slot %d, which differs in "
                          "this context", who, i, reinterpret_cast<const int32_t*>(pre + L.ids)[i], k);
                return EWK_ERR_STATE;
            }
        }
    }
    rc = ctx->flush_pending();                                // a pending host push belongs to the slots' old sessions
    if (rc) return rc;
    int cnt[2] = {0, 0};
    CK(cudaMemcpyAsync(cnt, B.ev_count, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (cnt[0] != 0 || cnt[1] != 0) {
        ctx->fail("%s: %d events are queued; poll first", who, cnt[0]);
        return EWK_ERR_STATE;
    }
    if (n == 0) return EWK_OK;
    if (need_det && !ctx->b_det_state.p) {
        CK(ctx->b_det_state.ensure(sizeof(DetState) * (size_t)B.n_streams));
        CK(cudaMemsetAsync(ctx->b_det_state.p, 0, sizeof(DetState) * (size_t)B.n_streams, ctx->stream));
    }
    if (need_tail > 0) {
        rc = ctx->ensure_rs_tail(need_tail);
        if (rc) return rc;
    }
    // one upload: the destination list, then the checked small state
    const size_t list_bytes = (size_t)align16(4LL * n);
    std::vector<char> up(list_bytes + sizeof(MigrateSmall) * (size_t)n, 0);
    std::memcpy(up.data(), streams, sizeof(int32_t) * (size_t)n);
    MigrateSmall* sm = reinterpret_cast<MigrateSmall*>(up.data() + list_bytes);
    for (int i = 0; i < n; i++) {
        sm[i].prm = meta[i].prm;
        sm[i].st = meta[i].st;
        sm[i].st.last_ev = -1;                                // a queue index of another context means nothing here
        sm[i].res = meta[i].res;
        sm[i].det = meta[i].det;
        sm[i].tail_len = meta[i].tail_len;
    }
    CK(ctx->b_mig.ensure(up.size()));
    CK(cudaMemcpyAsync(ctx->b_mig.p, up.data(), up.size(), cudaMemcpyHostToDevice, ctx->stream));
    const char* bulk = (const char*)blob + L.bulk;
    if (where == EWK_HOST) {
        CK(ctx->b_blob.ensure((size_t)(L.total - L.bulk)));
        CK(cudaMemcpyAsync(ctx->b_blob.p, bulk, (size_t)(L.total - L.bulk), cudaMemcpyHostToDevice, ctx->stream));
        bulk = (const char*)ctx->b_blob.p;
    }
    stream_import_kernel<<<migrate_grid(B, n), RESET_THREADS, 0, ctx->stream>>>(
        B, (const int*)ctx->b_mig.p, (const MigrateSmall*)((const char*)ctx->b_mig.p + list_bytes), n, bulk, L.g,
        (long long*)ctx->b_keep_end.p, (DetState*)ctx->b_det_state.p, ctx->d_rs_tail, ctx->rs_tail_cap);
    CK(cudaGetLastError());
    ctx->launches++;
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        const StreamMeta& m = meta[i];
        ctx->h_written[s] = m.written; ctx->h_visible_lb[s] = m.visible_lb; ctx->h_tick[s] = m.tick;
        ctx->h_dense_next[s] = m.dense_next; ctx->h_det_next[s] = m.det_next; ctx->h_frame_size[s] = m.frame_size;
        ctx->h_rate[s] = m.rate; ctx->h_inputs[s] = m.inputs; ctx->h_prm[s] = m.prm;
    }
    ctx->max_post = 0.0;
    for (int s = 0; s < B.n_streams; s++) ctx->max_post = std::max(ctx->max_post, ctx->h_prm[s].post_speech_silence);
    // K2 takes block sums of ticks at or past a stream's ss_from only when every push since the last tick formed them;
    // an imported stream's sums came from another context's pushes, so K2 reads its samples on the next tick
    ctx->all_presummed = false;
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

// ewk_tick / ewk_tick_trace, and paced: ewk_tick_ready (n_ticks = max_ticks; stream s takes taken[s] of them)
static int tick_impl(ewk_ctx* ctx, int n_ticks, bool paced, int32_t* taken, uint8_t* silent, uint8_t* state, double* thr,
                     double* rms) {
    const char* who = paced ? "ewk_tick_ready" : "ewk_tick";
    int rc = need_streams(ctx, who);
    if (rc) return rc;
    if (n_ticks < 1 || n_ticks > 4096) { ctx->fail("%s: %s must be in [1, 4096]", who, paced ? "max_ticks" : "n_ticks"); return EWK_ERR_ARG; }
    BankView& B = ctx->bank;
    CK(cudaSetDevice(ctx->device));
    // paced: the budgets depend on every landed sample
    if (paced) { rc = ctx->flush_pending(); if (rc) return rc; }
    if (ctx->pending.valid) {
        // land the in-flight host push only if these ticks reach into its samples
        bool need = false;
        const std::vector<RowDesc>& rows = ctx->pending.rows;
        for (int i = 0; !need && i < ctx->pending.n_streams; i++) {
            const int s = rows.empty() ? ctx->pending.stream0 + i : rows[i].stream;
            const int fs = ctx->h_frame_size[s] > 0 ? ctx->h_frame_size[s] : ctx->h_prm[s].frame_size;
            if (ctx->h_prm[s].live || fs <= 0) need = true;
            else need = ((ctx->h_tick[s] + n_ticks) * TICK / fs) * fs > ctx->h_written[s];
        }
        if (need) { rc = ctx->flush_pending(); if (rc) return rc; }
    }
    // the ticks each stream takes: the due rule of ewk_tick_ready on the host mirrors (K2 applies it to StreamState), and
    // only as many K2 rounds as the largest budget needs (one at least: K2 stores every stream's record in every call)
    std::vector<int> budget;
    int rounds_ticks = n_ticks;
    if (paced) {
        budget.resize((size_t)B.n_streams);
        int most = 0;
        for (int s = 0; s < B.n_streams; s++) {
            const long long due = ctx->h_written[s] / TICK - ctx->h_tick[s];
            budget[s] = (int)std::max(0LL, std::min((long long)n_ticks, due));
            most = std::max(most, budget[s]);
        }
        rounds_ticks = std::max(1, most);
    }
    TraceView tr{};
    const bool want = silent || state || thr || rms;
    const size_t cells = (size_t)B.n_streams * n_ticks;
    if (want) {
        CK(ctx->b_trace.ensure(cells * (2 + 16)));
        char* base = (char*)ctx->b_trace.p;
        tr.thr = (double*)base;
        tr.rms = (double*)(base + cells * 8);
        tr.silent = (unsigned char*)(base + cells * 16);
        tr.state = (unsigned char*)(base + cells * 17);
        // cells of ticks a stream does not take: silent = state = 255, thr = rms = NaN (all-ones bits)
        if (paced) CK(cudaMemsetAsync(ctx->b_trace.p, 0xFF, cells * (2 + 16), ctx->stream));
    }
    int smem_chunks = ctx->gate_chunks();
    if (smem_chunks > GATE_SMEM_CHUNKS) {
        ctx->fail("ewk_tick: ring_samples / frame_size = %d chunks; the gate keeps them in shared memory and supports at most %d "
                  "(use a larger frame_size or a shorter ring)", smem_chunks, GATE_SMEM_CHUNKS);
        return EWK_ERR_ARG;
    }
    if (smem_chunks & 1) smem_chunks++;                   // keeps the staging area 16-byte aligned
    // bulk staging of whole ticks pays when chunk arrays are small (frame_size 1600: 100 chunks)
    static const int stage_env = [] { const char* e = getenv("EWK_GATE_STAGE"); return e ? atoi(e) : 1; }();
    const int stage_bytes = (stage_env && smem_chunks <= 128 && !ctx->all_presummed) ? TICK * (B.fmt == 1 ? 2 : 4) : 0;
    if (B.n_pub > 0) {                                    // this call's sequence number and parity buffer at every destination
        ctx->publish_seq++;
        B.pub_seq = (unsigned long long)ctx->publish_seq;
        B.pub_parity = (int)((ctx->publish_seq - 1) & 1);
    }
    if (B.n_pub > 0 && ctx->ev_pub_valid[B.pub_parity])   // K2 rewrites this parity's copy: its sender (two calls ago) is long done
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_pub[B.pub_parity], 0));
    cudaEvent_t pe = ctx->prof_begin(1);
    for (int done = 0; done < rounds_ticks; done += GATE_MAX_TICKS) {
        const int nt = std::min(GATE_MAX_TICKS, rounds_ticks - done);
        auto k2 = paced ? tick_gate_kernel<true> : tick_gate_kernel<false>;
        k2<<<(B.n_streams + GATE_WARPS - 1) / GATE_WARPS, GATE_THREADS,
             sizeof(double) * 3 * (size_t)smem_chunks * GATE_WARPS + (size_t)2 * stage_bytes * GATE_WARPS,
             ctx->stream>>>(B, nt, tr, n_ticks, done, smem_chunks, stage_bytes);
        ctx->launches++;
    }
    ctx->prof_end(pe, 1);
    CK(cudaGetLastError());
    const int grid = ctx->queue_grid();
    // Overlap mode: K3 only reads ring samples of the last 3 s before the gated position and writes event / result
    // records, so the next push (K1) may run beside it; the next gate, poll or result read joins it first.  The push
    // guard keeps un-gated samples within the slack, which protects [visible - R, visible); the segments of these ticks
    // start at most 3 s + n_ticks x 0.1 s before it, hence the ring-length condition.
    cudaStream_t ks = ctx->stream;
    // ... plus the tail a cut drops: n_back = segment + n_drop, n_drop ~ (post_speech_silence + 0.05 s) and one tick of slop
    const long long drop_reserve = (long long)std::ceil((ctx->max_post + 0.15) * 16000.0);
    if (ctx->overlap && (long long)B.R >= MAX_SEG + (long long)(rounds_ticks + 2) * TICK + drop_reserve && !want) {
        CK(cudaEventRecord(ctx->ev_gate, ctx->stream));
        CK(cudaStreamWaitEvent(ctx->match_stream, ctx->ev_gate, 0));
        ks = ctx->match_stream;
    }
    ctx->last_match_stream = ks;
    pe = ctx->prof_begin(2, ks);
    if (ctx->k3_frames) {
        auto k3f = ctx->cfg.preemphasis != 0.f ? segment_frames_kernel<true> : segment_frames_kernel<false>;
        k3f<<<grid, SEG_THREADS, fq_smem_bytes(), ks>>>(ctx->d_tables, B, ctx->d_tmpl, ctx->cfg.max_templates);
    } else {
        auto k3q = ctx->cfg.preemphasis != 0.f ? segment_queue_kernel<true> : segment_queue_kernel<false>;
        k3q<<<grid, SEG_THREADS, seg_smem_bytes(SEG_SMEM_FRAMES), ks>>>(ctx->d_tables, B, ctx->d_tmpl, ctx->cfg.max_templates);
    }
    ctx->prof_end(pe, 2, ks);
    CK(cudaGetLastError());
    if (ks != ctx->stream) {
        CK(cudaEventRecord(ctx->ev_match, ks));
        ctx->match_inflight = true;
    }
    ctx->launches += 1;
    if (B.n_pub > 0) {
        // the sender: off everybody's critical path on its own stream, behind K3's snapshot of the records
        CK(cudaEventRecord(ctx->ev_k3, ks));
        CK(cudaStreamWaitEvent(ctx->pub_stream, ctx->ev_k3, 0));
        cudaEvent_t pp = ctx->prof_begin(6, ctx->pub_stream);
        publish_records_kernel<<<B.n_pub, 256, 0, ctx->pub_stream>>>(B);
        ctx->prof_end(pp, 6, ctx->pub_stream);
        CK(cudaGetLastError());
        ctx->launches += 1;
        CK(cudaEventRecord(ctx->ev_pub[B.pub_parity], ctx->pub_stream));
        ctx->ev_pub_valid[B.pub_parity] = true;
        ctx->launches += 1;
    }
    ctx->pushes_since_tick = 0;
    // host mirrors (audio clock): V after these ticks, given what has been pushed
    for (int s = 0; s < B.n_streams; s++) {
        const int k = paced ? budget[s] : n_ticks;
        if (taken) taken[s] = k;
        ctx->h_tick[s] += k;
        const StreamParams& p = ctx->h_prm[s];
        if (p.live) { ctx->h_visible_lb[s] = ctx->h_written[s]; continue; }
        const int fs = ctx->h_frame_size[s];
        if (fs > 0) {
            const long long v = std::min((ctx->h_tick[s] * TICK / fs) * fs, (ctx->h_written[s] / fs) * fs);
            ctx->h_visible_lb[s] = std::max(ctx->h_visible_lb[s], v);
        }
    }
    if (want) {
        if (thr) CK(cudaMemcpyAsync(thr, tr.thr, cells * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (rms) CK(cudaMemcpyAsync(rms, tr.rms, cells * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (silent) CK(cudaMemcpyAsync(silent, tr.silent, cells, cudaMemcpyDeviceToHost, ctx->stream));
        if (state) CK(cudaMemcpyAsync(state, tr.state, cells, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return EWK_OK;
}

extern "C" int ewk_tick(ewk_ctx* ctx, int n_ticks) {
    if (!ctx) return EWK_ERR_ARG;
    return tick_impl(ctx, n_ticks, false, nullptr, nullptr, nullptr, nullptr, nullptr);
}

extern "C" int ewk_tick_trace(ewk_ctx* ctx, int n_ticks, uint8_t* silent, uint8_t* state, double* thr, double* rms) {
    if (!ctx) return EWK_ERR_ARG;
    return tick_impl(ctx, n_ticks, false, nullptr, silent, state, thr, rms);
}

extern "C" int ewk_tick_ready(ewk_ctx* ctx, int max_ticks, int32_t* taken, uint8_t* silent, uint8_t* state, double* thr,
                              double* rms) {
    if (!ctx) return EWK_ERR_ARG;
    return tick_impl(ctx, max_ticks, true, taken, silent, state, thr, rms);
}

extern "C" int ewk_poll(ewk_ctx* ctx, ewk_event* out, int cap, int* dropped) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_poll");
    if (rc) return rc;
    if (cap < 0 || (cap > 0 && !out)) { ctx->fail("ewk_poll: bad output buffer"); return EWK_ERR_ARG; }
    BankView& B = ctx->bank;
    CK(cudaSetDevice(ctx->device));
    int cnt[2] = {0, 0};
    CK(cudaMemcpyAsync(cnt, B.ev_count, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    int n = std::min(cnt[0], B.max_events);
    if (dropped) *dropped = cnt[1];
    if (n > cap) { ctx->fail("ewk_poll: %d events pending but cap is %d", n, cap); return EWK_ERR_ARG; }
    if (n > 0) {
        CK(cudaMemcpyAsync(out, B.events, sizeof(EventRec) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaMemsetAsync(B.ev_count, 0, sizeof(int) * 7, ctx->stream));     // count, dropped, K3 work counter, scored watermark, frame table
    CK(cudaStreamSynchronize(ctx->stream));
    std::sort(out, out + n, [](const ewk_event& a, const ewk_event& b) {
        if (a.tick != b.tick) return a.tick < b.tick;
        if (a.stream != b.stream) return a.stream < b.stream;
        return a.kind < b.kind;
    });
    return n;
}

extern "C" int ewk_stream_status_get(ewk_ctx* ctx, int stream, ewk_stream_status* out) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_stream_status_get");
    if (rc) return rc;
    cudaSetDevice(ctx->device);
    rc = ctx->flush_pending();
    if (rc) return rc;
    if (!out || stream < 0 || stream >= ctx->bank.n_streams) { ctx->fail("ewk_stream_status_get: bad stream %d", stream); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    StreamState st;
    CK(cudaMemcpyAsync(&st, ctx->bank.st + stream, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    out->written = st.written; out->visible = st.visible; out->tick = st.tick;
    out->silence_threshold = st.thr; out->last_rms = st.last_rms; out->frame_size = st.frame_size;
    out->state = st.state; out->started = st.started; out->is_silent = st.last_silent;
    out->n_timeouts = st.n_timeouts; out->n_events = st.n_events;
    return EWK_OK;
}

// absolute samples [a0, a0+len) of one stream as float32 into `out` (host)
static int read_abs(ewk_ctx* ctx, int stream, long long a0, long long len, float* out) {
    BankView& B = ctx->bank;
    const size_t esz = B.fmt == 1 ? 2 : 4;
    std::vector<char> tmp((size_t)len * esz);
    const char* ring = (const char*)B.ring + (size_t)stream * B.P * esz;
    const long long p0 = ((a0 % B.P) + B.P) % B.P;
    const long long first = std::min<long long>(len, B.P - p0);
    CK(cudaMemcpyAsync(tmp.data(), ring + p0 * esz, (size_t)first * esz, cudaMemcpyDeviceToHost, ctx->stream));
    if (first < len)
        CK(cudaMemcpyAsync(tmp.data() + first * esz, ring, (size_t)(len - first) * esz, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (B.fmt == 1) {
        const short* q = (const short*)tmp.data();
        for (long long i = 0; i < len; i++) out[i] = (float)q[i] * (1.0f / 32768.0f);
    } else std::memcpy(out, tmp.data(), (size_t)len * 4);
    return EWK_OK;
}

extern "C" int ewk_read_last(ewk_ctx* ctx, int stream, int64_t n_samples, float* out) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_read_last");
    if (rc) return rc;
    cudaSetDevice(ctx->device);
    rc = ctx->flush_pending();
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (!out || stream < 0 || stream >= B.n_streams || n_samples < 0 || n_samples > B.R) {
        ctx->fail("ewk_read_last: bad arguments"); return EWK_ERR_ARG;
    }
    if (n_samples == 0) return EWK_OK;
    CK(cudaSetDevice(ctx->device));
    StreamState st;
    CK(cudaMemcpyAsync(&st, B.st + stream, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const long long V = ctx->h_prm[stream].live ? st.written : st.visible;
    // positions never written still hold the zeros of np.zeros (wakeword.py:428)
    const long long a0 = V - n_samples;
    long long lead = a0 < 0 ? -a0 : 0;
    for (long long i = 0; i < lead; i++) out[i] = 0.f;
    if (n_samples - lead > 0) return read_abs(ctx, stream, a0 + lead, n_samples - lead, out + lead);
    return EWK_OK;
}

extern "C" int ewk_read_segment(ewk_ctx* ctx, int stream, int64_t seg_start, int64_t seg_len, float* out) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_read_segment");
    if (rc) return rc;
    cudaSetDevice(ctx->device);
    rc = ctx->flush_pending();
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (!out || stream < 0 || stream >= B.n_streams || seg_len < 1 || seg_len > B.P || seg_start < 0) {
        ctx->fail("ewk_read_segment: bad arguments"); return EWK_ERR_ARG;
    }
    if (seg_start + seg_len > ctx->h_written[stream]) { ctx->fail("ewk_read_segment: segment not pushed yet"); return EWK_ERR_STATE; }
    if (ctx->h_written[stream] - seg_start > B.P) { ctx->fail("ewk_read_segment: segment already overwritten in the ring"); return EWK_ERR_STATE; }
    CK(cudaSetDevice(ctx->device));
    return read_abs(ctx, stream, seg_start, seg_len, out);
}

extern "C" int ewk_prepare_segments(ewk_ctx* ctx, int n_seg, const int32_t* streams, const int64_t* starts, const int64_t* lens,
                                    const int64_t* out_offsets, float* out, int64_t out_len, int where) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_prepare_segments");
    if (rc) return rc;
    cudaSetDevice(ctx->device);
    rc = ctx->flush_pending();
    if (rc) return rc;
    if (n_seg == 0) return EWK_OK;
    BankView& B = ctx->bank;
    if (n_seg < 0 || !streams || !starts || !lens || !out_offsets || !out || out_len < 1) {
        ctx->fail("ewk_prepare_segments: bad arguments");
        return EWK_ERR_ARG;
    }
    std::vector<PrepDesc> d(n_seg);
    for (int i = 0; i < n_seg; i++) {
        if (streams[i] < 0 || streams[i] >= B.n_streams || lens[i] < 1 || lens[i] > B.P || starts[i] < 0 ||
            out_offsets[i] < 0 || out_offsets[i] + lens[i] > out_len) {
            ctx->fail("ewk_prepare_segments: segment %d is out of range", i);
            return EWK_ERR_ARG;
        }
        if (starts[i] + lens[i] > ctx->h_written[streams[i]]) { ctx->fail("ewk_prepare_segments: segment %d not pushed yet", i); return EWK_ERR_STATE; }
        if (ctx->h_written[streams[i]] - starts[i] > B.P) { ctx->fail("ewk_prepare_segments: segment %d already overwritten in the ring", i); return EWK_ERR_STATE; }
        d[i] = PrepDesc{streams[i], (int)lens[i], starts[i], out_offsets[i]};
    }
    CK(cudaSetDevice(ctx->device));
    CK(ctx->b_desc.ensure(sizeof(PrepDesc) * (size_t)n_seg));
    CK(cudaMemcpyAsync(ctx->b_desc.p, d.data(), sizeof(PrepDesc) * (size_t)n_seg, cudaMemcpyHostToDevice, ctx->stream));
    float* d_out = out;
    if (where == EWK_HOST) { CK(ctx->b_read.ensure(sizeof(float) * (size_t)out_len)); d_out = (float*)ctx->b_read.p; }
    cudaEvent_t pe = ctx->prof_begin(5);
    segment_prepare_kernel<<<n_seg, 256, 0, ctx->stream>>>(B, (const PrepDesc*)ctx->b_desc.p, d_out);
    ctx->prof_end(pe, 5);
    CK(cudaGetLastError());
    ctx->launches++;
    if (where == EWK_HOST) {
        // copy back only the segments' ranges (merged where they touch): the scratch holds stale data elsewhere, and
        // floats of `out` between or after the segments are the caller's
        std::vector<std::pair<int64_t, int64_t>> iv(n_seg);
        for (int i = 0; i < n_seg; i++) iv[i] = {out_offsets[i], out_offsets[i] + lens[i]};
        std::sort(iv.begin(), iv.end());
        for (size_t i = 0; i < iv.size();) {
            int64_t a = iv[i].first, b = iv[i].second;
            for (++i; i < iv.size() && iv[i].first <= b; ++i) b = std::max(b, iv[i].second);
            CK(cudaMemcpyAsync(out + a, d_out + a, sizeof(float) * (size_t)(b - a), cudaMemcpyDeviceToHost, ctx->stream));
        }
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

extern "C" int ewk_set_templates_from_streams(ewk_ctx* ctx, const int32_t* slots, int n, const int32_t* streams,
                                              const int64_t* starts, const int64_t* lens, ewk_vad_result* vad) {
    if (!ctx) return EWK_ERR_ARG;
    const char* who = "ewk_set_templates_from_streams";
    int rc = need_streams(ctx, who);                         // overlap mode: K3 of the last tick still reads the table
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();                               // the ranges may reach into a pending push
    if (rc) return rc;
    rc = check_enrol(ctx, who, slots, n, starts, lens);
    if (rc) return rc;
    if (n == 0) return EWK_OK;
    if (!streams) { ctx->fail("%s: streams is NULL", who); return EWK_ERR_ARG; }
    const BankView& B = ctx->bank;
    std::vector<PrepDesc> g((size_t)n);
    std::vector<int64_t> off((size_t)n);
    int64_t packed = 0;
    for (int i = 0; i < n; i++) {                            // ewk_read_segment's checks, row by row
        const int s = streams[i];
        if (s < 0 || s >= B.n_streams || lens[i] > B.P) {
            ctx->fail("%s: row %d (stream %d): stream out of range [0, %d) or len %lld above the ring's %d samples", who, i,
                      s, B.n_streams, (long long)lens[i], B.P);
            return EWK_ERR_ARG;
        }
        if (starts[i] + lens[i] > ctx->h_written[s]) {
            ctx->fail("%s: row %d (stream %d): segment not pushed yet", who, i, s);
            return EWK_ERR_STATE;
        }
        if (ctx->h_written[s] - starts[i] > B.P) {
            ctx->fail("%s: row %d (stream %d): segment already overwritten in the ring", who, i, s);
            return EWK_ERR_STATE;
        }
        g[i] = PrepDesc{s, (int)lens[i], starts[i], packed};
        off[i] = packed;
        packed += lens[i];
    }
    return enrol_impl(ctx, who, slots, n, EnrolSource{nullptr, EWK_DEVICE, &g}, off.data(), lens, vad);
}

// ---- frame alignment: ewk_get_template_frames, ewk_align_segments, ewk_align_buffers (K3 + K11) ---------------------------
extern "C" int ewk_get_template_frames(ewk_ctx* ctx, int slot, float* out, int64_t cap, int32_t* n_frames) {
    if (!ctx) return EWK_ERR_ARG;
    const char* who = "ewk_get_template_frames";
    int rc = check_slot(ctx, slot, who);
    if (rc) return rc;
    if (!ctx->d_tfr) { ctx->fail("%s: the context keeps no template frames (ewk_config.template_frames = 0)", who); return EWK_ERR_STATE; }
    if (!ctx->h_tmpl[slot].valid) { ctx->fail("%s: template slot %d is empty. No reference word set. Call set_reference() first.", who, slot); return EWK_ERR_NO_TEMPLATE; }
    const int F = ctx->h_tfr_n[slot];
    if (out && cap < F) { ctx->fail("%s: cap %lld < %d frames", who, (long long)cap, F); return EWK_ERR_ARG; }
    if (n_frames) *n_frames = F;
    if (out && F) {
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpyAsync(out, ctx->d_tfr + (size_t)slot * ALIGN_MAX_FRAMES * N_MFCC, sizeof(float) * N_MFCC * (size_t)F,
                           cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return EWK_OK;
}

// Row i: segment descriptor seg[i] (base, start, ring, fmt set by the caller), set [first[i], first[i] + count[i]).  Checks
// the sets and the output capacity, then runs K3 over every segment (frames and features into workspaces) and K11, and
// copies the outputs back when where == EWK_HOST.  Every check comes before the first launch.
static int align_run(ewk_ctx* ctx, const char* who, int n, std::vector<SegDesc>& seg, const std::vector<int>& stream_of,
                     const int32_t* first, const int32_t* count, float* dist, int64_t dist_cap, int32_t* best_slot,
                     float* best_dist, int where, const void* h_pcm, size_t pcm_bytes) {
    std::vector<AlignRow> rows((size_t)n);
    long long frames = 0, packed = 0;
    int max_frames = 1;
    for (int i = 0; i < n; i++) {
        const int s = stream_of[i];
        const int f = first[i], c = count[i];
        if (c < 1 || c > ALIGN_MAX_T || f < 0 || f > ctx->cfg.max_templates - c) {
            ctx->fail("%s: row %d (stream %d) has a bad template range [%d, %d) (1..%d templates of %d slots)", who, i, s, f,
                      f + c, ALIGN_MAX_T, ctx->cfg.max_templates);
            return EWK_ERR_ARG;
        }
        for (int k = f; k < f + c; k++) {
            if (!ctx->h_tmpl[k].valid) {
                ctx->fail("%s: row %d (stream %d): template slot %d is empty. No reference word set. Call set_reference() first.",
                          who, i, s, k);
                return EWK_ERR_NO_TEMPLATE;
            }
            if (!ctx->h_tfr_n[k]) {
                ctx->fail("%s: row %d (stream %d): template slot %d has no frames (cleared, features only, or %lld samples: "
                          "over %d)", who, i, s, k, (long long)ctx->h_tmpl[k].n_samples, ALIGN_MAX_SAMPLES);
                return EWK_ERR_ARG;
            }
        }
        const int F = 1 + seg[i].len / HOP;
        seg[i].ws_frame_off = 0; seg[i].frames_off = frames; seg[i].lm_off = frames;
        rows[i] = AlignRow{frames, packed, F, f, c, 0};
        frames += F;
        packed += c;
        max_frames = std::max(max_frames, F);
    }
    if (dist_cap < packed) {
        ctx->fail("%s: dist_cap %lld is below the %lld distances of the rows", who, (long long)dist_cap, (long long)packed);
        return EWK_ERR_ARG;
    }
    // K3 keeps every frame's log-mel row (the top_db floor's input) only up to LM_WS_MAX_BYTES, as ewk_extract_mfcc does
    if (ctx->use_lm && sizeof(float) * (size_t)frames * LM_ROW > ewk_ctx::LM_WS_MAX_BYTES) {
        ctx->fail("%s: the segments hold %lld frames together; one call takes at most %lld (split the batch)", who,
                  (long long)frames, (long long)(ewk_ctx::LM_WS_MAX_BYTES / (sizeof(float) * LM_ROW)));
        return EWK_ERR_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    if (h_pcm) {                                            // host input: one copy, then the segments point into it
        CK(ctx->b_pcm.ensure(pcm_bytes));
        CK(cudaMemcpyAsync(ctx->b_pcm.p, h_pcm, pcm_bytes, cudaMemcpyHostToDevice, ctx->stream));
        for (int i = 0; i < n; i++) seg[i].base = ctx->b_pcm.p;
    }
    // descriptors, one upload: SegDesc [n] | AlignRow [n]
    const size_t o_row = sizeof(SegDesc) * (size_t)n;
    std::vector<char> desc(o_row + sizeof(AlignRow) * (size_t)n);
    std::memcpy(desc.data(), seg.data(), o_row);
    std::memcpy(desc.data() + o_row, rows.data(), sizeof(AlignRow) * (size_t)n);
    CK(ctx->b_desc.ensure(desc.size()));
    char* d_desc = (char*)ctx->b_desc.p;
    CK(cudaMemcpyAsync(d_desc, desc.data(), desc.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx->b_feat.ensure(sizeof(float) * FEAT * (size_t)n));
    CK(ctx->b_frames.ensure(sizeof(float) * N_MFCC * (size_t)frames));
    int rc = ctx->launch_segments((const SegDesc*)d_desc, n, max_frames, 0, frames, 0, 0, 0.f, (float*)ctx->b_feat.p,
                                  (float*)ctx->b_frames.p, nullptr, nullptr);
    if (rc != EWK_OK) return rc;
    // outputs: the caller's device memory, or scratch dist [packed] | best_dist [n] | best_slot [n] copied back
    float *o_dist = dist, *o_best = best_dist;
    int32_t* o_slot = best_slot;
    if (where == EWK_HOST) {
        CK(ctx->b_scores.ensure(sizeof(float) * (size_t)(packed + 2 * n)));
        o_dist = (float*)ctx->b_scores.p;
        o_best = best_dist ? o_dist + packed : nullptr;
        o_slot = best_slot ? (int32_t*)(o_dist + packed + n) : nullptr;
    }
    cudaEvent_t pe = ctx->prof_begin(3);
    segment_align_kernel<<<n, ALIGN_THREADS, 0, ctx->stream>>>((const AlignRow*)(d_desc + o_row), (const float*)ctx->b_frames.p,
                                                               (const float*)ctx->b_feat.p, ctx->d_tfr, ctx->d_tmpl,
                                                               ctx->cfg.n_mfcc > 0 ? ctx->cfg.n_mfcc : N_MFCC, o_dist,
                                                               o_best, o_slot);
    ctx->prof_end(pe, 3);
    CK(cudaGetLastError());
    ctx->launches++;
    if (where == EWK_HOST) {
        CK(cudaMemcpyAsync(dist, o_dist, sizeof(float) * (size_t)packed, cudaMemcpyDeviceToHost, ctx->stream));
        if (best_dist) CK(cudaMemcpyAsync(best_dist, o_best, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
        if (best_slot) CK(cudaMemcpyAsync(best_slot, o_slot, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

static int align_common_args(ewk_ctx* ctx, const char* who, int n, const int32_t* first, const int32_t* count,
                             const float* dist, int where) {
    if (!ctx->d_tfr) { ctx->fail("%s: the context keeps no template frames (ewk_config.template_frames = 0)", who); return EWK_ERR_STATE; }
    if (n < 0) { ctx->fail("%s: n = %d", who, n); return EWK_ERR_ARG; }
    if (!first != !count) {
        ctx->fail("%s: template_first and template_count must both be given or both be NULL", who);
        return EWK_ERR_ARG;
    }
    if (n > 0 && !dist) { ctx->fail("%s: dist must not be NULL", who); return EWK_ERR_ARG; }
    if (where != EWK_HOST && where != EWK_DEVICE) { ctx->fail("%s: where must be EWK_HOST or EWK_DEVICE", who); return EWK_ERR_ARG; }
    return EWK_OK;
}

extern "C" int ewk_align_segments(ewk_ctx* ctx, int n, const int32_t* streams, const int64_t* starts, const int64_t* lens,
                                  const int32_t* template_first, const int32_t* template_count, float* dist,
                                  int64_t dist_cap, int32_t* best_slot, float* best_dist, int where) {
    if (!ctx) return EWK_ERR_ARG;
    const char* who = "ewk_align_segments";
    int rc = align_common_args(ctx, who, n, template_first, template_count, dist, where);
    if (rc) return rc;
    rc = need_streams(ctx, who);                             // overlap mode: joins K3 of the last tick
    if (rc) return rc;
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();                               // the ranges may reach into a pending push
    if (rc) return rc;
    if (n == 0) return EWK_OK;
    if (!streams || !starts || !lens) { ctx->fail("%s: streams, starts and lens must not be NULL", who); return EWK_ERR_ARG; }
    const BankView& B = ctx->bank;
    const size_t esz = B.fmt == 1 ? 2 : 4;
    std::vector<SegDesc> seg((size_t)n);
    std::vector<int> st((size_t)n), f((size_t)n), c((size_t)n);
    for (int i = 0; i < n; i++) {                            // ewk_read_segment's checks, row by row
        const int s = streams[i];
        st[i] = s;
        if (s < 0 || s >= B.n_streams) {
            ctx->fail("%s: row %d (stream %d): stream out of range [0, %d)", who, i, s, B.n_streams);
            return EWK_ERR_ARG;
        }
        if (lens[i] < 1 || lens[i] > ALIGN_MAX_SAMPLES || starts[i] < 0) {
            ctx->fail("%s: row %d (stream %d): start %lld len %lld (need start >= 0, 1 <= len <= %d)", who, i, s,
                      (long long)starts[i], (long long)lens[i], ALIGN_MAX_SAMPLES);
            return EWK_ERR_ARG;
        }
        f[i] = template_first ? template_first[i] : ctx->h_prm[s].template_first;
        c[i] = template_count ? template_count[i] : ctx->h_prm[s].template_count;
    }
    for (int i = 0; i < n; i++) {
        const int s = st[i];
        if (starts[i] + lens[i] > ctx->h_written[s]) { ctx->fail("%s: row %d (stream %d): segment not pushed yet", who, i, s); return EWK_ERR_STATE; }
        if (ctx->h_written[s] - starts[i] > B.P) {
            ctx->fail("%s: row %d (stream %d): segment already overwritten in the ring", who, i, s);
            return EWK_ERR_STATE;
        }
        seg[i] = SegDesc{};
        seg[i].base = (const char*)B.ring + (size_t)s * B.P * esz;
        seg[i].start = starts[i] % B.P; seg[i].ring = B.P; seg[i].len = (int)lens[i]; seg[i].fmt = B.fmt;
    }
    return align_run(ctx, who, n, seg, st, f.data(), c.data(), dist, dist_cap, best_slot, best_dist, where, nullptr, 0);
}

extern "C" int ewk_align_buffers(ewk_ctx* ctx, int n, const void* pcm, int pcm_format, int where_in, const int64_t* offsets,
                                 const int64_t* lens, const int32_t* template_first, const int32_t* template_count,
                                 float* dist, int64_t dist_cap, int32_t* best_slot, float* best_dist, int where) {
    if (!ctx) return EWK_ERR_ARG;
    const char* who = "ewk_align_buffers";
    int rc = align_common_args(ctx, who, n, template_first, template_count, dist, where);
    if (rc) return rc;
    if (n == 0) return EWK_OK;
    if (!pcm || !offsets || !lens || !template_first || (pcm_format != EWK_PCM_F32 && pcm_format != EWK_PCM_I16) ||
        (where_in != EWK_HOST && where_in != EWK_DEVICE)) {
        ctx->fail("%s: need pcm, offsets, lens, template_first / template_count, pcm_format EWK_PCM_F32 or EWK_PCM_I16 and "
                  "where_in EWK_HOST or EWK_DEVICE", who);
        return EWK_ERR_ARG;
    }
    const size_t esz = pcm_format == EWK_PCM_I16 ? 2 : 4;
    std::vector<SegDesc> seg((size_t)n);
    std::vector<int> st((size_t)n, -1);
    int64_t extent = 0;
    for (int i = 0; i < n; i++) {
        if (offsets[i] < 0 || lens[i] < 1 || lens[i] > ALIGN_MAX_SAMPLES) {
            ctx->fail("%s: row %d (stream -1): offset %lld len %lld (need offset >= 0, 1 <= len <= %d)", who, i,
                      (long long)offsets[i], (long long)lens[i], ALIGN_MAX_SAMPLES);
            return EWK_ERR_ARG;
        }
        extent = std::max(extent, offsets[i] + lens[i]);
        seg[i] = SegDesc{};
        seg[i].base = pcm; seg[i].start = offsets[i]; seg[i].ring = 0; seg[i].len = (int)lens[i];
        seg[i].fmt = pcm_format == EWK_PCM_I16 ? 1 : 0;
    }
    rc = ctx->join_match();                                  // overlap mode: K3 of the last tick shares the K3 workspaces
    if (rc) return rc;
    return align_run(ctx, who, n, seg, st, template_first, template_count, dist, dist_cap, best_slot, best_dist, where,
                     where_in == EWK_HOST ? pcm : nullptr, esz * (size_t)extent);
}

static bool dense_plan(int T, int n_min, int n_max, int n_re_u, DensePlan& out) {
    const size_t SM_TOTAL = 233472, CTA_MAX = 232448, RESERVED = 1024;     // sm_100: 228 KB per SM, 227 KB per CTA
    auto bytes = [&](int DH, int threads) {
        return dense_smem_bytes(threads / 32, T, DH, DH + n_max + 2, DH + n_max - n_min, n_re_u);
    };
    for (int DH : {64, 32})
        for (int threads : {512, 448}) {
            const size_t b = bytes(DH, threads);
            if (2 * (b + RESERVED) <= SM_TOTAL) { out = {DH, threads, 2, b}; return true; }
        }
    for (int threads : {1024, 512})
        for (int DH : {64, 32}) {
            const size_t b = bytes(DH, threads);
            if (b <= CTA_MAX) { out = {DH, threads, 1, b}; return true; }
        }
    return false;
}

// Everything of a K4 call that follows from the template lengths alone (each in [DENSE_MIN_L, DENSE_MAX_L]): window
// geometry per template, the right-edge frames templates share, and the launch geometry.  ewk_dense_plan reports what
// the entry points launch because all go through here.  False: the set does not fit shared memory.
static bool dense_setup(const int64_t* lens, int n, DenseSetDev& S, DensePlan& plan) {
    S.T = n;
    int max_n = 0, min_n = 1 << 30, g_back = 1 << 30, n_re_u = 0;
    for (int k = 0; k < n; k++) {
        const int L = (int)lens[k];
        DenseTmplDev& t = S.t[k];
        t.L = L; t.n = (L + HOP - 1) / HOP; t.F = 1 + L / HOP; t.t_hi = (L - N_FFT / 2) / HOP; t.r = t.F - 1 - t.t_hi;
        t.inv_f = 1.0 / (double)t.F;
        max_n = std::max(max_n, t.n); min_n = std::min(min_n, t.n);
        g_back = std::min(g_back, t.n - t.t_hi);
        // right-edge frame e: stream-grid frame (hop - goff) cut at sample 160 hop - delta.  Templates with the same
        // (goff, delta) share it; the group is computed through the window of its shortest member
        const int delta = HOP * t.n - L;
        for (int e = 0; e < t.r; e++) {
            const int goff = t.n - (t.t_hi + 1 + e);
            int u = 0;
            while (u < n_re_u && !(S.re_goff[u] == goff && S.re_delta[u] == delta)) u++;
            if (u == n_re_u) {
                S.re_goff[u] = goff; S.re_delta[u] = delta; S.re_rep[u] = k; S.re_rep_e[u] = e; S.re_nfirst[u] = t.n;
                n_re_u++;
            } else if (t.n < S.re_nfirst[u]) { S.re_rep[u] = k; S.re_rep_e[u] = e; S.re_nfirst[u] = t.n; }
            t.re_u[e] = u;
        }
    }
    if (!dense_plan(n, min_n, max_n, n_re_u, plan)) return false;
    S.DH = plan.DH; S.DG = plan.DH + max_n + 2; S.DLE = plan.DH + max_n - min_n; S.n_re_u = n_re_u;
    S.n_min = min_n; S.n_max = max_n; S.g_back = g_back;
    return true;
}

extern "C" int ewk_dense_plan(const int64_t* template_lens, int n, int32_t out[4]) {
    if (!template_lens || !out || n < 1 || n > DENSE_MAX_T) return EWK_ERR_ARG;
    for (int k = 0; k < n; k++)
        if (template_lens[k] < DENSE_MIN_L || template_lens[k] > DENSE_MAX_L) return EWK_ERR_ARG;
    DenseSetDev S{};
    DensePlan plan;
    if (!dense_setup(template_lens, n, S, plan)) return EWK_ERR_ARG;
    out[0] = plan.DH; out[1] = plan.threads; out[2] = plan.per_sm; out[3] = (int32_t)plan.smem;
    return EWK_OK;
}

extern "C" int ewk_dense_last_plan(const ewk_ctx* ctx, int32_t out[4]) {
    if (!ctx || !out) return EWK_ERR_ARG;
    for (int i = 0; i < 4; i++) out[i] = ctx->dense_plan_info[i];
    return EWK_OK;
}

static bool dense_range_ok(const ewk_ctx* ctx, int first, int count) {
    return count >= 1 && count <= DENSE_MAX_T && first >= 0 && first <= ctx->cfg.max_templates - count;
}

// The template set [first, first + count) of a K4 call, with every check of it (errors name `who`): the range, each slot's
// presence and length, the fit in shared memory (dense_setup) and the ring length.
static int dense_set_build(ewk_ctx* ctx, const char* who, int first, int count, DenseSetHost& e) {
    if (!dense_range_ok(ctx, first, count)) {
        ctx->fail("%s: bad template range [%d, %d) (1..%d templates of %d slots)", who, first, first + count, DENSE_MAX_T,
                  ctx->cfg.max_templates);
        return EWK_ERR_ARG;
    }
    int64_t lens[DENSE_MAX_T];
    for (int k = first; k < first + count; k++) {
        const TemplateFeat& tf = ctx->h_tmpl[k];
        if (!tf.valid) {
            ctx->fail("%s: template slot %d is empty. No reference word set. Call set_reference() first.", who, k);
            return EWK_ERR_NO_TEMPLATE;
        }
        if (tf.n_samples < DENSE_MIN_L || tf.n_samples > DENSE_MAX_L) {
            ctx->fail("%s: template %d has %lld samples; dense scoring needs %d..%d", who, k, (long long)tf.n_samples,
                      DENSE_MIN_L, DENSE_MAX_L);
            return EWK_ERR_ARG;
        }
        lens[k - first] = tf.n_samples;
    }
    e = DenseSetHost{};
    DenseSetDev& d = e.dev;
    if (!dense_setup(lens, count, d, e.plan)) {
        ctx->fail("%s: this template set does not fit shared memory (%d templates, windows of %d..%d hops)", who, count,
                  (int)((*std::min_element(lens, lens + count) + HOP - 1) / HOP),
                  (int)((*std::max_element(lens, lens + count) + HOP - 1) / HOP));
        return EWK_ERR_ARG;
    }
    d.slot0 = first;
    for (int k = 0; k < count; k++) d.t[k].slot = first + k;
    if ((long long)ctx->bank.P < 160LL * (d.n_max + e.plan.DH + 4) + N_FFT) {        // the kernel wraps ring positions once
        ctx->fail("%s: ring of %d samples is too short for a template of %d hops", who, ctx->bank.P, d.n_max);
        return EWK_ERR_ARG;
    }
    return EWK_OK;
}

// the audio of every window of stream s at hops [hop0, hop0 + n_hops) (n_hops >= 1) must be resident
static int dense_resident(ewk_ctx* ctx, const char* who, int s, long long hop0, long long n_hops, int max_n) {
    const long long need_hi = 160LL * (hop0 + n_hops - 1);
    const long long need_lo = std::max<long long>(0, 160LL * (hop0 - max_n) - N_FFT / 2);
    if (ctx->h_written[s] < need_hi) {
        ctx->fail("%s: stream %d has %lld samples, hop %lld needs %lld", who, s, ctx->h_written[s], hop0 + n_hops - 1, need_hi);
        return EWK_ERR_STATE;
    }
    if (ctx->h_written[s] - need_lo > ctx->bank.P) {
        ctx->fail("%s: stream %d no longer holds sample %lld (ring of %d)", who, s, need_lo, ctx->bank.P);
        return EWK_ERR_STATE;
    }
    return EWK_OK;
}

// A host push whose copy is still in flight lands now only if the call's hops reach into its samples: otherwise the copy
// of the NEXT block keeps overlapping the call's kernel (offline sweeps: push block j + 1, then score block j).
// last_hop(s): the last hop the call scores on stream s (< 0: none).
template <class F>
static int dense_land_if_reached(ewk_ctx* ctx, F last_hop) {
    if (!ctx->pending.valid) return EWK_OK;
    const std::vector<RowDesc>& rows = ctx->pending.rows;
    for (int j = 0; j < ctx->pending.n_streams; j++) {
        const int s = rows.empty() ? ctx->pending.stream0 + j : rows[j].stream;
        const long long h = last_hop(s);
        if (h >= 0 && ctx->h_written[s] < 160LL * h) return ctx->flush_pending();
    }
    return EWK_OK;
}

// K4 over n_ctas CTAs into d_out: the uniform instance, or with A.rows set a row instance: the one-set instance when every
// row's set is A.set (one_set), else the per-row-set instance
static int dense_launch(ewk_ctx* ctx, DenseArgs& A, const DensePlan& plan, float* d_out, int n_ctas, bool one_set = true) {
    BankView& B = ctx->bank;
    A.out = d_out;
    if (!ctx->b_keep_rows.p) {
        CK(ctx->b_keep_rows.ensure(sizeof(float) * (size_t)B.n_streams * DENSE_KEEP * ROW));
        CK(ctx->b_keep_end.ensure(sizeof(long long) * 2 * (size_t)B.n_streams));
        CK(cudaMemsetAsync(ctx->b_keep_end.p, 0, sizeof(long long) * 2 * (size_t)B.n_streams, ctx->stream));
    }
    CK(ctx->b_g2.ensure(sizeof(float) * (size_t)B.n_streams * DENSE_WAYS * (one_set ? A.set.DG : A.DG) * N_MFCC));
    A.keep_rows = (float*)ctx->b_keep_rows.p;
    A.keep_end = (long long*)ctx->b_keep_end.p;
    A.g2 = (float*)ctx->b_g2.p;
    const bool pre = ctx->cfg.preemphasis != 0.f;
    auto k4 = !A.rows ? (pre ? dense_score_kernel<true, false, false> : dense_score_kernel<false, false, false>)
            : one_set ? (pre ? dense_score_kernel<true, true, false> : dense_score_kernel<false, true, false>)
                      : (pre ? dense_score_kernel<true, true, true> : dense_score_kernel<false, true, true>);
    CK(cudaFuncSetAttribute(k4, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan.smem));
    CK(cudaFuncSetAttribute(k4, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    cudaEvent_t pe = ctx->prof_begin(4);
    k4<<<n_ctas, plan.threads, plan.smem, ctx->stream>>>(ctx->d_tables, B, ctx->d_tmpl, A);
    ctx->prof_end(pe, 4);
    CK(cudaGetLastError());
    ctx->launches++;
    ctx->dense_plan_info[0] = plan.DH; ctx->dense_plan_info[1] = plan.threads; ctx->dense_plan_info[2] = plan.per_sm;
    ctx->dense_plan_info[3] = (int)plan.smem;
    return EWK_OK;
}

extern "C" int ewk_dense_scores(ewk_ctx* ctx, int64_t hop0, int n_hops, int tmpl_first, int tmpl_count, float* out, int where) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_dense_scores");
    if (rc) return rc;
    cudaSetDevice(ctx->device);
    BankView& B = ctx->bank;
    rc = dense_land_if_reached(ctx, [&](int) { return (long long)hop0 + n_hops - 1; });
    if (rc) return rc;
    if (!out || hop0 < 0 || n_hops < 1 || tmpl_count < 1 || tmpl_count > DENSE_MAX_T || tmpl_first < 0 ||
        tmpl_first + tmpl_count > ctx->cfg.max_templates) {
        ctx->fail("ewk_dense_scores: bad arguments (hop0=%lld n_hops=%d templates [%d, %d), at most %d per call)", (long long)hop0,
                  n_hops, tmpl_first, tmpl_first + tmpl_count, DENSE_MAX_T);
        return EWK_ERR_ARG;
    }
    DenseSetHost e;
    rc = dense_set_build(ctx, "ewk_dense_scores", tmpl_first, tmpl_count, e);
    if (rc) return rc;
    for (int s = 0; s < B.n_streams; s++) {
        rc = dense_resident(ctx, "ewk_dense_scores", s, hop0, n_hops, e.dev.n_max);
        if (rc) return rc;
    }
    CK(cudaSetDevice(ctx->device));
    const size_t n_out = (size_t)B.n_streams * n_hops * tmpl_count;
    float* d_out = out;
    if (where == EWK_HOST) { CK(ctx->b_dense.ensure(sizeof(float) * n_out)); d_out = (float*)ctx->b_dense.p; }
    DenseArgs A{};
    A.hop0 = hop0; A.n_hops = n_hops; A.set = e.dev;
    rc = dense_launch(ctx, A, e.plan, d_out, B.n_streams);
    if (rc) return rc;
    if (where == EWK_HOST) {
        CK(cudaMemcpyAsync(out, d_out, sizeof(float) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return EWK_OK;
}

// ---- template sets of the row calls: a table of descriptors on the device, built on first use ------------------------
static inline int dset_key(int first, int count) { return first * DENSE_MAX_T + count - 1; }

void ewk_ctx::dense_sets_forget(int slot) {
    for (int c = 1; c <= DENSE_MAX_T; c++)
        for (int f = std::max(0, slot - c + 1); f <= slot; f++)
            if ((size_t)dset_key(f, c) < h_dset.size()) h_dset[dset_key(f, c)].valid = false;
}

// The set of each row of a row call.  uniform (the single-set entry points): [first1, first1 + count1) for every row;
// otherwise row i's is [first[i], first[i] + count[i]), and with both arrays NULL its stream's own range.
struct RowSets {
    const int32_t* first;
    const int32_t* count;
    bool uniform;
    int first1, count1;
};

// Row i's set -> key[i] (its index in the context's table), with every check of the set; sets not cached yet are built
// into `fresh`, which dense_sets_commit uploads once the call has passed every check.  A uniform call resolves its one
// set, and its messages name `who`; otherwise they name the row and the stream.
static int dense_sets_resolve(ewk_ctx* ctx, const char* who, const int32_t* streams, int n, const RowSets& rs,
                              std::vector<int>& key, std::map<int, DenseSetHost>& fresh) {
    if (!rs.uniform && !rs.first != !rs.count) {
        ctx->fail("%s: template_first and template_count must both be given or both be NULL", who);
        return EWK_ERR_ARG;
    }
    if (ctx->h_dset.empty()) ctx->h_dset.resize((size_t)ctx->cfg.max_templates * DENSE_MAX_T);
    key.assign((size_t)n, -1);
    for (int i = 0; i < n; i++) {
        if (rs.uniform && i > 0) { key[i] = key[0]; continue; }
        const int s = streams[i];
        const int f = rs.uniform ? rs.first1 : rs.first ? rs.first[i] : ctx->h_prm[s].template_first;
        const int c = rs.uniform ? rs.count1 : rs.count ? rs.count[i] : ctx->h_prm[s].template_count;
        if (dense_range_ok(ctx, f, c)) {
            key[i] = dset_key(f, c);
            if (ctx->h_dset[key[i]].valid || fresh.count(key[i])) continue;
        }
        char w[192];
        snprintf(w, sizeof w, "%s: row %d (stream %d)", who, i, s);
        DenseSetHost e;
        const int rc = dense_set_build(ctx, rs.uniform ? who : w, f, c, e);
        if (rc) return rc;
        fresh[key[i]] = e;
    }
    return EWK_OK;
}

// the new descriptors -> a staging slot -> their places in the table (one copy per run of consecutive keys), in stream
// order behind every K4 / K4D that read an older descriptor at those places
static int dense_sets_commit(ewk_ctx* ctx, const std::map<int, DenseSetHost>& fresh) {
    if (!ctx->b_dset.p) CK(ctx->b_dset.ensure(sizeof(DenseSetDev) * ctx->h_dset.size()));
    if (fresh.empty()) return EWK_OK;
    std::vector<DenseSetDev> up;
    std::vector<int> keys;
    for (const auto& kv : fresh) { keys.push_back(kv.first); up.push_back(kv.second.dev); }
    SlotPair<DenseSetDev>& st = ctx->dset_stage;
    int k = -1;
    int rc = upload_slot(ctx, st.h, st.b, st.ev, st.ev_valid, st.idx, up, ctx->stream, &k);
    if (rc) return rc;
    DenseSetDev* tab = (DenseSetDev*)ctx->b_dset.p;
    const DenseSetDev* stage = (const DenseSetDev*)st.b[k].p;
    for (size_t a = 0; a < keys.size();) {
        size_t b = a + 1;
        while (b < keys.size() && keys[b] == keys[b - 1] + 1) b++;
        CK(cudaMemcpyAsync(tab + keys[a], stage + a, sizeof(DenseSetDev) * (b - a), cudaMemcpyDeviceToDevice, ctx->stream));
        a = b;
    }
    CK(cudaEventRecord(st.ev[k], ctx->stream));
    st.ev_valid[k] = true;
    for (const auto& kv : fresh) { ctx->h_dset[kv.first] = kv.second; ctx->h_dset[kv.first].valid = true; }
    return EWK_OK;
}

// Rows of ewk_dense_scores_streams, ewk_dense_ready, ewk_dense_detect and their _sets forms: row i scores stream
// streams[i] at hops [hop0[i], hop0[i] + n_hops[i]) against its set (rs), packed from float sum_{j < i} n_hops[j] T_j and
// laid out [n_hops[i]][T_i].  One K4 launch per launch geometry (DH, threads, CTAs per SM) among the rows' sets, each set
// at the geometry it has alone; the launch gets its group's largest shared memory and g2 stride, and runs its rows longest
// first so that it ends with short ones.  A group whose rows all share one set (every group of a single-set call) runs
// K4's one-set row instance with that set in its arguments, a group of several sets the per-row-set instance.  Every check comes before the first launch or copy, so an error changes no state.
// d_scores (the detect calls): the caller reads the scores on the device after K4 and copies host output itself; out may
// then be NULL (the scores stay in device scratch), and *d_scores receives where K4 wrote them (NULL when no row has
// hops).  *keys (when given) receives each row's key.
static int dense_rows(ewk_ctx* ctx, const char* who, const int32_t* streams, int n, const int64_t* hop0,
                      const int32_t* n_hops, const RowSets& rs, float* out, int64_t out_cap, int where,
                      float** d_scores = nullptr, std::vector<int>* keys = nullptr) {
    if (d_scores) *d_scores = nullptr;
    BankView& B = ctx->bank;
    if (n < 0 || (n > 0 && (!streams || !hop0 || !n_hops))) { ctx->fail("%s: bad row list (n=%d)", who, n); return EWK_ERR_ARG; }
    if (n == 0) return EWK_OK;
    std::vector<int> row_of((size_t)B.n_streams, -1);
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        if (s < 0 || s >= B.n_streams) { ctx->fail("%s: bad stream %d (context has %d)", who, s, B.n_streams); return EWK_ERR_ARG; }
        if (row_of[s] >= 0) { ctx->fail("%s: stream %d is listed twice", who, s); return EWK_ERR_ARG; }
        row_of[s] = i;
        if (hop0[i] < 0 || n_hops[i] < 0 || hop0[i] > ((int64_t)1 << 48)) {
            ctx->fail("%s: row %d of stream %d has bad hops (hop0=%lld n_hops=%d)", who, i, s, (long long)hop0[i], n_hops[i]);
            return EWK_ERR_ARG;
        }
    }
    std::vector<int> key;
    std::map<int, DenseSetHost> fresh;
    int rc = dense_sets_resolve(ctx, who, streams, n, rs, key, fresh);
    if (rc) return rc;
    auto set_of = [&](int i) -> const DenseSetHost& {
        if (fresh.empty()) return ctx->h_dset[key[i]];
        const auto it = fresh.find(key[i]);
        return it != fresh.end() ? it->second : ctx->h_dset[key[i]];
    };
    long long n_out = 0;
    for (int i = 0; i < n; i++) n_out += (long long)n_hops[i] * set_of(i).dev.T;
    if (n_out > 0 && (out || !d_scores) && (!out || out_cap < n_out)) {
        ctx->fail("%s: out holds %lld floats, the rows need %lld", who, out ? (long long)out_cap : 0LL, n_out);
        return EWK_ERR_ARG;
    }
    CK(cudaSetDevice(ctx->device));
    rc = dense_land_if_reached(ctx, [&](int s) {
        const int i = row_of[s];
        return i >= 0 && n_hops[i] > 0 ? (long long)hop0[i] + n_hops[i] - 1 : -1LL;
    });
    if (rc) return rc;
    for (int i = 0; i < n; i++) {
        if (n_hops[i] == 0) continue;
        rc = dense_resident(ctx, who, streams[i], hop0[i], n_hops[i], set_of(i).dev.n_max);
        if (rc) return rc;
    }
    if (keys) *keys = key;
    if (n_out == 0) return EWK_OK;
    rc = dense_sets_commit(ctx, fresh);
    if (rc) return rc;
    // geometry groups in order of first appearance
    struct Group { DensePlan plan; int DG, key; size_t n_rows; };   // key: the rows' one set, -1: several
    std::vector<Group> groups;
    std::vector<unsigned char> group_of((size_t)n);
    size_t n_rows = 0;
    int max_dg = 0;
    for (int i = 0; i < n; i++) {
        if (n_hops[i] == 0) continue;
        const DenseSetHost& e = ctx->h_dset[key[i]];
        size_t g = 0;
        while (g < groups.size() && !(groups[g].plan.DH == e.plan.DH && groups[g].plan.threads == e.plan.threads &&
                                      groups[g].plan.per_sm == e.plan.per_sm)) g++;
        if (g == groups.size()) groups.push_back(Group{DensePlan{e.plan.DH, e.plan.threads, e.plan.per_sm, 0}, 0, key[i], 0});
        if (groups[g].key != key[i]) groups[g].key = -1;
        groups[g].plan.smem = std::max(groups[g].plan.smem, e.plan.smem);
        groups[g].DG = std::max(groups[g].DG, e.dev.DG);
        groups[g].n_rows++;
        group_of[i] = (unsigned char)g;
        max_dg = std::max(max_dg, e.dev.DG);
        n_rows++;
    }
    // the descriptors group by group, each group's rows longest first
    const DenseSetDev* tab = (const DenseSetDev*)ctx->b_dset.p;
    std::vector<DenseRow> rows;
    rows.reserve(n_rows);
    for (size_t g = 0; g < groups.size(); g++) {
        const size_t first = rows.size();
        long long off = 0;
        for (int i = 0; i < n; i++) {
            if (n_hops[i] > 0 && group_of[i] == g) rows.push_back(DenseRow{hop0[i], off, streams[i], n_hops[i], tab + key[i]});
            off += (long long)n_hops[i] * ctx->h_dset[key[i]].dev.T;
        }
        auto longer = [](const DenseRow& a, const DenseRow& b) { return a.n_hops > b.n_hops; };
        if (!std::is_sorted(rows.begin() + first, rows.end(), longer))     // paced calls often give every row max_hops
            std::stable_sort(rows.begin() + first, rows.end(), longer);
    }
    SlotPair<DenseRow>& sp = ctx->drows;
    int k = -1;
    rc = upload_slot(ctx, sp.h, sp.b, sp.ev, sp.ev_valid, sp.idx, rows, ctx->stream, &k);
    if (rc) return rc;
    float* d_out = out;
    if (where == EWK_HOST || !out) { CK(ctx->b_dense.ensure(sizeof(float) * (size_t)n_out)); d_out = (float*)ctx->b_dense.p; }
    CK(ctx->b_g2.ensure(sizeof(float) * (size_t)B.n_streams * DENSE_WAYS * max_dg * N_MFCC));
    size_t base = 0;
    for (const Group& g : groups) {
        DenseArgs A{};
        A.DH = g.plan.DH;
        A.DG = g.DG;
        if (g.key >= 0) A.set = ctx->h_dset[g.key].dev;
        A.rows = (const DenseRow*)sp.b[k].p + base;
        rc = dense_launch(ctx, A, g.plan, d_out, (int)g.n_rows, g.key >= 0);
        if (rc) return rc;
        base += g.n_rows;
    }
    CK(cudaEventRecord(sp.ev[k], ctx->stream));               // the slot is free once these K4 launches have read it
    sp.ev_valid[k] = true;
    if (d_scores) { *d_scores = d_out; return EWK_OK; }
    if (where == EWK_HOST) {
        CK(cudaMemcpyAsync(out, d_out, sizeof(float) * (size_t)n_out, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return EWK_OK;
}

extern "C" int ewk_dense_scores_sets(ewk_ctx* ctx, const int32_t* streams, int n, const int64_t* hop0, const int32_t* n_hops,
                                     const int32_t* template_first, const int32_t* template_count, float* out, int64_t out_cap,
                                     int where) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_dense_scores_sets");
    if (rc) return rc;
    return dense_rows(ctx, "ewk_dense_scores_sets", streams, n, hop0, n_hops, RowSets{template_first, template_count, false, 0, 0},
                      out, out_cap, where);
}

extern "C" int ewk_dense_scores_streams(ewk_ctx* ctx, const int32_t* streams, int n, const int64_t* hop0, const int32_t* n_hops,
                                        int template_first, int template_count, float* out, int64_t out_cap, int where) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_dense_scores_streams");
    if (rc) return rc;
    return dense_rows(ctx, "ewk_dense_scores_streams", streams, n, hop0, n_hops,
                      RowSets{nullptr, nullptr, true, template_first, template_count}, out, out_cap, where);
}

// The rows a paced call (ewk_dense_ready, ewk_dense_detect and their _sets forms) scores: max_hops is checked, NULL streams
// means every stream, the list is checked (outs: the caller's per-row outputs are given); then the pending push lands,
// since the due hops depend on every landed sample, and the due rule runs on `cursor`: hop h is due once 160 h samples
// have landed, from the cursor on, at most max_hops.
struct DueRows {
    std::vector<int32_t> streams;
    std::vector<int64_t> h0;
    std::vector<int32_t> nh;
};

static int dense_due(ewk_ctx* ctx, const char* who, const int32_t* streams, int n, int max_hops, bool outs,
                     const std::vector<long long>& cursor, DueRows& d) {
    const int ns = ctx->bank.n_streams;
    if (max_hops < 1 || max_hops > (1 << 20)) { ctx->fail("%s: max_hops must be in [1, %d]", who, 1 << 20); return EWK_ERR_ARG; }
    if (!streams) {
        d.streams.resize((size_t)ns);
        for (int s = 0; s < ns; s++) d.streams[s] = s;
        streams = d.streams.data();
        n = ns;
    }
    if (n > 0 && !outs) { ctx->fail("%s: bad stream list (n=%d)", who, n); return EWK_ERR_ARG; }
    int rc = check_stream_list(ctx, who, streams, n);
    if (rc) return rc;
    d.streams.assign(streams, streams + n);
    CK(cudaSetDevice(ctx->device));
    rc = ctx->flush_pending();
    if (rc) return rc;
    d.h0.resize((size_t)n);
    d.nh.resize((size_t)n);
    for (int i = 0; i < n; i++) {
        const int s = streams[i];
        d.h0[i] = cursor[s];
        d.nh[i] = (int32_t)std::max<long long>(0, std::min<long long>(d.h0[i] + max_hops, ctx->h_written[s] / 160 + 1) - d.h0[i]);
    }
    return EWK_OK;
}

// ewk_dense_ready and ewk_dense_ready_sets
static int dense_ready_impl(ewk_ctx* ctx, const char* who, const int32_t* streams, int n, int max_hops, const RowSets& rs,
                            int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap, int where) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, who);
    if (rc) return rc;
    DueRows d;
    rc = dense_due(ctx, who, streams, n, max_hops, hop0_out && n_hops_out, ctx->h_dense_next, d);
    if (rc) return rc;
    n = (int)d.streams.size();
    rc = dense_rows(ctx, who, d.streams.data(), n, d.h0.data(), d.nh.data(), rs, out, out_cap, where);
    if (rc) return rc;
    for (int i = 0; i < n; i++) {
        hop0_out[i] = d.h0[i];
        n_hops_out[i] = d.nh[i];
        ctx->h_dense_next[d.streams[i]] += d.nh[i];
    }
    return EWK_OK;
}

extern "C" int ewk_dense_ready(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops, int template_first,
                               int template_count, int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap,
                               int where) {
    return dense_ready_impl(ctx, "ewk_dense_ready", streams, n, max_hops,
                            RowSets{nullptr, nullptr, true, template_first, template_count}, hop0_out, n_hops_out, out,
                            out_cap, where);
}

extern "C" int ewk_dense_ready_sets(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops, const int32_t* template_first,
                                    const int32_t* template_count, int64_t* hop0_out, int32_t* n_hops_out, float* out,
                                    int64_t out_cap, int where) {
    return dense_ready_impl(ctx, "ewk_dense_ready_sets", streams, n, max_hops,
                            RowSets{template_first, template_count, false, 0, 0}, hop0_out, n_hops_out, out, out_cap, where);
}

static_assert(sizeof(DetRecord) == sizeof(ewk_detection) && sizeof(ewk_detection) == 48, "ewk_detection layout");
static_assert(offsetof(DetRecord, score) == offsetof(ewk_detection, score), "ewk_detection layout");

// ewk_dense_detect and ewk_dense_detect_sets: ewk_dense_ready's due rule on the detector's own cursor, then K4 (one launch
// per geometry) and K4D behind it on the context's stream.
static int dense_detect_impl(ewk_ctx* ctx, const char* who, const int32_t* streams, int n, int max_hops, const RowSets& rs,
                             int hold_hops, int refractory_hops, ewk_detection* det, int det_cap, int64_t* hop0_out,
                             int32_t* n_hops_out, float* out, int64_t out_cap, int where) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, who);
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (hold_hops < 1 || refractory_hops < 0) {
        ctx->fail("%s: hold_hops must be >= 1 and refractory_hops >= 0 (got %d, %d)", who, hold_hops, refractory_hops);
        return EWK_ERR_ARG;
    }
    DueRows d;
    rc = dense_due(ctx, who, streams, n, max_hops, true, ctx->h_det_next, d);
    if (rc) return rc;
    n = (int)d.streams.size();
    const std::vector<int64_t>& h0 = d.h0;
    const std::vector<int32_t>& nh = d.nh;
    long long need = 0;                                      // emissions are >= 2 hops apart: ceil(n_i / 2) per row
    for (int i = 0; i < n; i++) need += (nh[i] + 1) / 2;
    if (det_cap < need || (need > 0 && !det)) {
        ctx->fail("%s: det holds %d records, the due hops need %lld", who, det ? det_cap : 0, need);
        return EWK_ERR_ARG;
    }
    // K4D's output: counts [n_streams], then the records of row i from offset sum_{j < i} ceil(n_j / 2)
    const size_t rec_off = ((size_t)4 * B.n_streams + 15) / 16 * 16, map_bytes = rec_off + sizeof(DetRecord) * (size_t)need;
    if (map_bytes > ctx->det_map_cap) {
        if (ctx->h_det_map) CK(ctx->pool.free(ctx->h_det_map, true));
        ctx->h_det_map = nullptr; ctx->det_map_cap = 0;
        const size_t want = ctx->pool.poison >= 0 ? map_bytes : map_bytes + map_bytes / 4 + 256;
        CK(ctx->pool.alloc_host(&ctx->h_det_map, want, cudaHostAllocMapped | cudaHostAllocPortable, "h_det_map"));
        ctx->det_map_cap = want;
    } else if (ctx->pool.poison >= 0) {
        CK(ctx->pool.refill(ctx->h_det_map));                // the previous call's records are dead
    }
    float* d_scores = nullptr;
    std::vector<int> keys;
    rc = dense_rows(ctx, who, d.streams.data(), n, h0.data(), nh.data(), rs, out, out_cap, where, &d_scores, &keys);
    if (rc) return rc;
    int n_det = 0;
    if (d_scores) {
        if (!ctx->b_det_state.p) {
            CK(ctx->b_det_state.ensure(sizeof(DetState) * (size_t)B.n_streams));
            CK(cudaMemsetAsync(ctx->b_det_state.p, 0, sizeof(DetState) * (size_t)B.n_streams, ctx->stream));
        }
        std::vector<DetRow> rows;
        rows.reserve((size_t)n);
        long long off = 0, doff = 0;
        for (int i = 0; i < n; i++) {
            if (nh[i] > 0) rows.push_back(DetRow{h0[i], off, doff, d.streams[i], nh[i], i, 0, (const DenseSetDev*)ctx->b_dset.p + keys[i]});
            off += (long long)nh[i] * ctx->h_dset[keys[i]].dev.T;
            doff += (nh[i] + 1) / 2;
        }
        SlotPair<DetRow>& sp = ctx->ddets;
        int k = -1;
        rc = upload_slot(ctx, sp.h, sp.b, sp.ev, sp.ev_valid, sp.idx, rows, ctx->stream, &k);
        if (rc) return rc;
        char* d_map = nullptr;
        CK(cudaHostGetDevicePointer((void**)&d_map, ctx->h_det_map, 0));
        DetArgs D{};
        D.hold = hold_hops; D.refractory = refractory_hops;
        D.rows = (const DetRow*)sp.b[k].p; D.n_rows = (int)rows.size();
        D.scores = d_scores; D.state = (DetState*)ctx->b_det_state.p;
        D.counts = (int*)d_map; D.rec = (DetRecord*)(d_map + rec_off);
        cudaEvent_t pe = ctx->prof_begin(4);
        dense_detect_kernel<<<(D.n_rows + DETECT_WARPS - 1) / DETECT_WARPS, 32 * DETECT_WARPS, 0, ctx->stream>>>(B.prm, D);
        ctx->prof_end(pe, 4);
        CK(cudaGetLastError());
        ctx->launches++;
        CK(cudaEventRecord(sp.ev[k], ctx->stream));
        sp.ev_valid[k] = true;
        if (out && where == EWK_HOST)
            CK(cudaMemcpyAsync(out, d_scores, sizeof(float) * (size_t)off, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        // list order, then emit order within a row
        const int* counts = (const int*)ctx->h_det_map;
        const DetRecord* rec = (const DetRecord*)((const char*)ctx->h_det_map + rec_off);
        for (const DetRow& r : rows) {
            std::memcpy((DetRecord*)det + n_det, rec + r.det, sizeof(DetRecord) * (size_t)counts[r.row]);
            n_det += counts[r.row];
        }
    }
    for (int i = 0; i < n; i++) {
        if (hop0_out) hop0_out[i] = h0[i];
        if (n_hops_out) n_hops_out[i] = nh[i];
        ctx->h_det_next[d.streams[i]] += nh[i];
    }
    return n_det;
}

extern "C" int ewk_dense_detect(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops, int template_first,
                                int template_count, int hold_hops, int refractory_hops, ewk_detection* det, int det_cap,
                                int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap, int where) {
    return dense_detect_impl(ctx, "ewk_dense_detect", streams, n, max_hops,
                             RowSets{nullptr, nullptr, true, template_first, template_count}, hold_hops, refractory_hops,
                             det, det_cap, hop0_out, n_hops_out, out, out_cap, where);
}

extern "C" int ewk_dense_detect_sets(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops, const int32_t* template_first,
                                     const int32_t* template_count, int hold_hops, int refractory_hops, ewk_detection* det,
                                     int det_cap, int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap,
                                     int where) {
    return dense_detect_impl(ctx, "ewk_dense_detect_sets", streams, n, max_hops,
                             RowSets{template_first, template_count, false, 0, 0}, hold_hops, refractory_hops, det, det_cap,
                             hop0_out, n_hops_out, out, out_cap, where);
}

extern "C" int ewk_stream_results(ewk_ctx* ctx, ewk_stream_result* out) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_stream_results");
    if (rc) return rc;
    if (!out) { ctx->fail("ewk_stream_results: null output"); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(out, ctx->bank.results, sizeof(StreamResult) * (size_t)ctx->bank.n_streams, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return EWK_OK;
}

extern "C" int ewk_results_device_ptr(ewk_ctx* ctx, void** out) {
    if (!ctx || !out) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_results_device_ptr");
    if (rc) return rc;
    *out = ctx->bank.results;
    return EWK_OK;
}

extern "C" int ewk_set_results_buffer(ewk_ctx* ctx, void* device_ptr) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_set_results_buffer");
    if (rc) return rc;
    if ((size_t)device_ptr & 7) { ctx->fail("ewk_set_results_buffer: the buffer must be 8-byte aligned (records are stored as one 64-bit word)"); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    StreamResult* dst = device_ptr ? (StreamResult*)device_ptr : (StreamResult*)ctx->own_results;
    if (dst != ctx->bank.results) {
        CK(cudaMemcpyAsync(dst, ctx->bank.results, sizeof(StreamResult) * (size_t)ctx->bank.n_streams, cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->bank.results = dst;
    }
    return EWK_OK;
}

extern "C" int ewk_set_results_peers(ewk_ctx* ctx, void* const* bases, int n_bases, int64_t stride_records, int64_t offset_records,
                                     void* const* signals, int slot) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_set_results_peers");
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (n_bases < 0 || n_bases > MAX_PUB || (n_bases > 0 && !bases)) {
        ctx->fail("ewk_set_results_peers: n_bases must be in [0, %d]", MAX_PUB);
        return EWK_ERR_ARG;
    }
    if (n_bases > 0 && (offset_records < 0 || stride_records < offset_records + B.n_streams)) {
        ctx->fail("ewk_set_results_peers: stride %lld cannot hold %d records at offset %lld",
                  (long long)stride_records, B.n_streams, (long long)offset_records);
        return EWK_ERR_ARG;
    }
    if (n_bases > 0 && signals && (slot < 0 || slot >= n_bases)) {
        ctx->fail("ewk_set_results_peers: slot %d outside [0, %d)", slot, n_bases);
        return EWK_ERR_ARG;
    }
    for (int p = 0; p < n_bases; p++) {
        if (!bases[p] || ((size_t)bases[p] & 7)) { ctx->fail("ewk_set_results_peers: destination %d is null or not 8-byte aligned", p); return EWK_ERR_ARG; }
        if (signals && (!signals[p] || ((size_t)signals[p] & 7))) { ctx->fail("ewk_set_results_peers: signal row %d is null or not 8-byte aligned", p); return EWK_ERR_ARG; }
    }
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));                // kernels in flight keep the destinations they were launched with
    for (int p = 0; p < MAX_PUB; p++) {
        B.pub[p] = p < n_bases ? (StreamResult*)bases[p] : nullptr;
        B.pub_sig[p] = (p < n_bases && signals) ? (unsigned long long*)signals[p] : nullptr;
    }
    B.n_pub = n_bases;
    B.pub_stride = n_bases ? stride_records : 0;
    B.pub_off = n_bases ? offset_records : 0;
    B.pub_slot = n_bases && signals ? slot : 0;
    B.pub_seq = 0;
    B.pub_parity = 0;
    ctx->publish_seq = 0;
    if (ctx->pub_stream) CK(cudaStreamSynchronize(ctx->pub_stream));
    ctx->ev_pub_valid[0] = ctx->ev_pub_valid[1] = false;
    if (n_bases && !ctx->pub_stream) {
        // highest priority: the sender is a handful of CTAs that should start the moment K3 ends, not queue behind the
        // full grids of the next push
        int prio_lo = 0, prio_hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CK(cudaStreamCreateWithPriority(&ctx->pub_stream, cudaStreamNonBlocking, prio_hi));
        CK(cudaEventCreateWithFlags(&ctx->ev_k3, cudaEventDisableTiming));
        for (int i = 0; i < 2; i++) CK(cudaEventCreateWithFlags(&ctx->ev_pub[i], cudaEventDisableTiming));
        CK(ctx->pool.alloc(&ctx->d_pub_snap, sizeof(StreamResult) * 2 * (size_t)B.n_streams, "d_pub_snap"));
    }
    B.pub_snap = (StreamResult*)ctx->d_pub_snap;
    if (n_bases && signals && !ctx->d_wait_flag) {
        CK(ctx->pool.alloc(&ctx->d_wait_flag, sizeof(int), "d_wait_flag"));
        CK(cudaMemsetAsync(ctx->d_wait_flag, 0, sizeof(int), ctx->stream));
    }
    return EWK_OK;
}

extern "C" int ewk_publish_parity(const ewk_ctx* ctx) { return ctx && ctx->publish_seq > 0 ? (int)((ctx->publish_seq - 1) & 1) : -1; }
extern "C" int64_t ewk_publish_seq(const ewk_ctx* ctx) { return ctx ? ctx->publish_seq : 0; }

extern "C" int ewk_wait_published(ewk_ctx* ctx, int n_slots, int64_t seq, int timeout_ms) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_wait_published", false);
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (!B.n_pub || !B.pub_sig[0]) { ctx->fail("ewk_wait_published: no signal rows installed (ewk_set_results_peers)"); return EWK_ERR_STATE; }
    if (n_slots < 1 || n_slots > B.n_pub || seq < 1 || timeout_ms < 1) { ctx->fail("ewk_wait_published: bad arguments"); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    // this rank's own sender (side stream, same GPU) first: the wait kernel then only spins on other GPUs' signals
    if (ctx->ev_pub_valid[(seq - 1) & 1]) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_pub[(seq - 1) & 1], 0));
    const unsigned long long* row = B.pub_sig[B.pub_slot] + (size_t)((seq - 1) & 1) * MAX_PUB;
    peer_wait_kernel<<<1, 32, 0, ctx->stream>>>(row, n_slots, (unsigned long long)seq, (unsigned long long)timeout_ms * 1000000ULL,
                                                ctx->d_wait_flag);
    CK(cudaGetLastError());
    ctx->launches++;
    return EWK_OK;
}

extern "C" int ewk_published_seq(ewk_ctx* ctx, int parity, uint64_t* out, int n_slots) {
    if (!ctx) return EWK_ERR_ARG;
    int rc = need_streams(ctx, "ewk_published_seq", false);
    if (rc) return rc;
    BankView& B = ctx->bank;
    if (!B.n_pub || !B.pub_sig[0]) { ctx->fail("ewk_published_seq: no signal rows installed (ewk_set_results_peers)"); return EWK_ERR_STATE; }
    if (!out || n_slots < 1 || n_slots > MAX_PUB || parity < 0 || parity > 1) { ctx->fail("ewk_published_seq: bad arguments"); return EWK_ERR_ARG; }
    CK(cudaSetDevice(ctx->device));
    int flag = 0;
    CK(cudaMemcpyAsync(out, B.pub_sig[B.pub_slot] + (size_t)parity * MAX_PUB, sizeof(uint64_t) * (size_t)n_slots, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&flag, ctx->d_wait_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_wait_flag, 0, sizeof(int), ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return flag ? 1 : 0;
}

extern "C" int ewk_match_stream(ewk_ctx* ctx, void** out) {
    if (!ctx || !out) return EWK_ERR_ARG;
    if (ctx->bank.n_pub > 0 && ctx->pub_stream) { *out = (void*)ctx->pub_stream; return EWK_OK; }   // where the call's records are sent
    *out = (void*)(ctx->last_match_stream ? ctx->last_match_stream : ctx->stream);
    return EWK_OK;
}

extern "C" int ewk_host_alloc(void** out, int64_t bytes) {
    if (!out || bytes < 1) return EWK_ERR_ARG;
    return cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault) == cudaSuccess ? EWK_OK : EWK_ERR_NOMEM;
}

extern "C" int ewk_host_free(void* p) {
    if (!p) return EWK_ERR_ARG;
    return cudaFreeHost(p) == cudaSuccess ? EWK_OK : EWK_ERR_CUDA;
}

// ==========================================================================================
// per-kernel event timing
// ==========================================================================================
cudaEvent_t ewk_ctx::prof_begin(int, cudaStream_t on) {
    if (!prof_on) return nullptr;
    cudaEvent_t e;
    if (!prof_free.empty()) { e = prof_free.back(); prof_free.pop_back(); }
    else if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    cudaEventRecord(e, on ? on : stream);
    return e;
}

void ewk_ctx::prof_end(cudaEvent_t a, int cls, cudaStream_t on) {
    if (!a) return;
    cudaEvent_t b;
    if (!prof_free.empty()) { b = prof_free.back(); prof_free.pop_back(); }
    else if (cudaEventCreate(&b) != cudaSuccess) { prof_free.push_back(a); return; }
    cudaEventRecord(b, on ? on : stream);
    prof_pairs.push_back({a, b, cls});
}

int ewk_ctx::prof_collect() {
    ewk_ctx* ctx = this;
    int jr = join_match();
    if (jr) return jr;
    CK(cudaStreamSynchronize(stream));
    if (pub_stream) CK(cudaStreamSynchronize(pub_stream));
    for (auto& p : prof_pairs) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) { prof_ms[p.cls] += ms; prof_n[p.cls]++; }
        prof_free.push_back(p.a);
        prof_free.push_back(p.b);
    }
    prof_pairs.clear();
    return EWK_OK;
}

extern "C" int ewk_profile(ewk_ctx* ctx, int enable) {
    if (!ctx) return EWK_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    int rc = ctx->prof_collect();
    if (rc) return rc;
    for (int i = 0; i < 8; i++) { ctx->prof_ms[i] = 0; ctx->prof_n[i] = 0; }
    ctx->prof_on = enable != 0;
    return EWK_OK;
}

extern "C" int ewk_profile_read(ewk_ctx* ctx, double* ms, int64_t* launches) {
    if (!ctx || !ms || !launches) return EWK_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    int rc = ctx->prof_collect();
    if (rc) return rc;
    for (int i = 0; i < 8; i++) { ms[i] = ctx->prof_ms[i]; launches[i] = ctx->prof_n[i]; ctx->prof_ms[i] = 0; ctx->prof_n[i] = 0; }
    return EWK_OK;
}
