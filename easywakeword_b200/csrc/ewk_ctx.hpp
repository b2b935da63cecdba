// Context object behind the opaque ewk_ctx handle of include/ewk.h.
#pragma once
#include <cuda_runtime.h>

#include <map>
#include <string>
#include <vector>

#include "ewk_frame.cuh"
#include "ewk_segment.cuh"
#include "ewk_streams.cuh"
#include "ewk_dense.cuh"
#include "ewk_vad.cuh"
#include "ewk_resample.cuh"
#include "ewk_resample_push.cuh"
#include "ewk_align.cuh"
#include "ewk_tables.hpp"

namespace ewk {

// Every device allocation of a context, and every pinned host buffer it owns, comes from its Pool.  EWK_POISON=<byte>
// (read per context by ewk_create) is a test mode: each allocation is filled with the byte before anything initialises
// it and is followed by a guard band of GUARD bytes of it, per-call scratch is refilled at every ensure, and
// ewk_debug_check reports guard bands that changed.  So a read of memory nobody wrote sees the byte instead of the zeros a
// fresh cudaMalloc usually holds, and a write past a buffer's end is found.  Unset, an allocation is a plain cudaMalloc /
// cudaHostAlloc of the size asked for.  Poison mode synchronises the device around every fill and check.
struct Pool {
    static constexpr size_t GUARD = 256;
    int poison = -1;                           // the fill byte; -1: off
    struct Block { const char* name; size_t bytes; bool host; };
    std::map<void*, Block> blocks;             // poison mode: every live allocation and its requested size
    std::string damage;                        // guard damage found when a block was freed, kept for ewk_debug_check
    cudaStream_t stream = nullptr;             // poison mode: fills and guard read-backs (created by the first fill)
    cudaError_t alloc(void** p, size_t bytes, const char* name);
    cudaError_t alloc_host(void** p, size_t bytes, unsigned flags, const char* name);
    template <class T> cudaError_t alloc(T** p, size_t bytes, const char* name) { return alloc((void**)p, bytes, name); }
    template <class T> cudaError_t alloc_host(T** p, size_t bytes, unsigned flags, const char* name) {
        return alloc_host((void**)p, bytes, flags, name);
    }
    cudaError_t refill(void* p);               // poison mode: the whole block (not its guard) holds the byte again
    cudaError_t free(void* p, bool host = false);   // cudaFree / cudaFreeHost, after checking the guard in poison mode
    cudaError_t check(std::string* report);    // every live guard; damage found at free time included
    cudaError_t check_block(void* p, const Block& b, std::string* report);
    cudaError_t fill(void* p, size_t bytes, bool host);
};

// scratch: the content is dead whenever ensure is called (per-call workspaces), so poison mode refills it every time;
// otherwise (staging slots that may hold a pending push, descriptor slots, state kept across calls) only at allocation
struct DevBuf {
    Pool* pool;
    const char* name;
    bool scratch;
    void* p = nullptr;
    size_t cap = 0;
    DevBuf(Pool* pool_, const char* name_, bool scratch_) : pool(pool_), name(name_), scratch(scratch_) {}
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return scratch && pool->poison >= 0 && p ? pool->refill(p) : cudaSuccess;
        free();
        // poison mode: exactly the bytes asked for, so that a read past them lands in the guard band
        size_t want = pool->poison >= 0 ? bytes : bytes + bytes / 4 + 256;
        cudaError_t e = pool->alloc(&p, want, name);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void free() { if (p) pool->free(p); p = nullptr; cap = 0; }
};

// two slots of pinned host + device memory for descriptors (upload_slot), each reused only once its reader has run (ev)
template <class D>
struct SlotPair {
    D* h[2] = {nullptr, nullptr};
    DevBuf b[2];
    cudaEvent_t ev[2] = {nullptr, nullptr};
    bool ev_valid[2] = {false, false};
    int idx = 0;
    SlotPair(Pool* pool, const char* name) : b{{pool, name, false}, {pool, name, false}} {}
    void free() {
        for (int i = 0; i < 2; i++) {
            if (ev[i]) cudaEventDestroy(ev[i]);
            if (h[i]) b[i].pool->free(h[i], true);
            ev[i] = nullptr; h[i] = nullptr; ev_valid[i] = false;
            b[i].free();
        }
    }
};

// Launch geometry of K4 for a template set: hops per sub-chunk, threads per CTA and CTAs per SM that fit shared memory.
struct DensePlan { int DH, threads, per_sm; size_t smem; };

// A template set's descriptor for K4 / K4D (valid: built and on the device) and the launch geometry it has alone
struct DenseSetHost {
    bool valid = false;
    DensePlan plan{};
    DenseSetDev dev{};
};

}  // namespace ewk

struct ewk_ctx {
    ewk::Pool pool;              // declared first: the buffers below allocate from it
    int device = 0;
    int sm_count = 0;
    bool use_lm = true;          // keep log-mel rows of K3 frames in a global workspace (EWK_SEG_LM=0 disables)
    bool k3_frames = false;      // EWK_K3=2: queue-form K3 with frames as the unit of work (default: one CTA per segment)
    ewk_config cfg{};
    std::string err;
    cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    bool ev_free_valid[2] = {false, false};
    // optional overlap of K3 (level-2 matching) with the next push: K3 runs on match_stream after the gate (ev_gate) and the
    // context's stream joins it (ev_match) at the next call that needs level-2 results
    cudaStream_t match_stream = nullptr;
    cudaEvent_t ev_gate = nullptr, ev_match = nullptr;
    bool overlap = false, match_inflight = false;
    long long publish_seq = 0;               // ewk_tick calls since ewk_set_results_peers (peer publication); parity = (seq - 1) & 1
    int* d_wait_flag = nullptr;              // set by peer_wait_kernel when it gave up
    cudaStream_t pub_stream = nullptr;       // publish_records_kernel: the call's records -> every destination, then the signal
    cudaEvent_t ev_k3 = nullptr, ev_pub[2] = {nullptr, nullptr};
    bool ev_pub_valid[2] = {false, false};
    void* d_pub_snap = nullptr;              // StreamResult [2][n_streams]: K3's snapshots, one per parity
    cudaStream_t last_match_stream = nullptr;   // where the latest ewk_tick launched K3
    int join_match();
    int stage_idx = 0;
    // n: samples that land in the rings; rs_rate != 0 marks a native-rate push (K8) of rs_n_in inputs at that rate, from
    // input position rs_c.  rows_slot >= 0: a push of per-row descriptors `rows` (device copy in that slot) of n_items
    // work items from the raw input (format rs_fmt): K8 when rs_rate != 0, else K1L (ewk_push_streams at 16 kHz)
    struct Pending {
        bool valid = false; int slot = 0, stream0 = 0, n_streams = 0; long long n = 0;
        int rs_rate = 0, rs_fmt = 0; long long rs_n_in = 0, rs_c = 0;
        int rows_slot = -1; long long n_items = 0; std::vector<ewk::RowDesc> rows;
    } pending;
    int land(int stream0, int n_streams, const void* d_src, long long d_stride, long long n, int stage_slot);
    // rows_slot < 0: rows i < n_streams (d_stride apart) go to streams stream0 + i, all at input position c (uniform K8).
    // rows_slot >= 0: per-row descriptors rows[0 .. n_streams) (host) and their device copy in that slot, n_items tiles
    int land_resampled(int stream0, int n_streams, const void* d_src, long long d_stride, int in_fmt, long long n_in,
                       int sr_in, long long c, const ewk::RowDesc* rows, int rows_slot, long long n_items, int stage_slot);
    // K1L: the rows of a list push at 16 kHz (descriptors on the host and in slot rows_slot), from d_src in format in_fmt
    int land_list(const std::vector<ewk::RowDesc>& rows, int rows_slot, long long n_items, const void* d_src, int in_fmt,
                  int stage_slot);
    // per-row descriptors -> the next slot (copied on stream `on`); *slot receives its index
    int upload_rows(const std::vector<ewk::RowDesc>& rows, cudaStream_t on, int* slot);
    // per-row descriptors of a list push (ewk_push_streams) or of a push at different input positions
    // (ewk_push_resampled_each): two slots of pinned host + device memory for n_streams rows, each reused only once the
    // kernel that read it has finished (ev_pos)
    ewk::RowDesc* h_pos[2] = {nullptr, nullptr};
    ewk::DevBuf b_pos[2]{{&pool, "b_pos", false}, {&pool, "b_pos", false}};
    cudaEvent_t ev_pos[2] = {nullptr, nullptr};
    bool ev_pos_valid[2] = {false, false};
    int pos_idx = 0;
    ewk::DevBuf b_det_state{&pool, "b_det_state", false};                 // K4D's DetState [n_streams], allocated (zeroed) by the first detect call
    // the template sets of K4 row calls and K4D: the descriptor of set [first, first + count) sits at index
    // first * DENSE_MAX_T + count - 1 of a device table; h_dset mirrors it.  A set is built and uploaded on first use and
    // kept until a template slot of its range changes (dense_sets_forget).  New descriptors go through dset_stage.
    std::vector<ewk::DenseSetHost> h_dset;
    ewk::DevBuf b_dset{&pool, "b_dset", false};
    ewk::SlotPair<ewk::DenseSetDev> dset_stage{&pool, "dset_stage"};
    ewk::SlotPair<ewk::DenseRow> drows{&pool, "drows"};   // K4 row descriptors of a row call
    ewk::SlotPair<ewk::DetRow> ddets{&pool, "ddets"};     // K4D row descriptors
    void dense_sets_forget(int slot);
    // K4D's output, pinned and mapped into the device: per-row record counts [n_streams], then records (row i at its offset)
    void* h_det_map = nullptr;
    size_t det_map_cap = 0;
    ewk::DevBuf b_reset{&pool, "b_reset", true};                     // K9's stream list
    ewk::DevBuf b_blob{&pool, "b_blob", true};                      // K10: a host blob's device copy (export: the whole blob; import: its bulk rows)
    ewk::DevBuf b_mig{&pool, "b_mig", true};                       // K10 import: the destination list and the checked small state, one upload
    int flush_pending();
    ewk::DevBuf b_stage2[2]{{&pool, "b_stage2", false}, {&pool, "b_stage2", false}};
    ewk::DevBuf b_raw[2]{{&pool, "b_raw", false}, {&pool, "b_raw", false}};                    // compact host input: G.711 codes (ewk_push_g711, decoded into b_stage2) or a native-rate feed
    ewk::DeviceTables* d_tables = nullptr;
    ewk::TemplateFeat* d_tmpl = nullptr;
    std::vector<ewk::TemplateFeat> h_tmpl;
    // template frame store (ewk_config.template_frames = 1): slot k's K3 frames at d_tfr + k * ALIGN_MAX_FRAMES * N_MFCC;
    // h_tfr_n[k] frames (0: none: an empty slot, features only, or a template over ALIGN_MAX_SAMPLES samples)
    float* d_tfr = nullptr;
    std::vector<int> h_tfr_n;
    void store_frames(int slot, const float* d_src, long long n_samples);   // the frames of a template of n_samples
    ewk::DevBuf b_pcm{&pool, "b_pcm", true}, b_desc{&pool, "b_desc", true}, b_ws{&pool, "b_ws", true}, b_lm{&pool, "b_lm", true}, b_feat{&pool, "b_feat", true}, b_scores{&pool, "b_scores", true}, b_matched{&pool, "b_matched", true}, b_frames{&pool, "b_frames", true}, b_off{&pool, "b_off", true};

    void fail(const char* fmt, ...);
    int init();
    void release();
    // stream bank
    ewk::BankView bank{};
    void* own_results = nullptr;
    ewk::DevBuf b_trace{&pool, "b_trace", true}, b_read{&pool, "b_read", true}, b_dense{&pool, "b_dense", true}, b_keep_rows{&pool, "b_keep_rows", false}, b_keep_end{&pool, "b_keep_end", false}, b_g2{&pool, "b_g2", true};
    int dense_plan_info[4] = {0, 0, 0, 0};  // K4 geometry of the latest K4 call: hops per sub-chunk, threads, CTAs per SM, smem bytes (ewk_dense_last_plan)
    int chunk_cap = 0;
    bool all_presummed = false;            // K1's block sums cover every sample pushed since the last tick
    int pushes_since_tick = 0;
    long long launches = 0;
    std::vector<ewk::StreamParams> h_prm;
    double max_post = 0.4;                 // largest post_speech_silence of any stream (overlap-mode ring reserve)
    std::vector<long long> h_written;      // host mirror of StreamState.written
    std::vector<long long> h_visible_lb;   // lower bound of StreamState.visible (audio-clock overrun check)
    std::vector<long long> h_tick;
    std::vector<long long> h_dense_next;   // ewk_dense_ready's cursor: the next hop it scores (1 after create / reset)
    std::vector<long long> h_det_next;     // ewk_dense_detect's own cursor, independent of ewk_dense_ready's
    std::vector<int> h_frame_size;         // latched frame size per stream (0: no push yet)
    std::vector<int> h_rate;               // input rate latched by the stream's first push (0: none yet; 16000: ewk_push)
    std::vector<long long> h_inputs;       // input samples the stream received (at its own rate)
    float* d_rs_tail = nullptr;            // K8 input tails [n_streams][rs_tail_cap], sized by the rates in use
    int rs_tail_cap = 0;
    int ensure_rs_tail(int cap);           // grows the tails to cap floats per stream
    int gate_chunks() const;               // largest R / frame_size in use
    // per-kernel event timing (ewk_profile)
    bool prof_on = false;
    struct ProfPair { cudaEvent_t a, b; int cls; };
    std::vector<ProfPair> prof_pairs;
    std::vector<cudaEvent_t> prof_free;
    double prof_ms[8] = {0};
    long long prof_n[8] = {0};
    cudaEvent_t prof_begin(int cls, cudaStream_t on = nullptr);
    void prof_end(cudaEvent_t a, int cls, cudaStream_t on = nullptr);
    int prof_collect();
    int init_streams();
    void release_streams();
    int launch_segments(const ewk::SegDesc* d_segs, int n_seg, int max_frames, long long spill_frames,
                        long long lm_frames, int n_tmpl, int tmpl_first, float threshold, float* d_feat, float* d_frames,
                        float* d_scores, unsigned char* d_matched);
    int queue_grid() const { return sm_count > 0 ? 2 * sm_count : 1; }     // persistent K3 CTAs (2 per SM)
    static constexpr size_t LM_WS_MAX_BYTES = (size_t)4 << 30;
    // K7 filter tables, one per input rate seen
    struct ResampleTable { ewk::ResampleDesign d; float* H = nullptr; };
    std::map<int, ResampleTable> rs_tables;
    ewk::DevBuf b_rs_in{&pool, "b_rs_in", true}, b_rs_out{&pool, "b_rs_out", true};
    int resample_table(int sr_in, const ResampleTable** out);
    // A.rows set: the grid is the descriptors' n_items flat output tiles (fir_tiles per row)
    int launch_fir(const ResampleTable& t, ewk::RsPushArgs& A, int n_rows, int prof_cls, const char* who,
                   long long n_items = 0);
};
