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
#include "ewk_tables.hpp"

#define EWK_MAX_TEMPLATES 64

namespace ewk {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void free() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

}  // namespace ewk

struct ewk_ctx {
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
    ewk::DevBuf b_pos[2];
    cudaEvent_t ev_pos[2] = {nullptr, nullptr};
    bool ev_pos_valid[2] = {false, false};
    int pos_idx = 0;
    // per-row descriptors of a ragged K4 call (ewk_dense_scores_streams, ewk_dense_ready): two slots of the same kind
    ewk::DenseRow* h_drow[2] = {nullptr, nullptr};
    ewk::DevBuf b_drow[2];
    cudaEvent_t ev_drow[2] = {nullptr, nullptr};
    bool ev_drow_valid[2] = {false, false};
    int drow_idx = 0;
    // per-row descriptors of K4D (ewk_dense_detect): two slots of the same kind
    ewk::DetRow* h_ddet[2] = {nullptr, nullptr};
    ewk::DevBuf b_ddet[2];
    cudaEvent_t ev_ddet[2] = {nullptr, nullptr};
    bool ev_ddet_valid[2] = {false, false};
    int ddet_idx = 0;
    ewk::DevBuf b_det_state;                 // K4D's DetState [n_streams], allocated (zeroed) by the first detect call
    // K4D's output, pinned and mapped into the device: per-row record counts [n_streams], then records (row i at its offset)
    void* h_det_map = nullptr;
    size_t det_map_cap = 0;
    ewk::DevBuf b_reset;                     // K9's stream list
    ewk::DevBuf b_blob;                      // K10: a host blob's device copy (export: the whole blob; import: its bulk rows)
    ewk::DevBuf b_mig;                       // K10 import: the destination list and the checked small state, one upload
    int flush_pending();
    ewk::DevBuf b_stage2[2];
    ewk::DevBuf b_raw[2];                    // compact host input: G.711 codes (ewk_push_g711, decoded into b_stage2) or a native-rate feed
    ewk::DeviceTables* d_tables = nullptr;
    ewk::TemplateFeat* d_tmpl = nullptr;
    std::vector<ewk::TemplateFeat> h_tmpl;
    ewk::DevBuf b_pcm, b_desc, b_ws, b_lm, b_feat, b_scores, b_matched, b_frames, b_off;

    void fail(const char* fmt, ...);
    int init();
    void release();
    // stream bank
    ewk::BankView bank{};
    void* own_results = nullptr;
    ewk::DevBuf b_trace, b_read, b_dense, b_keep_rows, b_keep_end, b_g2;
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
    ewk::DevBuf b_rs_in, b_rs_out;
    int resample_table(int sr_in, const ResampleTable** out);
    // A.rows set: the grid is the descriptors' n_items flat output tiles (fir_tiles per row)
    int launch_fir(const ResampleTable& t, ewk::RsPushArgs& A, int n_rows, int prof_cls, const char* who,
                   long long n_items = 0);
};
