// K1 ring_push and K2 tick_gate: the level-1 data plane of the reference, batched over streams.
//
//   K1  SoundBuffer._add_sound_to_buffer   (/root/reference/easywakeword/wakeword.py:454-465)
//   K2  SoundBuffer._adjust_silence_threshold + is_silent (wakeword.py:472-496) and the 4-state
//       timing machine + segment cut of WakeWord._detect_word (wakeword.py:1036-1118, 1155-1157)
//
// Device layout (all SoA over streams): a PHYSICAL ring of P = ring + slack samples per stream
// (int16 or f32) holding absolute sample a at a % P.  The reference's logical ring of R samples is
// the most recent R samples visible at a tick; keeping `slack` older samples lets one push run
// ahead of the ticks that consume it while every intermediate tick still sees exactly the ring
// content the reference would have had (chunk RMS values are recomputed from samples, never
// updated incrementally, so there is no drift).
//
// Time is the audio clock: tick k has time k*0.1 (float64, computed with the same IEEE operations
// as the oracle, no FMA contraction) and sees V_k = floor(1600 k / frame_size) * frame_size samples.
#pragma once
#include "ewk_frame.cuh"
#include "ewk_segment.cuh"

#ifndef EWK_MAX_TEMPLATES
#define EWK_MAX_TEMPLATES 64
#endif

namespace ewk {

constexpr int GATE_THREADS = 128;
constexpr int TICK = 1600;              // int(0.1 * 16000)            wakeword.py:492, 500
constexpr int MAX_SEG = 48000;          // 3.0 s cap                   wakeword.py:1114-1118

enum : int { ST_WAITING = 0, ST_IN_SILENCE = 1, ST_IN_SOUND = 2, ST_AFTER_SOUND = 3 };
enum : int { EV_PENDING = 0, EV_TIMEOUT = 1, EV_SCORED = 2 };

struct StreamParams {               // mirrors ewk_stream_params (include/ewk.h)
    float similarity_threshold;
    int frame_size;
    double pre_speech_silence, speech_duration_min, speech_duration_max, post_speech_silence;
    double timeout;
    double min_threshold;
    int template_first, template_count;
    int live;
    int reserved;
};

struct StreamState {
    long long written;      // samples pushed so far (absolute index of the next sample)
    long long visible;      // V of the last processed tick
    long long tick;         // k of the last processed tick
    double thr;             // SoundBuffer.silence_threshold (init 0.01, wakeword.py:431)
    double silence_start, sound_start, sound_end, start_time;
    double last_rms;
    int frame_size;         // 0 until the first push (wakeword.py:457-458)
    int state;
    int started;            // _detect_word entered (buffer was full at some tick)
    int last_silent;
    int chunks_valid;       // chunk mean-squares reflect the ring at `visible`
    int n_timeouts;
    int n_events;
    int last_ev;            // queue index of the stream's newest level-2 candidate in the current queue epoch (-1: none):
                            // K3 lets only that event write the per-stream result record, so the record always carries the
                            // LATEST evaluation however the CTAs that score a stream's events are ordered
    long long ss_from;      // block_ss holds the sum of squares of every aligned 1600-sample block in [ss_from, written)
};

struct EventRec {           // mirrors ewk_event
    int stream;
    int kind;
    long long tick;
    long long seg_start;    // absolute sample index of the segment's first sample
    int seg_len;
    int tmpl;
    float score;
    int matched;
};

struct StreamResult {       // dense per-stream record (what multi-GPU runs gather)
    float score;            // score of the stream's latest level-2 evaluation (NaN before the first)
    unsigned flags;         // bit0 matched(latest) | bit1 silent | bits2-3 state | bit4 event this call | bits 8.. event count
};

constexpr int MAX_PUB = 16;  // destinations of a peer publication (GPUs of one NVLink domain)
constexpr int SEG_NB = 24;   // length classes of queued candidates: ceil(frames / SEG_WARPS) <= ceil(301 / 14) = 22
constexpr int FROW = 24;     // floats per frame row of the frame-parallel K3: mfcc[20], log-mel min, log-mel max, pad (96 B)

struct BankView {
    void* ring;             // [n_streams][P]
    StreamState* st;
    StreamParams* prm;
    double* chunk_ms;       // [n_streams][chunk_cap] mean square per storage-order chunk
    EventRec* events;
    int* ev_count;          // [0] count, [1] dropped, [2] K3 work counter, [3] events below this index are scored, [4] K3 CTAs done,
                            // [5] frames below this index are done, [6] frames allocated to queued candidates (frame-parallel K3)
    int* frame_ev;          // [frow_cap] event index of every allocated frame (-1: a hole left by a dropped candidate)
    int* ev_done;           // [max_events] frames of the event computed so far: whoever completes the last one scores the event
    float* frow;            // [frow_cap][FROW] un-floored MFCC rows (+ log-mel min / max) of the queued candidates' frames
    int frow_cap;
    StreamResult* results;
    double* block_ss;       // [n_streams][NB]: sum of squares of absolute block b = a / 1600 at b % NB (written by K1)
    float* lm_ws;           // K3 log-mel workspace: [segment_queue CTAs][SEG_SMEM_FRAMES][LM_ROW]
    int* bk_count;          // [SEG_NB] candidates queued since the last K3 launch, by length class (rounds of SEG_WARPS frames)
    int* bk_list;           // [SEG_NB][max_events] their event indices: K3 takes the longest class first
    long long* k3_trace;    // measuring builds (-DEWK_K3_TRACE) with EWK_K3_TRACE=<file> set: per-CTA timeline of the last K3 launch
    int n_streams, R, P, fmt, chunk_cap, max_events, NB;
    // peer publication (ewk_set_results_peers): K2 and K3 store every record they write into `results` also into the
    // call's local copy pub_snap[pub_parity] (K2 writes every stream's record in every call, so the copy is complete when
    // K3 ends); behind K3, on a side stream, a small kernel sends that copy to pub[p] + pub_parity * pub_stride + pub_off
    // for each destination p — local or NVLink peer-mapped memory — and releases the call's sequence number into every
    // destination's signal row: a put-with-signal that is on nobody's critical path (the next push and the next gate
    // depend on nothing of it; the call after next, which reuses the copy, finds the sender long done).
    StreamResult* pub[MAX_PUB];
    int n_pub, pub_parity;
    long long pub_stride, pub_off;
    unsigned long long* pub_sig[MAX_PUB];   // per destination: uint64 [2][MAX_PUB] signal rows (optional)
    unsigned long long pub_seq;
    int pub_slot;
    int pad_pub;
    StreamResult* pub_snap;                 // [2][n_streams] local snapshots, one per parity
};

// Peer publication, the sending side: CTA p copies the call's snapshot of this rank's records into destination p with
// plain (weak) 8-byte stores — remote destinations travel over NVLink as posted writes that pipeline behind each other —
// then every thread orders its stores at system scope and thread 0 releases the call's sequence number into slot
// `pub_slot` of the destination's signal row: whoever reads that number (ld.acquire.sys) holds all records of the call.
__global__ void __launch_bounds__(256)
publish_records_kernel(BankView B) {
    const int p = blockIdx.x;
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(B.pub_snap + (size_t)B.pub_parity * B.n_streams);
    unsigned long long* dst = reinterpret_cast<unsigned long long*>(B.pub[p] + (size_t)B.pub_parity * (size_t)B.pub_stride + (size_t)B.pub_off);
    for (int i0 = threadIdx.x; i0 < B.n_streams; i0 += 8 * blockDim.x) {
        unsigned long long v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { const int i = i0 + u * blockDim.x; v[u] = i < B.n_streams ? __ldcg(src + i) : 0ull; }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int i = i0 + u * blockDim.x;
            if (i < B.n_streams) asm volatile("st.weak.global.b64 [%0], %1;" :: "l"(dst + i), "l"(v[u]) : "memory");
        }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0 && B.pub_sig[p]) {
        unsigned long long* sg = B.pub_sig[p] + (size_t)B.pub_parity * MAX_PUB + B.pub_slot;
        asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(sg), "l"(B.pub_seq) : "memory");
    }
}

// the record as ONE 8-byte store (readers — peers, an all-gather, the host — never see half of it)
__device__ __forceinline__ void store_result(StreamResult* dst, StreamResult r) {
    const unsigned long long bits = ((unsigned long long)r.flags << 32) | (unsigned long long)__float_as_uint(r.score);
    *reinterpret_cast<unsigned long long*>(dst) = bits;
}

struct TraceView {          // optional per-tick trace for parity tests: [n_streams][n_ticks]
    unsigned char* silent;
    unsigned char* state;
    double* thr;
    double* rms;
};

// ------------------------------------------------------------------------------------ K0 (G.711 ingest)
// the 16-bit linear value of G.711 code c (mu-law, or A-law when alaw), from the standard's bit layout
__device__ __forceinline__ short g711_linear(int c, int alaw) {
    int v;
    if (alaw) {
        const int a = c ^ 0x55, e = (a >> 4) & 7, m = a & 0x0F;
        v = e == 0 ? (m << 4) + 8 : ((m << 4) + 0x108) << (e - 1);
        v = (a & 0x80) ? v : -v;
    } else {
        const int u = ~c & 0xFF;
        v = ((((u & 0x0F) << 3) + 0x84) << ((u >> 4) & 7)) - 0x84;
        v = (u & 0x80) ? -v : v;
    }
    return (short)v;
}

// 8-bit mu-law / A-law codes -> the 16-bit linear samples of ITU-T G.711 (what libsndfile hands librosa.load for such
// files, and what a telephony feed carries): in[r * stride + i] -> out[r * n + i], i < n.  The 256-entry expansion table is
// formed in shared memory; 16 codes per thread per step (one 16-byte load, two stores).
// HBM-bound: 1 byte read + 2 bytes written per sample.  It runs on the copy stream right behind the H2D copy of the
// codes, so a host feed crosses PCIe at half the bytes of PCM16.
__global__ void __launch_bounds__(256)
g711_decode_kernel(const unsigned char* __restrict__ in, short* __restrict__ out, int n_rows, long long n, long long stride, int alaw) {
    __shared__ short lut[256];
    lut[threadIdx.x] = g711_linear(threadIdx.x, alaw);
    __syncthreads();
    const bool vec = (n % 16) == 0 && (stride % 16) == 0 && ((size_t)in & 15) == 0 && ((size_t)out & 15) == 0;
    const long long per_row = vec ? n / 16 : n;
    const long long total = per_row * n_rows;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long r = i / per_row, j = i - r * per_row;
        if (vec) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(in + r * stride) + j);
            const unsigned w[4] = {q.x, q.y, q.z, q.w};
            unsigned o[8];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                o[2 * k] = (unsigned)(unsigned short)lut[w[k] & 0xFF] | ((unsigned)(unsigned short)lut[(w[k] >> 8) & 0xFF] << 16);
                o[2 * k + 1] = (unsigned)(unsigned short)lut[(w[k] >> 16) & 0xFF] | ((unsigned)(unsigned short)lut[w[k] >> 24] << 16);
            }
            uint4* d = reinterpret_cast<uint4*>(out + r * n) + 2 * j;
            d[0] = make_uint4(o[0], o[1], o[2], o[3]);
            d[1] = make_uint4(o[4], o[5], o[6], o[7]);
        } else {
            out[r * n + j] = lut[in[r * stride + j]];
        }
    }
}

// ------------------------------------------------------------------------------------ K1
// src[s * stride + i] (i < n) -> ring of stream stream0 + s at absolute index written + i.
// 16-byte vector path when source and destination runs are 16-byte aligned, scalar otherwise.
template <typename T>
__global__ void ring_push_kernel(BankView B, int stream0, const T* __restrict__ src, long long stride, int n) {
    const int s = blockIdx.y;
    constexpr int V = 16 / sizeof(T);
    T* ring = (T*)B.ring + (size_t)(stream0 + s) * B.P;
    const T* in = src + (size_t)s * stride;
    const long long w = B.st[stream0 + s].written;
    const int p0 = (int)(w % B.P);
    const bool vec = (p0 % V == 0) && (n % V == 0) && (B.P % V == 0) && ((((size_t)in) & 15) == 0);
    if (vec) {
        const int nv = n / V;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += gridDim.x * blockDim.x) {
            int p = p0 + i * V;
            if (p >= B.P) p -= B.P;
            *reinterpret_cast<int4*>(ring + p) = __ldg(reinterpret_cast<const int4*>(in) + i);
        }
    } else {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            int p = p0 + i;
            if (p >= B.P) p -= B.P;
            ring[p] = in[i];
        }
    }
}

// K1, fused form: the copy of a device-resident push also produces the sum of squares of every 0.1 s block
// it writes (what K2 needs for the adaptive threshold and is_silent), so the samples are read once for both.
// One warp per (stream, 1600-sample block).  Preconditions (checked per stream, identical in the commit
// kernel): the stream's `written` and `n` are multiples of 1600, 16-byte aligned source rows.
__device__ __forceinline__ long long sq8(const int4 q);
__device__ __forceinline__ double sq4(const float4 q, double acc);

template <typename T>
__global__ void __launch_bounds__(128)
ring_push_sums_kernel(BankView B, int stream0, const T* __restrict__ src, long long stride, int n) {
    constexpr int V = 16 / sizeof(T);                 // samples per 16-byte word
    constexpr int NV = TICK / V;                      // words per block: 200 (int16) / 400 (f32)
    constexpr int PER = (NV + 31) / 32;
    const int lane = threadIdx.x & 31;
    const int blk = blockIdx.x * 4 + (threadIdx.x >> 5);
    const int s = stream0 + blockIdx.y;
    if (blk * TICK >= n) return;
    const long long w = B.st[s].written;
    const T* in = src + (size_t)blockIdx.y * stride + (size_t)blk * TICK;
    T* ring = (T*)B.ring + (size_t)s * B.P;
    const long long a0 = w + (long long)blk * TICK;
    const int p0 = (int)(a0 % B.P);
    const int4* vin = reinterpret_cast<const int4*>(in);
    int4 q[PER];
#pragma unroll
    for (int u = 0; u < PER; u++) {
        const int k = lane + 32 * u;
        q[u] = k < NV ? __ldg(vin + k) : make_int4(0, 0, 0, 0);
    }
    if (p0 + TICK <= B.P) {
        int4* vout = reinterpret_cast<int4*>(ring + p0);
#pragma unroll
        for (int u = 0; u < PER; u++) { const int k = lane + 32 * u; if (k < NV) vout[k] = q[u]; }
    } else {
#pragma unroll
        for (int u = 0; u < PER; u++) {
            const int k = lane + 32 * u;
            if (k < NV) { int p = p0 + k * V; if (p >= B.P) p -= B.P; *reinterpret_cast<int4*>(ring + p) = q[u]; }
        }
    }
    double acc;
    if (sizeof(T) == 2) {
        long long iacc = 0;
#pragma unroll
        for (int u = 0; u < PER; u++) iacc += sq8(q[u]);
        acc = (double)iacc;
    } else {
        double a0d = 0.0, a1d = 0.0;
#pragma unroll
        for (int u = 0; u < PER; u++) {
            const float4 f = make_float4(__int_as_float(q[u].x), __int_as_float(q[u].y), __int_as_float(q[u].z), __int_as_float(q[u].w));
            if (u & 1) a1d = sq4(f, a1d); else a0d = sq4(f, a0d);
        }
        acc = a0d + a1d;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    if (lane == 0) B.block_ss[(size_t)s * B.NB + (size_t)((a0 / TICK) % B.NB)] = acc;
}

// bookkeeping after the payload of a push landed (kernel or 2-D copy): written += n, frame_size latch,
// validity range of the per-block sums (with_sums: the fused kernel produced them for this push)
__global__ void ring_commit_kernel(BankView B, int stream0, int n_streams, int n, int with_sums) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_streams) return;
    StreamState& st = B.st[stream0 + s];
    if (st.frame_size == 0) {
        const int fs = B.prm[stream0 + s].frame_size;
        st.frame_size = fs > 0 ? fs : n;                               // wakeword.py:457-458
    }
    if (!with_sums) st.ss_from = st.written + n;                        // nothing known about these samples
    else if (st.ss_from > st.written) st.ss_from = st.written;          // sums restart at this push
    st.written += n;
}

// ------------------------------------------------------------------------------------ K1L (list push)
// One row of a list push (ewk_push_streams; K8's per-row instance reads the same descriptors).  The rows' work is one flat
// list of items — K1L: LIST_CHUNK-sample chunks, K8: output tiles — and row y owns items [item0, next row's item0).
struct RowDesc {
    long long off;          // first input sample of the row in the call's buffer
    long long len;          // input samples of the row (> 0)
    long long pos;          // K1L: samples the stream had landed (its `written`); K8: input samples it had received
    int stream;
    int item0;
    int latch;              // frame size latched by a stream's first push when frame_size is 0
    int pad;
};

// the row that owns flat item `item` (rows' item0 ascend, every row owns at least one item)
__device__ __forceinline__ int row_of_item(const RowDesc* __restrict__ rows, int n_rows, int item) {
    int lo = 0, hi = n_rows - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(&rows[mid].item0) <= item) lo = mid; else hi = mid - 1;
    }
    return lo;
}

constexpr int LIST_THREADS = 256, LIST_PER = 16;
constexpr int LIST_CHUNK = LIST_THREADS * LIST_PER;     // samples per K1L item

// K1L: row y's samples in[off, off + len) -> ring of stream `stream` at absolute index pos + i, with wrap.  in_fmt: the
// ring's format (0 f32, 1 int16), or G.711 codes (2 mu-law, 3 A-law) expanded through a shared-memory table into int16
// rings, as K0 does.  The row's first item commits it: written = pos + len, the frame-size latch, and ss_from past the
// new samples (no block sums: K2 reads them).  Nothing in the launch reads `written`, so the commit needs no barrier.
// Rows start at any sample, so accesses are per sample; each thread issues its LIST_PER loads before its stores, which
// keeps enough bytes in flight to stream at HBM rate.
template <typename T>
__global__ void __launch_bounds__(LIST_THREADS)
ring_push_list_kernel(BankView B, const void* __restrict__ in, int in_fmt, const RowDesc* __restrict__ rows, int n_rows) {
    __shared__ short lut[256];
    if (in_fmt >= 2) lut[threadIdx.x] = g711_linear(threadIdx.x, in_fmt == 3);
    __syncthreads();
    const int y = row_of_item(rows, n_rows, blockIdx.x);
    const RowDesc d = rows[y];
    const long long i0 = (long long)(blockIdx.x - d.item0) * LIST_CHUNK;
    const int n = (int)min((long long)LIST_CHUNK, d.len - i0);
    T* ring = (T*)B.ring + (size_t)d.stream * B.P;
    const int p0 = (int)((d.pos + i0) % B.P);
    T v[LIST_PER];
#pragma unroll
    for (int u = 0; u < LIST_PER; u++) {
        const int i = threadIdx.x + u * LIST_THREADS;
        if (i < n) {
            if (in_fmt >= 2) v[u] = (T)lut[__ldg((const unsigned char*)in + d.off + i0 + i)];
            else v[u] = __ldg((const T*)in + d.off + i0 + i);
        }
    }
#pragma unroll
    for (int u = 0; u < LIST_PER; u++) {
        const int i = threadIdx.x + u * LIST_THREADS;
        int p = p0 + i;
        if (p >= B.P) p -= B.P;
        if (i < n) ring[p] = v[u];
    }
    if (i0 == 0 && threadIdx.x == 0) {
        StreamState& st = B.st[d.stream];
        if (st.frame_size == 0) {
            const int fs = B.prm[d.stream].frame_size;
            st.frame_size = fs > 0 ? fs : d.latch;
        }
        st.written = d.pos + d.len;
        st.ss_from = d.pos + d.len;
    }
}

// ------------------------------------------------------------------------------------ K2 helpers
constexpr int GATE_WARPS = GATE_THREADS / 32;
constexpr int GATE_MAX_TICKS = 16;     // ticks per launch (the host splits longer requests)
constexpr int GATE_MAXP = 12;          // chunk pieces planned per tick; more -> the tick is "heavy"

// sum of the squares of the eight int16 samples of a 16-byte word, exact (64-bit integer): per 32-bit
// word one sign-extracting BFE, one arithmetic shift and two signed 32x32+64 multiply-adds.
__device__ __forceinline__ long long sq8(const int4 q) {
    long long acc = 0;
    asm("{\n\t.reg .s32 lo, hi;\n\t"
        "bfe.s32 lo, %1, 0, 16;\n\tshr.s32 hi, %1, 16;\n\tmad.wide.s32 %0, lo, lo, %0;\n\tmad.wide.s32 %0, hi, hi, %0;\n\t"
        "bfe.s32 lo, %2, 0, 16;\n\tshr.s32 hi, %2, 16;\n\tmad.wide.s32 %0, lo, lo, %0;\n\tmad.wide.s32 %0, hi, hi, %0;\n\t"
        "bfe.s32 lo, %3, 0, 16;\n\tshr.s32 hi, %3, 16;\n\tmad.wide.s32 %0, lo, lo, %0;\n\tmad.wide.s32 %0, hi, hi, %0;\n\t"
        "bfe.s32 lo, %4, 0, 16;\n\tshr.s32 hi, %4, 16;\n\tmad.wide.s32 %0, lo, lo, %0;\n\tmad.wide.s32 %0, hi, hi, %0;\n\t}"
        : "+l"(acc) : "r"(q.x), "r"(q.y), "r"(q.z), "r"(q.w));
    return acc;
}

__device__ __forceinline__ double sq4(const float4 q, double acc) {
    acc = fma((double)q.x, (double)q.x, acc); acc = fma((double)q.y, (double)q.y, acc);
    acc = fma((double)q.z, (double)q.z, acc); acc = fma((double)q.w, (double)q.w, acc);
    return acc;
}

// Sum of squares of absolute samples [a0, a0+len) of one stream, in double; whole warp cooperates,
// result in every lane.  int16 sums are exact integers (the caller scales by 2^-30).  The aligned
// body keeps up to eight independent 16-byte loads per lane in flight (a 0.1 s tick of int16 PCM is
// 200 such loads per warp), which is what lets a single resident wave of warps saturate HBM.
__device__ __noinline__ double warp_sumsq(const void* ring_s, int P, int fmt, long long a0, int len, int lane) {
    double acc = 0.0;
    if (len <= 0) return 0.0;
    const int p0 = (int)(a0 % P);
    if (fmt == 1) {
        const short* ring = (const short*)ring_s;
        int i = 0;
        long long iacc = 0;
        if ((p0 & 7) == 0 && p0 + len <= P) {
            const int nv = len >> 3;
            const int4* v = reinterpret_cast<const int4*>(ring + p0);
            for (int k0 = 0; k0 < nv; k0 += 256) {
                int4 q[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int k = k0 + lane + 32 * u;
                    q[u] = k < nv ? __ldg(v + k) : make_int4(0, 0, 0, 0);
                }
#pragma unroll
                for (int u = 0; u < 8; u++) iacc += sq8(q[u]);
            }
            i = nv << 3;
        }
        for (int k = i + lane; k < len; k += 32) {
            int p = p0 + k;
            if (p >= P) p -= P;
            const int q = ring[p];
            iacc += (long long)(q * q);
        }
        acc = (double)iacc;
    } else {
        const float* ring = (const float*)ring_s;
        int i = 0;
        if ((p0 & 3) == 0 && p0 + len <= P) {
            const int nv = len >> 2;
            const float4* v = reinterpret_cast<const float4*>(ring + p0);
            double a1 = 0.0;
            for (int k0 = 0; k0 < nv; k0 += 256) {
                float4 q[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int k = k0 + lane + 32 * u;
                    q[u] = k < nv ? __ldg(v + k) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 8; u += 2) { acc = sq4(q[u], acc); a1 = sq4(q[u + 1], a1); }
            }
            acc += a1;
            i = nv << 2;
        }
        for (int k = i + lane; k < len; k += 32) {
            int p = p0 + k;
            if (p >= P) p -= P;
            const double x = (double)ring[p];
            acc = fma(x, x, acc);
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    return acc;
}

// mean square of storage-order chunk c as the reference's ring holds it when V samples are visible:
// logical position p < V % R was written in the current lap, p >= V % R in the previous one.
__device__ __forceinline__ double warp_chunk_ms(const BankView& B, int s, long long V, int fs, int c, int lane) {
    const void* ring_s = (const char*)B.ring + (size_t)s * B.P * (B.fmt == 1 ? 2 : 4);
    const long long lap = V / B.R;
    const int q = (int)(V % B.R);
    const int lo = c * fs, hi = lo + fs;
    const int split = min(max(q, lo), hi);            // [lo, split) current lap, [split, hi) previous lap
    double ss = 0.0;
    if (split > lo) ss += warp_sumsq(ring_s, B.P, B.fmt, lap * B.R + lo, split - lo, lane);
    if (hi > split) ss += warp_sumsq(ring_s, B.P, B.fmt, (lap - 1) * B.R + split, hi - split, lane);
    if (B.fmt == 1) ss *= (1.0 / 1073741824.0);       // (q/32768)^2, exact power of two
    return ss / (double)fs;                           // np.mean(frame**2)            wakeword.py:481
}

// sorted[] <- ascending order of ms[0..n) (rank by counting; ties broken by index).  One warp.
__device__ __forceinline__ void warp_sort_build(const double* ms, double* sorted, int n, int lane) {
    for (int i = lane; i < n; i += 32) {
        const long long vi = __double_as_longlong(ms[i]);
        int r = 0;
        for (int j = 0; j < n; j++) {
            const long long vj = __double_as_longlong(ms[j]);
            r += (vj < vi) || (vj == vi && j < i);
        }
        sorted[r] = ms[i];
    }
    __syncwarp();
}

// Replace one occurrence of `oldv` by `newv` in the ascending array S[0..n) (one warp; T is a second
// buffer; returns with the result in S).  Non-negative doubles order like their bit patterns.
__device__ __forceinline__ void warp_sorted_replace(double*& S, double*& T, int n, double oldv, double newv, int lane) {
    const long long bo = __double_as_longlong(oldv), bn = __double_as_longlong(newv);
    if (bo == bn) return;
    if (n <= 128) {
        // in place: the lane keeps its (up to four) elements from the counting pass in registers; the elements between
        // the old and the new position move by one slot — every lane stores its own element into the neighbouring slot —
        // and one lane drops the new value into the gap.  No second pass of loads, no second buffer.
        long long v[4];
        int lo = 0, ln = 0;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int i = 32 * r + lane;
            v[r] = i < n ? __double_as_longlong(S[i]) : 0x7fffffffffffffffLL;
            lo += __popc(__ballot_sync(FULL, v[r] < bo));
            ln += __popc(__ballot_sync(FULL, v[r] < bn));
        }
        const int pos_old = lo;
        const int pos_new = ln - (bo < bn ? 1 : 0);    // index in the array with `oldv` removed
        __syncwarp();
        if (pos_new > pos_old) {                       // (pos_old, pos_new] move down
#pragma unroll
            for (int r = 0; r < 4; r++) {
                const int i = 32 * r + lane;
                if (i > pos_old && i <= pos_new) S[i - 1] = __longlong_as_double(v[r]);
            }
        } else if (pos_new < pos_old) {                // [pos_new, pos_old) move up
#pragma unroll
            for (int r = 0; r < 4; r++) {
                const int i = 32 * r + lane;
                if (i >= pos_new && i < pos_old) S[i + 1] = __longlong_as_double(v[r]);
            }
        }
        __syncwarp();
        if (lane == 0) S[pos_new] = newv;
        __syncwarp();
        return;
    }
    int lo = 0, ln = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        const long long v = i < n ? __double_as_longlong(S[i]) : 0x7fffffffffffffffLL;
        lo += __popc(__ballot_sync(FULL, v < bo));
        ln += __popc(__ballot_sync(FULL, v < bn));
    }
    const int pos_old = lo;
    const int pos_new = ln - (bo < bn ? 1 : 0);        // index in the array with `oldv` removed
    for (int i = lane; i < n; i += 32) {
        double v;
        if (i == pos_new) v = newv;
        else {
            const int r = i > pos_new ? i - 1 : i;     // position in the "removed" array
            v = S[r >= pos_old ? r + 1 : r];
        }
        T[i] = v;
    }
    __syncwarp();
    double* t = S; S = T; T = t;
}

// np.percentile(rms, 25), numpy's default 'linear' method and its _lerp, from the ascending
// mean-square array (sqrt is monotone: order statistics of the RMS are sqrt of those of the ms).
__device__ __forceinline__ double percentile25_rms_sorted(const double* S, int n) {
    const double vi = (double)n * 0.25 - 0.25;        // n*q + (alpha + q*(1-alpha-beta)) - 1, alpha=beta=1
    const int k_lo = (int)floor(vi);
    const int k_hi = min(k_lo + 1, n - 1);
    const double a = sqrt(S[k_lo]), b = sqrt(S[k_hi]);
    const double t = vi - (double)k_lo;
    const double diff = __dsub_rn(b, a);
    double r = __dadd_rn(a, __dmul_rn(diff, t));
    if (t >= 0.5) r = __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, t)));
    return r;
}

// ---- TMA-style bulk staging (cp.async.bulk + mbarrier): one lane moves a whole 0.1 s tick of PCM from the
// ring into shared memory with a single instruction; the warp overlaps the copy of tick j+2 with the
// arithmetic of tick j.
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.release.cta.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    }
}

// sum of squares of one staged tick (TICK samples in shared memory), whole warp, result in every lane
__device__ __forceinline__ double warp_sumsq_smem(const void* buf, int fmt, int lane) {
    double acc;
    if (fmt == 1) {
        const int4* v = reinterpret_cast<const int4*>(buf);
        long long iacc = 0;
#pragma unroll
        for (int u = 0; u < 7; u++) {
            const int k = lane + 32 * u;
            if (k < TICK / 8) iacc += sq8(v[k]);
        }
        acc = (double)iacc;
    } else {
        const float4* v = reinterpret_cast<const float4*>(buf);
        double a0 = 0.0, a1 = 0.0;
#pragma unroll
        for (int u = 0; u < 13; u++) {
            const int k = lane + 32 * u;
            if (k < TICK / 4) { if (u & 1) a1 = sq4(v[k], a1); else a0 = sq4(v[k], a0); }
        }
        acc = a0 + a1;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(FULL, acc, o);
    return acc;
}

// ------------------------------------------------------------------------------------ K1 (bulk form)
// The same push + per-block sums as ring_push_sums_kernel, moved by the TMA engine: a persistent kernel of small
// CTAs whose warps each run a ring of `stages` shared-memory slots — cp.async.bulk global -> shared (mbarrier
// completion), sum of squares of the staged 0.1 s block, cp.async.bulk shared -> ring (bulk group).  Bandwidth comes
// from bytes in flight (stages x 3.2 KB per warp), not from resident threads, so the kernel needs ~2 k registers and
// no issue slots to speak of: it can run beside K3 on the same SMs (ewk_set_overlap) as well as alone.
// Requires what the fused kernel requires (whole blocks, 16-byte aligned rows) plus rings that are a whole number
// of blocks, so a block never wraps.
constexpr int PUSH_BULK_WARPS = 2;

__device__ __forceinline__ void bulk_s2g(void* dst, const void* src_smem, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}

template <typename T>
__global__ void __launch_bounds__(PUSH_BULK_WARPS * 32)
ring_push_bulk_kernel(BankView B, int stream0, int n_streams, const T* __restrict__ src, long long stride, int n, int stages) {
    extern __shared__ __align__(128) unsigned char push_smem[];
    constexpr unsigned BYTES = TICK * sizeof(T);
    const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
    unsigned char* buf = push_smem + (size_t)wl * stages * BYTES;
    unsigned long long* full = reinterpret_cast<unsigned long long*>(push_smem + (size_t)PUSH_BULK_WARPS * stages * BYTES) + wl * stages;
    const int nb = n / TICK;
    // a warp takes whole streams (gw, gw + GW, ...) and walks their nb blocks in order: its k-th item is block k % nb
    // of its (k / nb)-th stream
    const int gw = blockIdx.x * PUSH_BULK_WARPS + wl, GW = gridDim.x * PUSH_BULK_WARPS;
    const int my_streams = gw < n_streams ? (n_streams - gw + GW - 1) / GW : 0;
    const long long my_items = (long long)my_streams * nb;
    if (lane == 0) {
        for (int i = 0; i < stages; i++) mbar_init(full + i, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    // all indices are carried incrementally (no divisions on the single warp's critical path)
    int ij = 0, ib = 0, ist = 0;                                  // issue cursor: stream ordinal, block, stage
    long long issued = 0;
    auto issue = [&]() {                                          // lane 0: start the load of the warp's next item
        if (issued >= my_items) return;
        mbar_expect_tx(full + ist, BYTES);
        bulk_g2s(buf + (size_t)ist * BYTES, src + (size_t)(gw + ij * GW) * stride + (size_t)ib * TICK, BYTES, full + ist);
        issued++;
        if (++ist == stages) ist = 0;
        if (++ib == nb) { ib = 0; ij++; }
    };
    if (lane == 0) for (int k = 0; k < stages; k++) issue();
    long long w_next = my_streams ? B.st[stream0 + gw].written : 0;
    int j = 0, b = 0, st = 0, p0 = 0, bi = 0;
    unsigned phase = 0;
    for (long long k = 0; k < my_items; k++) {
        const int s = stream0 + gw + j * GW;
        if (b == 0) {
            const long long w_cur = w_next;
            p0 = (int)(w_cur % B.P);                                        // once per stream
            bi = (int)((w_cur / TICK) % B.NB);
            if (j + 1 < my_streams) w_next = B.st[s + GW].written;          // needed nb items from now
        }
        mbar_wait(full + st, phase);
        const double acc = warp_sumsq_smem(buf + (size_t)st * BYTES, sizeof(T) == 2 ? 1 : 0, lane);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic reads of the slot precede its async reuse
        __syncwarp();
        if (lane == 0) {
            bulk_s2g((T*)B.ring + (size_t)s * B.P + p0, buf + (size_t)st * BYTES, BYTES);   // P % TICK == 0: no wrap inside the block
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            B.block_ss[(size_t)s * B.NB + bi] = acc;
            if (k >= 1) {
                // the store of the previous item has read its slot: refill it
                asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                issue();
            }
        }
        __syncwarp();
        if (++st == stages) { st = 0; phase ^= 1u; }
        p0 += TICK; if (p0 >= B.P) p0 -= B.P;
        if (++bi == B.NB) bi = 0;
        if (++b == nb) { b = 0; j++; }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

struct GatePlan {                                   // one per warp (= per stream)
    long long V[GATE_MAX_TICKS];                    // samples visible at each tick
    double pv[GATE_MAX_TICKS][GATE_MAXP + 1];       // piece values; [GATE_MAXP] = recent-window sum of squares
    short pc[GATE_MAX_TICKS][GATE_MAXP];            // chunk index of each piece
    unsigned char np[GATE_MAX_TICKS];               // chunk pieces; 255: heavy tick (all chunks, done in phase 2)
    unsigned char alias[GATE_MAX_TICKS];            // recent window == piece 0 (frame_size 1600, aligned)
    unsigned char full[GATE_MAX_TICKS];
    double rms[GATE_MAX_TICKS];                     // is_silent's RMS per tick, formed by lane j ahead of the replay (not staged ticks)
};

// The 4-state timing machine + segment cut of WakeWord._detect_word for one tick (lane 0 only).
__device__ __forceinline__ unsigned gate_state_step(const BankView& B, int s, StreamState& st, const StreamParams& prm,
                                                    long long k, long long V, bool full, int silent) {
    unsigned evflag = 0;
    const double now = __dmul_rn((double)k, 0.1);
    if (full && !st.started) {                                  // _wait_for_buffer done -> _detect_word entry
        st.started = 1;
        st.state = silent ? ST_IN_SILENCE : ST_WAITING;        // wakeword.py:1048, 1055-1057
        st.start_time = now;                                    // :1052
        if (silent) st.silence_start = now;
        return 0;
    }
    if (!st.started) return 0;
    // loop top: the timeout check uses time() before the sleep (:1061), i.e. the previous tick's time
    const double prev = __dmul_rn((double)(k - 1), 0.1);
    if (prm.timeout > 0.0 && __dsub_rn(prev, st.start_time) > prm.timeout) {
        // TimeoutError -> the listen loop re-enters _detect_word at `prev` (:1205-1211)
        const int idx = atomicAdd(B.ev_count, 1);
        if (idx < B.max_events) {
            EventRec e{};
            e.stream = s; e.kind = EV_TIMEOUT; e.tick = k - 1; e.score = __int_as_float(0x7fc00000);
            B.events[idx] = e;
        } else { atomicAdd(B.ev_count + 1, 1); atomicSub(B.ev_count, 1); }
        st.n_timeouts++;
        st.state = st.last_silent ? ST_IN_SILENCE : ST_WAITING;
        st.start_time = prev;
        if (st.last_silent) st.silence_start = prev;
    }
    switch (st.state) {
        case ST_WAITING:                                        // :1069-1072
            if (silent) { st.state = ST_IN_SILENCE; st.silence_start = now; }
            break;
        case ST_IN_SILENCE:                                     // :1074-1081
            if (!silent) {
                if (__dsub_rn(now, st.silence_start) >= prm.pre_speech_silence) {
                    st.state = ST_IN_SOUND; st.sound_start = now;
                } else st.state = ST_WAITING;
            }
            break;
        case ST_IN_SOUND: {                                     // :1083-1094
            const double dur = __dsub_rn(now, st.sound_start);
            if (!silent) { if (dur > prm.speech_duration_max) st.state = ST_WAITING; }
            else if (prm.speech_duration_min <= dur && dur <= prm.speech_duration_max) {
                st.state = ST_AFTER_SOUND; st.sound_end = now;
            } else st.state = ST_WAITING;
            break;
        }
        case ST_AFTER_SOUND:                                    // :1096-1157
            if (silent) {
                if (__dsub_rn(now, st.sound_end) >= prm.post_speech_silence) {
                    const double es = __dsub_rn(__dsub_rn(st.sound_start, now), 0.05);   // :1102
                    const double ee = __dadd_rn(__dsub_rn(st.sound_end, now), 0.05);     // :1103
                    long long n_back = (long long)__dmul_rn(fabs(es), 16000.0);          // :500
                    const long long n_drop = (long long)__dmul_rn(fabs(ee), 16000.0);    // :1108
                    if (n_back > B.R) n_back = B.R;                                      // :501-502
                    const long long len = n_back - n_drop;
                    if (len >= 1 && len <= MAX_SEG) {                                    // :1114-1118
                        const int idx = atomicAdd(B.ev_count, 1);
                        // frame-parallel K3: the candidate's 1 + len/160 frames get a contiguous range of the frame table
                        const int nf = 1 + (int)len / HOP;
                        const int f0 = B.frame_ev ? atomicAdd(B.ev_count + 6, nf) : 0;
                        const bool fits = !B.frame_ev || (f0 >= 0 && f0 + nf <= B.frow_cap);
                        if (idx < B.max_events && fits) {
                            EventRec e{};
                            e.stream = s; e.kind = EV_PENDING; e.tick = k;
                            e.seg_start = V - n_back; e.seg_len = (int)len;
                            e.tmpl = f0;                                 // first frame of the range until K3 writes the best template
                            e.score = __int_as_float(0x7fc00000); e.matched = 0;
                            B.events[idx] = e;
                            if (B.frame_ev) {
                                B.ev_done[idx] = 0;
                                for (int t = 0; t < nf; t++) B.frame_ev[f0 + t] = idx;
                            }
                            {   // length class for K3's longest-first order (no tail of one long segment started last)
                                const int b = min(SEG_NB - 1, (nf + SEG_WARPS - 1) / SEG_WARPS);
                                const int q = atomicAdd(B.bk_count + b, 1);
                                if (q < B.max_events) B.bk_list[(size_t)b * B.max_events + q] = idx;
                            }
                            st.n_events++;
                            st.last_ev = idx;
                            evflag = 16u;
                        } else {
                            atomicAdd(B.ev_count + 1, 1); atomicSub(B.ev_count, 1);
                            if (B.frame_ev && f0 >= 0)                   // the range stays allocated: mark what exists of it as a hole
                                for (int t = 0; t < nf && f0 + t < B.frow_cap; t++) B.frame_ev[f0 + t] = -1;
                        }
                    }
                    st.state = ST_WAITING;                      // :1117, 1155
                }
            } else st.state = ST_WAITING;                       // :1157
            break;
    }
    return evflag;
}

// ------------------------------------------------------------------------------------ K2
// One WARP per stream, GATE_WARPS streams per CTA, no block-level barrier: a bank of 4096 streams is a
// single resident wave of warps.  Phase 0: lane j plans tick j (which sample ranges it needs);
// phase 1: the warp sums every planned range (the only HBM traffic: each new sample is read once,
// 16-byte loads, eight in flight per lane); phase 2: the ticks are replayed in order — chunk updates
// into an incrementally maintained sorted array, percentile, threshold, is_silent, state machine.
// PACED (ewk_tick_ready): each stream takes only the ticks its landed audio pays for, min(n_ticks, written / 1600 - tick),
// possibly none; its result record is stored all the same, since peer publication relies on every record in every call.
template <bool PACED>
__global__ void __launch_bounds__(GATE_THREADS, 7)
tick_gate_kernel(BankView B, int n_ticks, TraceView tr, int trace_stride, int trace_off, int smem_chunks, int stage_bytes) {
    extern __shared__ __align__(16) double sm_d[];
    __shared__ GatePlan plans[GATE_WARPS];
    __shared__ __align__(8) unsigned long long mbar[GATE_WARPS][2];
    char* stage = reinterpret_cast<char*>(sm_d + (size_t)GATE_WARPS * 3 * smem_chunks);   // [warp][2][stage_bytes], 16-byte aligned
    __shared__ StreamState st_s[GATE_WARPS];
    __shared__ StreamParams prm_s[GATE_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s = blockIdx.x * GATE_WARPS + warp;
    if (s >= B.n_streams) return;
    double* ms = sm_d + (size_t)warp * 3 * smem_chunks;   // [n_chunks] storage order
    double* SA = ms + smem_chunks;                       // sorted buffers
    double* SB = SA + smem_chunks;
    GatePlan& plan = plans[warp];

    // per-stream state and parameters live in shared memory (only lane 0 mutates them)
    StreamState& st = st_s[warp];
    const StreamParams& prm = prm_s[warp];
    double* g_ms = B.chunk_ms + (size_t)s * 2 * B.chunk_cap;
    double* g_sorted = g_ms + B.chunk_cap;
    {
        // one round trip: state, parameters and (speculatively, up to the shared-memory capacity) the chunk arrays
        static_assert(sizeof(StreamState) % 8 == 0 && sizeof(StreamParams) % 8 == 0, "8-byte words");
        const unsigned long long* gs = reinterpret_cast<const unsigned long long*>(B.st + s);
        const unsigned long long* gp = reinterpret_cast<const unsigned long long*>(B.prm + s);
        unsigned long long* ds = reinterpret_cast<unsigned long long*>(&st_s[warp]);
        unsigned long long* dp = reinterpret_cast<unsigned long long*>(&prm_s[warp]);
        if (lane < (int)(sizeof(StreamState) / 8)) ds[lane] = gs[lane];
        if (lane < (int)(sizeof(StreamParams) / 8)) dp[lane] = gp[lane];
        const int spec = min(smem_chunks, B.chunk_cap);
        for (int i = lane; i < spec; i += 32) { ms[i] = g_ms[i]; SA[i] = g_sorted[i]; }
    }
    __syncwarp();
    if (PACED) n_ticks = (int)max(0LL, min((long long)n_ticks, st.written / TICK - st.tick));
    const int fs = st.frame_size;
    const long long tick0 = st.tick, visible0 = st.visible, written0 = st.written;
    const int valid0 = st.chunks_valid;
    const int n_chunks = fs > 0 ? B.R / fs : 0;
    const bool use_chunks = n_chunks > 0 && n_chunks <= B.chunk_cap && n_chunks <= smem_chunks;

    // ---- phase 0: lane j plans tick j
    {
        const int j = lane;
        long long V = visible0, Vp = visible0;
        if (fs > 0 && j < n_ticks) {
            const long long avail = (written0 / fs) * fs;
            const long long k = tick0 + j + 1;
            V = prm.live ? written0 : min((k * TICK / fs) * fs, avail);
            if (V < visible0) V = visible0;
            if (j > 0) {
                Vp = prm.live ? written0 : min(((k - 1) * TICK / fs) * fs, avail);
                if (Vp < visible0) Vp = visible0;
            }
        }
        const bool full = fs > 0 && V >= B.R;                           // is_buffer_full   wakeword.py:515-517
        const bool upd = j < n_ticks && full && use_chunks && V > Vp;
        const unsigned updmask = __ballot_sync(FULL, upd);
        const bool valid_before = valid0 || (updmask & ((1u << j) - 1u));
        if (j < n_ticks) {
            int np = 0, alias = 0;
            if (upd) {
                const long long dv = V - Vp;
                if (!valid_before || dv >= B.R) np = 255;
                else {
                    // storage-order chunks touched by the new samples: logical positions [q0, q0+dv) mod R
                    const int q0 = (int)(Vp % B.R);
                    const long long e = q0 + dv;
                    const int e1 = (int)min(e, (long long)B.R);
                    const int c1 = q0 / fs;
                    const int n1 = (e1 - 1) / fs - c1 + 1;
                    const int n2 = e > B.R ? (int)((e - B.R - 1) / fs) + 1 : 0;
                    for (int i = 0; i < n1 + n2; i++) {
                        const int c = i < n1 ? c1 + i : i - n1;
                        if (c >= n_chunks) continue;                    // the tail R - n_chunks*fs is in no chunk
                        if (np == GATE_MAXP) { np = 255; break; }
                        plan.pc[j][np++] = (short)c;
                    }
                    // the recent window IS chunk pc[0] only when the tick's 1600 new samples sit inside the logical ring:
                    // with R % 1600 != 0 the tick at q0 = floor(R / 1600) * 1600 lands in the tail and wraps into chunk 0
                    if (np == 1 && fs == TICK && dv == TICK && (q0 % TICK) == 0 && q0 + TICK <= B.R) alias = 1;
                }
            }
            plan.V[j] = V;
            plan.full[j] = full;
            plan.np[j] = (unsigned char)np;
            plan.alias[j] = (unsigned char)alias;
        }
    }
    __syncwarp();

    const int nrec = min(TICK, B.R);
    unsigned evflag = 0;
    int valid = valid0;
    long long key_lo = -1, key_hi = -1;            // bit patterns of the order statistics behind st.thr (lane 0)

    // ---- one tick of phase 2: chunk updates into the sorted array, percentile, threshold, is_silent, state machine
    bool rms_ahead = false;                        // plan.rms[] holds every tick's RMS (set below once the sums are known)
    auto replay_tick = [&](int j) {
        const long long k = tick0 + j + 1;
        const long long V = plan.V[j];
        const bool full = plan.full[j];
        const int np = plan.np[j];
        if (np == 255) {
            // heavy tick (first full ring, or a jump of a whole ring): every chunk from samples, then sort
            for (int c = 0; c < n_chunks; c++) {
                const double v = warp_chunk_ms(B, s, V, fs, c, lane);
                if (lane == 0) ms[c] = v;
            }
            __syncwarp();
            warp_sort_build(ms, SA, n_chunks, lane);
            valid = 1;
        } else {
            for (int i = 0; i < np; i++) {
                const int c = plan.pc[j][i];
                const double nv = plan.pv[j][i];
                const double ov = ms[c];
                __syncwarp();
                warp_sorted_replace(SA, SB, n_chunks, ov, nv, lane);
                if (lane == 0) ms[c] = nv;
                __syncwarp();
            }
        }
        if (lane == 0) {
            if (np != 0) {
                // the threshold only moves when one of the two order statistics np.percentile reads moved
                const int k_lo = (int)floor((double)n_chunks * 0.25 - 0.25), k_hi = min(k_lo + 1, n_chunks - 1);
                const long long b_lo = __double_as_longlong(SA[k_lo]), b_hi = __double_as_longlong(SA[k_hi]);
                if (b_lo != key_lo || b_hi != key_hi) {
                    key_lo = b_lo; key_hi = b_hi;
                    const double p25 = percentile25_rms_sorted(SA, n_chunks);
                    const double nt = __dmul_rn(p25, 1.5);                  // wakeword.py:485
                    st.thr = nt > prm.min_threshold ? nt : prm.min_threshold;   // max(new, MIN_THRESHOLD)  :486
                }
            }
            // ---- is_silent (wakeword.py:488-496)
            int silent = 1;
            double rms = 0.0;
            if (fs > 0) {
                if (rms_ahead) rms = plan.rms[j];
                else {
                    double ss;
                    if (plan.alias[j]) ss = plan.pv[j][0] * (double)fs;     // same 1600 samples as the chunk
                    else { ss = plan.pv[j][GATE_MAXP]; if (B.fmt == 1) ss *= (1.0 / 1073741824.0); }
                    rms = sqrt(ss / (double)nrec);
                }
                silent = rms < st.thr;
            }
            st.last_rms = rms;
            evflag |= gate_state_step(B, s, st, prm, k, V, full, silent);
            st.last_silent = silent;
            if (tr.silent) {
                const size_t o = (size_t)s * trace_stride + trace_off + j;
                tr.silent[o] = (unsigned char)silent;
                tr.state[o] = (unsigned char)(st.started ? st.state : 255);
                tr.thr[o] = st.thr;
                tr.rms[o] = rms;
            }
            st.tick = k; st.visible = V;
        }
    };

    // Is every tick the aligned case (frame_size 1600: the tick's new block is one storage chunk and also the
    // RMS window) with its 1600 samples contiguous in the physical ring?  Then stage ticks through shared
    // memory with bulk copies, two ticks ahead, and replay tick j while ticks j+1, j+2 are in flight.
    const size_t esz = B.fmt == 1 ? 2 : 4;
    const bool mine_ok = lane >= n_ticks || (plan.alias[lane] && plan.np[lane] == 1);
    const bool all_alias = (B.P % TICK) == 0 && __all_sync(FULL, mine_ok);
    // block sums from the fused push kernel cover these ticks? then no PCM is read here at all
    const bool presummed = all_alias && B.NB > 0 && n_ticks > 0 && plan.V[0] - TICK >= st.ss_from;
    if (presummed) {
        if (lane < n_ticks) {
            double ss = B.block_ss[(size_t)s * B.NB + (size_t)(((plan.V[lane] - TICK) / TICK) % B.NB)];
            if (B.fmt == 1) ss *= (1.0 / 1073741824.0);
            plan.pv[lane][0] = ss / (double)fs;                          // np.mean(frame**2)   wakeword.py:481
        }
        __syncwarp();
    }
    const bool pipelined = !presummed && stage_bytes > 0 && all_alias && (!PACED || n_ticks > 0);
    unsigned long long* bar = mbar[warp];
    char* buf = stage + (size_t)warp * 2 * stage_bytes;
    const char* ring_s = (const char*)B.ring + (size_t)s * B.P * esz;
    int pos0 = 0;
    auto issue = [&](int j) {                                      // lane 0: bulk-copy tick j into stage j & 1
        int pos = pos0 + j * TICK;
        while (pos >= B.P) pos -= B.P;
        mbar_expect_tx(bar + (j & 1), (unsigned)(TICK * esz));
        bulk_g2s(buf + (size_t)(j & 1) * stage_bytes, ring_s + (size_t)pos * esz, (unsigned)(TICK * esz), bar + (j & 1));
    };
    if (pipelined) {
        pos0 = (int)((plan.V[0] - TICK) % B.P);                    // every tick advances by exactly TICK samples
        if (lane == 0) {
            mbar_init(bar, 1); mbar_init(bar + 1, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            issue(0);
            if (n_ticks > 1) issue(1);
        }
        __syncwarp();
    } else if (!presummed) {
        // ---- phase 1: every planned range (generic: any frame size, wrap, first-full and live streams)
        for (int j = 0; j < n_ticks; j++) {
            const long long V = plan.V[j];
            const int np = plan.np[j] == 255 ? 0 : plan.np[j];
            for (int i = 0; i < np; i++) {
                const double v = warp_chunk_ms(B, s, V, fs, plan.pc[j][i], lane);
                if (lane == 0) plan.pv[j][i] = v;
            }
            if (fs > 0 && !plan.alias[j]) {
                // RMS window of is_silent: the last min(1600, R) samples; zeros before the stream began
                const long long a0 = V - nrec;
                const double ss = warp_sumsq(ring_s, B.P, B.fmt, a0 < 0 ? 0 : a0, (int)(a0 < 0 ? V : nrec), lane);
                if (lane == 0) plan.pv[j][GATE_MAXP] = ss;
            }
        }
        __syncwarp();
    }
    if (!pipelined) {
        // every tick's sum of squares is known: lane j forms tick j's RMS (a double division and square root, ~35
        // instructions) once, instead of lane 0 doing it tick after tick inside the serial replay; same operations
        if (lane < n_ticks && fs > 0) {
            double ss;
            if (plan.alias[lane]) ss = plan.pv[lane][0] * (double)fs;
            else { ss = plan.pv[lane][GATE_MAXP]; if (B.fmt == 1) ss *= (1.0 / 1073741824.0); }
            plan.rms[lane] = sqrt(ss / (double)nrec);
        }
        rms_ahead = true;
        __syncwarp();
    }
    // ---- phase 2: replay the ticks in order (pipelined: tick j's sum first, copies of j+1, j+2 in flight)
    for (int j = 0; j < n_ticks; j++) {
        if (pipelined) {
            mbar_wait(bar + (j & 1), (unsigned)((j >> 1) & 1));
            double ss = warp_sumsq_smem(buf + (size_t)(j & 1) * stage_bytes, B.fmt, lane);
            __syncwarp();
            if (lane == 0) {
                if (j + 2 < n_ticks) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    issue(j + 2);
                }
                if (B.fmt == 1) ss *= (1.0 / 1073741824.0);
                plan.pv[j][0] = ss / (double)fs;                     // np.mean(frame**2)   wakeword.py:481
            }
            __syncwarp();
        }
        replay_tick(j);
    }
    __syncwarp();

    if (use_chunks && valid)
        for (int i = lane; i < n_chunks; i += 32) { g_ms[i] = ms[i]; g_sorted[i] = SA[i]; }
    if (lane == 0) {
        st.chunks_valid = valid;
        B.st[s] = st;
        StreamResult r = B.results[s];
        r.flags = (r.flags & 1u) | (st.last_silent ? 2u : 0u) | ((unsigned)st.state << 2) | evflag |
                  ((unsigned)st.n_events << 8);
        store_result(B.results + s, r);
        if (B.n_pub) store_result(B.pub_snap + (size_t)B.pub_parity * B.n_streams + s, r);   // the call's copy for the sender
    }
}

// ------------------------------------------------------------------------------------ K5 (level-3 hand-off)
struct PrepDesc { int stream; int len; long long start; long long out_off; };

// One CTA per segment: mean (double), max |x - mean|, then (x - mean) / max * 1.5 clipped to [-1, 1]
// (wakeword.py:1020-1025; the reference works in float64 on the float64 ring, the result here is its float32).
__global__ void __launch_bounds__(256)
segment_prepare_kernel(BankView B, const PrepDesc* __restrict__ d, float* __restrict__ out) {
    __shared__ double red[8];
    __shared__ double bc[2];
    const PrepDesc pd = d[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const short* q = B.fmt == 1 ? (const short*)B.ring + (size_t)pd.stream * B.P : nullptr;
    const float* f = B.fmt == 0 ? (const float*)B.ring + (size_t)pd.stream * B.P : nullptr;
    const int p0 = (int)(pd.start % B.P);
    auto at = [&](int i) -> double {
        int p = p0 + i;
        if (p >= B.P) p -= B.P;
        return q ? (double)q[p] * (1.0 / 32768.0) : (double)f[p];
    };
    double s = 0.0;
    for (int i = tid; i < pd.len; i += 256) s += at(i);
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (tid == 0) { double t = 0.0; for (int w = 0; w < 8; w++) t += red[w]; bc[0] = t / (double)pd.len; }
    __syncthreads();
    const double mean = bc[0];
    double m = 0.0;
    for (int i = tid; i < pd.len; i += 256) m = fmax(m, fabs(at(i) - mean));
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmax(m, __shfl_xor_sync(FULL, m, o));
    __syncthreads();
    if (lane == 0) red[warp] = m;
    __syncthreads();
    if (tid == 0) { double t = 0.0; for (int w = 0; w < 8; w++) t = fmax(t, red[w]); bc[1] = t; }
    __syncthreads();
    const double mx = bc[1];
    for (int i = tid; i < pd.len; i += 256) {
        double v = at(i) - mean;
        if (mx > 0.0) v = v / mx;
        v = v * 1.5;
        v = v < -1.0 ? -1.0 : (v > 1.0 ? 1.0 : v);
        out[pd.out_off + i] = (float)v;
    }
}

// ------------------------------------------------------------------------------------ K3 (queue form)
// Persistent CTAs drain the segments K2 queued: PCM straight from the stream's device ring ->
// fused MFCC + template match -> score written back into the event record and the per-stream result.
// Scheduling: segments differ in length (0.3 .. 3 s) and there are only a few per CTA (555 over 296 in the bench
// workload), so (1) CTAs take them dynamically — first task = blockIdx.x, then an atomic counter (ev_count[2]) — and
// (2) in LONGEST-FIRST order: K2 files every candidate it queues under its length class (rounds of SEG_WARPS frames,
// bk_count / bk_list), and task t is the t-th candidate counted from the longest class down.  The kernel then ends
// with its shortest segments instead of whatever came last (list scheduling, longest processing time first).
// The lists hold the candidates queued since the previous K3 launch; the last CTA to finish zeroes the counters and
// advances the scored watermark ev_count[3].

#ifdef EWK_K3_TRACE
// timeline of one launch (a measuring build only: -DEWK_K3_TRACE, profiles/tools/k3_timeline.py): per CTA
// [0] SM id, [1] start, [2] tables loaded, [3] exit, [4] segments taken; then per segment start, end, samples, event index
constexpr int K3_TRACE_SEGS = 14, K3_TRACE_WORDS = 8 + 4 * K3_TRACE_SEGS;
__device__ __forceinline__ long long k3_now() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#endif

template <bool PRE>
__global__ void __launch_bounds__(512, 2)
segment_queue_kernel(const DeviceTables* __restrict__ T, BankView B, const TemplateFeat* __restrict__ tmpl, int n_tmpl_slots) {
    extern __shared__ __align__(16) float smem[];
    const SegSmem m = seg_carve(smem, SEG_SMEM_FRAMES);
    __shared__ float sc_s[EWK_MAX_TEMPLATES];
    __shared__ int next_s;
    __shared__ int cum_s[SEG_NB + 1];
    const int tid = threadIdx.x;
    const int n = min(B.ev_count[0], B.max_events);
    // task t of this launch = the t-th candidate in longest-class-first order (K2 filed them by class)
    auto task_event = [&](int t) -> int {
        if (t >= cum_s[SEG_NB]) return -1;
        int j = 0;
        while (t >= cum_s[j + 1]) j++;
        return B.bk_list[(size_t)(SEG_NB - 1 - j) * B.max_events + (t - cum_s[j])];
    };
#ifdef EWK_K3_TRACE
    long long* trc = B.k3_trace ? B.k3_trace + (size_t)blockIdx.x * K3_TRACE_WORDS : nullptr;
    int trc_n = 0;
    if (trc && tid == 0) { unsigned sm; asm("mov.u32 %0, %%smid;" : "=r"(sm)); trc[0] = sm; trc[1] = k3_now(); }
#endif
    if (tid == 0) {
        int c = 0;
        for (int j = 0; j < SEG_NB; j++) { cum_s[j] = c; c += min(B.bk_count[SEG_NB - 1 - j], B.max_events); }
        cum_s[SEG_NB] = c;
        next_s = task_event(blockIdx.x);
    }
    __syncthreads();
    int r = next_s;
    if (r >= 0) seg_prologue(T, m);                                      // tables; ends with __syncthreads()
    const size_t esz = B.fmt == 1 ? 2 : 4;
    float* lm = B.lm_ws ? B.lm_ws + (size_t)blockIdx.x * SEG_SMEM_FRAMES * LM_ROW : nullptr;
#ifdef EWK_K3_TRACE
    if (trc && tid == 0) trc[2] = k3_now();
#endif
    while (r >= 0) {
        const int i = r;
        const EventRec e = B.events[i];
#ifdef EWK_K3_TRACE
        if (trc && tid == 0 && trc_n < K3_TRACE_SEGS) { trc[8 + 4 * trc_n] = k3_now(); trc[8 + 4 * trc_n + 2] = e.seg_len; trc[8 + 4 * trc_n + 3] = i; }
#endif
        int t_next = 0;
        if (tid == 0) t_next = (int)gridDim.x + atomicAdd(B.ev_count + 2, 1);     // its latency hides behind the segment
        SegDesc sd;
        sd.base = (const char*)B.ring + (size_t)e.stream * B.P * esz;
        sd.start = e.seg_start % B.P; sd.ring = B.P; sd.len = e.seg_len; sd.fmt = B.fmt;
        sd.ws_frame_off = 0; sd.frames_off = 0; sd.lm_off = 0;
        const float* feat = segment_features<PRE>(sd, m, SEG_SMEM_FRAMES, nullptr, nullptr, lm);
        const StreamParams& prm = B.prm[e.stream];
        const int t0 = max(0, prm.template_first);
        const int nt = max(0, min(prm.template_count, n_tmpl_slots - t0));
        if (tid < nt) {
            const TemplateFeat& tf = tmpl[t0 + tid];
            sc_s[tid] = tf.valid ? similarity_score(tf.mean, tf.std, feat, feat + N_MFCC) : __int_as_float(0x7fc00000);
        }
        __syncthreads();
        if (tid == 0) {
            const int nx = task_event(t_next);                           // the list load overlaps the record updates below
            // best score over the stream's template set (NaN never wins: NaN >= x is false, as in wakeword.py:638-639)
            float best = __int_as_float(0x7fc00000);
            int arg = nt > 0 ? t0 : -1;
            for (int k = 0; k < nt; k++)
                if (!(sc_s[k] != sc_s[k]) && (best != best || sc_s[k] > best)) { best = sc_s[k]; arg = t0 + k; }
            const int ok = best >= prm.similarity_threshold ? 1 : 0;
            EventRec* o = B.events + i;
            o->score = best; o->tmpl = arg; o->matched = ok; o->kind = EV_SCORED;
            if (B.st[e.stream].last_ev == i) {
                // only the stream's newest candidate of this queue epoch reaches the 8-byte record (one owner per stream:
                // no read-modify-write race between CTAs that score two events of one stream in arbitrary order)
                StreamResult res = B.results[e.stream];
                res.score = best;
                res.flags = (res.flags & ~1u) | (unsigned)ok;
                store_result(B.results + e.stream, res);
                if (B.n_pub) store_result(B.pub_snap + (size_t)B.pub_parity * B.n_streams + e.stream, res);
            }
            next_s = nx;
        }
        __syncthreads();
#ifdef EWK_K3_TRACE
        if (trc && tid == 0 && trc_n < K3_TRACE_SEGS) { trc[8 + 4 * trc_n + 1] = k3_now(); trc_n++; }
#endif
        r = next_s;
    }
#ifdef EWK_K3_TRACE
    if (trc && tid == 0) { trc[3] = k3_now(); trc[4] = trc_n; }
#endif
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(B.ev_count + 4, 1) == (int)gridDim.x - 1) {       // every other CTA has read the counters
            B.ev_count[3] = n;
            B.ev_count[2] = 0;
            B.ev_count[4] = 0;
            for (int j = 0; j < SEG_NB; j++) B.bk_count[j] = 0;
        }
    }
}

// ------------------------------------------------------------------------------------ K3 (frame-parallel queue form)
// The same result as segment_queue_kernel, with FRAMES as the unit of work instead of segments: the queued candidates'
// frames (K2 gave every candidate a contiguous range of a frame table) are taken in small chunks by any warp of the
// grid, so the kernel has no block barrier and no tail of whole segments.  A warp turns its frames into un-floored MFCC
// rows (+ log-mel min / max) in a global row table that stays L2-resident (96 B per frame), counts them on the
// candidate's completion counter, and the warp that delivers a candidate's LAST frame runs its epilogue alone:
// max over frames -> power_to_db floor, frames below it recomputed with the floor, mean / std over frames with the very
// operation order of segment_features (14 strided partials, Chan pooling — so the features are bit-identical to the
// one-CTA form and to what ewk_extract_mfcc / ewk_set_template produce), cosine scores, event and result records.
constexpr int FQ_CHUNK = 2;                    // frames a warp takes per visit of the work counter
__host__ __device__ inline size_t fq_smem_bytes() { return sizeof(FrameTables) + sizeof(float) * (size_t)SEG_WARPS * (SCR_WARP + FEAT); }

struct FqView {                                // what the epilogue needs of the bank, by value (the kernel's BankView stays in
    const void* ring;                          // parameter space: a non-inlined callee must not take its address)
    EventRec* events;
    float* frow;
    const StreamParams* prm;
    const StreamState* st;
    StreamResult* results;
    StreamResult* pub_snap;                    // this call's snapshot for the publication sender (null: publication off)
    int P, fmt;
};

template <bool PRE>
__device__ __forceinline__ void fq_reader(const void* ring, int P, int fmt, int stream, long long seg_start, int seg_len, float pre,
                                          PcmReader& rd) {
    const size_t esz = fmt == 1 ? 2 : 4;
    const char* base = (const char*)ring + (size_t)stream * P * esz;
    rd.f = fmt == 0 ? (const float*)base : nullptr;
    rd.q = fmt == 1 ? (const short*)base : nullptr;
    rd.ring = P; rd.len = seg_len; rd.start = seg_start % P; rd.pre = PRE ? pre : 0.f;
}

// epilogue of one candidate by one warp: rows -> features -> scores -> records
template <bool PRE>
__device__ __noinline__ void fq_finish(const FqView B, int idx, const FrameTables* ft, float* scr, float* feat,
                                       const TemplateFeat* __restrict__ tmpl, int n_tmpl_slots) {
    const int lane = threadIdx.x & 31;
    const EventRec e = B.events[idx];
    const int F = 1 + e.seg_len / HOP;
    float* rows = B.frow + (size_t)e.tmpl * FROW;              // e.tmpl still holds the candidate's first frame
    // floor = (max over frames of the log-mel max) - 80.  The (min, max) of up to 320 frames are fetched with ten
    // independent loads per lane: one L2 latency instead of one per frame
    constexpr int MMR = (SEG_SMEM_FRAMES + 31) / 32;
    float2 mm[MMR];
#pragma unroll
    for (int i = 0; i < MMR; i++) {
        const int t = lane + 32 * i;
        mm[i] = t < F ? __ldcg(reinterpret_cast<const float2*>(rows + (size_t)t * FROW + N_MFCC)) : make_float2(INFINITY, -INFINITY);
    }
    float vmax = -INFINITY;
#pragma unroll
    for (int i = 0; i < MMR; i++) vmax = fmaxf(vmax, mm[i].y);
#pragma unroll
    for (int o = 16; o; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(FULL, vmax, o));
    const float floor_db = vmax - 80.0f;                        // librosa.power_to_db(top_db=80)
    // frames that reach below the floor are recomputed with it (same function, same bits as the one-CTA form's re-floor)
    {
        PcmReader rd;
        fq_reader<PRE>(B.ring, B.P, B.fmt, e.stream, e.seg_start, e.seg_len, ft->preemph, rd);
#pragma unroll
        for (int i = 0; i < MMR; i++) {
            unsigned m = __ballot_sync(FULL, mm[i].x < floor_db);
            while (m) {
                const int tt = 32 * i + __ffs(m) - 1;
                m &= m - 1;
                float2 x[8];
                load_frame_pairs<PRE>(rd, tt, lane, x);
                float mn, mx;
                warp_frame_mfcc(x, *ft, scr, lane, floor_db, rows + (size_t)tt * FROW, mn, mx);
            }
        }
    }
    __syncwarp();
    // mean / std over frames, operation for operation as segment_features: partial w owns frames w, w + 14, ... (its sum,
    // then its M2 about its own mean, each in frame order), the 14 partials pooled in order (Chan et al.).  The rows come
    // through the warp's scratch in tiles of FQ_TILE frames, fetched with independent 16-byte loads.
    constexpr int FQ_TILE = 24;                                  // 24 frames x 96 B = 2304 B of the 2560 B scratch
    float acc[SEG_WARPS], mu[SEG_WARPS];
#pragma unroll
    for (int w = 0; w < SEG_WARPS; w++) { acc[w] = 0.f; mu[w] = 0.f; }
    const int cl = lane < N_MFCC ? lane : 0;
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
#pragma unroll 1
        for (int t0 = 0; t0 < F; t0 += FQ_TILE) {
            const int nt = min(FQ_TILE, F - t0);
            __syncwarp();
            {
                const float4* src = reinterpret_cast<const float4*>(rows + (size_t)t0 * FROW);
                float4* dst = reinterpret_cast<float4*>(scr);
                const int n4 = nt * (FROW / 4);
                float4 v[5];                                     // 24 * 6 = 144 words of 16 bytes: at most 5 per lane
#pragma unroll
                for (int u = 0; u < 5; u++) { const int i = lane + 32 * u; v[u] = i < n4 ? __ldcg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f); }
#pragma unroll
                for (int u = 0; u < 5; u++) { const int i = lane + 32 * u; if (i < n4) dst[i] = v[u]; }
            }
            __syncwarp();
            const int ph = t0 % SEG_WARPS;
#pragma unroll
            for (int w = 0; w < SEG_WARPS; w++) {
                int j = w - ph; if (j < 0) j += SEG_WARPS;       // first frame of the tile that belongs to partial w
                for (; j < nt; j += SEG_WARPS) {
                    const float v = scr[j * FROW + cl];
                    if (pass == 0) acc[w] += v;
                    else { const float d = v - mu[w]; acc[w] = fmaf(d, d, acc[w]); }
                }
            }
        }
        if (pass == 0) {
#pragma unroll
            for (int w = 0; w < SEG_WARPS; w++) {
                const int nw = (F - w + SEG_WARPS - 1) / SEG_WARPS;
                mu[w] = w < F ? acc[w] / (float)nw : 0.f;
                acc[w] = 0.f;
            }
        }
    }
    __syncwarp();
    if (lane < N_MFCC) {
        float n = 0.f, mean = 0.f, M2 = 0.f;
#pragma unroll
        for (int w = 0; w < SEG_WARPS; w++) {
            if (w < F) {
                const float cw = (float)((F - w + SEG_WARPS - 1) / SEG_WARPS);
                const float delta = mu[w] - mean, nn = n + cw;
                mean = fmaf(delta, cw / nn, mean);
                M2 += acc[w] + delta * delta * (n * cw / nn);
                n = nn;
            }
        }
        const bool kept = lane < ft->n_mfcc;
        feat[lane] = kept ? mean : 0.f;
        feat[N_MFCC + lane] = kept ? sqrtf(M2 / (float)F) : 0.f;
    }
    __syncwarp();
    // best score over the stream's template set (NaN never wins: NaN >= x is false, as in wakeword.py:638-639)
    const StreamParams& prm = B.prm[e.stream];
    const int t0 = max(0, prm.template_first);
    const int nt = max(0, min(prm.template_count, n_tmpl_slots - t0));
    float best = __int_as_float(0x7fc00000);
    int arg = nt > 0 ? t0 : -1;
    for (int k0 = 0; k0 < nt; k0 += 32) {
        const int k = k0 + lane;
        float sc = __int_as_float(0x7fc00000);
        if (k < nt) {
            const TemplateFeat& tf = tmpl[t0 + k];
            if (tf.valid) sc = similarity_score(tf.mean, tf.std, feat, feat + N_MFCC);
        }
        // sequential order over k (the first best wins), as the one-CTA form
        for (int j = 0; j < 32 && k0 + j < nt; j++) {
            const float v = __shfl_sync(FULL, sc, j);
            if (!(v != v) && (best != best || v > best)) { best = v; arg = t0 + k0 + j; }
        }
    }
    if (lane == 0) {
        const int ok = best >= prm.similarity_threshold ? 1 : 0;
        EventRec* o = B.events + idx;
        o->score = best; o->tmpl = arg; o->matched = ok; o->kind = EV_SCORED;
        if (B.st[e.stream].last_ev == idx) {
            StreamResult res = B.results[e.stream];
            res.score = best;
            res.flags = (res.flags & ~1u) | (unsigned)ok;
            store_result(B.results + e.stream, res);
            if (B.pub_snap) store_result(B.pub_snap + e.stream, res);
        }
    }
    __syncwarp();
}

template <bool PRE>
__global__ void __launch_bounds__(512, 2)
segment_frames_kernel(const DeviceTables* __restrict__ T, BankView B, const TemplateFeat* __restrict__ tmpl, int n_tmpl_slots) {
    extern __shared__ __align__(16) float smem[];
    FrameTables* ft = reinterpret_cast<FrameTables*>(smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float* scr = smem + sizeof(FrameTables) / sizeof(float) + (size_t)warp * (SCR_WARP + FEAT);
    float* feat = scr + SCR_WARP;
    const int n = min(B.ev_count[0], B.max_events);
    const int f_lo = min(B.ev_count[5], B.frow_cap), f_hi = min(max(B.ev_count[6], 0), B.frow_cap);
    if (f_hi > f_lo) {
        copy_frame_tables(*ft, T, tid, blockDim.x);
        __syncthreads();
        for (;;) {
            int c0 = 0;
            if (lane == 0) c0 = atomicAdd(B.ev_count + 2, FQ_CHUNK);
            c0 = f_lo + __shfl_sync(FULL, c0, 0);
            if (c0 >= f_hi) break;
            const int c1 = min(c0 + FQ_CHUNK, f_hi);
            int done_ev = -1, done_cnt = 0, done_F = 0;            // frames of one candidate computed in this chunk, not yet delivered
            auto deliver = [&]() {
                int old = 0;
                __threadfence();
                if (lane == 0) old = atomicAdd(B.ev_done + done_ev, done_cnt);
                old = __shfl_sync(FULL, old, 0);
                if (old + done_cnt == done_F) {                    // this warp delivered the candidate's last frame: it scores it
                    __threadfence();
                    fq_finish<PRE>(FqView{B.ring, B.events, B.frow, B.prm, B.st, B.results,
                                          B.n_pub ? B.pub_snap + (size_t)B.pub_parity * B.n_streams : nullptr, B.P, B.fmt}, done_ev, ft, scr, feat, tmpl,
                                   n_tmpl_slots);
                }
                done_cnt = 0;
            };
            for (int f = c0; f < c1; f++) {
                const int idx = B.frame_ev[f];
                if (idx != done_ev && done_cnt) deliver();          // leaving a candidate
                if (idx < 0) continue;                             // hole left by a dropped candidate
                float2 x[8];
                {
                    // the candidate's descriptor is re-read per frame (L1 / L2 hits) rather than kept live across the pipeline call
                    const EventRec* ep = B.events + idx;
                    const int len = ep->seg_len;
                    PcmReader rd;
                    fq_reader<PRE>(B.ring, B.P, B.fmt, ep->stream, ep->seg_start, len, ft->preemph, rd);
                    done_F = 1 + len / HOP;
                    load_frame_pairs<PRE>(rd, f - ep->tmpl, lane, x);
                }
                float mn, mx;
                float* row = B.frow + (size_t)f * FROW;
                warp_frame_mfcc(x, *ft, scr, lane, -INFINITY, row, mn, mx);
                if (lane == 0) { row[N_MFCC] = mn; row[N_MFCC + 1] = mx; }
                done_ev = idx;
                done_cnt++;
            }
            if (done_cnt) deliver();
        }
    }
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(B.ev_count + 4, 1) == (int)gridDim.x - 1) {       // every other CTA is done: nobody reads the counters any more
            B.ev_count[3] = n;
            B.ev_count[5] = 0;                                           // rows are scratch of one launch: the frame table restarts,
            B.ev_count[6] = 0;                                           // so it stays small and L2-resident
            B.ev_count[2] = 0;
            B.ev_count[4] = 0;
            for (int j = 0; j < SEG_NB; j++) B.bk_count[j] = 0;
        }
    }
}

// Device-side consumer gate for peer publication: returns once slots [0, n_slots) of the local signal row hold a sequence
// number >= seq (all records of those ranks up to that call have landed), or after timeout_ns (then *timed_out = 1):
// it can never hang the device.  One warp, lane p watches slot p.
__global__ void peer_wait_kernel(const unsigned long long* __restrict__ sig_row, int n_slots, unsigned long long seq,
                                 unsigned long long timeout_ns, int* timed_out) {
    const int p = threadIdx.x;
    if (p >= n_slots) return;
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(sig_row + p) : "memory");
        if (v >= seq) break;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > timeout_ns) { atomicExch(timed_out, 1); break; }
        __nanosleep(256);
    }
}

// ------------------------------------------------------------------------------------ K9 (stream recycling)
// ewk_reset_streams: every listed stream back to the state init_streams gives it.  CTA (x, y) clears byte slice x of the
// ring row of list[y] with 16-byte stores (rows are P * esz bytes, P a multiple of 64: 16-byte aligned); the CTAs of
// slice 0 also write the StreamState, the block_ss and chunk_ms rows, the result record, K4's carried-row range and
// K4D's detector state.
// The K8 input tail needs no clearing: a stream at input position 0 reads none of it and rewrites it on its next push.
// HBM-bound: P * esz bytes per stream plus a few KB.
constexpr int RESET_THREADS = 256;
constexpr int RESET_SLICE = RESET_THREADS * 16 * 8;       // bytes of a ring row per CTA (8 stores per thread)

// Per-stream state of the dense detector (K4D, ewk_dense_detect; ewk_dense.cuh).  All zeros is the initial state:
// IDLE, quiet_until 0, no pending record.
enum : int { DET_IDLE = 0, DET_ARMED = 1, DET_SPENT = 2 };
struct DetState {
    int mode, slot;                    // slot: template slot of the pending peak
    long long quiet_until, peak, run_start, seg_start;
    int seg_len;
    float score;                       // pending peak score
};

__global__ void __launch_bounds__(RESET_THREADS)
stream_reset_kernel(BankView B, const int* __restrict__ list, int n, long long* keep_end, DetState* det) {
    const size_t row_bytes = (size_t)B.P * (B.fmt == 1 ? 2 : 4);
    for (int y = blockIdx.y; y < n; y += gridDim.y) {
        const int s = list[y];
        int4* row = reinterpret_cast<int4*>(reinterpret_cast<char*>(B.ring) + (size_t)s * row_bytes);
        const size_t w0 = (size_t)blockIdx.x * (RESET_SLICE / 16), w1 = min(w0 + RESET_SLICE / 16, row_bytes / 16);
        for (size_t w = w0 + threadIdx.x; w < w1; w += RESET_THREADS) row[w] = make_int4(0, 0, 0, 0);   // np.zeros  wakeword.py:428
        if (blockIdx.x != 0) continue;
        if (threadIdx.x == 0) {
            StreamState z;
            memset(&z, 0, sizeof(z));
            z.thr = 0.01; z.last_ev = -1;                                       // wakeword.py:431
            B.st[s] = z;
            store_result(B.results + s, StreamResult{__int_as_float(0x7fc00000), 0u});   // nanf(""), as init_streams
            if (keep_end) { keep_end[2 * s] = 0; keep_end[2 * s + 1] = 0; }
            if (det) det[s] = DetState{};
        }
        double* ss = B.block_ss + (size_t)s * B.NB;
        for (int i = threadIdx.x; i < B.NB; i += RESET_THREADS) ss[i] = 0.0;
        double* ms = B.chunk_ms + (size_t)s * 2 * B.chunk_cap;                 // ms[cap] ++ sorted[cap]
        for (int i = threadIdx.x; i < 2 * B.chunk_cap; i += RESET_THREADS) ms[i] = 0.0;
    }
}

// ------------------------------------------------------------------------------------ K10 (stream migration)
// ewk_export_streams / ewk_import_streams (include/ewk.h): a stream's whole device state to and from row y of a blob's
// bulk section, in K9's grid shape.  CTA (x, y) copies 32 KB slice x of the ring row with 16-byte loads and stores;
// the CTAs of slice 0 also copy the block_ss, chunk_ms and K8 tail rows and the small state (StreamState, result record, DetState).  One read and one
// write per byte: HBM-bound.  Rings hold absolute sample a at a % P in every context with the same ring_samples and
// slack_samples, and block_ss holds block b at b % NB, so every row moves verbatim.
// A bulk row (all parts 16-byte aligned): ring [P * esz] | block_ss [NB] doubles, zero-padded | chunk_ms [2 chunk_cap]
// doubles | K8 input tail [tail_floats] floats: the stream's live inputs [t0, c) (StreamMeta.tail_len of them), zeros
// beyond, so a blob carries nothing an earlier occupant of the slot left in its tail row.
struct MigrateGeom { long long row_bytes, ss_off, ms_off, tail_off; int tail_floats, pad; };

// One record per stream of a blob's meta section.  The host fills the mirrors and the parameters; on export K10 fills
// st, res and det.  Import reads it on the host only: the kernel takes the checked copy (MigrateSmall).
struct StreamMeta {
    long long written, visible_lb, tick, dense_next, det_next, inputs;   // host mirrors of the context
    int frame_size, rate, tail_len, pad;                                 // tail_len: live K8 tail inputs c - t0 (0 at 16 kHz)
    StreamParams prm;
    StreamState st;
    StreamResult res;
    DetState det;                                                        // zeros when the source had no detector state
};
static_assert(sizeof(StreamMeta) == 304, "StreamMeta is part of blob version 1");

// the small state is copied by the CTA's threads in 8-byte words (every struct here is a multiple of 8 bytes)
template <class T> __device__ __forceinline__ void copy_words(T* dst, const T* src) {
    static_assert(sizeof(T) % 8 == 0, "8-byte words");
    const long long* a = reinterpret_cast<const long long*>(src);
    long long* b = reinterpret_cast<long long*>(dst);
    for (int i = threadIdx.x; i < (int)(sizeof(T) / 8); i += blockDim.x) b[i] = a[i];
}

struct MigrateSmall {       // import: the checked small state of one stream (last_ev already -1)
    StreamParams prm;
    StreamState st;
    StreamResult res;
    DetState det;
    int tail_len, pad;
};

__global__ void __launch_bounds__(RESET_THREADS)
stream_export_kernel(BankView B, const int* __restrict__ list, int n, const DetState* __restrict__ det,
                     const float* __restrict__ tail, int tail_cap, StreamMeta* meta, char* bulk, MigrateGeom g) {
    const size_t ring_bytes = (size_t)B.P * (B.fmt == 1 ? 2 : 4);
    for (int y = blockIdx.y; y < n; y += gridDim.y) {
        const int s = list[y];
        const int4* src = reinterpret_cast<const int4*>(reinterpret_cast<const char*>(B.ring) + (size_t)s * ring_bytes);
        char* row = bulk + (size_t)y * g.row_bytes;
        int4* dst = reinterpret_cast<int4*>(row);
        const size_t w0 = (size_t)blockIdx.x * (RESET_SLICE / 16), w1 = min(w0 + RESET_SLICE / 16, ring_bytes / 16);
        for (size_t w = w0 + threadIdx.x; w < w1; w += RESET_THREADS) dst[w] = src[w];
        if (blockIdx.x != 0) continue;
        copy_words(&meta[y].st, B.st + s);
        copy_words(&meta[y].res, B.results + s);
        if (det) copy_words(&meta[y].det, det + s);
        else if (threadIdx.x == 0) meta[y].det = DetState{};
        const double* ss = B.block_ss + (size_t)s * B.NB;
        double* oss = reinterpret_cast<double*>(row + g.ss_off);
        const int n_ss = (int)((g.ms_off - g.ss_off) / 8);
        for (int i = threadIdx.x; i < n_ss; i += RESET_THREADS) oss[i] = i < B.NB ? ss[i] : 0.0;
        const double* ms = B.chunk_ms + (size_t)s * 2 * B.chunk_cap;
        double* oms = reinterpret_cast<double*>(row + g.ms_off);
        for (int i = threadIdx.x; i < 2 * B.chunk_cap; i += RESET_THREADS) oms[i] = ms[i];
        float* ot = reinterpret_cast<float*>(row + g.tail_off);
        for (int i = threadIdx.x; i < g.tail_floats; i += RESET_THREADS)
            ot[i] = (tail && i < meta[y].tail_len) ? tail[(size_t)s * tail_cap + i] : 0.f;   // tail_len <= tail_cap (host)
    }
}

// list and small: the host's checked copy (one upload); bulk values are copied, never used as an index or a length
__global__ void __launch_bounds__(RESET_THREADS)
stream_import_kernel(BankView B, const int* __restrict__ list, const MigrateSmall* __restrict__ small, int n,
                     const char* __restrict__ bulk, MigrateGeom g, long long* keep_end, DetState* det, float* tail,
                     int tail_cap) {
    const size_t ring_bytes = (size_t)B.P * (B.fmt == 1 ? 2 : 4);
    for (int y = blockIdx.y; y < n; y += gridDim.y) {
        const int s = list[y];
        const char* row = bulk + (size_t)y * g.row_bytes;
        const int4* src = reinterpret_cast<const int4*>(row);
        int4* dst = reinterpret_cast<int4*>(reinterpret_cast<char*>(B.ring) + (size_t)s * ring_bytes);
        const size_t w0 = (size_t)blockIdx.x * (RESET_SLICE / 16), w1 = min(w0 + RESET_SLICE / 16, ring_bytes / 16);
        for (size_t w = w0 + threadIdx.x; w < w1; w += RESET_THREADS) dst[w] = src[w];
        if (blockIdx.x != 0) continue;
        const MigrateSmall& m = small[y];
        copy_words(B.prm + s, &m.prm);
        copy_words(B.st + s, &m.st);
        if (det) copy_words(det + s, &m.det);
        if (threadIdx.x == 0) {
            store_result(B.results + s, m.res);
            if (keep_end) { keep_end[2 * s] = 0; keep_end[2 * s + 1] = 0; }    // K4 rebuilds its carried rows
        }
        const double* ss = reinterpret_cast<const double*>(row + g.ss_off);
        double* oss = B.block_ss + (size_t)s * B.NB;
        for (int i = threadIdx.x; i < B.NB; i += RESET_THREADS) oss[i] = ss[i];
        const double* ms = reinterpret_cast<const double*>(row + g.ms_off);
        double* oms = B.chunk_ms + (size_t)s * 2 * B.chunk_cap;
        for (int i = threadIdx.x; i < 2 * B.chunk_cap; i += RESET_THREADS) oms[i] = ms[i];
        if (tail) {
            const float* t = reinterpret_cast<const float*>(row + g.tail_off);
            for (int i = threadIdx.x; i < m.tail_len; i += RESET_THREADS) tail[(size_t)s * tail_cap + i] = t[i];
        }
    }
}

}  // namespace ewk
