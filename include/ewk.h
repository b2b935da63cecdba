/* libewk — C ABI of the B200-native EasyWakeWord hot path (level-1 energy gate + level-2 MFCC/cosine
 * matcher, batched over independent 16 kHz audio streams).
 *
 * The reference (raymondclowe/EasyWakeWord) has no FFI of its own: its seam is two duck-typed Python
 * attributes of WakeWord, `_sound_buffer` and `_matcher` (easywakeword/wakeword.py:989-997; used at
 * 1004, 1055, 1066, 1105, 1121, 1225).  Each entry point below cites the reference method it replaces.
 * easywakeword_b200/_lib.py is the ctypes binding; INTEGRATION.md shows the stub a reference
 * maintainer would add.
 *
 * Conventions: every call returns 0 (EWK_OK) or a negative ewk_status; the message is read with
 * ewk_last_error().  The caller owns all host buffers; the library owns device memory; no callbacks
 * cross the ABI.  One context per GPU; one consumer thread per context.  There is no CPU fallback:
 * without a CUDA device ewk_create fails with EWK_ERR_CUDA.
 */
#ifndef EWK_H
#define EWK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EWK_ABI_VERSION 2

typedef struct ewk_ctx ewk_ctx;

typedef enum ewk_status {
    EWK_OK = 0,
    EWK_ERR_ARG = -1,         /* bad argument                                    -> ValueError   */
    EWK_ERR_NO_TEMPLATE = -2, /* wakeword.py:608-609 "No reference word set..."  -> ValueError   */
    EWK_ERR_CUDA = -3,        /* CUDA runtime failure / no device                -> RuntimeError */
    EWK_ERR_STATE = -4,       /* call made in the wrong state                    -> RuntimeError */
    EWK_ERR_NOMEM = -5
} ewk_status;

typedef enum ewk_pcm_format { EWK_PCM_F32 = 0, EWK_PCM_I16 = 1 } ewk_pcm_format;
typedef enum ewk_mem { EWK_HOST = 0, EWK_DEVICE = 1 } ewk_mem;

enum { EWK_N_MFCC = 20, EWK_N_MELS = 128, EWK_N_FFT = 512, EWK_HOP = 160, EWK_SAMPLE_RATE = 16000,
       EWK_TICK_SAMPLES = 1600 };

/* Template slots: a context holds up to EWK_MAX_TEMPLATE_SLOTS (ewk_config.max_templates), enough for one personal
 * word per stream of a full B200 bank; one stream is scored against at most EWK_MAX_STREAM_TEMPLATES consecutive slots
 * (ewk_stream_params.template_count). */
#define EWK_MAX_TEMPLATE_SLOTS 4096
#define EWK_MAX_STREAM_TEMPLATES 64

typedef struct ewk_config {
    int32_t n_streams;      /* independent audio streams resident on this GPU (0: matcher only)       */
    int32_t ring_samples;   /* SoundBuffer.buffer_length = seconds * 16000       wakeword.py:426-428  */
    int32_t slack_samples;  /* extra physical ring so that one ewk_push may run ahead of ewk_tick      */
    int32_t pcm_format;     /* ewk_pcm_format of the device rings                                     */
    int32_t max_templates;  /* template slots, 1..EWK_MAX_TEMPLATE_SLOTS (reference: one WordMatcher) */
    int32_t max_events;     /* capacity of the device event queue between two ewk_poll calls          */
    /* --- ABI 2: front-end parameters the reference hard-codes (wakeword.py:561-563; exposing them is on its own
     * wish list, LEARNINGS.md:87, README-CODE-ALIGNMENT.md:84-107).  0 selects the reference's value. */
    float preemphasis;      /* coefficient a of y[n] = x[n] - a x[n-1], applied to every segment / dense window
                               handed to the MFCC front-end, before centring (librosa.effects.preemphasis incl.
                               its zi = 2 x[0] - x[1] initial state).  The reference applies none: 0 = identity
                               is the parity default and leaves every result bit-identical                    */
    int32_t n_mfcc;         /* MFCC coefficients kept, 1..20; 0 = 20                      wakeword.py:562     */
    int32_t template_frames;/* 1: keep every template slot's MFCC frame matrix for frame alignment (ewk_align_*);
                               max_templates x 301 x 20 floats of device memory (24 KB per slot).  0: none        */
    int32_t reserved1;
} ewk_config;

/* ---- library ------------------------------------------------------------------------------ */
int ewk_abi_version(void);
/* message of the last failing call on `ctx` (or, with ctx == NULL, of the last failing ewk_create
 * on this thread).  Never NULL. */
const char* ewk_last_error(const ewk_ctx* ctx);
/* Host-only (no GPU needed): copies a read-only table the kernels use into out[cap] and returns its
 * length: 0 hann[512], 1 mel filterbank dense [128*257], 2 dct [20*128] (row k, column b). */
int ewk_host_table(int which, float* out, int cap);

/* ---- context ------------------------------------------------------------------------------ */
/* WakeWord._initialize_audio (wakeword.py:989-1000) for a whole bank of streams on CUDA `device`. */
int ewk_create(int device, const ewk_config* cfg, ewk_ctx** out);
int ewk_destroy(ewk_ctx* ctx);
/* Run all kernels of `ctx` on an existing cudaStream_t (e.g. torch's current stream); NULL restores
 * the context's own stream. */
int ewk_set_cuda_stream(ewk_ctx* ctx, void* cuda_stream);
int ewk_synchronize(ewk_ctx* ctx);

/* ---- level 2: WordMatcher (wakeword.py:520-639) -------------------------------------------- */
/* WordMatcher.extract_mfcc (wakeword.py:544-567): n float32 samples -> mean[20], std[20] over the
 * 1 + n/160 MFCC frames; when frames != NULL also the frame matrix, row-major [n_frames][20]
 * (frames_cap = capacity in frames).  pcm is a host or device pointer according to `where`. */
int ewk_extract_mfcc(ewk_ctx* ctx, const float* pcm, int64_t n, int where, float* mean20, float* std20,
                     float* frames, int64_t frames_cap);
/* WordMatcher.set_reference (wakeword.py:569-578) into template slot `slot`. */
int ewk_set_template(ewk_ctx* ctx, int slot, const float* pcm, int64_t n);
/* Install precomputed features (mean[20], std[20]) for a template of n_samples samples. */
int ewk_set_template_features(ewk_ctx* ctx, int slot, const float* mean20, const float* std20, int64_t n_samples);
int ewk_get_template(ewk_ctx* ctx, int slot, float* mean20, float* std20, int64_t* n_samples);
int ewk_clear_template(ewk_ctx* ctx, int slot);
/* WordMatcher.calculate_similarity / matches (wakeword.py:591-639) for n_seg segments of one PCM
 * buffer (segment i = pcm[offsets[i] : offsets[i] + lens[i]]) against template `slot`:
 * scores[i] in [0, 100] or NaN; matched[i] = scores[i] >= threshold (NaN -> 0).  features may be NULL;
 * otherwise [n_seg][40] = mean, std per segment.  EWK_ERR_NO_TEMPLATE if the slot is empty. */
int ewk_similarity_batch(ewk_ctx* ctx, int slot, const void* pcm, int pcm_format, int where,
                         const int64_t* offsets, const int64_t* lens, int n_seg, float threshold,
                         float* scores, uint8_t* matched, float* features);

/* ---- level 1: SoundBuffer (wakeword.py:405-517) + _detect_word timing (wakeword.py:1036-1159) --- */
typedef struct ewk_stream_params {
    float similarity_threshold;     /* WakeWord(similarity_threshold=75.0)              wakeword.py:676  */
    int32_t frame_size;             /* PortAudio callback length; 0: length of the first push  :457-458 */
    double pre_speech_silence;      /* 0.8                                                :38, 677       */
    double speech_duration_min;     /* auto from the template WAV (fallback 0.3)          :39, 678       */
    double speech_duration_max;     /* 2 x min (fallback 2.0)                             :40, 679       */
    double post_speech_silence;     /* 0.4                                                :41, 680       */
    double timeout;                 /* seconds before _detect_word raises and the listen loop re-enters
                                       it (:1061-1062, 1205-1211); <= 0: never                          */
    double min_threshold;           /* SoundBuffer.MIN_THRESHOLD = 0.005                  :409           */
    int32_t template_first;         /* the stream is scored against template slots                      */
    int32_t template_count;         /*   [template_first, template_first + template_count), best wins;  
                                       at most EWK_MAX_STREAM_TEMPLATES                                  */
    int32_t live;                   /* 1: a tick sees every pushed sample (SoundBuffer facade driven by
                                       wall-clock polls); 0: audio clock, tick k sees
                                       floor(1600 k / frame_size) * frame_size samples                  */
    int32_t reserved;
} ewk_stream_params;

typedef struct ewk_event {
    int32_t stream;
    int32_t kind;          /* 2: level-2 evaluation of a level-1 candidate (wakeword.py:1121); 1: timeout */
    int64_t tick;          /* tick index k (time = k * 0.1 s) at which the reference would have acted     */
    int64_t seg_start;     /* absolute sample index of the first sample of the extracted word_audio       */
    int32_t seg_len;       /* len(word_audio)                                       wakeword.py:1109-1111 */
    int32_t template_slot; /* best-scoring template slot                                                  */
    float score;           /* WordMatcher.calculate_similarity                      wakeword.py:591-625   */
    int32_t matched;       /* score >= similarity_threshold                         wakeword.py:638-639   */
} ewk_event;

typedef struct ewk_stream_status {
    int64_t written;            /* samples pushed                                                       */
    int64_t visible;            /* samples the last tick saw                                            */
    int64_t tick;               /* ticks processed                                                      */
    double silence_threshold;   /* SoundBuffer.silence_threshold                     wakeword.py:431,486 */
    double last_rms;            /* RMS of the last 0.1 s at the last tick            wakeword.py:495     */
    int32_t frame_size;         /* SoundBuffer.frame_size                                               */
    int32_t state;              /* 0 waiting, 1 in_silence, 2 in_sound, 3 after_sound                   */
    int32_t started;            /* buffer was full and _detect_word is running                          */
    int32_t is_silent;          /* SoundBuffer.is_silent() at the last tick          wakeword.py:488-496 */
    int32_t n_timeouts;
    int32_t n_events;
} ewk_stream_status;

typedef struct ewk_stream_result {  /* dense per-stream record, 8 bytes: what multi-GPU runs gather      */
    float score;                    /* latest level-2 score of the stream (NaN before the first)         */
    uint32_t flags;                 /* bit0 matched | bit1 silent | bits2-3 state | bit4 event in the last
                                       ewk_tick | bits 8..31 events so far                               */
} ewk_stream_result;

typedef struct ewk_detection {      /* dense detector decision (ewk_dense_detect), 48 bytes               */
    int32_t stream, template_slot;  /* slot of the peak score                                             */
    int64_t hop;                    /* peak hop                                                           */
    int64_t run_start;              /* first hop of the run                                               */
    int64_t emit_hop;               /* hop at which it was decided (run end, or peak + hold)              */
    int64_t seg_start;              /* 160 * (hop - n_k): the peak window, for ewk_read_segment /          */
    int32_t seg_len;                /*   ewk_prepare_segments (level 3); seg_len = L_k                    */
    float score;                    /* peak score                                                         */
} ewk_detection;

typedef struct ewk_vad_result {     /* template voice-activity analysis, 32 bytes                          */
    double duration_s;              /* max((last - first) * 160 / 16000, 0.2); 0 when voiced == 0         */
    float max_rms, threshold;       /* max frame RMS and max_rms * 0.1 (float32)                          */
    int32_t first_frame, last_frame;/* first / last frame with rms > threshold (-1 when none)             */
    int32_t n_frames;               /* 1 + len / 160                                                      */
    int32_t voiced;                 /* 0: no frame above the threshold (the reference returns None)       */
} ewk_vad_result;

/* defaults of the reference (wakeword.py:31-48, 408-409, 676) with audio-clock ticks */
int ewk_default_stream_params(ewk_stream_params* out);
/* stream == -1 applies to every stream. */
int ewk_set_stream_params(ewk_ctx* ctx, int stream, const ewk_stream_params* p);
/* SoundBuffer._add_sound_to_buffer (wakeword.py:454-465) for n_streams streams at once: n samples per
 * stream, stream s reads pcm + s*stride (in samples, format = the ring's).  `where` tells whether pcm is
 * a host pointer (pinned memory makes the copy asynchronous) or a device pointer.  Host PCM is copied on a
 * dedicated copy stream into one of two staging buffers and lands in the rings (K1) when something needs it:
 * the next push, a tick that reaches into it, or a read of stream state; a PINNED host buffer must therefore
 * stay unchanged until one of those calls (or ewk_synchronize) returns.  Pageable buffers are safe on return. */
int ewk_push(ewk_ctx* ctx, int stream0, int n_streams, const void* pcm, int64_t n, int64_t stride, int where);
/* The same for a G.711 feed: 8-bit mu-law (law = 0) / A-law (law = 1) codes — the telephony wire format, and WAV format
 * tags 7 / 6 that libsndfile decodes under librosa.load (wakeword.py:588).  The codes are expanded on the device to the
 * standard's 16-bit linear samples and pushed like PCM16, so a host feed crosses PCIe at one byte per sample.  The
 * context's rings must be EWK_PCM_I16.  Results equal those of pushing the expanded samples with ewk_push, bit for bit. */
int ewk_push_g711(ewk_ctx* ctx, int stream0, int n_streams, const uint8_t* codes, int64_t n, int64_t stride, int where, int law);
/* n_ticks polls of WakeWord._detect_word (wakeword.py:1064-1157) for every stream: adaptive threshold,
 * is_silent, timing state machine, segment cut, then the fused MFCC+match kernel on every candidate.
 * Asynchronous; results are read with ewk_poll / ewk_stream_results. */
int ewk_tick(ewk_ctx* ctx, int n_ticks);
/* Same, also recording per-tick traces [n_streams][n_ticks] (any pointer may be NULL; host memory). */
int ewk_tick_trace(ewk_ctx* ctx, int n_ticks, uint8_t* silent, uint8_t* state, double* thr, double* rms);
/* Drain the event queue into out[cap] (sorted by tick, then stream); returns the number of events
 * (>= 0) or a negative status.  *dropped (may be NULL) counts events lost to a full queue. */
int ewk_poll(ewk_ctx* ctx, ewk_event* out, int cap, int* dropped);
int ewk_stream_status_get(ewk_ctx* ctx, int stream, ewk_stream_status* out);
/* SoundBuffer.return_last_n_seconds (wakeword.py:498-513): the last n_samples visible samples. */
int ewk_read_last(ewk_ctx* ctx, int stream, int64_t n_samples, float* out);
/* word_audio of an event (wakeword.py:1105-1111) for the level-3 hand-off; EWK_ERR_STATE if overwritten. */
int ewk_read_segment(ewk_ctx* ctx, int stream, int64_t seg_start, int64_t seg_len, float* out);
/* Level-3 hand-off, batched (SURVEY §8(f) N1): what WakeWord._transcribe_audio does to word_audio before the
 * speech-to-text call (wakeword.py:1020-1025): x - mean(x), / max|.| when > 0, * 1.5, clip to [-1, 1] — for
 * n_seg segments of the rings at once (typically the matched events of one ewk_poll).  Segment i is
 * streams[i], absolute samples [starts[i], starts[i] + lens[i]); its float32 result is written at
 * out + out_offsets[i]; no other float of `out` is written.  `where` tells whether `out` is host or device memory.
 * EWK_ERR_STATE if a segment was already overwritten in its ring.  A failed call writes nothing to `out`. */
int ewk_prepare_segments(ewk_ctx* ctx, int n_seg, const int32_t* streams, const int64_t* starts, const int64_t* lens,
                         const int64_t* out_offsets, float* out, int64_t out_len, int where);
/* Overlap of level-2 matching with the next push (off by default).  When enabled, ewk_tick launches K3 on a second
 * stream right after the gate: the next ewk_push (K1, HBM-bound) then runs beside K3's tail instead of behind it.
 * K3 only reads ring samples that the push guard already protects and writes event / result records, and every other
 * stream-bank call (the next ewk_tick, ewk_poll, ewk_stream_results, ewk_read_*, ...) first makes the context's
 * stream wait for it, so results are unchanged.  The one visible difference: work that the CALLER enqueues on the
 * context's stream right after ewk_tick (e.g. an NCCL all-gather of ewk_results_device_ptr) must be preceded by
 * ewk_join, which enqueues that wait without blocking the host.  Rings shorter than 3 s + the ticks of a call keep the
 * sequential order. */
int ewk_set_overlap(ewk_ctx* ctx, int enable);
int ewk_join(ewk_ctx* ctx);
/* Template analysis, batched (SURVEY §8(f) N2): WakeWord._analyze_reference_audio_duration
 * (wakeword.py:872-893) for n templates at once — librosa.feature.rms with 25 ms frames every 10 ms (zero-padded
 * centring), frames above 0.1 * max RMS, first-to-last span, floor 0.2 s.  Template i is the float32 samples
 * pcm[offsets[i] : offsets[i] + lens[i]] (16 kHz; `where` says host or device).  rms_out (nullable, host) receives
 * the frame RMS values of all templates back to back (n_frames each; rms_cap = its capacity in floats).  The
 * caller derives speech_duration_min/max from duration_s as the reference's tests pin it
 * (tests/test_wakeword_simulated.py:687-775: min = duration or 0.3, max = 2 * min or 2.0). */
int ewk_analyze_templates(ewk_ctx* ctx, const float* pcm, int where, const int64_t* offsets, const int64_t* lens,
                          int n, ewk_vad_result* out, float* rms_out, int64_t rms_cap);
/* Template enrolment, batched: template slots[i] gets the float32 16 kHz samples pcm[offsets[i] : offsets[i] + lens[i]]
 * (`where` says host or device), for n templates in one call.  Every field each slot receives (K3's mean / std, the
 * dense kernel's dmean / dstd, n_samples) is bit-identical to what ewk_set_template(ctx, slots[i], that audio) installs,
 * and vad (nullable, host) receives vad[i] bit-identical to ewk_analyze_templates of the same audio.  One K3 launch over
 * all n templates (templates over 48 000 samples take K3's workspace path, as in ewk_set_template), one dense-feature
 * launch that also writes the table entries, one K6 launch when vad is given, one copy of the features back and one
 * synchronisation: the number of launches does not grow with n.  Dense sets (ewk_dense_*_sets) covering a written slot
 * are rebuilt on their next use.  In overlap mode the call joins K3 first.  n = 0 is a no-op.
 * EWK_ERR_ARG, naming the entry, for a slot out of [0, max_templates) or listed twice, lens[i] < 1 or > 2^30, a negative
 * offset, or a NULL array with n > 0.  Every check comes before the first launch: a failed call changes no slot. */
int ewk_set_templates(ewk_ctx* ctx, const int32_t* slots, int n, const float* pcm, int where,
                      const int64_t* offsets, const int64_t* lens, ewk_vad_result* vad);
/* Template enrolment from the rings: template slots[i] gets stream streams[i]'s absolute samples
 * [starts[i], starts[i] + lens[i]) — the coordinates of ewk_event.seg_start / seg_len, ewk_detection.seg_start / seg_len
 * and ewk_read_segment.  The result equals ewk_set_templates of what ewk_read_segment returns for those ranges, bit for
 * bit (int16 rings convert as q / 32768).  One gather launch copies the ranges into a float32 device scratch, then the
 * call runs as ewk_set_templates on it.  Streams may repeat (one stream enrolling several utterances).  A pending host
 * push lands first; in overlap mode the call joins K3 first.  Errors, named by row and stream, all before the first
 * launch (a failed call changes no slot): those of ewk_set_templates, EWK_ERR_ARG for a stream out of range or
 * lens[i] > the physical ring, EWK_ERR_STATE for a range not yet pushed or already overwritten in its ring and for a
 * context with n_streams = 0. */
int ewk_set_templates_from_streams(ewk_ctx* ctx, const int32_t* slots, int n, const int32_t* streams,
                                   const int64_t* starts, const int64_t* lens, ewk_vad_result* vad);
/* Frame alignment (second stage after level 2, before level 3): dynamic time warping of a segment's MFCC frames against
 * a template's, which tells the word from the same sounds in another order (pooled mean / std cannot).  Needs a context
 * created with ewk_config.template_frames = 1: ewk_set_template, ewk_set_templates and ewk_set_templates_from_streams then
 * also keep each slot's frame matrix (the K3 frames of its audio, at no extra launch); a template over 48 000 samples
 * (the longest segment alignment takes: 301 frames), ewk_set_template_features and ewk_clear_template leave the slot without frames.
 * ewk_get_template_frames: *n_frames (nullable) receives the slot's frame count (0: none) and out[cap frames][20] (nullable)
 * the frames, bit-identical to ewk_extract_mfcc's `frames` for the slot's audio.  EWK_ERR_STATE with template_frames = 0,
 * EWK_ERR_NO_TEMPLATE for an empty slot, EWK_ERR_ARG for cap below the count. */
int ewk_get_template_frames(ewk_ctx* ctx, int slot, float* out, int64_t cap, int32_t* n_frames);
/* ewk_align_segments: row i is stream streams[i]'s absolute samples [starts[i], starts[i] + lens[i]) (the coordinates of
 * ewk_event and ewk_detection, with ewk_read_segment's checks), aligned against slots [template_first[i], template_first[i]
 * + template_count[i]); with both arrays NULL, row i takes its stream's own range (ewk_stream_params).  For a segment with
 * frames f_0..f_{n-1} (exactly ewk_extract_mfcc's frames of that audio) and mean `mean` (its ewk_extract_mfcc mean), a
 * template with stored frames g_0..g_{m-1} and its mean, and C = the context's n_mfcc (coefficients c < C only):
 *   u_i = f_i - mean, v_j = g_j - template mean;  r_i = 1 / sqrt(sum_c u_i[c]^2) (0 when the sum is 0), s_j alike;
 *   cost_ij = 1 - (dot(u_i, v_j) * r_i) * s_j  (cosine distance; an all-constant segment costs 1 everywhere);
 *   D_00 = cost_00, D_i0 = D_{i-1,0} + cost_i0, D_0j = D_{0,j-1} + cost_0j,
 *   D_ij = cost_ij + min(D_{i-1,j-1}, D_{i-1,j}, D_{i,j-1});   distance = D_{n-1,m-1} / (n + m),
 * in float32 with every dot product and sum of squares a serial fma chain over c from +0 and every other operation rounded
 * once (oracle/align_model.py is the bit-exact model).  0 is a perfect match; the word against itself gives 0.  There
 * is no default threshold: a distance is not on the 0-100 score scale.
 * dist is packed as the _sets forms pack rows: row i starts at sum_{j < i} T_j and holds T_i = template_count[i] values,
 * in slot order; dist_cap is its capacity in floats.  best_slot[i] (nullable) receives the absolute slot of the lowest
 * distance (the lowest slot on ties) and best_dist[i] (nullable) that distance.  `where` says whether the three outputs
 * are host or device memory.  The call reads the rings and changes no stream, cursor, detector or event.  A pending host
 * push lands first; in overlap mode the call joins K3 first.  One K3 launch (frames and means of every segment) and one
 * K11 launch (one CTA per row), whatever n; synchronises with the context's stream.  n = 0 is a no-op.
 * Errors, all before the first launch (a failed call writes no output), naming the row and the stream:
 *   EWK_ERR_STATE: template_frames = 0; a range not yet pushed or already overwritten; a context with n_streams = 0.
 *   EWK_ERR_ARG: a stream out of range; lens[i] outside 1..48000 or a negative start; T_i outside 1..64; a slot range
 *   outside [0, max_templates); one of the two set arrays without the other; dist NULL or dist_cap below the packed
 *   length; a slot without frames (cleared, features only, or over 48 000 samples).
 *   EWK_ERR_NO_TEMPLATE: an empty slot. */
int ewk_align_segments(ewk_ctx* ctx, int n, const int32_t* streams, const int64_t* starts, const int64_t* lens,
                       const int32_t* template_first, const int32_t* template_count,
                       float* dist, int64_t dist_cap, int32_t* best_slot, float* best_dist, int where);
/* The same for caller audio (offline evaluation, threshold tuning): row i is pcm[offsets[i] : offsets[i] + lens[i]] in
 * pcm_format (EWK_PCM_F32, or EWK_PCM_I16 read as q / 32768), host or device memory according to where_in; host input
 * crosses in one copy.  The set arrays are required.  Works on any context (n_streams may be 0); the errors are those of
 * ewk_align_segments that apply, rows named with stream -1. */
int ewk_align_buffers(ewk_ctx* ctx, int n, const void* pcm, int pcm_format, int where_in,
                      const int64_t* offsets, const int64_t* lens,
                      const int32_t* template_first, const int32_t* template_count,
                      float* dist, int64_t dist_cap, int32_t* best_slot, float* best_dist, int where);
/* Ingest at other sample rates (SURVEY §8(f) N3): conversion to 16 kHz on the device, the step the reference
 * delegates to librosa.load(sr=16000) / librosa.resample (wakeword.py:588, 866-870; examples/tune_threshold.py:
 * 33-47; soxr HQ).  The filter meets soxr HQ's published specification (linear phase, pass-band to 0.913 of the
 * lower Nyquist, stop-band from 1.0, 125 dB) as one Kaiser-windowed-sinc polyphase stage; it is NOT soxr bit for
 * bit (oracle/resample_restated.py: parity unpinned).  Framing follows librosa.resample: output sample n sits at
 * input time n * sr_in / 16000, zeros outside the input, no gain rescale, one-shot length ceil(n_in*16000/sr_in).
 *
 * ewk_resample computes, for each of n_rows rows, absolute output samples [out_first, out_first + n_out) from
 * the absolute input samples [in_first, in_first + n_in) it is given (zeros elsewhere): one-shot use passes
 * in_first = out_first = 0; streaming use passes each chunk with half_width samples of history and emits only
 * outputs whose half_width samples of look-ahead are present, which reproduces the one-shot result exactly.
 * in: float32 or int16 (pcm_format), rows in_stride samples apart; out: float32, rows out_stride apart.
 * Supported rates: 1000 to 768000 Hz with 16000 / gcd(sr_in, 16000) <= 4096 (every standard rate).
 * Arithmetic: output n is the sequential fmaf chain, from +0, over taps j = 0 .. 2W-1 of H[j][p] * x[k_c - W + 1 + j]
 * with the float32 table H (k_c = floor(n M / L), p = n M mod L), the same on every code path.  Its rounding error
 * against the float64 sum of the same products grows with the filter length; measured on one B200 (1000 W) on full-scale
 * square waves, worst output: at most 1.2e-6 (-118 dBFS) up to 24 kHz, 1.8e-6 up to 64 kHz, 2.2e-6 at 96 kHz,
 * 1.5e-6 at 192 kHz, 5.5e-6 at 384 kHz and 8.1e-6 (-102 dBFS) at 768 kHz (DESIGN.md, K8).  The 125 dB above is the
 * filter's stop-band design, not the arithmetic's noise floor. */
int ewk_resample_info(int sr_in, int32_t* half_width, int32_t* up, int32_t* down);
int64_t ewk_resample_out_len(int64_t n_in, int sr_in);
int ewk_resample(ewk_ctx* ctx, const void* in, int pcm_format, int where_in, int n_rows, int64_t n_in, int64_t in_stride,
                 int sr_in, int64_t in_first, int64_t out_first, int64_t n_out, float* out, int64_t out_stride,
                 int where_out);
/* Native-rate feeds into the rings (K8): telephony G.711 at 8 kHz, 44.1 / 48 kHz from WebRTC or sound cards.
 * ewk_push_resampled takes n_in samples per stream at sr_in Hz (stream s reads in + s*stride, in samples of in_format:
 * EWK_PCM_F32, EWK_PCM_I16 = int16 / 32768, or 8-bit G.711 codes EWK_IN_ULAW / EWK_IN_ALAW = the standard's 16-bit
 * value / 32768; any format into either ring format) and lands their 16 kHz conversion in the rings in one fused launch.
 * Sample a of a stream's ring is exactly output a of a one-shot ewk_resample of everything pushed to the stream (int16
 * rings store rint(y * 32768) clamped to [-32768, 32767], ties to even).  After c input samples, outputs
 * [0, ready(c)) are in the ring, ready(c) = max(0, ceil((c - W) * up / down)) with W, up, down of ewk_resample_info:
 * an output lands once its W input samples of look-ahead have arrived (the last W inputs wait for the next push; there
 * is no final flush).  Returns the number of samples landed per stream (>= 0) or a status.
 * A stream's input rate is fixed by its first push of any kind.  EWK_ERR_STATE: streams of one call that have received
 * different numbers of input samples, a different rate than the stream's, a 16 kHz stream, and ewk_push /
 * ewk_push_g711 onto a native-rate stream.  EWK_ERR_ARG: sr_in = 16000 or a rate ewk_resample rejects.
 * With frame_size 0 the stream latches ewk_resample_out_len(n_in, sr_in) of its first call, so the audio clock stays on
 * the nominal 16 kHz grid.  Push guards, host staging (pinned or pageable, on the copy stream, landing lazily) and
 * overlap mode behave as for ewk_push, on the landed count.  The device keeps each stream's last <= 2W input samples. */
enum { EWK_IN_ULAW = 2, EWK_IN_ALAW = 3 };
int ewk_push_resampled(ewk_ctx* ctx, int stream0, int n_streams, const void* in, int in_format, int64_t n_in, int64_t stride,
                       int where, int sr_in);
/* ewk_push_resampled for streams at their own input positions (recycled streams restart at 0): the same in every respect
 * except that the streams of one call may have received different numbers of input samples, still in one launch.
 * landed (host, required: EWK_ERR_ARG when NULL) receives, for stream stream0 + i, the number of 16 kHz samples landed,
 * ready(c_i + n_in) - ready(c_i) for its position c_i.  Rings and input tails are bit-identical to one ewk_push_resampled
 * per group of equal positions.  Returns EWK_OK or a status. */
int ewk_push_resampled_each(ewk_ctx* ctx, int stream0, int n_streams, const void* in, int in_format, int64_t n_in,
                            int64_t stride, int where, int sr_in, int64_t* landed);
/* Ragged push to a list of streams.  Row i is in[offsets[i] .. offsets[i] + lens[i]) (in samples of in_format; the
 * buffer holds in_len samples) and goes to stream streams[i].  sr_in = 16000 lands the samples directly (in_format = the
 * ring's format, or EWK_IN_ULAW / EWK_IN_ALAW into int16 rings, as ewk_push / ewk_push_g711); any other rate converts
 * them with K8, any input format into either ring format, as ewk_push_resampled.  landed[i] (host, required) receives
 * the 16 kHz samples landed on streams[i] (lens[i] at 16 kHz).  lens[i] = 0 is allowed; n = 0 is a no-op.
 * The result is bit-identical to pushing each row alone with ewk_push / ewk_push_g711 / ewk_push_resampled onto
 * [streams[i], streams[i] + 1): rings, K8 input tails, rate and frame-size latches, ewk_stream_input.  A row of length 0
 * changes nothing.  With frame_size 0 a stream latches its row's length (other rates: ewk_resample_out_len of it).
 * EWK_ERR_ARG: a stream out of range or listed twice, a negative length or a row outside [0, in_len), landed = NULL, an
 * unsupported rate, G.711 at 16 kHz into f32 rings, another in_format than the rings' at 16 kHz, a row larger than the
 * ring.  EWK_ERR_STATE: a stream latched to another rate, and the push guards of ewk_push, per stream on its landed
 * count.  Host input crosses PCIe as one copy of [0, in_len) on the copy stream and lands lazily (pinned or pageable), as
 * with ewk_push; overlap mode behaves as for ewk_push.  Streams not listed are untouched and cost no bytes. */
int ewk_push_streams(ewk_ctx* ctx, const int32_t* streams, int n, const void* in, int in_format,
                     const int64_t* offsets, const int64_t* lens, int64_t in_len, int where, int sr_in, int64_t* landed);
/* Ticks paced by each stream's own audio: stream s takes taken[s] = min(max_ticks, max(0, written_s / 1600 - tick_s))
 * ticks (written_s after any pending host push has landed), i.e. tick k is taken once 1600 k samples have landed.
 * Otherwise the same as ewk_tick_trace: any of taken / silent / state / thr / rms may be NULL; trace cells are
 * [n_streams][max_ticks], and cells of ticks a stream did not take hold silent = 255, state = 255, thr = rms = NaN.
 * A stream with nothing due (a parked slot) takes no tick and raises no event; its result record is still rewritten
 * (bit 4 cleared) and published.  The same audio gives the same events however it was split into pushes.  Mixing with
 * ewk_tick on one context is allowed: ewk_tick moves every stream.  max_ticks in [1, 4096]. */
int ewk_tick_ready(ewk_ctx* ctx, int max_ticks, int32_t* taken, uint8_t* silent, uint8_t* state, double* thr, double* rms);
/* rate latched by the stream's first push (0: none yet; 16000: ewk_push / ewk_push_g711) and input samples received */
int ewk_stream_input(ewk_ctx* ctx, int stream, int32_t* sr_in, int64_t* n_in);
/* Stream recycling (a call ends, the slot takes the next one) without rebuilding the bank: return streams[0..n) to the
 * state ewk_create gives a stream.  Afterwards stream s behaves exactly like stream s of a new context with the same
 * ewk_config, templates and stream parameters given the same calls: events, result records, tick traces,
 * ewk_stream_status, ewk_stream_input, ewk_read_last (zeros before the ring fills), ewk_read_segment, dense scores.  Its
 * ticks and sample indices count from the reset; its detector (ewk_dense_detect) is back to cursor 1, IDLE,
 * quiet_until 0.  Streams not listed are untouched.  Stream parameters are kept (change them with
 * ewk_set_stream_params); the input-rate latch is cleared, so the next session may come at any rate.  A pending
 * host push lands first (its samples belong to the old session and are cleared with it); in overlap mode the call joins
 * K3 first.  One launch (K9) for the whole list; duplicates are harmless, n = 0 is a no-op.
 * EWK_ERR_STATE while the event queue is not empty ("poll first": events carry no session, so an old session's event
 * polled afterwards would point ewk_read_segment at the new session's audio) and for a context with n_streams = 0;
 * EWK_ERR_ARG for a stream out of range or streams = NULL with n > 0.  Synchronises with the context's stream. */
int ewk_reset_streams(ewk_ctx* ctx, const int32_t* streams, int n);
/* Stream migration: move live sessions between slots, contexts and GPUs (rebalancing, draining a GPU, checkpoints).
 * ewk_export_streams snapshots streams[0..n) into a blob; ewk_import_streams makes blob stream i stream streams[i] of a
 * context.  Afterwards stream streams[i] behaves exactly like the exported stream would have in its source context
 * given the same calls from then on: events (with the destination's stream id), result records, tick traces,
 * ewk_stream_status, ewk_stream_input, ewk_read_last, ewk_read_segment / ewk_prepare_segments of segments still in the
 * ring, dense scores, the cursors of ewk_dense_ready and ewk_dense_detect, and the detector's state with a pending
 * ARMED run.  Stream parameters travel with the stream (the destination's overlap-mode ring reserve follows them, as
 * with ewk_set_stream_params).  Streams not listed are untouched.
 * A blob may be imported into the same context (other slots, any permutation: exporting [a, b] and importing into
 * [b, a] swaps two live calls) or into another context with the same ring_samples, slack_samples, pcm_format, n_mfcc
 * and preemphasis, of any n_streams, max_events or max_templates, on the same GPU or another.  `where` says whether
 * the blob is host memory (pinned or pageable) or device memory of the context's device (16-byte aligned; copy it
 * across GPUs with your own copy, e.g. torch .to()).  A device blob must be complete when ewk_import_streams is called:
 * the call reads it on the context's stream and does not wait for copies queued on other streams, so synchronise with
 * the copy first (e.g. torch.cuda.synchronize(device), or make the context's stream wait for an event recorded behind
 * it).  A blob is position-independent and may be saved to a file.  A host blob goes through a device scratch buffer of
 * its size (export: the whole blob; import: its bulk rows), which the context keeps for later calls until it is
 * destroyed: about 360 KB per stream of a 10 s int16 ring; device blobs need none.
 * ewk_export_streams is read-only: the source goes on exactly as without it.  It lands a pending host push first (its
 * samples belong to the stream) and in overlap mode joins K3 first; events already raised stay in the source's queue
 * with the source's ids, so it needs no poll.
 * ewk_import_streams lands a pending push first (its samples belong to the slots' old sessions) and joins K3.  The
 * imported streams' newest-event link is cleared, K4 rebuilds their carried rows, and the detector state and K8 input
 * tails are allocated or grown as needed.
 * Both are one launch (K10) plus plain copies, and synchronise with the context's stream.  Every check comes before the
 * first launch: on any error no stream of the context changes.
 * EWK_ERR_ARG: a stream out of range or listed twice, n different from the blob's count, blob_cap / blob_len too small,
 * bad magic or version, a fingerprint field different from the context's (named), a device blob that is not 16-byte
 * aligned memory of the context's device, and a meta field outside what the entry points produce (named).
 * EWK_ERR_STATE: import while the context's event queue holds events ("poll first", as ewk_reset_streams), a context
 * with n_streams = 0, and a template slot a stream is scored against whose features or n_samples in the context are not
 * bit-identical to the blob's (named): a moved call never scores silently against another word. */
#define EWK_STREAM_BLOB_MAGIC 0x534B5745u      /* "EWKS" */
#define EWK_STREAM_BLOB_VERSION 1
typedef struct ewk_stream_blob {               /* at offset 0 of every blob, 96 bytes; the rest of a blob is opaque    */
    uint32_t magic, version;
    int32_t n_streams;                         /* streams in the blob                                                  */
    int32_t ring_samples, slack_samples;       /* fingerprint: the importing context's ewk_config must have the same   */
    int32_t pcm_format, n_mfcc;                /*   values (n_mfcc 0 is stored as 20)                                  */
    uint32_t preemphasis_bits;                 /*   and the same float32 bit pattern of preemphasis                    */
    int32_t meta_bytes;                        /* per-stream record of the meta section                                */
    int32_t n_templates;                       /* records of the template section: every slot a stream is scored on    */
    int32_t tail_floats;                       /* K8 input tail floats per bulk row                                     */
    int32_t reserved;
    int64_t ids_offset;                        /* int32 source stream ids [n_streams]                                  */
    int64_t meta_offset, template_offset, bulk_offset;   /* sections, 16-byte aligned                                  */
    int64_t bulk_row_bytes;                    /* one row per stream: ring, block sums, chunk mean squares, K8 tail    */
    int64_t total_bytes;                       /* length of the blob                                                   */
} ewk_stream_blob;
/* An upper bound of the bytes ewk_export_streams(ctx, .., n, ..) writes, for the input rates the context has seen so
 * far (host code: no device work). */
int64_t ewk_stream_blob_bytes(const ewk_ctx* ctx, int n);
int ewk_export_streams(ewk_ctx* ctx, const int32_t* streams, int n, void* blob, int64_t blob_cap, int where);
int ewk_import_streams(ewk_ctx* ctx, const int32_t* streams, int n, const void* blob, int64_t blob_len, int where);
/* Dense per-hop scoring (SURVEY §8(a) A9; usage shape of examples/tune_threshold.py:86-116 at hop
 * granularity): for every stream, every hop h in [hop0, hop0 + n_hops) (hop h <-> 160*h samples pushed)
 * and every template slot k in [template_first, template_first + template_count), the value
 * WordMatcher.calculate_similarity (wakeword.py:591-625) returns for the window
 *     x[160*(h - n_k) : 160*(h - n_k) + L_k],  n_k = ceil(L_k / 160)
 * i.e. the latest template-length window that starts on the hop grid and is complete at hop h
 * (window-local zero-pad centring and top_db floor).  out[(stream * n_hops + (h - hop0)) * template_count
 * + k], NaN where the window starts before the stream.  The audio must have been pushed and still be in
 * the ring (EWK_ERR_STATE otherwise).  Templates must have 640 <= L_k <= 48000 samples (the reference's own 3.0 s
 * segment cap, wakeword.py:1114-1118); template_count <= 8 per call.  Left-edge frames are shared by all templates, right-
 * edge frames by templates with the same padding to the hop grid; every call may continue where the previous one stopped.
 * `where` tells whether `out` is host or device memory. */
int ewk_dense_scores(ewk_ctx* ctx, int64_t hop0, int n_hops, int template_first, int template_count,
                     float* out, int where);
/* Ragged dense scoring: row i scores stream streams[i] at hops [hop0[i], hop0[i] + n_hops[i]) against templates
 * [template_first, template_first + template_count), each score the value ewk_dense_scores gives for that stream, hop
 * and template (NaN where the window starts before the stream).  out is packed in list order: row i starts at float
 * T * (n_hops[0] + .. + n_hops[i - 1]) (T = template_count) and is laid out [n_hops[i]][T]; out_cap is its capacity in
 * floats, and host output is copied back over the used length only.  n_hops[i] = 0 scores nothing for that row and
 * costs no CTA; n = 0 is a no-op.  One K4 launch, one CTA per non-empty row, longest rows first.  A pending host push
 * lands first only if some row reaches into it; overlap mode behaves as for ewk_dense_scores.
 * EWK_ERR_ARG (naming the stream): a stream out of range or listed twice, hop0 or n_hops negative, out_cap below the
 * packed length, a template range ewk_dense_scores rejects (EWK_ERR_NO_TEMPLATE for an empty slot).  EWK_ERR_STATE
 * (naming the stream): a row whose hops are not yet pushed, or whose oldest needed sample has left the ring.  On an
 * error nothing is scored.  Neither reads nor moves the cursors of ewk_dense_ready. */
int ewk_dense_scores_streams(ewk_ctx* ctx, const int32_t* streams, int n, const int64_t* hop0, const int32_t* n_hops,
                             int template_first, int template_count, float* out, int64_t out_cap, int where);
/* Dense scores paced by each stream's own audio.  The context keeps a cursor next_s per stream, 1 after ewk_create and
 * after ewk_reset_streams of the stream (hop 0 holds no sample).  Each listed stream (streams = NULL: every stream of the
 * bank, n ignored) is scored at hops [next_s, min(next_s + max_hops, written_s / 160 + 1)), written_s read after any
 * pending host push has landed, i.e. hop h is scored once 160 h samples have landed; hop0_out[i] = next_s and
 * n_hops_out[i] = the count, then next_s moves past them.  Output as ewk_dense_scores_streams, packed in list order;
 * n * max_hops * template_count floats always suffice.  A stream with nothing due gets 0 hops and costs no CTA.  The same
 * audio gives the same per-hop scores however it was split into pushes and calls.  max_hops in [1, 1 << 20].
 * Errors as ewk_dense_scores_streams; on any error no cursor moves (EWK_ERR_STATE for a stream whose cursor's windows
 * have left the ring: score it more often, or reset it).  ewk_dense_scores and ewk_dense_scores_streams leave the
 * cursors alone. */
int ewk_dense_ready(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops, int template_first, int template_count,
                    int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap, int where);
/* Wake-word detections from per-hop scores, on the device: a peak picker per stream that needs no gate.  The context
 * keeps a second cursor per stream for it, 1 after ewk_create and after ewk_reset_streams, independent of
 * ewk_dense_ready's.  Each listed stream (streams = NULL: every stream, n ignored) is scored at the hops ewk_dense_ready's
 * due rule gives from this cursor (at most max_hops), and those hops go in order through a state machine whose state
 * the context keeps per stream between calls:
 *   b_h = max over the call's templates of score[h][k], ignoring NaN (NaN when all are); k* the lowest k reaching it;
 *   above_h = b_h >= the stream's similarity_threshold (ewk_stream_params; NaN is never above).
 *   IDLE,  above_h and h >= quiet_until -> ARMED; pending = {peak h, run_start h, score b_h, slot template_first + k*,
 *                                          seg_start 160 (h - n_k*), seg_len L_k*}
 *   ARMED, above_h      -> if b_h > pending score (strictly: the first maximum wins) the peak fields move to h; then if
 *                          h - peak >= hold_hops the pending record is emitted with emit_hop h -> SPENT
 *   ARMED, not above_h  -> emit with emit_hop h, quiet_until = h + refractory_hops -> IDLE
 *   SPENT, not above_h  -> quiet_until = h + refractory_hops -> IDLE
 * quiet_until is 0 initially.  Any two emissions are >= 2 hops apart, so a call emits at most sum_i ceil(n_hops_i / 2)
 * records and n * ceil(max_hops / 2) always suffice.  A run still ARMED at the end of a call carries to the next; every
 * pending run is emitted at most hold_hops hops after its peak, so feed hold_hops more hops of audio (e.g. trailing
 * silence) to finish a recording.  The same audio gives the same detections however it was split into pushes and calls.
 * Returns the number of records written to det[0 .. det_cap), in list order and within a stream in emit_hop order, or a
 * status.  hop0_out / n_hops_out (either may be NULL) receive the hops scored per listed stream.  out may be NULL: the
 * scores then stay in device scratch and cross no PCIe; otherwise they are packed and laid out as by ewk_dense_ready, in
 * host or device memory (`where`).  One K4 launch plus one K4D launch (one warp per non-empty row) on the context's
 * stream; only the emitted records and a count per row cross PCIe.  Synchronises with the context's stream.
 * Errors as ewk_dense_ready, and EWK_ERR_ARG for hold_hops < 1, refractory_hops < 0 or det_cap below
 * sum_i ceil(n_hops_i / 2).  Every check comes before the first launch: on any error no cursor, detector state or score
 * moves.  ewk_dense_scores, ewk_dense_scores_streams and ewk_dense_ready neither read nor move the detector; pending
 * pushes and overlap mode behave as for ewk_dense_ready. */
int ewk_dense_detect(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops, int template_first, int template_count,
                     int hold_hops, int refractory_hops, ewk_detection* det, int det_cap,
                     int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap, int where);
/* Per-row template sets: the forms above with a template set of its own for every row, in one call.  Row i is scored
 * against slots [template_first[i], template_first[i] + template_count[i]); with both arrays NULL, row i takes its
 * stream's own range (ewk_stream_params.template_first / template_count, the gate's range).  streams = NULL in the ready
 * and detect forms means every stream, as there (the arrays then have n_streams entries).
 *   Results: every score of row i is bit-identical to what ewk_dense_scores_streams gives for that stream and those hops
 *   with row i's set (NaN where the window starts before the stream); every detection equals what ewk_dense_detect emits
 *   for that stream with that set (template_slot is the absolute slot; within a set the lowest k wins ties).
 *   Packing: rows in list order; row i starts at float sum_{j < i} n_hops[j] T_j and is laid out [n_hops[i]][T_i],
 *   T_i = template_count[i].  n * max_hops * max_i T_i floats always suffice for the ready and detect forms; the
 *   detection bound stays sum_i ceil(n_hops_i / 2).
 *   Cursors and state: ewk_dense_ready_sets reads and moves ewk_dense_ready's cursor, ewk_dense_detect_sets the
 *   detector's cursor and state of ewk_dense_detect, so a stream may switch between the forms, and between sets, from one
 *   call to the next.  ewk_reset_streams and ewk_export_streams / ewk_import_streams treat them as before.
 *   Launches: one K4 launch per distinct launch geometry (ewk_dense_plan of the set alone: hops per sub-chunk, threads,
 *   CTAs per SM; at most 8) among the rows' sets, each row at the geometry its set has alone, plus one K4D launch for
 *   ewk_dense_detect_sets.  The number of launches does not grow with the number of distinct sets.
 *   ewk_dense_last_plan reports the call's last K4 launch.  A set's descriptor is built on its first use and kept on
 *   the device until ewk_set_template, ewk_set_template_features or ewk_clear_template changes a slot of its range, so
 *   a steady-state call uploads only its row descriptors.
 *   Errors, all before the first launch (no cursor, detector state or score moves), naming the row and the stream:
 *   EWK_ERR_ARG for a set of a count outside 1..8 or a range outside [0, max_templates), a template length outside
 *   640..48000, a set that does not fit shared memory alone (ewk_dense_plan refuses it), or only one of the two arrays
 *   given; EWK_ERR_NO_TEMPLATE for an empty slot; otherwise the errors of the single-set form. */
int ewk_dense_scores_sets(ewk_ctx* ctx, const int32_t* streams, int n, const int64_t* hop0, const int32_t* n_hops,
                          const int32_t* template_first, const int32_t* template_count,
                          float* out, int64_t out_cap, int where);
int ewk_dense_ready_sets(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops,
                         const int32_t* template_first, const int32_t* template_count,
                         int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap, int where);
int ewk_dense_detect_sets(ewk_ctx* ctx, const int32_t* streams, int n, int max_hops,
                          const int32_t* template_first, const int32_t* template_count,
                          int hold_hops, int refractory_hops, ewk_detection* det, int det_cap,
                          int64_t* hop0_out, int32_t* n_hops_out, float* out, int64_t out_cap, int where);
/* Launch geometry ewk_dense_scores chooses for templates of these lengths (samples, n <= 8, each 640..48000):
 * out = {hops per sub-chunk (32 or 64), threads per CTA, CTAs per SM, dynamic shared memory bytes}.  Host code only
 * (no context, no device): the function ewk_dense_scores itself plans with.  EWK_ERR_ARG for lengths out of range or a
 * set that does not fit shared memory. */
int ewk_dense_plan(const int64_t* template_lens, int n, int32_t out[4]);
/* The geometry (same layout) the context's latest K4 call (ewk_dense_scores, ewk_dense_scores_streams, ewk_dense_ready)
 * launched; zeros before the first call.  All three plan alike for the same template set. */
int ewk_dense_last_plan(const ewk_ctx* ctx, int32_t out[4]);
/* Copy the dense per-stream results [n_streams] to host memory. */
int ewk_stream_results(ewk_ctx* ctx, ewk_stream_result* out);
/* Device pointer of that array (ewk_stream_result[n_streams]); or make the kernels write into a
 * caller-owned device buffer instead (e.g. a registered NCCL send buffer). */
int ewk_results_device_ptr(ewk_ctx* ctx, void** out);
int ewk_set_results_buffer(ewk_ctx* ctx, void* device_ptr);
/* Peer publication — the multi-GPU "gather" without a collective (SURVEY §8(e); the reference's multiroom shape,
 * examples/multiroom_async.py:14-35, has no exchange at all: N objects report to one host thread).
 * bases[p], p < n_bases <= 16, are device pointers — local, or peer-mapped over NVLink (CUDA IPC / VMM /
 * torch symmetric memory) — to arrays of 2 * stride_records ewk_stream_result.  After this call every ewk_tick ends
 * with the last K3 CTA snapshotting the per-stream records, and a small sender kernel on a side stream of the context
 * (nothing of the next push / gate waits for it) storing the snapshot at
 *     bases[p][parity * stride_records + offset_records + stream]      for every p,
 * where the k-th ewk_tick call after this one (k = 1, 2, ...; ewk_publish_seq returns the latest k) uses
 * parity = (k - 1) & 1 (ewk_publish_parity), so a consumer reads a complete, stable copy of call k while call k + 1
 * is being produced.
 * signals (optional, may be NULL): signals[p] points to uint64_t[2][16] at destination p.  Behind its stores to
 * destination p the sender stores k at signals[p][parity][slot] with release semantics at system scope
 * (a put-with-signal): whoever reads k in slot r of its own copy holds every record rank r published up to call k.
 * bases[slot] / signals[slot] must be this context's own copy (ewk_wait_published / ewk_published_seq read it).
 * Without signals the records are globally visible once the sender of the call has completed on ewk_match_stream()
 * and a cross-GPU barrier enqueued there does the job.  n_bases = 0 switches publication off. */
int ewk_set_results_peers(ewk_ctx* ctx, void* const* bases, int n_bases, int64_t stride_records, int64_t offset_records,
                          void* const* signals, int slot);
int ewk_publish_parity(const ewk_ctx* ctx);
int64_t ewk_publish_seq(const ewk_ctx* ctx);
/* Enqueue, on the context's stream, a wait until slots [0, n_slots) of the local signal row of call `seq` hold a
 * value >= seq — everything enqueued afterwards sees all those ranks' records of that call.  The wait gives up after
 * timeout_ms (it never hangs the device); ewk_published_seq then shows which slot is behind. */
int ewk_wait_published(ewk_ctx* ctx, int n_slots, int64_t seq, int timeout_ms);
/* Synchronous read of the local signal row of `parity`: out[0 .. n_slots).  Returns 1 if an earlier
 * ewk_wait_published timed out since the last call of this function, else 0 (negative: error). */
int ewk_published_seq(ewk_ctx* ctx, int parity, uint64_t* out, int n_slots);
/* The cudaStream_t on which the latest ewk_tick's results become complete: the sender's stream while peer publication is
 * on, else the stream K3 was launched on (the match stream in overlap mode, else the context's stream). */
int ewk_match_stream(ewk_ctx* ctx, void** out);
/* Pinned host memory for asynchronous pushes. */
int ewk_host_alloc(void** out, int64_t bytes);
int ewk_host_free(void* p);
/* Kernel launches issued by this context so far (for bench accounting). */
int64_t ewk_launch_count(const ewk_ctx* ctx);
/* Memory check of the poison test mode.  With EWK_POISON=<byte> (0..255, decimal or 0x..) set when the context is
 * created, every device allocation of the context and every pinned host buffer it owns is filled with the byte before
 * the library initialises it and is followed by a guard band of the byte; per-call workspaces are refilled at every call
 * and allocated at exactly the size the call needs.  ewk_debug_check synchronises the device and reads every guard band
 * back: EWK_OK if none changed, else EWK_ERR_STATE with ewk_last_error naming each damaged buffer and the first damaged
 * byte (damage found when a buffer was freed or regrown is kept and reported here).  EWK_ERR_STATE also when poison mode
 * is off.  Poison mode synchronises the device at every allocation; it is for tests, not for serving. */
int ewk_debug_check(ewk_ctx* ctx);
/* Per-kernel device timing with CUDA events on the context's stream.  ewk_profile(ctx, 1) starts
 * bracketing every kernel launch with an event pair; ewk_profile_read synchronises and returns, per
 * kernel class (0 ring_push, 1 tick_gate, 2 segment_queue, 3 segment_batch (K3 of explicit segments, K6 and K11),
 * 4 dense_score, 5 segment_prepare, 6 publish, 7 resample_push), the summed
 * milliseconds and the number of launches since profiling was enabled, then resets the sums. */
enum { EWK_PROF_CLASSES = 8 };
int ewk_profile(ewk_ctx* ctx, int enable);
int ewk_profile_read(ewk_ctx* ctx, double* ms, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* EWK_H */
