"""ctypes binding of libewk.so (include/ewk.h).  Fails loudly when the CUDA library is missing —
there is no CPU fallback in this package."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libewk.so")

EWK_OK, EWK_ERR_ARG, EWK_ERR_NO_TEMPLATE, EWK_ERR_CUDA, EWK_ERR_STATE, EWK_ERR_NOMEM = 0, -1, -2, -3, -4, -5
PCM_F32, PCM_I16 = 0, 1
IN_ULAW, IN_ALAW = 2, 3          # input formats of ewk_push_resampled beside PCM_F32 / PCM_I16
HOST, DEVICE = 0, 1


class EwkError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("n_streams", C.c_int32), ("ring_samples", C.c_int32), ("slack_samples", C.c_int32),
                ("pcm_format", C.c_int32), ("max_templates", C.c_int32), ("max_events", C.c_int32),
                ("preemphasis", C.c_float), ("n_mfcc", C.c_int32), ("reserved0", C.c_int32), ("reserved1", C.c_int32)]


_lib = None


def _p(t):
    return C.POINTER(t)


def load():
    """dlopen libewk.so (built in-tree by easywakeword_b200.build) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EwkError(f"{LIB_PATH} is missing: build it with `python -m easywakeword_b200.build` "
                       "(nvcc, sm_100a). easywakeword_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32p = C.c_void_p, C.c_int, C.c_int64, _p(C.c_float)
    protos = {
        "ewk_abi_version": (C.c_int, []),
        "ewk_last_error": (C.c_char_p, [vp]),
        "ewk_host_table": (C.c_int, [i32, f32p, i32]),
        "ewk_create": (C.c_int, [i32, _p(Config), _p(vp)]),
        "ewk_destroy": (C.c_int, [vp]),
        "ewk_set_cuda_stream": (C.c_int, [vp, vp]),
        "ewk_synchronize": (C.c_int, [vp]),
        "ewk_extract_mfcc": (C.c_int, [vp, vp, i64, i32, f32p, f32p, f32p, i64]),
        "ewk_set_template": (C.c_int, [vp, i32, f32p, i64]),
        "ewk_set_template_features": (C.c_int, [vp, i32, f32p, f32p, i64]),
        "ewk_get_template": (C.c_int, [vp, i32, f32p, f32p, _p(i64)]),
        "ewk_clear_template": (C.c_int, [vp, i32]),
        "ewk_similarity_batch": (C.c_int, [vp, i32, vp, i32, i32, _p(i64), _p(i64), i32, C.c_float, f32p,
                                           _p(C.c_uint8), f32p]),
        "ewk_analyze_templates": (C.c_int, [vp, f32p, i32, _p(i64), _p(i64), i32, vp, f32p, i64]),
        "ewk_resample_info": (C.c_int, [i32, _p(C.c_int32), _p(C.c_int32), _p(C.c_int32)]),
        "ewk_resample_out_len": (i64, [i64, i32]),
        "ewk_resample": (C.c_int, [vp, vp, i32, i32, i32, i64, i64, i32, i64, i64, i64, vp, i64, i32]),
        "ewk_dense_plan": (C.c_int, [_p(i64), i32, _p(C.c_int32)]),
        "ewk_dense_last_plan": (C.c_int, [vp, _p(C.c_int32)]),
    }
    for name, (res, args) in protos.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    lib._protos = protos
    _lib = lib
    return lib


def f32ptr(a):
    return a.ctypes.data_as(_p(C.c_float))


def i64ptr(a):
    return a.ctypes.data_as(_p(C.c_int64))


def u8ptr(a):
    return a.ctypes.data_as(_p(C.c_uint8))


def host_table(which):
    lib = load()
    n = lib.ewk_host_table(which, None, 0)
    out = np.empty(n, dtype=np.float32)
    lib.ewk_host_table(which, f32ptr(out), n)
    return out


def dense_plan(lens):
    """(DH, threads, CTAs per SM, shared-memory bytes) that ewk_dense_scores launches for templates of these lengths
    (samples).  Host code: needs no GPU."""
    lib = load()
    a = np.ascontiguousarray(lens, dtype=np.int64)
    out = (C.c_int32 * 4)()
    if lib.ewk_dense_plan(i64ptr(a), len(a), out) != EWK_OK:
        raise ValueError(f"no dense plan for template lengths {a.tolist()} (1..8 templates of 640..48000 samples that fit "
                         "shared memory)")
    return tuple(int(v) for v in out)


def check(lib, ctx, rc):
    """Map ewk_status to the reference's exception types (SURVEY §8(b) 'Errors')."""
    if rc == EWK_OK:
        return
    msg = lib.ewk_last_error(ctx).decode("utf-8", "replace")
    if rc in (EWK_ERR_ARG, EWK_ERR_NO_TEMPLATE):
        raise ValueError(msg)
    if rc == EWK_ERR_NOMEM:
        raise MemoryError(msg)
    raise EwkError(f"libewk error {rc}: {msg}")


class Context:
    """Owns one ewk_ctx (one GPU)."""

    def __init__(self, device=0, n_streams=0, ring_samples=160000, slack_samples=16000, pcm_format=PCM_I16,
                 max_templates=4, max_events=0, preemphasis=0.0, n_mfcc=0):
        self.lib = load()
        self.cfg = Config(n_streams, ring_samples, slack_samples, pcm_format, max_templates,
                          max_events or max(1024, 4 * n_streams), float(preemphasis), int(n_mfcc), 0, 0)
        h = C.c_void_p()
        rc = self.lib.ewk_create(device, C.byref(self.cfg), C.byref(h))
        if rc != EWK_OK:
            msg = self.lib.ewk_last_error(None).decode("utf-8", "replace")
            if rc == EWK_ERR_ARG:
                raise ValueError(msg)
            raise EwkError(f"libewk error {rc}: {msg}")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.ewk_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        check(self.lib, self.h, rc)

    # ---- level 2
    def extract_mfcc(self, audio, want_frames=False):
        a = np.ascontiguousarray(audio, dtype=np.float32).reshape(-1)
        mean = np.empty(20, np.float32)
        std = np.empty(20, np.float32)
        frames = None
        if want_frames:
            nf = 1 + len(a) // 160
            frames = np.empty((nf, 20), np.float32)
        self._ck(self.lib.ewk_extract_mfcc(self.h, a.ctypes.data, len(a), HOST, f32ptr(mean), f32ptr(std),
                                           f32ptr(frames) if want_frames else None, 0 if frames is None else len(frames)))
        return (mean, std, frames) if want_frames else (mean, std)

    def set_template(self, slot, audio):
        a = np.ascontiguousarray(audio, dtype=np.float32).reshape(-1)
        self._ck(self.lib.ewk_set_template(self.h, slot, f32ptr(a), len(a)))

    def set_template_features(self, slot, mean, std, n_samples):
        m = np.ascontiguousarray(mean, dtype=np.float32)
        s = np.ascontiguousarray(std, dtype=np.float32)
        self._ck(self.lib.ewk_set_template_features(self.h, slot, f32ptr(m), f32ptr(s), int(n_samples)))

    def get_template(self, slot):
        m = np.empty(20, np.float32)
        s = np.empty(20, np.float32)
        n = C.c_int64()
        self._ck(self.lib.ewk_get_template(self.h, slot, f32ptr(m), f32ptr(s), C.byref(n)))
        return m, s, n.value

    def clear_template(self, slot):
        self._ck(self.lib.ewk_clear_template(self.h, slot))

    def similarity_batch(self, slot, pcm, offsets, lens, threshold=75.0, want_features=False):
        pcm = np.ascontiguousarray(pcm).reshape(-1)
        if pcm.dtype == np.int16:
            fmt = PCM_I16
        else:
            pcm = pcm.astype(np.float32, copy=False)
            fmt = PCM_F32
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        ln = np.ascontiguousarray(lens, dtype=np.int64)
        n = len(off)
        scores = np.empty(n, np.float32)
        matched = np.empty(n, np.uint8)
        feats = np.empty((n, 40), np.float32) if want_features else None
        self._ck(self.lib.ewk_similarity_batch(self.h, slot, pcm.ctypes.data, fmt, HOST, i64ptr(off), i64ptr(ln), n,
                                               float(threshold), f32ptr(scores), u8ptr(matched),
                                               f32ptr(feats) if want_features else None))
        return (scores, matched.astype(bool), feats) if want_features else (scores, matched.astype(bool))

    def analyze_templates(self, audios, want_rms=False):
        """Batched WakeWord._analyze_reference_audio_duration (wakeword.py:872-893) on the device (K6).
        audios: sequence of float32 16 kHz arrays.  -> structured array (VAD_DTYPE), one row per template
        [, list of per-template frame-RMS arrays]."""
        audios = [np.ascontiguousarray(a, dtype=np.float32).reshape(-1) for a in audios]
        n = len(audios)
        out = np.zeros(n, dtype=VAD_DTYPE)
        if n == 0:
            return (out, []) if want_rms else out
        lens = np.array([len(a) for a in audios], np.int64)
        offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
        pcm = np.concatenate(audios) if lens.sum() else np.zeros(1, np.float32)
        frames = 1 + lens // 160
        rms = np.empty(int(frames.sum()), np.float32) if want_rms else None
        self._ck(self.lib.ewk_analyze_templates(self.h, f32ptr(pcm), HOST, i64ptr(offs), i64ptr(lens), n,
                                                out.ctypes.data, f32ptr(rms) if want_rms else None,
                                                len(rms) if want_rms else 0))
        if want_rms:
            cuts = np.cumsum(frames)[:-1]
            return out, np.split(rms, cuts)
        return out

    def resample(self, y, sr_in, *, in_first=0, out_first=0, n_out=None, out_device_ptr=None):
        """K7: y[rows, n] or y[n] (float32 / int16, host) at sr_in -> float32 at 16 kHz (absolute output samples
        [out_first, out_first + n_out); default: the one-shot length ceil(n * 16000 / sr_in)).  A device input is
        (ptr, rows, n, stride) with the dtype given as a 5th element (np.int16 / np.float32)."""
        if isinstance(y, tuple):
            ptr, rows, n, stride, dt = y
            fmt, where_in, one_d = (PCM_I16 if np.dtype(dt) == np.int16 else PCM_F32), DEVICE, False
        else:
            y = np.asarray(y)
            one_d = y.ndim == 1
            y = np.ascontiguousarray(y.reshape(1, -1) if one_d else y)
            if y.dtype != np.int16:
                y = y.astype(np.float32, copy=False)
            fmt, where_in = (PCM_I16 if y.dtype == np.int16 else PCM_F32), HOST
            ptr, rows, n, stride = y.ctypes.data, y.shape[0], y.shape[1], y.shape[1]
        if n_out is None:
            n_out = max(0, int(self.lib.ewk_resample_out_len(n, int(sr_in))) - out_first)
        if out_device_ptr is not None:
            self._ck(self.lib.ewk_resample(self.h, ptr, fmt, where_in, rows, n, stride, int(sr_in), in_first, out_first,
                                           n_out, out_device_ptr, n_out, DEVICE))
            return None
        out = np.empty((rows, n_out), np.float32)
        self._ck(self.lib.ewk_resample(self.h, ptr, fmt, where_in, rows, n, stride, int(sr_in), in_first, out_first,
                                       n_out, out.ctypes.data, n_out, HOST))
        return out[0] if one_d else out

    def set_overlap(self, enable=True):
        """K3 on a second stream so that the next push runs beside it (see include/ewk.h: ewk_set_overlap)."""
        self._ck(self.lib.ewk_set_overlap(self.h, 1 if enable else 0))

    def join(self):
        """Enqueue (no host sync) the wait for an in-flight K3 on the context's stream."""
        self._ck(self.lib.ewk_join(self.h))

    def synchronize(self):
        self._ck(self.lib.ewk_synchronize(self.h))


def resample_info(sr_in):
    """-> (half_width, up, down) of the 16 kHz conversion filter for sr_in, or raises ValueError."""
    w, up, dn = C.c_int32(), C.c_int32(), C.c_int32()
    if load().ewk_resample_info(int(sr_in), C.byref(w), C.byref(up), C.byref(dn)) != 0:
        raise ValueError(f"{sr_in} Hz -> 16000 Hz is not supported")
    return w.value, up.value, dn.value


VAD_DTYPE = np.dtype([("duration_s", "<f8"), ("max_rms", "<f4"), ("threshold", "<f4"), ("first_frame", "<i4"),
                      ("last_frame", "<i4"), ("n_frames", "<i4"), ("voiced", "<i4")])      # ewk_vad_result


# ------------------------------------------------------------------------------------------
# stream bank bindings
class StreamParams(C.Structure):
    _fields_ = [("similarity_threshold", C.c_float), ("frame_size", C.c_int32),
                ("pre_speech_silence", C.c_double), ("speech_duration_min", C.c_double),
                ("speech_duration_max", C.c_double), ("post_speech_silence", C.c_double),
                ("timeout", C.c_double), ("min_threshold", C.c_double),
                ("template_first", C.c_int32), ("template_count", C.c_int32),
                ("live", C.c_int32), ("reserved", C.c_int32)]


class Event(C.Structure):
    _fields_ = [("stream", C.c_int32), ("kind", C.c_int32), ("tick", C.c_int64), ("seg_start", C.c_int64),
                ("seg_len", C.c_int32), ("template_slot", C.c_int32), ("score", C.c_float), ("matched", C.c_int32)]


class StreamStatus(C.Structure):
    _fields_ = [("written", C.c_int64), ("visible", C.c_int64), ("tick", C.c_int64),
                ("silence_threshold", C.c_double), ("last_rms", C.c_double), ("frame_size", C.c_int32),
                ("state", C.c_int32), ("started", C.c_int32), ("is_silent", C.c_int32),
                ("n_timeouts", C.c_int32), ("n_events", C.c_int32)]


EVENT_DTYPE = np.dtype([("stream", "<i4"), ("kind", "<i4"), ("tick", "<i8"), ("seg_start", "<i8"),
                        ("seg_len", "<i4"), ("template_slot", "<i4"), ("score", "<f4"), ("matched", "<i4")])
RESULT_DTYPE = np.dtype([("score", "<f4"), ("flags", "<u4")])
DETECTION_DTYPE = np.dtype([("stream", "<i4"), ("template_slot", "<i4"), ("hop", "<i8"), ("run_start", "<i8"),
                            ("emit_hop", "<i8"), ("seg_start", "<i8"), ("seg_len", "<i4"), ("score", "<f4")])
EV_TIMEOUT, EV_SCORED = 1, 2
# ewk_stream_blob: the 96-byte header at offset 0 of a stream blob (ewk_export_streams); the rest of a blob is opaque
STREAM_BLOB_HEADER_DTYPE = np.dtype([
    ("magic", "<u4"), ("version", "<u4"), ("n_streams", "<i4"), ("ring_samples", "<i4"), ("slack_samples", "<i4"),
    ("pcm_format", "<i4"), ("n_mfcc", "<i4"), ("preemphasis_bits", "<u4"), ("meta_bytes", "<i4"),
    ("n_templates", "<i4"), ("tail_floats", "<i4"), ("reserved", "<i4"), ("ids_offset", "<i8"), ("meta_offset", "<i8"),
    ("template_offset", "<i8"), ("bulk_offset", "<i8"), ("bulk_row_bytes", "<i8"), ("total_bytes", "<i8")])
STREAM_BLOB_MAGIC, STREAM_BLOB_VERSION = 0x534B5745, 1
STREAM_META_BYTES, STREAM_TEMPLATE_BYTES = 304, 176       # per-stream meta record, per-slot template record


def stream_blob_layout(ring_samples, slack_samples, pcm_format, n, n_templates, tail_floats):
    """Section offsets of a version-1 stream blob of n streams (what ewk_export_streams writes and ewk_import_streams
    recomputes): header | int32 ids | meta records | template records | bulk rows, each 16-byte aligned.  A bulk row is
    the raw ring (P = ring + slack rounded up to 64 samples), the block sums (P // 1600 doubles), the chunk mean squares
    (2 * (ring // 160) doubles) and tail_floats K8 input-tail floats.  ewk_stream_blob_bytes is this total with
    n_templates = max_templates and tail_floats = the context's widest K8 tail, rounded up to 4."""
    a16 = lambda v: (v + 15) // 16 * 16                                          # noqa: E731
    P = (ring_samples + slack_samples + 63) // 64 * 64
    esz = 2 if pcm_format == PCM_I16 else 4
    ss_off = P * esz
    ms_off = ss_off + a16(8 * (P // 1600))
    tail_off = ms_off + 16 * max(1, ring_samples // 160)
    row = a16(tail_off + 4 * tail_floats)
    ids = STREAM_BLOB_HEADER_DTYPE.itemsize
    meta = a16(ids + 4 * n)
    tmpl = meta + STREAM_META_BYTES * n
    bulk = tmpl + STREAM_TEMPLATE_BYTES * n_templates
    return dict(ids_offset=ids, meta_offset=meta, template_offset=tmpl, bulk_offset=bulk, bulk_row_bytes=row,
                total_bytes=bulk + row * n, ss_off=ss_off, ms_off=ms_off, tail_off=tail_off)


def _declare_stream_protos(lib):
    vp, i32, i64, f32p = C.c_void_p, C.c_int, C.c_int64, _p(C.c_float)
    protos = {
        "ewk_default_stream_params": (C.c_int, [_p(StreamParams)]),
        "ewk_set_stream_params": (C.c_int, [vp, i32, _p(StreamParams)]),
        "ewk_push": (C.c_int, [vp, i32, i32, vp, i64, i64, i32]),
        "ewk_push_g711": (C.c_int, [vp, i32, i32, vp, i64, i64, i32, i32]),
        "ewk_push_resampled": (C.c_int, [vp, i32, i32, vp, i32, i64, i64, i32, i32]),
        "ewk_push_resampled_each": (C.c_int, [vp, i32, i32, vp, i32, i64, i64, i32, i32, _p(i64)]),
        "ewk_push_streams": (C.c_int, [vp, _p(C.c_int32), i32, vp, i32, _p(i64), _p(i64), i64, i32, i32, _p(i64)]),
        "ewk_tick_ready": (C.c_int, [vp, i32, _p(C.c_int32), vp, vp, vp, vp]),
        "ewk_stream_input": (C.c_int, [vp, i32, _p(C.c_int32), _p(i64)]),
        "ewk_reset_streams": (C.c_int, [vp, _p(C.c_int32), i32]),
        "ewk_stream_blob_bytes": (C.c_int64, [vp, i32]),
        "ewk_export_streams": (C.c_int, [vp, _p(C.c_int32), i32, vp, i64, i32]),
        "ewk_import_streams": (C.c_int, [vp, _p(C.c_int32), i32, vp, i64, i32]),
        "ewk_tick": (C.c_int, [vp, i32]),
        "ewk_set_overlap": (C.c_int, [vp, i32]),
        "ewk_join": (C.c_int, [vp]),
        "ewk_tick_trace": (C.c_int, [vp, i32, vp, vp, vp, vp]),
        "ewk_poll": (C.c_int, [vp, vp, i32, _p(C.c_int)]),
        "ewk_stream_status_get": (C.c_int, [vp, i32, _p(StreamStatus)]),
        "ewk_read_last": (C.c_int, [vp, i32, i64, f32p]),
        "ewk_read_segment": (C.c_int, [vp, i32, i64, i64, f32p]),
        "ewk_stream_results": (C.c_int, [vp, vp]),
        "ewk_dense_scores": (C.c_int, [vp, i64, i32, i32, i32, vp, i32]),
        "ewk_dense_scores_streams": (C.c_int, [vp, _p(C.c_int32), i32, _p(i64), _p(C.c_int32), i32, i32, vp, i64, i32]),
        "ewk_dense_ready": (C.c_int, [vp, _p(C.c_int32), i32, i32, i32, i32, _p(i64), _p(C.c_int32), vp, i64, i32]),
        "ewk_dense_detect": (C.c_int, [vp, _p(C.c_int32), i32, i32, i32, i32, i32, i32, vp, i32, _p(i64), _p(C.c_int32),
                                       vp, i64, i32]),
        "ewk_prepare_segments": (C.c_int, [vp, i32, _p(C.c_int32), _p(i64), _p(i64), _p(i64), f32p, i64, i32]),
        "ewk_results_device_ptr": (C.c_int, [vp, _p(vp)]),
        "ewk_set_results_buffer": (C.c_int, [vp, vp]),
        "ewk_set_results_peers": (C.c_int, [vp, _p(vp), i32, i64, i64, _p(vp), i32]),
        "ewk_publish_parity": (C.c_int, [vp]),
        "ewk_publish_seq": (C.c_int64, [vp]),
        "ewk_wait_published": (C.c_int, [vp, i32, i64, i32]),
        "ewk_published_seq": (C.c_int, [vp, i32, _p(C.c_uint64), i32]),
        "ewk_match_stream": (C.c_int, [vp, _p(vp)]),
        "ewk_host_alloc": (C.c_int, [_p(vp), i64]),
        "ewk_host_free": (C.c_int, [vp]),
        "ewk_launch_count": (C.c_int64, [vp]),
        "ewk_profile": (C.c_int, [vp, i32]),
        "ewk_profile_read": (C.c_int, [vp, _p(C.c_double), _p(C.c_int64)]),
    }
    for name, (res, args) in protos.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    lib._protos.update(protos)


_orig_load = load


def load():  # noqa: F811  (extends the loader above with the stream-bank prototypes)
    lib = _orig_load()
    if "ewk_push" not in lib._protos:
        _declare_stream_protos(lib)
    return lib


def default_stream_params(**over):
    lib = load()
    p = StreamParams()
    lib.ewk_default_stream_params(C.byref(p))
    for k, v in over.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown stream parameter {k!r}")
        setattr(p, k, v)
    return p


class PinnedArray:
    """numpy view over cudaHostAlloc memory (asynchronous H2D pushes)."""

    def __init__(self, shape, dtype):
        lib = load()
        self.lib = lib
        dt = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dt.itemsize
        ptr = C.c_void_p()
        rc = lib.ewk_host_alloc(C.byref(ptr), max(1, nbytes))
        if rc != EWK_OK:
            raise MemoryError("cudaHostAlloc failed")
        self.ptr = ptr
        buf = (C.c_char * nbytes).from_address(ptr.value)
        self.array = np.frombuffer(buf, dtype=dt).reshape(shape)

    def free(self):
        if getattr(self, "ptr", None):
            self.array = None
            self.lib.ewk_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _resampled_input(pcm_or_codes, fmt):
    """(ptr, n_streams, n, stride, in_format) of a native-rate feed: an array [n_streams, n] (float32, int16, or uint8
    G.711 codes with fmt "ulaw" / "alaw") or a device input (ptr, n_streams, n, stride, dtype), and the array behind
    ptr, which the caller keeps alive across the call."""
    a = None
    if isinstance(pcm_or_codes, tuple):
        ptr, ns, n, stride, dt = pcm_or_codes
        dt = np.dtype(dt)
    else:
        a = pcm_or_codes if pcm_or_codes.ndim == 2 else pcm_or_codes.reshape(1, -1)
        if a.strides[1] != a.itemsize:
            a = np.ascontiguousarray(a)
        ns, n = a.shape
        stride = a.strides[0] // a.itemsize if ns > 1 else n
        ptr, dt = a.ctypes.data, a.dtype
    if dt == np.uint8:
        if fmt not in ("ulaw", "alaw"):
            raise ValueError('uint8 input is G.711: fmt must be "ulaw" or "alaw"')
        code = IN_ULAW if fmt == "ulaw" else IN_ALAW
    elif fmt is not None:
        raise ValueError("fmt selects G.711 for uint8 input only")
    elif dt == np.int16:
        code = PCM_I16
    elif dt == np.float32:
        code = PCM_F32
    else:
        raise TypeError(f"push_resampled takes float32, int16 or uint8 G.711 input, got {dt}")
    return ptr, ns, n, stride, code, a


def _stream_list(streams):
    """int32 array of stream indices (ValueError for values no int32 holds: the library names the others)."""
    st = np.asarray(streams, dtype=np.int64).reshape(-1)
    if st.size and (st.min() < -2**31 or st.max() >= 2**31):
        raise ValueError("stream index out of range")
    return np.ascontiguousarray(st, dtype=np.int32)


def _unpack_rows(out, n_hops, T):
    """Packed [sum n_i][T] scores -> list of [n_i, T] views, in list order."""
    ends = np.cumsum(n_hops, dtype=np.int64)
    return [out[(e - n) * T:e * T].reshape(n, T) for e, n in zip(ends.tolist(), [int(v) for v in n_hops])]


def _bank_methods():
    def set_stream_params(self, stream=-1, params=None, **over):
        p = params if params is not None else default_stream_params(**over)
        self._ck(self.lib.ewk_set_stream_params(self.h, stream, C.byref(p)))

    def push(self, pcm, stream0=0, where=HOST):
        """pcm: [n_streams, n] array in the ring's dtype (rows may be strided), or (ptr, n_streams, n, stride)."""
        if isinstance(pcm, tuple):
            ptr, ns, n, stride = pcm
        else:
            want = np.int16 if self.cfg.pcm_format == PCM_I16 else np.float32
            a = pcm if pcm.ndim == 2 else pcm.reshape(1, -1)
            if a.dtype != want:
                raise TypeError(f"push expects {np.dtype(want)} PCM for this context, got {a.dtype}")
            if a.strides[1] != a.itemsize:
                a = np.ascontiguousarray(a)
            ns, n = a.shape
            stride = a.strides[0] // a.itemsize if ns > 1 else n
            ptr = a.ctypes.data
        self._ck(self.lib.ewk_push(self.h, stream0, ns, ptr, n, stride, where))

    def push_g711(self, codes, stream0=0, where=HOST, law="ulaw"):
        """codes: uint8 [n_streams, n] G.711 mu-law ("ulaw") / A-law ("alaw") codes, or (ptr, n_streams, n, stride):
        expanded to 16-bit samples on the device and pushed like PCM16 (int16 rings only)."""
        if law not in ("ulaw", "alaw"):
            raise ValueError("law must be 'ulaw' or 'alaw'")
        if isinstance(codes, tuple):
            ptr, ns, n, stride = codes
        else:
            a = codes if codes.ndim == 2 else codes.reshape(1, -1)
            if a.dtype != np.uint8:
                raise TypeError(f"push_g711 expects uint8 codes, got {a.dtype}")
            if a.strides[1] != 1:
                a = np.ascontiguousarray(a)
            ns, n = a.shape
            stride = a.strides[0] if ns > 1 else n
            ptr = a.ctypes.data
        self._ck(self.lib.ewk_push_g711(self.h, stream0, ns, ptr, n, stride, where, 1 if law == "alaw" else 0))

    def push_resampled(self, pcm_or_codes, sr_in, stream0=0, where=HOST, fmt=None):
        """A native-rate feed [n_streams, n] at sr_in Hz, converted to 16 kHz on the device and landed in the rings (K8;
        include/ewk.h: ewk_push_resampled).  The input format follows the dtype: float32, int16, or uint8 G.711 codes with
        fmt="ulaw" / "alaw" (into either ring format).  A device input is (ptr, n_streams, n, stride, dtype).
        Returns the number of 16 kHz samples landed per stream."""
        ptr, ns, n, stride, code, _keep = _resampled_input(pcm_or_codes, fmt)
        rc = self.lib.ewk_push_resampled(self.h, stream0, ns, ptr, code, n, stride, where, int(sr_in))
        if rc < 0:
            self._ck(rc)
        return rc

    def push_resampled_each(self, pcm_or_codes, sr_in, stream0=0, where=HOST, fmt=None):
        """push_resampled for streams at their own input positions (recycled streams restart at 0), in one launch
        (include/ewk.h: ewk_push_resampled_each).  Returns int64 [n_streams]: the 16 kHz samples landed per stream."""
        ptr, ns, n, stride, code, _keep = _resampled_input(pcm_or_codes, fmt)
        landed = np.zeros(ns, np.int64)
        self._ck(self.lib.ewk_push_resampled_each(self.h, stream0, ns, ptr, code, n, stride, where, int(sr_in),
                                                  landed.ctypes.data_as(_p(C.c_int64))))
        return landed

    def push_streams(self, streams, rows, sr_in=16000, fmt=None, where=HOST):
        """Ragged push (include/ewk.h: ewk_push_streams): rows[i], a 1-D array of any length (0 included), goes to stream
        streams[i]; the rows are packed into one buffer that crosses PCIe in one copy.  The format follows the dtype as in
        push_resampled (uint8: G.711 with fmt "ulaw" / "alaw"); at sr_in = 16000 it must be the rings' dtype or G.711 into
        int16 rings.  A device input is (ptr, offsets, lens, in_len, dtype).  Returns int64 [len(streams)]: the 16 kHz
        samples landed per row."""
        st = np.asarray(streams, dtype=np.int64).reshape(-1)
        if st.size and (st.min() < -2**31 or st.max() >= 2**31):
            raise ValueError("stream index out of range")
        st = np.ascontiguousarray(st, dtype=np.int32)
        if isinstance(rows, tuple):
            ptr, off, ln, in_len, dt = rows
            off = np.ascontiguousarray(off, dtype=np.int64)
            ln = np.ascontiguousarray(ln, dtype=np.int64)
            dt = np.dtype(dt)
            buf = None
        else:
            rows = [np.asarray(r) for r in rows]
            if len(rows) != len(st):
                raise ValueError("one row per stream")
            dts = {r.dtype for r in rows}
            if len(dts) > 1:
                raise TypeError(f"rows of one call share a dtype, got {sorted(map(str, dts))}")
            dt = dts.pop() if dts else np.dtype(np.uint8 if fmt is not None else
                                                np.int16 if self.cfg.pcm_format == PCM_I16 else np.float32)
            ln = np.array([r.size for r in rows], np.int64)
            off = np.zeros(len(rows), np.int64)
            if len(rows) > 1:
                off[1:] = np.cumsum(ln)[:-1]
            buf = np.concatenate([r.reshape(-1) for r in rows]) if rows else np.zeros(0, dt)
            ptr, in_len = (buf.ctypes.data if buf.size else None), int(buf.size)
        if len(off) != len(st) or len(ln) != len(st):
            raise ValueError("one offset and one length per stream")
        _, _, _, _, code, _keep = _resampled_input((0, 1, 0, 0, dt), fmt)
        landed = np.zeros(len(st), np.int64)
        self._ck(self.lib.ewk_push_streams(self.h, st.ctypes.data_as(_p(C.c_int32)), len(st), ptr, code, i64ptr(off),
                                           i64ptr(ln), int(in_len), where, int(sr_in), i64ptr(landed)))
        return landed

    def tick_ready(self, max_ticks, trace=False):
        """Ticks paced by each stream's own landed audio (include/ewk.h: ewk_tick_ready): stream s takes
        min(max_ticks, written_s // 1600 - tick_s) ticks (resample.due_ticks).  Returns taken (int32 [n_streams]), and
        with trace=True also the trace dict of tick(trace=True) over [n_streams, max_ticks] (cells of ticks not taken:
        state 255, thr / rms NaN; "silent" is then the raw uint8 with 255)."""
        ns = self.cfg.n_streams
        taken = np.zeros(ns, np.int32)
        tp = taken.ctypes.data_as(_p(C.c_int32))
        if not trace:
            self._ck(self.lib.ewk_tick_ready(self.h, int(max_ticks), tp, None, None, None, None))
            return taken
        silent = np.empty((ns, max_ticks), np.uint8)
        state = np.empty((ns, max_ticks), np.uint8)
        thr = np.empty((ns, max_ticks), np.float64)
        rms = np.empty((ns, max_ticks), np.float64)
        self._ck(self.lib.ewk_tick_ready(self.h, int(max_ticks), tp, silent.ctypes.data, state.ctypes.data,
                                         thr.ctypes.data, rms.ctypes.data))
        return taken, {"silent": silent, "state": state, "thr": thr, "rms": rms}

    def reset_streams(self, streams):
        """Return the listed streams to the state of a new context (include/ewk.h: ewk_reset_streams); their parameters
        stay.  The event queue must be empty (poll first)."""
        lst = np.ascontiguousarray(np.asarray(streams, dtype=np.int64).reshape(-1))
        if lst.size and (lst.min() < -2**31 or lst.max() >= 2**31):
            raise ValueError("stream index out of range")
        lst = lst.astype(np.int32)
        self._ck(self.lib.ewk_reset_streams(self.h, lst.ctypes.data_as(_p(C.c_int32)), int(lst.size)))

    def stream_blob_bytes(self, n):
        """Bytes that always hold a blob of n of this context's streams (include/ewk.h: ewk_stream_blob_bytes), for the
        input rates the context has seen so far."""
        v = int(self.lib.ewk_stream_blob_bytes(self.h, int(n)))
        if v < 0:
            self._ck(v)
        return v

    def export_streams(self, streams, where=HOST, out=None):
        """Snapshot the listed streams into a blob (include/ewk.h: ewk_export_streams); the streams go on untouched.
        where=HOST returns the blob as a np.uint8 array of its exact length (save it with np.save).  where=DEVICE writes
        it into out = (ptr, cap), 16-byte aligned memory of this context's device, and returns None: the blob's length is
        its header's total_bytes, and import_streams takes (ptr, cap) as it is."""
        st = _stream_list(streams)
        sp = st.ctypes.data_as(_p(C.c_int32))
        if where == DEVICE:
            if out is None:
                raise ValueError("a device export takes out=(ptr, cap)")
            ptr, cap = out
            self._ck(self.lib.ewk_export_streams(self.h, sp, len(st), C.c_void_p(int(ptr)), int(cap), DEVICE))
            return None
        if out is not None:
            raise ValueError("out is for where=DEVICE; a host export returns its array")
        cap = self.stream_blob_bytes(len(st))
        buf = np.zeros(cap, np.uint8)
        self._ck(self.lib.ewk_export_streams(self.h, sp, len(st), buf.ctypes.data, cap, HOST))
        n = int(buf[:STREAM_BLOB_HEADER_DTYPE.itemsize].view(STREAM_BLOB_HEADER_DTYPE)[0]["total_bytes"])
        return buf[:n]

    def import_streams(self, streams, blob, where=HOST):
        """Make blob stream i stream streams[i] of this context (include/ewk.h: ewk_import_streams).  blob: a host
        np.uint8 array (any exported blob, e.g. np.load of a saved one), or with where=DEVICE (ptr, length) in this
        context's device memory.  The event queue must be empty (poll first)."""
        st = _stream_list(streams)
        sp = st.ctypes.data_as(_p(C.c_int32))
        if where == DEVICE:
            ptr, length = blob
            self._ck(self.lib.ewk_import_streams(self.h, sp, len(st), C.c_void_p(int(ptr)), int(length), DEVICE))
            return
        b = np.ascontiguousarray(blob).view(np.uint8).reshape(-1)
        self._ck(self.lib.ewk_import_streams(self.h, sp, len(st), b.ctypes.data if b.size else None, int(b.size), HOST))

    def stream_input(self, stream):
        """-> (input rate latched by the stream's first push (0: none yet), input samples received)."""
        sr, n = C.c_int32(), C.c_int64()
        self._ck(self.lib.ewk_stream_input(self.h, int(stream), C.byref(sr), C.byref(n)))
        return sr.value, n.value

    def tick(self, n_ticks=1, trace=False):
        if not trace:
            self._ck(self.lib.ewk_tick(self.h, n_ticks))
            return None
        ns = self.cfg.n_streams
        silent = np.empty((ns, n_ticks), np.uint8)
        state = np.empty((ns, n_ticks), np.uint8)
        thr = np.empty((ns, n_ticks), np.float64)
        rms = np.empty((ns, n_ticks), np.float64)
        self._ck(self.lib.ewk_tick_trace(self.h, n_ticks, silent.ctypes.data, state.ctypes.data, thr.ctypes.data,
                                         rms.ctypes.data))
        return {"silent": silent.astype(bool), "state": state, "thr": thr, "rms": rms}

    def poll(self):
        cap = self.cfg.max_events
        out = np.zeros(cap, dtype=EVENT_DTYPE)
        dropped = C.c_int()
        n = self.lib.ewk_poll(self.h, out.ctypes.data, cap, C.byref(dropped))
        if n < 0:
            self._ck(n)
        self.dropped = dropped.value
        return out[:n]

    def status(self, stream):
        st = StreamStatus()
        self._ck(self.lib.ewk_stream_status_get(self.h, stream, C.byref(st)))
        return st

    def read_last(self, stream, n_samples):
        out = np.empty(int(n_samples), np.float32)
        if n_samples:
            self._ck(self.lib.ewk_read_last(self.h, stream, int(n_samples), f32ptr(out)))
        return out

    def read_segment(self, stream, seg_start, seg_len):
        out = np.empty(int(seg_len), np.float32)
        self._ck(self.lib.ewk_read_segment(self.h, stream, int(seg_start), int(seg_len), f32ptr(out)))
        return out

    def dense_scores(self, hop0, n_hops, template_first=0, template_count=1, out_device_ptr=None):
        """[n_streams, n_hops, template_count] float32 scores for hops [hop0, hop0 + n_hops)."""
        if out_device_ptr is not None:
            self._ck(self.lib.ewk_dense_scores(self.h, int(hop0), int(n_hops), template_first, template_count,
                                               C.c_void_p(out_device_ptr), DEVICE))
            return None
        out = np.empty((self.cfg.n_streams, int(n_hops), template_count), np.float32)
        self._ck(self.lib.ewk_dense_scores(self.h, int(hop0), int(n_hops), template_first, template_count,
                                           out.ctypes.data, HOST))
        return out

    def dense_scores_streams(self, streams, hop0, n_hops, template_first=0, template_count=1, out_device_ptr=None,
                             out_cap=None):
        """Ragged dense scoring (include/ewk.h: ewk_dense_scores_streams): row i scores stream streams[i] at hops
        [hop0[i], hop0[i] + n_hops[i]) (0 included).  Returns a list of float32 [n_hops[i], template_count] arrays; with
        out_device_ptr the rows go there packed back to back in list order (out_cap floats, default exactly what they
        need) and None is returned."""
        st = _stream_list(streams)
        h0 = np.ascontiguousarray(np.asarray(hop0, dtype=np.int64).reshape(-1))
        nh64 = np.asarray(n_hops, dtype=np.int64).reshape(-1)
        if len(h0) != len(st) or len(nh64) != len(st):
            raise ValueError("one hop0 and one n_hops per stream")
        if nh64.size and (nh64.min() < -2**31 or nh64.max() >= 2**31):
            raise ValueError("n_hops out of range")
        nh = np.ascontiguousarray(nh64, dtype=np.int32)
        T = int(template_count)
        need = max(0, int(nh64[nh64 > 0].sum()) * T)
        args = (st.ctypes.data_as(_p(C.c_int32)), len(st), i64ptr(h0), nh.ctypes.data_as(_p(C.c_int32)), template_first, T)
        if out_device_ptr is not None:
            self._ck(self.lib.ewk_dense_scores_streams(self.h, *args, C.c_void_p(out_device_ptr),
                                                       need if out_cap is None else int(out_cap), DEVICE))
            return None
        out = np.empty(need, np.float32)
        self._ck(self.lib.ewk_dense_scores_streams(self.h, *args, out.ctypes.data if need else None,
                                                   need if out_cap is None else int(out_cap), HOST))
        return _unpack_rows(out, nh64, T)

    def dense_ready(self, streams=None, max_hops=100, template_first=0, template_count=1, out_device_ptr=None,
                    out_cap=None):
        """Dense scores paced by each stream's own audio (include/ewk.h: ewk_dense_ready): each listed stream (None: every
        stream) is scored from its cursor at every hop its landed audio completes, at most max_hops, and its cursor moves
        on.  Returns (hop0, scores): int64 [n] first hops and a list of float32 [n_i, template_count] arrays.  With
        out_device_ptr (out_cap floats, default n * max_hops * template_count) the rows go there packed in list order and
        (hop0, n_hops) is returned."""
        st = None if streams is None else _stream_list(streams)
        n = self.cfg.n_streams if st is None else len(st)
        T = int(template_count)
        h0 = np.zeros(n, np.int64)
        nh = np.zeros(n, np.int32)
        cap = n * int(max_hops) * T if out_cap is None else int(out_cap)
        args = (None if st is None else st.ctypes.data_as(_p(C.c_int32)), n, int(max_hops), template_first, T, i64ptr(h0),
                nh.ctypes.data_as(_p(C.c_int32)))
        if out_device_ptr is not None:
            self._ck(self.lib.ewk_dense_ready(self.h, *args, C.c_void_p(out_device_ptr), cap, DEVICE))
            return h0, nh
        out = np.empty(max(0, cap), np.float32)
        self._ck(self.lib.ewk_dense_ready(self.h, *args, out.ctypes.data if out.size else None, cap, HOST))
        return h0, _unpack_rows(out, nh, T)

    def dense_detect(self, streams=None, max_hops=100, template_first=0, template_count=1, hold_hops=20,
                     refractory_hops=50, scores=False, out_device_ptr=None, det_cap=None, out_cap=None, hops=False):
        """Detections from per-hop scores on the device (include/ewk.h: ewk_dense_detect): each listed stream (None: every
        stream) is scored from the detector's own cursor at every hop its landed audio completes, at most max_hops, and
        those hops go through the stream's peak picker (threshold: its similarity_threshold).  Returns a DETECTION_DTYPE
        array in list order, then emit_hop order.  det holds n * ceil(max_hops / 2) records unless det_cap is given.
        scores=True also returns (hop0, list of float32 [n_i, template_count] arrays); with out_device_ptr the scores go
        there packed in list order (out_cap floats, default n * max_hops * template_count) and (hop0, n_hops) is returned
        with the detections.  Otherwise the scores stay on the device; hops=True then returns (hop0, n_hops) with them."""
        st = None if streams is None else _stream_list(streams)
        n = self.cfg.n_streams if st is None else len(st)
        T = int(template_count)
        cap = n * ((min(int(max_hops), 1 << 20) + 1) // 2) if det_cap is None else int(det_cap)
        det = np.empty(max(0, cap), DETECTION_DTYPE)
        h0 = np.zeros(n, np.int64)
        nh = np.zeros(n, np.int32)
        ocap = n * int(max_hops) * T if out_cap is None else int(out_cap)
        buf = None
        if out_device_ptr is not None:
            out, where = C.c_void_p(out_device_ptr), DEVICE
        elif scores:
            buf = np.empty(max(0, ocap), np.float32)
            out, where = (buf.ctypes.data if buf.size else None), HOST
        else:
            out, ocap, where = None, 0, HOST
        rc = self.lib.ewk_dense_detect(self.h, None if st is None else st.ctypes.data_as(_p(C.c_int32)), n, int(max_hops),
                                       int(template_first), T, int(hold_hops), int(refractory_hops),
                                       det.ctypes.data if det.size else None, cap, i64ptr(h0),
                                       nh.ctypes.data_as(_p(C.c_int32)), out, ocap, where)
        if rc < 0:
            self._ck(rc)
        d = det[:rc].copy()
        if out_device_ptr is not None:
            return d, (h0, nh)
        if scores:
            return d, (h0, _unpack_rows(buf, nh, T))
        return (d, (h0, nh)) if hops else d

    def dense_last_plan(self):
        """(DH, threads, CTAs per SM, shared-memory bytes) of the latest K4 launch (dense_scores, dense_scores_streams or
        dense_ready; zeros before the first)."""
        out = (C.c_int32 * 4)()
        self._ck(self.lib.ewk_dense_last_plan(self.h, out))
        return tuple(int(v) for v in out)

    def prepare_segments(self, streams, starts, lens):
        """Level-3 pre-processing (wakeword.py:1020-1025) of many ring segments at once -> list of float32 arrays."""
        st = np.ascontiguousarray(streams, dtype=np.int32)
        a = np.ascontiguousarray(starts, dtype=np.int64)
        ln = np.ascontiguousarray(lens, dtype=np.int64)
        if len(st) == 0:
            return []
        off = np.concatenate([[0], np.cumsum(ln)[:-1]]).astype(np.int64)
        out = np.empty(int(ln.sum()), np.float32)
        self._ck(self.lib.ewk_prepare_segments(self.h, len(st), st.ctypes.data_as(_p(C.c_int32)), i64ptr(a), i64ptr(ln),
                                               i64ptr(off), f32ptr(out), len(out), HOST))
        return [out[o:o + n] for o, n in zip(off, ln)]

    def results(self):
        out = np.empty(self.cfg.n_streams, dtype=RESULT_DTYPE)
        self._ck(self.lib.ewk_stream_results(self.h, out.ctypes.data))
        return out

    def results_device_ptr(self):
        p = C.c_void_p()
        self._ck(self.lib.ewk_results_device_ptr(self.h, C.byref(p)))
        return p.value

    def set_results_buffer(self, device_ptr):
        self._ck(self.lib.ewk_set_results_buffer(self.h, C.c_void_p(device_ptr)))

    def set_results_peers(self, bases, stride_records=0, offset_records=0, signals=None, slot=0):
        """Peer publication: K2 / K3 also store every result record at bases[p][parity * stride + offset + stream]
        (device pointers, local or NVLink peer-mapped); `signals[p]` (uint64 [2][16] per destination) additionally get
        the call's sequence number in `slot` when K3 is done.  An empty list switches it off."""
        bases = list(bases)
        arr = (C.c_void_p * max(1, len(bases)))(*[C.c_void_p(int(b)) for b in bases])
        sig = None
        if signals is not None:
            signals = list(signals)
            if len(signals) != len(bases):
                raise ValueError("one signal row per destination")
            sig = (C.c_void_p * max(1, len(signals)))(*[C.c_void_p(int(b)) for b in signals])
        self._ck(self.lib.ewk_set_results_peers(self.h, arr, len(bases), int(stride_records), int(offset_records), sig, int(slot)))

    def publish_parity(self):
        return int(self.lib.ewk_publish_parity(self.h))

    def publish_seq(self):
        return int(self.lib.ewk_publish_seq(self.h))

    def wait_published(self, n_slots, seq, timeout_ms=2000):
        """Enqueue (context's stream) a bounded device-side wait for the records of call `seq` from slots [0, n_slots)."""
        self._ck(self.lib.ewk_wait_published(self.h, int(n_slots), int(seq), int(timeout_ms)))

    def published_seq(self, parity, n_slots):
        """-> (uint64 [n_slots] sequence numbers in this context's own signal row, timed_out flag)."""
        out = np.zeros(n_slots, np.uint64)
        rc = self.lib.ewk_published_seq(self.h, int(parity), out.ctypes.data_as(_p(C.c_uint64)), int(n_slots))
        if rc < 0:
            self._ck(rc)
        return out, bool(rc)

    def match_stream(self):
        """cudaStream_t (as int) the latest tick launched K3 on."""
        p = C.c_void_p()
        self._ck(self.lib.ewk_match_stream(self.h, C.byref(p)))
        return p.value or 0

    def set_cuda_stream(self, handle):
        self._ck(self.lib.ewk_set_cuda_stream(self.h, C.c_void_p(handle)))

    def launch_count(self):
        return int(self.lib.ewk_launch_count(self.h))

    def profile(self, enable=True):
        self._ck(self.lib.ewk_profile(self.h, 1 if enable else 0))

    def profile_read(self):
        ms = (C.c_double * 8)()
        n = (C.c_int64 * 8)()
        self._ck(self.lib.ewk_profile_read(self.h, ms, n))
        names = ["ring_push", "tick_gate", "segment_queue", "segment_batch", "dense_score", "segment_prepare", "publish",
                 "resample_push"]
        return {names[i]: {"ms": ms[i], "launches": int(n[i])} for i in range(len(names))}

    for f in (prepare_segments, dense_scores, dense_scores_streams, dense_ready, dense_detect, dense_last_plan, profile, profile_read, set_stream_params, push, push_g711, push_resampled,
              push_resampled_each, push_streams, tick_ready, reset_streams, stream_blob_bytes, export_streams, import_streams, stream_input, tick, poll, status, read_last, read_segment, results, results_device_ptr,
              set_results_buffer, set_results_peers, publish_parity, publish_seq, wait_published, published_seq, match_stream, set_cuda_stream, launch_count):
        setattr(Context, f.__name__, f)


_bank_methods()
