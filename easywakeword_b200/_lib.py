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
                ("preemphasis", C.c_float), ("n_mfcc", C.c_int32), ("template_frames", C.c_int32), ("reserved1", C.c_int32)]


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
        "ewk_set_templates": (C.c_int, [vp, _p(C.c_int32), i32, vp, i32, _p(i64), _p(i64), vp]),
        "ewk_resample_info": (C.c_int, [i32, _p(C.c_int32), _p(C.c_int32), _p(C.c_int32)]),
        "ewk_resample_out_len": (i64, [i64, i32]),
        "ewk_resample": (C.c_int, [vp, vp, i32, i32, i32, i64, i64, i32, i64, i64, i64, vp, i64, i32]),
        "ewk_dense_plan": (C.c_int, [_p(i64), i32, _p(C.c_int32)]),
        "ewk_dense_last_plan": (C.c_int, [vp, _p(C.c_int32)]),
        "ewk_get_template_frames": (C.c_int, [vp, i32, f32p, i64, _p(C.c_int32)]),
        "ewk_align_segments": (C.c_int, [vp, i32, _p(C.c_int32), _p(i64), _p(i64), _p(C.c_int32), _p(C.c_int32), f32p, i64,
                                         _p(C.c_int32), f32p, i32]),
        "ewk_align_buffers": (C.c_int, [vp, i32, vp, i32, i32, _p(i64), _p(i64), _p(C.c_int32), _p(C.c_int32), f32p, i64,
                                        _p(C.c_int32), f32p, i32]),
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
                 max_templates=4, max_events=0, preemphasis=0.0, n_mfcc=0, template_frames=False):
        """template_frames=True keeps every template slot's MFCC frames for frame alignment (align_segments /
        align_buffers): 24 KB of device memory per slot."""
        self.lib = load()
        self.cfg = Config(n_streams, ring_samples, slack_samples, pcm_format, max_templates,
                          max_events or max(1024, 4 * n_streams), float(preemphasis), int(n_mfcc),
                          1 if template_frames else 0, 0)
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

    def set_templates(self, slots, audios, want_vad=False):
        """Batched enrolment (include/ewk.h: ewk_set_templates): template slots[i] <- audios[i], each slot bit-identical
        to set_template(slots[i], audios[i]), in one K3 launch.  audios: a sequence of float32 16 kHz arrays, or a
        device input (ptr, offsets, lens): template i is the float32 device samples ptr[offsets[i] : offsets[i] +
        lens[i]].  want_vad: also return analyze_templates of the same audio (VAD_DTYPE [n])."""
        sl = _int32_list(slots, "template slot")
        if isinstance(audios, tuple):
            ptr, offs, lens = audios
            offs = np.ascontiguousarray(np.asarray(offs, dtype=np.int64).reshape(-1))
            lens = np.ascontiguousarray(np.asarray(lens, dtype=np.int64).reshape(-1))
            pcm, where = C.c_void_p(ptr), DEVICE
        else:
            audios = [np.ascontiguousarray(a, dtype=np.float32).reshape(-1) for a in audios]
            lens = np.array([len(a) for a in audios], np.int64)
            offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64) if len(lens) else lens
            host = np.concatenate(audios) if lens.sum() else np.zeros(1, np.float32)
            pcm, where = host.ctypes.data, HOST
        if len(offs) != len(sl) or len(lens) != len(sl):
            raise ValueError("one audio per template slot")
        vad = np.zeros(len(sl), dtype=VAD_DTYPE) if want_vad else None
        self._ck(self.lib.ewk_set_templates(self.h, sl.ctypes.data_as(_p(C.c_int32)), len(sl), pcm, where, i64ptr(offs),
                                            i64ptr(lens), vad.ctypes.data if want_vad else None))
        return vad

    def template_frames(self, slot):
        """The frames stored for a template slot (include/ewk.h: ewk_get_template_frames): float32 [n_frames, 20],
        bit-identical to extract_mfcc(audio, want_frames=True)[2]; 0 rows for a slot without frames (features only,
        cleared, or over 48 000 samples).  Needs Context(template_frames=True)."""
        nf = C.c_int32()
        self._ck(self.lib.ewk_get_template_frames(self.h, int(slot), None, 0, C.byref(nf)))
        out = np.empty((nf.value, 20), np.float32)
        if nf.value:
            self._ck(self.lib.ewk_get_template_frames(self.h, int(slot), f32ptr(out), nf.value, C.byref(nf)))
        return out

    def _align(self, fn, n, head, template_first, template_count, T, out_device_ptrs, dist_cap):
        """Shared tail of align_segments / align_buffers: the set arrays, outputs and unpacking."""
        need = int(T.sum())
        if out_device_ptrs is not None:
            d, bs, bd = out_device_ptrs
            self._ck(fn(self.h, n, *head, template_first, template_count, C.cast(C.c_void_p(d), _p(C.c_float)),
                        need if dist_cap is None else int(dist_cap),
                        None if bs is None else C.cast(C.c_void_p(bs), _p(C.c_int32)),
                        None if bd is None else C.cast(C.c_void_p(bd), _p(C.c_float)), DEVICE))
            return None
        dist = np.empty(max(1, need), np.float32)
        best_slot = np.empty(n, np.int32)
        best_dist = np.empty(n, np.float32)
        self._ck(fn(self.h, n, *head, template_first, template_count, f32ptr(dist), need if dist_cap is None else int(dist_cap),
                    best_slot.ctypes.data_as(_p(C.c_int32)), f32ptr(best_dist), HOST))
        off, _ = sets_offsets(np.ones(n, np.int64), T)
        return [dist[o:o + int(t)] for o, t in zip(off.tolist(), T)], best_slot, best_dist

    def align_buffers(self, pcm, offsets, lens, template_first, template_count, out_device_ptrs=None, dist_cap=None):
        """Frame-alignment distances of caller audio (include/ewk.h: ewk_align_buffers): row i is pcm[offsets[i] :
        offsets[i] + lens[i]] (float32 or int16, host) against slots [template_first[i], template_first[i] +
        template_count[i]) (scalars broadcast).  Returns (list of float32 [T_i] distances, best_slot int32 [n], best_dist
        float32 [n]); with out_device_ptrs = (dist, best_slot or None, best_dist or None) device pointers the outputs go
        there packed and None is returned."""
        pcm = np.ascontiguousarray(pcm).reshape(-1)
        if pcm.dtype == np.int16:
            fmt = PCM_I16
        else:
            pcm = pcm.astype(np.float32, copy=False)
            fmt = PCM_F32
        off = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1))
        ln = np.ascontiguousarray(np.asarray(lens, dtype=np.int64).reshape(-1))
        n = len(off)
        if len(ln) != n:
            raise ValueError("one offset and one length per row")
        tf = _int32_list(np.broadcast_to(np.asarray(template_first, np.int64), (n,)), "template_first")
        tc = _int32_list(np.broadcast_to(np.asarray(template_count, np.int64), (n,)), "template_count")
        return self._align(self.lib.ewk_align_buffers, n, (pcm.ctypes.data, fmt, HOST, i64ptr(off), i64ptr(ln)),
                           tf.ctypes.data_as(_p(C.c_int32)), tc.ctypes.data_as(_p(C.c_int32)), tc.astype(np.int64),
                           out_device_ptrs, dist_cap)

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
        "ewk_set_templates_from_streams": (C.c_int, [vp, _p(C.c_int32), i32, _p(C.c_int32), _p(i64), _p(i64), vp]),
        "ewk_stream_results": (C.c_int, [vp, vp]),
        "ewk_dense_scores": (C.c_int, [vp, i64, i32, i32, i32, vp, i32]),
        "ewk_dense_scores_streams": (C.c_int, [vp, _p(C.c_int32), i32, _p(i64), _p(C.c_int32), i32, i32, vp, i64, i32]),
        "ewk_dense_ready": (C.c_int, [vp, _p(C.c_int32), i32, i32, i32, i32, _p(i64), _p(C.c_int32), vp, i64, i32]),
        "ewk_dense_detect": (C.c_int, [vp, _p(C.c_int32), i32, i32, i32, i32, i32, i32, vp, i32, _p(i64), _p(C.c_int32),
                                       vp, i64, i32]),
        "ewk_dense_scores_sets": (C.c_int, [vp, _p(C.c_int32), i32, _p(i64), _p(C.c_int32), _p(C.c_int32),
                                            _p(C.c_int32), vp, i64, i32]),
        "ewk_dense_ready_sets": (C.c_int, [vp, _p(C.c_int32), i32, i32, _p(C.c_int32), _p(C.c_int32), _p(i64),
                                           _p(C.c_int32), vp, i64, i32]),
        "ewk_dense_detect_sets": (C.c_int, [vp, _p(C.c_int32), i32, i32, _p(C.c_int32), _p(C.c_int32), i32, i32, vp, i32,
                                            _p(i64), _p(C.c_int32), vp, i64, i32]),
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
        "ewk_debug_check": (C.c_int, [vp]),
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


def _int32_list(values, what):
    """int32 array of indices (ValueError for values no int32 holds: the library names the others)."""
    v = np.asarray(values, dtype=np.int64).reshape(-1)
    if v.size and (v.min() < -2**31 or v.max() >= 2**31):
        raise ValueError(f"{what} out of range")
    return np.ascontiguousarray(v, dtype=np.int32)


def _stream_list(streams):
    """int32 array of stream indices (ValueError for values no int32 holds: the library names the others)."""
    return _int32_list(streams, "stream index")


def sets_offsets(n_hops, T):
    """Float offset of each row of a per-row-set call (include/ewk.h: ewk_dense_scores_sets): row i starts at
    sum_{j < i} n_hops[j] T[j].  Returns (offsets int64 [n], total floats)."""
    sizes = np.asarray(n_hops, np.int64).reshape(-1) * np.asarray(T, np.int64).reshape(-1)
    ends = np.cumsum(sizes)
    return ends - sizes, int(ends[-1]) if sizes.size else 0


def _unpack_rows_sets(out, n_hops, T):
    """Packed rows of a per-row-set call -> list of [n_i, T_i] views, in list order."""
    off, _ = sets_offsets(n_hops, T)
    return [out[o:o + int(n) * int(t)].reshape(int(n), int(t)) for o, n, t in zip(off.tolist(), n_hops, T)]


def _one_set(n, template_first, template_count):
    """-> the (template_first, template_count) arguments of a single-set entry point and T int64 [n]: every row's"""
    return int(template_first), int(template_count), np.full(n, int(template_count), np.int64)


def sets_launches(set_lens):
    """The K4 launches of a per-row-set call whose rows have template sets of these lengths: {(DH, threads, CTAs per
    SM): row indices}, one launch per geometry each set has alone (dense_plan), in order of first appearance."""
    groups = {}
    for i, lens in enumerate(set_lens):
        groups.setdefault(dense_plan(lens)[:3], []).append(i)
    return groups


def _bank_methods():
    def set_stream_params(self, stream=-1, params=None, **over):
        p = params if params is not None else default_stream_params(**over)
        self._ck(self.lib.ewk_set_stream_params(self.h, stream, C.byref(p)))
        ranges = self._template_ranges()
        ranges[slice(None) if stream < 0 else stream] = (p.template_first, p.template_count)

    def _template_ranges(self):
        """[n_streams, 2] (template_first, template_count) of each stream as set through set_stream_params; -1: not
        known here (never set, or the stream was imported)."""
        if getattr(self, "_ranges", None) is None:
            self._ranges = np.full((self.cfg.n_streams, 2), -1, np.int32)
        return self._ranges

    def _row_sets(self, st, n, template_first, template_count):
        """-> (first int32 [n] or None, count int32 [n] or None, T int64 [n]) of a per-row-set call's rows (st None:
        every stream).  Both None: each stream's own range, NULL to the library, T from set_stream_params."""
        if (template_first is None) != (template_count is None):
            raise ValueError("give both template_first and template_count, or neither")
        if template_first is None:
            idx = np.arange(n) if st is None else st
            r = self._template_ranges()[idx]
            if n and r[:, 1].min() < 0:
                raise ValueError(f"stream {int(idx[np.argmax(r[:, 1] < 0)])} has a template range this Context did not "
                                 "set (imported stream): pass template_first / template_count")
            return None, None, r[:, 1].astype(np.int64)
        tf = np.ascontiguousarray(np.broadcast_to(np.asarray(template_first, np.int64), (n,)), np.int32)
        tc = np.ascontiguousarray(np.broadcast_to(np.asarray(template_count, np.int64), (n,)), np.int32)
        return tf, tc, tc.astype(np.int64)

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
            self._template_ranges()[st] = -1
            return
        b = np.ascontiguousarray(blob).view(np.uint8).reshape(-1)
        self._ck(self.lib.ewk_import_streams(self.h, sp, len(st), b.ctypes.data if b.size else None, int(b.size), HOST))
        self._template_ranges()[st] = -1                  # parameters travel with the streams

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

    def set_templates_from_streams(self, slots, streams, starts, lens, want_vad=False):
        """Enrolment from the rings (include/ewk.h: ewk_set_templates_from_streams): template slots[i] <- stream
        streams[i]'s absolute samples [starts[i], starts[i] + lens[i]) (an event's or a detection's seg_start /
        seg_len), bit-identical to set_templates of what read_segment returns.  want_vad: also return the VAD analysis
        of each segment (VAD_DTYPE [n])."""
        sl = _int32_list(slots, "template slot")
        st = _stream_list(streams)
        a0 = np.ascontiguousarray(np.asarray(starts, dtype=np.int64).reshape(-1))
        ln = np.ascontiguousarray(np.asarray(lens, dtype=np.int64).reshape(-1))
        if not (len(st) == len(a0) == len(ln) == len(sl)):
            raise ValueError("one stream, start and length per template slot")
        vad = np.zeros(len(sl), dtype=VAD_DTYPE) if want_vad else None
        self._ck(self.lib.ewk_set_templates_from_streams(self.h, sl.ctypes.data_as(_p(C.c_int32)), len(sl),
                                                         st.ctypes.data_as(_p(C.c_int32)), i64ptr(a0), i64ptr(ln),
                                                         vad.ctypes.data if want_vad else None))
        return vad

    def align_segments(self, streams, starts, lens, template_first=None, template_count=None, out_device_ptrs=None,
                       dist_cap=None):
        """Frame-alignment distances of ring segments (include/ewk.h: ewk_align_segments): row i is stream streams[i]'s
        absolute samples [starts[i], starts[i] + lens[i]) (an event's or a detection's seg_start / seg_len) against slots
        [template_first[i], template_first[i] + template_count[i]) (both None: its stream's own range).  Returns (list of
        float32 [T_i] distances, best_slot int32 [n], best_dist float32 [n]); with out_device_ptrs = (dist, best_slot or
        None, best_dist or None) device pointers the outputs go there packed and None is returned."""
        st = _stream_list(streams)
        a0 = np.ascontiguousarray(np.asarray(starts, dtype=np.int64).reshape(-1))
        ln = np.ascontiguousarray(np.asarray(lens, dtype=np.int64).reshape(-1))
        n = len(st)
        if len(a0) != n or len(ln) != n:
            raise ValueError("one stream, start and length per row")
        tf, tc, T = self._row_sets(st, n, template_first, template_count)
        return self._align(self.lib.ewk_align_segments, n, (st.ctypes.data_as(_p(C.c_int32)), i64ptr(a0), i64ptr(ln)),
                           None if tf is None else tf.ctypes.data_as(_p(C.c_int32)),
                           None if tc is None else tc.ctypes.data_as(_p(C.c_int32)), T, out_device_ptrs, dist_cap)

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

    def _sets_args(self, st, n, template_first, template_count):
        """-> the (template_first, template_count) arguments of a *_sets entry point and T int64 [n] (see _row_sets)"""
        tf, tc, T = self._row_sets(st, n, template_first, template_count)
        return (None if tf is None else tf.ctypes.data_as(_p(C.c_int32)),
                None if tc is None else tc.ctypes.data_as(_p(C.c_int32)), T)

    def _scores_rows(self, fn, sets, streams, hop0, n_hops, out_device_ptr, out_cap):
        """dense_scores_streams / dense_scores_sets through entry point fn; sets(st, n) -> its two template arguments
        and each row's T"""
        st = _stream_list(streams)
        h0 = np.ascontiguousarray(np.asarray(hop0, dtype=np.int64).reshape(-1))
        nh64 = np.asarray(n_hops, dtype=np.int64).reshape(-1)
        if len(h0) != len(st) or len(nh64) != len(st):
            raise ValueError("one hop0 and one n_hops per stream")
        if nh64.size and (nh64.min() < -2**31 or nh64.max() >= 2**31):
            raise ValueError("n_hops out of range")
        nh = np.ascontiguousarray(nh64, dtype=np.int32)
        tf, tc, T = sets(st, len(st))
        need = max(0, int(np.maximum(nh64, 0) @ T))
        cap = need if out_cap is None else int(out_cap)
        args = (st.ctypes.data_as(_p(C.c_int32)), len(st), i64ptr(h0), nh.ctypes.data_as(_p(C.c_int32)), tf, tc)
        if out_device_ptr is not None:
            self._ck(fn(self.h, *args, C.c_void_p(out_device_ptr), cap, DEVICE))
            return None
        out = np.empty(need, np.float32)
        self._ck(fn(self.h, *args, out.ctypes.data if need else None, cap, HOST))
        return _unpack_rows_sets(out, nh64, T)

    def _ready(self, fn, sets, streams, max_hops, out_device_ptr, out_cap):
        """dense_ready / dense_ready_sets through entry point fn (sets as in _scores_rows)"""
        st = None if streams is None else _stream_list(streams)
        n = self.cfg.n_streams if st is None else len(st)
        tf, tc, T = sets(st, n)
        h0 = np.zeros(n, np.int64)
        nh = np.zeros(n, np.int32)
        cap = n * int(max_hops) * (int(T.max()) if n else 0) if out_cap is None else int(out_cap)
        args = (None if st is None else st.ctypes.data_as(_p(C.c_int32)), n, int(max_hops), tf, tc, i64ptr(h0),
                nh.ctypes.data_as(_p(C.c_int32)))
        if out_device_ptr is not None:
            self._ck(fn(self.h, *args, C.c_void_p(out_device_ptr), cap, DEVICE))
            return h0, nh
        out = np.empty(max(0, cap), np.float32)
        self._ck(fn(self.h, *args, out.ctypes.data if out.size else None, cap, HOST))
        return h0, _unpack_rows_sets(out, nh, T)

    def _detect(self, fn, sets, streams, max_hops, hold_hops, refractory_hops, scores, out_device_ptr, det_cap, out_cap,
                hops):
        """dense_detect / dense_detect_sets through entry point fn (sets as in _scores_rows)"""
        st = None if streams is None else _stream_list(streams)
        n = self.cfg.n_streams if st is None else len(st)
        tf, tc, T = sets(st, n)
        cap = n * ((min(int(max_hops), 1 << 20) + 1) // 2) if det_cap is None else int(det_cap)
        det = np.empty(max(0, cap), DETECTION_DTYPE)
        h0 = np.zeros(n, np.int64)
        nh = np.zeros(n, np.int32)
        ocap = n * int(max_hops) * (int(T.max()) if n else 0) if out_cap is None else int(out_cap)
        buf = None
        if out_device_ptr is not None:
            out, where = C.c_void_p(out_device_ptr), DEVICE
        elif scores:
            buf = np.empty(max(0, ocap), np.float32)
            out, where = (buf.ctypes.data if buf.size else None), HOST
        else:
            out, ocap, where = None, 0, HOST
        rc = fn(self.h, None if st is None else st.ctypes.data_as(_p(C.c_int32)), n, int(max_hops), tf, tc, int(hold_hops),
                int(refractory_hops), det.ctypes.data if det.size else None, cap, i64ptr(h0), nh.ctypes.data_as(_p(C.c_int32)),
                out, ocap, where)
        if rc < 0:
            self._ck(rc)
        d = det[:rc].copy()
        if out_device_ptr is not None:
            return d, (h0, nh)
        if scores:
            return d, (h0, _unpack_rows_sets(buf, nh, T))
        return (d, (h0, nh)) if hops else d

    def dense_scores_streams(self, streams, hop0, n_hops, template_first=0, template_count=1, out_device_ptr=None,
                             out_cap=None):
        """Ragged dense scoring (include/ewk.h: ewk_dense_scores_streams): row i scores stream streams[i] at hops
        [hop0[i], hop0[i] + n_hops[i]) (0 included).  Returns a list of float32 [n_hops[i], template_count] arrays; with
        out_device_ptr the rows go there packed back to back in list order (out_cap floats, default exactly what they
        need) and None is returned."""
        return self._scores_rows(self.lib.ewk_dense_scores_streams,
                                 lambda st, n: _one_set(n, template_first, template_count), streams, hop0, n_hops,
                                 out_device_ptr, out_cap)

    def dense_scores_sets(self, streams, hop0, n_hops, template_first=None, template_count=None, out_device_ptr=None,
                          out_cap=None):
        """dense_scores_streams with a template set per row (include/ewk.h: ewk_dense_scores_sets): row i is scored
        against slots [template_first[i], template_first[i] + template_count[i]) (both None: its stream's own range).
        Returns a list of float32 [n_hops[i], T_i] arrays; with out_device_ptr the rows go there packed as the header
        says (out_cap floats, default exactly what they need) and None is returned."""
        return self._scores_rows(self.lib.ewk_dense_scores_sets,
                                 lambda st, n: self._sets_args(st, n, template_first, template_count), streams, hop0, n_hops,
                                 out_device_ptr, out_cap)

    def dense_ready(self, streams=None, max_hops=100, template_first=0, template_count=1, out_device_ptr=None,
                    out_cap=None):
        """Dense scores paced by each stream's own audio (include/ewk.h: ewk_dense_ready): each listed stream (None: every
        stream) is scored from its cursor at every hop its landed audio completes, at most max_hops, and its cursor moves
        on.  Returns (hop0, scores): int64 [n] first hops and a list of float32 [n_i, template_count] arrays.  With
        out_device_ptr (out_cap floats, default n * max_hops * template_count) the rows go there packed in list order and
        (hop0, n_hops) is returned."""
        return self._ready(self.lib.ewk_dense_ready, lambda st, n: _one_set(n, template_first, template_count),
                           streams, max_hops, out_device_ptr, out_cap)

    def dense_ready_sets(self, streams=None, max_hops=100, template_first=None, template_count=None,
                         out_device_ptr=None, out_cap=None):
        """dense_ready with a template set per row (include/ewk.h: ewk_dense_ready_sets; arguments as dense_scores_sets,
        one entry per listed stream, or per stream when streams is None).  Moves dense_ready's cursor.  Returns (hop0,
        list of float32 [n_i, T_i] arrays), or (hop0, n_hops) with out_device_ptr (out_cap floats, default
        n * max_hops * max T_i)."""
        return self._ready(self.lib.ewk_dense_ready_sets,
                           lambda st, n: self._sets_args(st, n, template_first, template_count), streams, max_hops,
                           out_device_ptr, out_cap)

    def dense_detect(self, streams=None, max_hops=100, template_first=0, template_count=1, hold_hops=20,
                     refractory_hops=50, scores=False, out_device_ptr=None, det_cap=None, out_cap=None, hops=False):
        """Detections from per-hop scores on the device (include/ewk.h: ewk_dense_detect): each listed stream (None: every
        stream) is scored from the detector's own cursor at every hop its landed audio completes, at most max_hops, and
        those hops go through the stream's peak picker (threshold: its similarity_threshold).  Returns a DETECTION_DTYPE
        array in list order, then emit_hop order.  det holds n * ceil(max_hops / 2) records unless det_cap is given.
        scores=True also returns (hop0, list of float32 [n_i, template_count] arrays); with out_device_ptr the scores go
        there packed in list order (out_cap floats, default n * max_hops * template_count) and (hop0, n_hops) is returned
        with the detections.  Otherwise the scores stay on the device; hops=True then returns (hop0, n_hops) with them."""
        return self._detect(self.lib.ewk_dense_detect, lambda st, n: _one_set(n, template_first, template_count),
                            streams, max_hops, hold_hops, refractory_hops, scores, out_device_ptr, det_cap, out_cap, hops)

    def dense_detect_sets(self, streams=None, max_hops=100, template_first=None, template_count=None, hold_hops=20,
                          refractory_hops=50, scores=False, out_device_ptr=None, det_cap=None, out_cap=None, hops=False):
        """dense_detect with a template set per row (include/ewk.h: ewk_dense_detect_sets; sets as dense_ready_sets).
        Moves dense_detect's cursor and detector state; returns what dense_detect returns, score rows [n_i, T_i]."""
        return self._detect(self.lib.ewk_dense_detect_sets,
                            lambda st, n: self._sets_args(st, n, template_first, template_count), streams, max_hops,
                            hold_hops, refractory_hops, scores, out_device_ptr, det_cap, out_cap, hops)

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

    def debug_check(self):
        """Poison mode (EWK_POISON set at creation): raise unless every guard band of the context is intact."""
        self._ck(self.lib.ewk_debug_check(self.h))

    def profile(self, enable=True):
        self._ck(self.lib.ewk_profile(self.h, 1 if enable else 0))

    def profile_read(self):
        ms = (C.c_double * 8)()
        n = (C.c_int64 * 8)()
        self._ck(self.lib.ewk_profile_read(self.h, ms, n))
        names = ["ring_push", "tick_gate", "segment_queue", "segment_batch", "dense_score", "segment_prepare", "publish",
                 "resample_push"]
        return {names[i]: {"ms": ms[i], "launches": int(n[i])} for i in range(len(names))}

    for f in (align_segments, _template_ranges, _row_sets, _sets_args, _scores_rows, _ready, _detect, dense_scores_sets,
              dense_ready_sets, dense_detect_sets, set_templates_from_streams):
        setattr(Context, f.__name__, f)
    for f in (prepare_segments, dense_scores, dense_scores_streams, dense_ready, dense_detect, dense_last_plan, profile, profile_read, set_stream_params, push, push_g711, push_resampled,
              push_resampled_each, push_streams, tick_ready, reset_streams, stream_blob_bytes, export_streams, import_streams, stream_input, tick, poll, status, read_last, read_segment, results, results_device_ptr,
              set_results_buffer, set_results_peers, publish_parity, publish_seq, wait_published, published_seq, match_stream, set_cuda_stream, launch_count,
              debug_check):
        setattr(Context, f.__name__, f)


_bank_methods()
