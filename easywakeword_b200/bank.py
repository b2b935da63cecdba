"""WakeWordBank — the batched ("multiroom") form of the reference's detector.

The reference runs N rooms as N independent WakeWord objects and N threads
(/root/reference/examples/multiroom_async.py:14-35).  Here N streams share one device context:
rings in HBM, and per 100 ms tick of audio one K2 launch (adaptive threshold, is_silent, timing state
machine for every stream) plus one persistent K3 launch (fused MFCC + template match on every candidate
segment).  Host code only pushes PCM, ticks, and polls events; level 3 (Whisper) is handed
`read_segment(event)` audio on the host, exactly where the reference calls `_transcribe_audio`
(wakeword.py:1126-1128).
"""
from __future__ import annotations

from typing import Callable, Iterable, Optional, Sequence

import numpy as np

from . import _lib
from .wakeword import WakeWord, load_wav_16k

TICK_SAMPLES = 1600
DENSE_ROUND = 500                 # hops per ewk_dense_ready call of WakeWordBank.dense_ready (5 s of audio)
EV_TIMEOUT, EV_SCORED = _lib.EV_TIMEOUT, _lib.EV_SCORED
VERIFY_DTYPE = np.dtype([("stream", "<i4"), ("seg_start", "<i8"), ("seg_len", "<i4"), ("best_slot", "<i4"),
                         ("distance", "<f4")])


def _segment_rows(segments):
    """(streams, starts, lens) int64 arrays of structured rows with stream / seg_start / seg_len or of a tuple."""
    if isinstance(segments, tuple):
        return tuple(np.asarray(a, dtype=np.int64).reshape(-1) for a in segments)
    rows = [e for e in segments]
    return (np.array([int(e["stream"]) for e in rows], np.int64), np.array([int(e["seg_start"]) for e in rows], np.int64),
            np.array([int(e["seg_len"]) for e in rows], np.int64))


def stream_blob_rates(blob) -> np.ndarray:
    """The input rate each stream of a host blob (export_streams) is latched to (0: none yet), from its meta records."""
    b = np.ascontiguousarray(blob).view(np.uint8).reshape(-1)
    hsz = _lib.STREAM_BLOB_HEADER_DTYPE.itemsize
    if b.size < hsz:
        raise ValueError("not a stream blob")
    h = b[:hsz].view(_lib.STREAM_BLOB_HEADER_DTYPE)[0]
    if int(h["magic"]) != _lib.STREAM_BLOB_MAGIC or int(h["meta_bytes"]) != _lib.STREAM_META_BYTES:
        raise ValueError("not a stream blob of version 1")
    n, off = int(h["n_streams"]), int(h["meta_offset"])
    if n < 0 or off + n * _lib.STREAM_META_BYTES > b.size:
        raise ValueError("truncated stream blob")
    rec = b[off:off + n * _lib.STREAM_META_BYTES].reshape(n, _lib.STREAM_META_BYTES)
    return np.ascontiguousarray(rec[:, 52:56]).view("<i4").reshape(-1)      # StreamMeta.rate


def enroll_ranges(streams, starts, lens, slots) -> dict:
    """{stream: (first slot, slot count, row of its first segment)} of an enrolment (WakeWordBank.enroll), in order of
    first appearance; ValueError unless the lists have one entry per segment and every stream's slots, in list order,
    are consecutive (at most 64 of them: include/ewk.h EWK_MAX_STREAM_TEMPLATES)."""
    n = len(slots)
    if not (len(streams) == len(starts) == len(lens) == n):
        raise ValueError(f"enroll: {len(streams)} streams, {len(starts)} starts, {len(lens)} lengths and {n} slots; "
                         "give one of each per segment")
    ranges, last = {}, {}
    for i in range(n):
        s, k = int(streams[i]), int(slots[i])
        if s not in ranges:
            ranges[s] = (k, 1, i)
        elif k != last[s] + 1:
            raise ValueError(f"enroll: stream {s} is listed again at segment {i} with slot {k}; its segments must take "
                             f"consecutive slots (expected {last[s] + 1})")
        else:
            first, count, row = ranges[s]
            if count == 64:
                raise ValueError(f"enroll: stream {s} takes more than 64 slots (EWK_MAX_STREAM_TEMPLATES)")
            ranges[s] = (first, count + 1, row)
        last[s] = k
    return ranges


class WakeWordBank:
    """N independent audio streams, one GPU.

    sample_rate: the rate of the blocks push / push_g711 / step / run take.  Any rate other than 16000 (8 kHz telephony,
    44.1 / 48 kHz devices) is converted to 16 kHz on the device as it lands (K8); the rings, the timing and
    samples_pushed are in 16 kHz samples.

    Streams are recycled with reset(streams): a stream that served one call takes the next without touching the others.
    A recycled stream's event ticks and seg_start count from its reset, as in a new bank.  At a sample_rate other than
    16000 its input restarts at position 0 while the others go on, and one push still serves them all;
    samples_pushed (the clock step() ticks by) then advances by the largest count landed, and status(s).written holds a
    stream's own count.

    Feeds with jitter or a sparse set of active calls use push_streams / step_streams: any list of streams, each with its
    own amount of audio, in one push, and ticks paced by each stream's own landed audio (include/ewk.h: ewk_push_streams,
    ewk_tick_ready).  The same audio then gives the same events however it was split into pushes, and a slot that is not
    fed takes no ticks and costs no PCIe bytes.  samples_pushed and ticks describe push / step only; read a stream's own
    clock with status(s) (written, tick).

    templates: list of float32 arrays or WAV paths (slot i = templates[i]); every stream is scored
    against all of them (best score wins) unless set_stream(..., template_first=, template_count=).
    Timing defaults are the reference's (wakeword.py:38-41); speech_duration_min/max default to the
    auto-calculated values of the first template (tests/test_wakeword_simulated.py:687-775).

    template_slots: the context's template slots (default len(templates), at most 4096 = include/ewk.h
    EWK_MAX_TEMPLATE_SLOTS); slots past the constructor's templates are filled later with enroll(), e.g. one personal
    word per stream spoken by its own user.

    alignment: keep every template's MFCC frames (24 KB of device memory per slot) so that verify() can check level-2
    candidates by frame alignment (DTW) before level 3: pooled level-2 features match the right sounds in the wrong
    order, an alignment does not."""

    def __init__(self, n_streams: int, templates: Sequence, *, device: int = 0, buffer_seconds: int = 10,
                 pcm_dtype=np.int16, frame_size: int = TICK_SAMPLES, similarity_threshold: float = 75.0,
                 pre_speech_silence: float = 0.8, speech_duration_min: Optional[float] = None,
                 speech_duration_max: Optional[float] = None, post_speech_silence: float = 0.4,
                 timeout: float = 30.0, max_push_seconds: float = 1.0, max_events: int = 0,
                 cuda_stream: Optional[int] = None, overlap: bool = False, preemphasis: float = 0.0, n_mfcc: int = 20,
                 sample_rate: int = 16000, template_slots: Optional[int] = None, alignment: bool = False):
        if n_streams < 1:
            raise ValueError("n_streams must be at least 1")
        if buffer_seconds <= 0:
            raise ValueError("buffer_seconds must be positive")
        if not templates:
            raise ValueError("at least one template is required")
        self.n_streams = n_streams
        self.sample_rate = int(sample_rate)
        if self.sample_rate != 16000:
            _lib.resample_info(self.sample_rate)                 # ValueError for rates the device filter does not support
        self.pcm_dtype = np.dtype(pcm_dtype)
        if self.pcm_dtype not in (np.dtype(np.int16), np.dtype(np.float32)):
            raise ValueError("pcm_dtype must be int16 or float32")
        fmt = _lib.PCM_I16 if self.pcm_dtype == np.int16 else _lib.PCM_F32
        n_slots = len(templates) if template_slots is None else int(template_slots)
        if n_slots < len(templates):
            raise ValueError(f"template_slots {n_slots} is below the {len(templates)} templates given")
        slack = int(max_push_seconds * 16000) + 2 * max(frame_size, TICK_SAMPLES)
        self.ctx = _lib.Context(device=device, n_streams=n_streams, ring_samples=buffer_seconds * 16000,
                                slack_samples=slack, pcm_format=fmt, max_templates=max(1, n_slots),
                                max_events=max_events or max(4096, 2 * n_streams), preemphasis=preemphasis,
                                n_mfcc=n_mfcc, template_frames=alignment)
        self.alignment = bool(alignment)
        if cuda_stream is not None:
            self.ctx.set_cuda_stream(cuda_stream)
        if overlap:
            # level-2 matching on a second stream beside the next push (include/ewk.h: ewk_set_overlap); work that the
            # caller enqueues on `cuda_stream` after tick() and that reads the results must follow self.ctx.join()
            self.ctx.set_overlap(True)
        self.templates = []
        for slot, t in enumerate(templates):
            audio = load_wav_16k(t) if isinstance(t, (str, bytes)) or hasattr(t, "__fspath__") else \
                np.ascontiguousarray(t, dtype=np.float32)
            self.ctx.set_template(slot, audio)
            self.templates.append(audio)
        # voice-activity duration of every template on the device (K6); the bank's default timing follows the first
        # template, as the reference's single-template WakeWord does (tests/test_wakeword_simulated.py:687-775)
        self.template_vad = self.ctx.analyze_templates(self.templates)
        if speech_duration_min is None:
            d = float(self.template_vad["duration_s"][0]) if self.template_vad["voiced"][0] else None
            speech_duration_min = d if d is not None else 0.3
            if speech_duration_max is None:
                speech_duration_max = 2.0 * speech_duration_min if d is not None else 2.0
        elif speech_duration_max is None:
            speech_duration_max = 2.0 * speech_duration_min
        self.params = dict(frame_size=frame_size, similarity_threshold=similarity_threshold,
                           pre_speech_silence=pre_speech_silence, speech_duration_min=speech_duration_min,
                           speech_duration_max=speech_duration_max, post_speech_silence=post_speech_silence,
                           timeout=float(timeout), template_first=0, template_count=len(templates))
        self.ctx.set_stream_params(-1, **self.params)
        self.ticks = 0
        self.samples_pushed = 0

    # ---- configuration
    def set_stream(self, stream: int, **overrides):
        """Per-stream parameters (any field of ewk_stream_params)."""
        p = dict(self.params)
        p.update(overrides)
        self.ctx.set_stream_params(stream, **p)

    def reset(self, streams, **overrides) -> np.ndarray:
        """Recycle `streams` (a new call on each slot): drains the event queue and returns those events (handle them as
        poll()'s; no event of the old sessions can surface afterwards), then returns the streams to the state of a new
        bank in one launch (include/ewk.h: ewk_reset_streams).  Their parameters stay unless `overrides` are given:
        those are applied to each stream through set_stream (e.g. another template range or threshold)."""
        events = self.poll()
        lst = [int(s) for s in np.asarray(streams, dtype=np.int64).reshape(-1)]
        self.ctx.reset_streams(lst)
        if overrides:
            for s in dict.fromkeys(lst):
                self.set_stream(s, **overrides)
        return events

    # ---- enrolment
    def enroll(self, segments, slots, set_durations: bool = True) -> np.ndarray:
        """Personal wake words from audio the bank has heard: template slots[i] <- segment i, for all segments in one
        call on the device (include/ewk.h: ewk_set_templates_from_streams), and each listed stream scored against its
        own slots from then on (gate, and dense_ready / dense_detect with own_templates=True).
        segments: structured rows with stream / seg_start / seg_len (poll()'s events, a dense_detect result, as
        prepare_for_transcription takes them) or a (streams, starts, lens) tuple; the ranges must still be in the rings.
        A stream listed k times takes k consecutive slots, in list order, and its range becomes those k slots (several
        recordings of one word, best score wins); ValueError before anything is installed otherwise.  Each listed stream
        is set through set_stream (the bank's parameters plus its new range); with set_durations its
        speech_duration_min / max also follow the first of its recordings, by the rule the constructor applies to the
        first template.  self.templates stays the constructor's list.  Returns the VAD analysis of every segment
        (_lib.VAD_DTYPE, or None without set_durations)."""
        streams, starts, lens = _segment_rows(segments)
        sl = np.asarray(slots, dtype=np.int64).reshape(-1)
        ranges = enroll_ranges(streams, starts, lens, sl)
        vad = self.ctx.set_templates_from_streams(sl, streams, starts, lens, want_vad=set_durations)
        for s, (first, count, row) in ranges.items():
            over = dict(template_first=first, template_count=count)
            if set_durations:
                d = float(vad["duration_s"][row]) if vad["voiced"][row] else None
                over["speech_duration_min"] = d if d is not None else 0.3
                over["speech_duration_max"] = 2.0 * d if d is not None else 2.0
            self.set_stream(s, **over)
        return vad

    # ---- migration
    def export_streams(self, streams) -> np.ndarray:
        """A host blob (np.uint8) holding the listed streams' whole live state (include/ewk.h: ewk_export_streams): ring,
        gate, timing, dense cursors, detector and K8 input tails.  The streams go on untouched and their queued events
        stay here.  Save it with np.save for a checkpoint; import_streams on any bank with the same buffer_seconds,
        max_push_seconds / frame_size (the slack), pcm_dtype, n_mfcc and preemphasis takes it."""
        return self.ctx.export_streams(streams)

    def import_streams(self, streams, blob) -> np.ndarray:
        """Blob stream i becomes stream streams[i] of this bank and goes on exactly as it would have where it was
        exported (include/ewk.h: ewk_import_streams); its parameters come with it.  Drains the event queue first and
        returns those events (handle them as poll()'s), as reset does.  ValueError for a stream latched to an input rate
        other than this bank's sample_rate (a later push would fail).  Moved streams sit at their own positions: feed
        them with push_streams / step_streams, as after staggered resets."""
        lst = [int(s) for s in np.asarray(streams, dtype=np.int64).reshape(-1)]
        for i, rate in enumerate(stream_blob_rates(blob)):
            if rate not in (0, self.sample_rate):
                raise ValueError(f"blob stream {i} takes {rate} Hz input; this bank takes {self.sample_rate} Hz")
        events = self.poll()
        self.ctx.import_streams(lst, blob)
        return events

    def move_streams(self, streams, dst: "WakeWordBank", dst_streams):
        """Move live calls: streams of this bank become dst_streams of dst (dst may be this bank).  In order: drain dst's
        queue, export, import, drain this bank's queue, reset the source slots that did not receive a stream.  Returns
        (source_events, destination_events): the drained events, with the ids of the bank that raised them.  A stream
        latched to another rate than dst's sample_rate is refused before anything is drained; if the import itself fails
        (e.g. banks of another geometry), the exception carries dst's drained events as `drained_events` and the source
        is untouched."""
        src = [int(s) for s in np.asarray(streams, dtype=np.int64).reshape(-1)]
        dst_l = [int(s) for s in np.asarray(dst_streams, dtype=np.int64).reshape(-1)]
        if len(src) != len(dst_l):
            raise ValueError("one destination stream per source stream")
        for s in src:                                  # refused before anything is drained
            rate = self.ctx.stream_input(s)[0]
            if rate not in (0, dst.sample_rate):
                raise ValueError(f"stream {s} takes {rate} Hz input; the destination bank takes {dst.sample_rate} Hz")
        dst_events = dst.poll()
        blob = self.export_streams(src)
        try:
            more = dst.import_streams(dst_l, blob)
        except Exception as e:                         # the caller still gets what was drained
            e.drained_events = dst_events
            raise
        if len(more):
            dst_events = np.concatenate([dst_events, more])
        src_events = self.poll()
        free = [s for s in src if dst is not self or s not in dst_l]
        if free:
            self.ctx.reset_streams(free)
        return src_events, dst_events

    # ---- data plane
    def push(self, pcm, where=_lib.HOST):
        """pcm[n_streams, n]: n new samples for every stream (K1 / direct H2D) in the bank's dtype; at another
        sample_rate, float32 or int16 at that rate (K8; a device input is (ptr, n_streams, n, stride, dtype))."""
        if self.sample_rate != 16000:
            self.samples_pushed += int(self.ctx.push_resampled_each(pcm, self.sample_rate, stream0=0, where=where).max())
            return
        self.ctx.push(pcm, stream0=0, where=where)
        self.samples_pushed += pcm[2] if isinstance(pcm, tuple) else pcm.shape[-1]

    def push_g711(self, codes, law: str = "ulaw", where=_lib.HOST):
        """codes[n_streams, n] uint8: a G.711 mu-law / A-law feed, expanded on the device (16 kHz: int16 banks only; at
        another sample_rate the codes are converted by K8 into either ring format)."""
        if self.sample_rate != 16000:
            if law not in ("ulaw", "alaw"):
                raise ValueError("law must be 'ulaw' or 'alaw'")
            if isinstance(codes, tuple):
                codes = (*codes[:4], np.uint8)
            self.samples_pushed += int(self.ctx.push_resampled_each(codes, self.sample_rate, stream0=0, where=where,
                                                                    fmt=law).max())
            return
        self.ctx.push_g711(codes, stream0=0, where=where, law=law)
        self.samples_pushed += codes[2] if isinstance(codes, tuple) else codes.shape[-1]

    def tick(self, n_ticks: int = 1, trace: bool = False):
        """n_ticks x 100 ms of the reference's poll loop for every stream (K2 + K3)."""
        self.ticks += n_ticks
        return self.ctx.tick(n_ticks, trace=trace)

    def step(self, pcm, where=_lib.HOST):
        """push + as many ticks as the landed audio covers."""
        self.push(pcm, where)
        due = self.samples_pushed // TICK_SAMPLES - self.ticks
        if due > 0:
            self.tick(due)

    def push_streams(self, streams, blocks, where=_lib.HOST):
        """blocks[i]: 1-D audio at the bank's sample_rate for stream streams[i], any length (0 included), in the bank's
        dtype at 16 kHz (float32 or int16 at other rates).  One push for the whole list.  Returns the 16 kHz samples landed
        per stream."""
        return self.ctx.push_streams(streams, blocks, sr_in=self.sample_rate, where=where)

    def step_streams(self, streams, blocks, where=_lib.HOST):
        """push_streams, then every tick the landed audio pays for, stream by stream (ewk_tick_ready): no stream has a
        due tick left when it returns.  Returns the ticks each stream took (int64 [n_streams])."""
        self.push_streams(streams, blocks, where)
        taken = np.zeros(self.n_streams, np.int64)
        while True:
            t = self.ctx.tick_ready(4096)
            taken += t
            if t.max() < 4096:
                return taken

    def poll(self) -> np.ndarray:
        """Structured array of events since the last poll, sorted by (tick, stream):
        kind 2 = level-2 evaluation (score, matched), kind 1 = timeout."""
        return self.ctx.poll()

    def results(self) -> np.ndarray:
        return self.ctx.results()

    def dense_scores(self, hop0: int, n_hops: int, template_first: int = 0, template_count: Optional[int] = None):
        """Per-hop scores [n_streams, n_hops, T] for hops [hop0, hop0 + n_hops) (hop h = 160*h samples
        pushed): calculate_similarity of the latest template-length window complete at each hop (K4)."""
        T = len(self.templates) - template_first if template_count is None else template_count
        return self.ctx.dense_scores(hop0, n_hops, template_first, T)

    def dense_ready(self, streams=None, template_first: int = 0, template_count: Optional[int] = None,
                    own_templates: bool = False):
        """Per-hop scores paced by each stream's own audio (include/ewk.h: ewk_dense_ready): every hop of the listed
        streams (None: all) that their landed audio completes and no earlier call scored, in rounds of DENSE_ROUND hops,
        so that no due hop is left when it returns.  Returns (hop0, scores): int64 first hop of each listed stream's
        scores and a list of float32 [n_i, T] arrays.  A stream recycled with reset() starts again at hop 1.
        own_templates=True scores each stream against its own set_stream(..., template_first=, template_count=) range
        in the same calls (ewk_dense_ready_sets); its arrays are then [n_i, T_i]."""
        T = len(self.templates) - template_first if template_count is None else template_count
        hop0, parts = None, None
        while True:
            if own_templates:
                h0, rows = self.ctx.dense_ready_sets(streams, DENSE_ROUND)
            else:
                h0, rows = self.ctx.dense_ready(streams, DENSE_ROUND, template_first, T)
            if hop0 is None:
                hop0, parts = h0, [[r] for r in rows]
            else:
                for p, r in zip(parts, rows):
                    p.append(r)
            if not rows or max(len(r) for r in rows) < DENSE_ROUND:
                return hop0, [p[0] if len(p) == 1 else np.concatenate(p) for p in parts]

    def dense_detect(self, streams=None, template_first: int = 0, template_count: Optional[int] = None,
                     hold_hops: int = 20, refractory_hops: int = 50, own_templates: bool = False) -> np.ndarray:
        """Wake-word detections from per-hop scores, without the energy gate (include/ewk.h: ewk_dense_detect): every hop
        of the listed streams (None: all) that their landed audio completes and no earlier dense_detect took, in rounds of
        DENSE_ROUND hops, so that no due hop is left when it returns.  A stream detects where its best per-hop score
        reaches its similarity_threshold; a run reports its first peak once it ends or hold_hops after the peak, and a
        stream stays quiet for refractory_hops after a run.  Returns a _lib.DETECTION_DTYPE array sorted by
        (emit_hop, stream); prepare_for_transcription takes it as it is.  The detector has its own cursor (dense_ready's is
        untouched); reset() restarts it.  Feed hold_hops hops of trailing audio to finish a recording's last run.
        own_templates=True detects each stream against its own set_stream(..., template_first=, template_count=) range
        in the same calls (ewk_dense_detect_sets): personal wake words, one launch per geometry."""
        T = len(self.templates) - template_first if template_count is None else template_count
        parts = []
        while True:
            if own_templates:
                d, (_, nh) = self.ctx.dense_detect_sets(streams, DENSE_ROUND, hold_hops=hold_hops,
                                                        refractory_hops=refractory_hops, hops=True)
            else:
                d, (_, nh) = self.ctx.dense_detect(streams, DENSE_ROUND, template_first, T, hold_hops, refractory_hops,
                                                   hops=True)
            parts.append(d)
            if nh.size == 0 or nh.max() < DENSE_ROUND:
                break
        det = np.concatenate(parts)
        return det[np.lexsort((det["stream"], det["emit_hop"]))]

    def read_segment(self, event) -> np.ndarray:
        """word_audio of a level-2 event as float32 (what level 3 transcribes)."""
        return self.ctx.read_segment(int(event["stream"]), int(event["seg_start"]), int(event["seg_len"]))

    def dense_sweep(self, blocks: Iterable[np.ndarray], template_first: int = 0, template_count: Optional[int] = None):
        """Offline sweep (BASELINE config 5): push each [n_streams, n] block (at 16 kHz, n a multiple of 160; at another
        sample_rate, any n) and yield (first_hop, scores[n_streams, hops, T]) for the hops the landed audio completes —
        every template scored at every hop."""
        self.ctx.set_stream_params(-1, **dict(self.params, live=1))     # no ticks here: pushes run free of the gate's guard
        for blk in blocks:
            if self.sample_rate == 16000 and blk.shape[-1] % 160:
                raise ValueError("dense_sweep blocks must hold a multiple of 160 samples")
            hop0 = self.samples_pushed // 160 + 1
            self.push(blk)
            n_hops = self.samples_pushed // 160 + 1 - hop0
            if n_hops == 0:
                T = len(self.templates) - template_first if template_count is None else template_count
                yield hop0, np.zeros((self.n_streams, 0, T), np.float32)
                continue
            yield hop0, self.dense_scores(hop0, n_hops, template_first, template_count)

    def prepare_for_transcription(self, events) -> list:
        """Batched level-3 pre-processing on the device (wakeword.py:1020-1025) of the word_audio of `events`
        (any structured rows with stream / seg_start / seg_len): list of float32 arrays ready for the STT backend."""
        ev = [e for e in events]
        return self.ctx.prepare_segments([int(e["stream"]) for e in ev], [int(e["seg_start"]) for e in ev],
                                         [int(e["seg_len"]) for e in ev])

    def verify(self, segments, own_templates: bool = True, template_first=None, template_count=None):
        """Frame-alignment distances of ring segments (include/ewk.h: ewk_align_segments; needs alignment=True): a second
        stage for level-2 candidates before level 3.  segments: poll()'s events, a dense_detect result or a (streams,
        starts, lens) tuple; the ranges must still be in the rings.  Each segment is aligned against its stream's own
        template range (own_templates=True), or against [template_first, template_first + template_count) (scalars or
        one per segment).  Returns (VERIFY_DTYPE array: stream, seg_start, seg_len, best_slot and its distance; list of
        float32 [T_i] distances per template of each segment's set).  0 is a perfect match; the distance is not on the
        score's 0-100 scale, so pick a threshold from your own recordings."""
        streams, starts, lens = _segment_rows(segments)
        if own_templates and template_first is None and template_count is None:
            dist, slot, best = self.ctx.align_segments(streams, starts, lens)
        else:
            if template_first is None or template_count is None:
                raise ValueError("give template_first and template_count, or neither with own_templates=True")
            dist, slot, best = self.ctx.align_segments(streams, starts, lens, template_first, template_count)
        out = np.zeros(len(streams), VERIFY_DTYPE)
        out["stream"], out["seg_start"], out["seg_len"] = streams, starts, lens
        out["best_slot"], out["distance"] = slot, best
        return out, dist

    def status(self, stream: int):
        return self.ctx.status(stream)

    # ---- convenience: the reference's callback surface over the whole bank
    def run(self, blocks: Iterable[np.ndarray], on_match: Optional[Callable] = None, transcriber=None,
            textword: str = "", numberofwords: int = 1, max_distance: Optional[float] = None):
        """Feed an iterable of [n_streams, n] blocks; for every level-2 match call
        on_match(stream, tick, score, text) where text is the level-3 confirmation (None without a
        transcriber).  Returns the list of all events.  max_distance (needs alignment=True): level-2 matches whose
        verify() distance against their stream's own templates exceeds it are dropped before level 3 and on_match."""
        log = []
        for blk in blocks:
            self.step(blk)
            ev = self.poll()
            log.extend(e.copy() for e in ev)
            hits = [e for e in ev if e["kind"] == EV_SCORED and e["matched"]]
            if not hits or on_match is None:
                continue
            if max_distance is not None:
                d = self.verify(hits)[0]["distance"]
                hits = [e for e, x in zip(hits, d) if x <= max_distance]
            audio = self.prepare_for_transcription(hits) if transcriber is not None else [None] * len(hits)
            for e, a in zip(hits, audio):
                text = transcriber.transcribe(a) if transcriber is not None else None
                on_match(int(e["stream"]), int(e["tick"]), float(e["score"]), text)
        return log

    def close(self):
        self.ctx.close()
