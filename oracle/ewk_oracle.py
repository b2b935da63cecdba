"""ORACLE — TEST INFRASTRUCTURE ONLY.  Not shipped, not on the product path.

CPU (numpy) restatement of the reference's level-1/level-2 hot path, function by
function, citing /root/reference/easywakeword/wakeword.py.  It exists to CHECK the
CUDA path (tests/, __graft_entry__.smoke()) and to be TIMED as the CPU baseline
(bench.py `cpu_baseline` / `--impl reference`); the product (easywakeword_b200/)
never imports it and has no CPU fallback.

Pinning (see tests/test_oracle.py, tests/golden/MANIFEST.json):
  * against the reference's own classes run UNMODIFIED in the build container
    (oracle/ref_harness.py -> tests/golden/*.npz written by oracle/gen_golden.py);
  * against every known-answer test the reference holds for this path
    (self-similarity == 100.0, shapes, inequalities: tests/test_wakeword_simulated.py:
    104-205, 298-360; tests/test_cross_platform.py:69-109) and the two doc pins
    (LEARNINGS.md:92-93);
  * the librosa arithmetic underneath is itself a restatement (librosa is not
    installable here): oracle/librosa_restated.py.  Beyond the items above the
    reference stores no MFCC vector or score, so MFCC values are pinned by that
    restatement + torchaudio cross-checks only (DESIGN.md §Oracle).

Time model ("audio clock"): tick k is the k-th 100 ms poll of WakeWord._detect_word
(wakeword.py:1064); time() == k * 0.1 in float64; 1600 samples of audio arrive per
tick, delivered to the ring in `block`-sample callbacks, so floor(1600 k / block)
callbacks have run when tick k samples the buffer.
"""
from __future__ import annotations

import math

import numpy as np
from scipy.spatial.distance import cosine

from . import librosa_restated as L

FREQUENCY = 16000          # SoundBuffer.FREQUENCY            wakeword.py:408
MIN_THRESHOLD = 0.005      # SoundBuffer.MIN_THRESHOLD        wakeword.py:409
INITIAL_THRESHOLD = 0.01   # SoundBuffer.silence_threshold    wakeword.py:431
TICK_SECONDS = 0.1         # time.sleep(0.1)                  wakeword.py:1064
TICK_SAMPLES = 1600        # int(0.1 * 16000)                 wakeword.py:492,500
SEGMENT_PADDING = 0.05     # padding                          wakeword.py:1101
MAX_SEGMENT_SECONDS = 3.0  # audio_duration > 3.0 -> skip     wakeword.py:1114-1118

DEFAULTS = dict(similarity_threshold=75.0, pre_speech_silence=0.8, speech_duration_min=0.3,
                speech_duration_max=2.0, post_speech_silence=0.4, timeout=30.0)


# ------------------------------------------------------------------ A4-A7  WordMatcher
def mfcc_frames(audio, preemphasis=0.0, n_mfcc=20):
    """The [20 x (1 + n//160)] matrix extract_mfcc pools (wakeword.py:561-563).
    preemphasis / n_mfcc are the build's exposed front-end parameters (ewk_config, ABI 2); the reference's values are
    0 (none) and 20, and with them this is the reference's call, statement for statement."""
    y = np.asarray(audio)
    if preemphasis:
        y = L.preemphasis(y, coef=preemphasis)
    return L.mfcc(y=y, sr=FREQUENCY, n_mfcc=n_mfcc, n_fft=512, hop_length=160)


def extract_mfcc(audio, preemphasis=0.0, n_mfcc=20):
    """WordMatcher.extract_mfcc (wakeword.py:544-567): MFCC[20 x frames] -> mean, std (ddof 0)."""
    m = mfcc_frames(audio, preemphasis, n_mfcc)
    return np.mean(m, axis=1), np.std(m, axis=1)


def similarity_from_features(ref_mean, ref_std, cand_mean, cand_std):
    """WordMatcher.calculate_similarity after feature extraction (wakeword.py:613-625)."""
    sim_mean = 1 - cosine(ref_mean, cand_mean)
    sim_std = 1 - cosine(ref_std, cand_std)
    combined_similarity = sim_mean * 0.7 + sim_std * 0.3
    similarity_percent = combined_similarity * 100
    return (similarity_percent ** 1.5) / (100 ** 0.5)


class WordMatcherOracle:
    """Restates WordMatcher (wakeword.py:520-639)."""

    def __init__(self, sample_rate=16000, preemphasis=0.0, n_mfcc=20):
        self.sample_rate = sample_rate
        self.reference_mfcc_mean = None
        self.reference_mfcc_std = None
        self.reference_word = None
        self.preemphasis, self.n_mfcc = preemphasis, n_mfcc

    def extract_mfcc(self, audio):
        return extract_mfcc(audio, self.preemphasis, self.n_mfcc)

    def set_reference(self, audio, word_name="target"):                # :569-578
        self.reference_word = word_name
        self.reference_mfcc_mean, self.reference_mfcc_std = self.extract_mfcc(audio)

    def load_reference_from_file(self, filepath, word_name="target"):  # :580-589
        audio, _ = L.load(filepath, sr=self.sample_rate)
        self.set_reference(audio, word_name)

    def calculate_similarity(self, audio):                              # :591-625
        if self.reference_mfcc_mean is None:
            raise ValueError("No reference word set. Call set_reference() first.")
        m, s = self.extract_mfcc(audio)
        with np.errstate(all="ignore"):
            return similarity_from_features(self.reference_mfcc_mean, self.reference_mfcc_std, m, s)

    def matches(self, audio, threshold=75.0):                           # :627-639
        similarity = self.calculate_similarity(audio)
        return similarity >= threshold, similarity


# ------------------------------------------------------------------ A1-A3  SoundBuffer
class SoundBufferOracle:
    """Restates SoundBuffer (wakeword.py:405-517) minus the PortAudio stream.

    fast=False follows the reference statement by statement (per-sample ring loop :461-465,
    per-chunk RMS loop :479-482) and is what the CPU baseline times; fast=True writes the ring
    with slice assignments and batches the chunk RMS with one reshape — bit-identical results
    (numpy reduces each contiguous row with the same pairwise sum), checked in tests.
    """

    FREQUENCY = FREQUENCY
    MIN_THRESHOLD = MIN_THRESHOLD

    def __init__(self, seconds=10, fast=False, ring_samples=None):
        # ring_samples: a ring of any integer length (the reference's seconds * 16000 cannot say 20000 samples)
        self.buffer_seconds = seconds
        self.buffer_length = int(ring_samples) if ring_samples is not None else self.buffer_seconds * self.FREQUENCY
        self.data = np.zeros(self.buffer_length)
        self.pointer = 0
        self.frame_size = 0
        self.silence_threshold = INITIAL_THRESHOLD
        self.samples_collected = 0
        self.fast = fast

    def add_block(self, indata):                                        # :454-470
        new_data = np.array(indata).flatten()
        if self.frame_size == 0:
            self.frame_size = len(new_data)
        n = len(new_data)
        R = self.buffer_length
        if not self.fast:                # the reference's own per-sample loop (:461-465)
            for sample in new_data:
                self.data[self.pointer] = sample
                self.pointer = (self.pointer + 1) % R
                if self.samples_collected < R:
                    self.samples_collected += 1
            if self.samples_collected < R:
                return
            self._adjust_silence_threshold()
            return
        if n >= R:                       # only the last R samples survive the loop
            keep = new_data[n - R:]
            start = (self.pointer + n - R) % R
            first = min(R - start, R)
            self.data[start:start + first] = keep[:first]
            self.data[:R - first] = keep[first:]
        else:
            first = min(n, R - self.pointer)
            self.data[self.pointer:self.pointer + first] = new_data[:first]
            self.data[:n - first] = new_data[first:]
        self.pointer = (self.pointer + n) % R
        self.samples_collected = min(R, self.samples_collected + n)
        if self.samples_collected < R:
            return
        self._adjust_silence_threshold()

    def _adjust_silence_threshold(self):                                # :472-486
        if self.frame_size == 0:
            return
        num_frames = len(self.data) // self.frame_size
        if num_frames == 0:
            return
        if self.fast:
            chunks = self.data[: num_frames * self.frame_size].reshape(num_frames, self.frame_size)
            all_rms = np.sqrt(np.mean(chunks ** 2, axis=1))
        else:
            all_rms = []
            for i in range(num_frames):
                frame = self.data[i * self.frame_size:(i + 1) * self.frame_size]
                all_rms.append(np.sqrt(np.mean(frame ** 2)))
        new_threshold = np.percentile(all_rms, 25) * 1.5
        self.silence_threshold = max(new_threshold, self.MIN_THRESHOLD)

    def recent_rms(self):
        recent = self.return_last_n_seconds(0.1)
        return np.sqrt(np.mean(recent ** 2))

    def is_silent(self):                                                # :488-496
        if len(self.data) == 0 or self.frame_size == 0:
            return True
        recent = self.return_last_n_seconds(0.1)
        if len(recent) == 0:
            return True
        rms = np.sqrt(np.mean(recent ** 2))
        return bool(rms < self.silence_threshold)

    def return_last_n_seconds(self, n):                                 # :498-513
        n_samples = int(n * self.FREQUENCY)
        if n_samples > len(self.data):
            n_samples = len(self.data)
        if n_samples == 0:
            return np.array([])
        start_index = (self.pointer - n_samples) % self.buffer_length
        if start_index < self.pointer:
            return self.data[start_index:self.pointer].copy()
        return np.concatenate((self.data[start_index:], self.data[: self.pointer])).copy()

    def is_buffer_full(self):                                           # :515-517
        return self.samples_collected >= self.buffer_length


# ------------------------------------------------------------------ A8  _detect_word
WAITING, IN_SILENCE, IN_SOUND, AFTER_SOUND = 0, 1, 2, 3
STATE_NAMES = ("waiting", "in_silence", "in_sound", "after_sound")


def segment_bounds(sound_start_time, sound_end_time, current_time):
    """The float64 arithmetic of wakeword.py:1101-1111 -> (n_back, n_drop): the segment is
    the last n_back samples of the ring minus its final n_drop samples."""
    padding = SEGMENT_PADDING
    extract_start = sound_start_time - current_time - padding
    extract_end = sound_end_time - current_time + padding
    n_back = int(abs(extract_start) * FREQUENCY)       # return_last_n_seconds(abs(extract_start))
    n_drop = int((abs(extract_end)) * FREQUENCY)       # word_end_idx
    return n_back, n_drop


def detect_stream(stream, template, *, block=512, buffer_seconds=10, max_ticks=None,
                  restart_on_timeout=True, fast=False, matcher=None, keep_audio=False, timing=None, ring_samples=None,
                  **params):
    """SoundBuffer + WordMatcher + WakeWord._wait_for_buffer/_detect_word (wakeword.py:1002-1007,
    1036-1159, listen loop 1202-1211) over one stream under the audio clock.

    stream: float32 samples.  template: float32 samples (set_reference).  Level 3 is stubbed to
    "no transcription" (wakeword.py:1152-1155), so a level-2 match only produces an event.
    Returns the same dict layout as oracle.ref_harness.run_reference_stream, plus per-tick state.
    ring_samples: ring length in samples instead of buffer_seconds * 16000.  template=None with a matcher that is None
    skips level 2 (events keep their tick and length, score NaN): the gate's own decisions at any ring length.
    """
    p = dict(DEFAULTS)
    p.update(params)
    thr = p["similarity_threshold"]
    pre, dmin, dmax, post = (p["pre_speech_silence"], p["speech_duration_min"],
                             p["speech_duration_max"], p["post_speech_silence"])
    timeout = p["timeout"]
    stream = np.asarray(stream, dtype=np.float32)
    buf = SoundBufferOracle(seconds=buffer_seconds, fast=fast, ring_samples=ring_samples)
    if matcher is None and template is not None:
        matcher = WordMatcherOracle()
        matcher.set_reference(np.asarray(template, dtype=np.float32))

    k = 0
    fed = 0

    class _Exhausted(Exception):
        pass

    def sleep():
        nonlocal k, fed
        if max_ticks is not None and k >= max_ticks:
            raise _Exhausted
        target = ((k + 1) * TICK_SAMPLES // block) * block
        if target > len(stream):
            raise _Exhausted
        k += 1
        while fed < target:
            buf.add_block(stream[fed:fed + block])
            fed += block

    t_tick, t_silent, t_thr, t_state, t_rms = [], [], [], [], []
    events, timeouts = [], []
    full_tick = None

    def sample():
        silent = buf.is_silent()
        t_tick.append(k)
        t_silent.append(silent)
        t_thr.append(float(buf.silence_threshold))
        t_rms.append(float(buf.recent_rms()) if buf.frame_size else 0.0)
        return silent

    try:
        while not buf.is_buffer_full():                                 # :1002-1007
            sleep()
        full_tick = k
        if timing is not None:
            import time as _time
            timing["t_full"] = _time.perf_counter()
        while True:                                                     # listen loop :1205-1211
            state = WAITING                                             # :1048
            silence_start_time = sound_start_time = sound_end_time = None
            start_time = k * TICK_SECONDS                               # :1052
            if sample():                                                # :1055-1057
                state = IN_SILENCE
                silence_start_time = k * TICK_SECONDS
            t_state.append(state)
            while True:
                if k * TICK_SECONDS - start_time > timeout:             # :1061-1062
                    timeouts.append(k)
                    break
                sleep()                                                 # :1064
                silent = sample()                                       # :1066
                current_time = k * TICK_SECONDS                         # :1067
                if state == WAITING:                                    # :1069-1072
                    if silent:
                        state = IN_SILENCE
                        silence_start_time = current_time
                elif state == IN_SILENCE:                               # :1074-1081
                    if not silent:
                        if current_time - silence_start_time >= pre:
                            state = IN_SOUND
                            sound_start_time = current_time
                        else:
                            state = WAITING
                elif state == IN_SOUND:                                 # :1083-1094
                    sound_duration = current_time - sound_start_time
                    if not silent:
                        if sound_duration > dmax:
                            state = WAITING
                    else:
                        if dmin <= sound_duration <= dmax:
                            state = AFTER_SOUND
                            sound_end_time = current_time
                        else:
                            state = WAITING
                elif state == AFTER_SOUND:                              # :1096-1157
                    if silent:
                        if current_time - sound_end_time >= post:
                            n_back, n_drop = segment_bounds(sound_start_time, sound_end_time, current_time)
                            seg = buf.return_last_n_seconds(abs(sound_start_time - current_time - SEGMENT_PADDING))
                            assert len(seg) == min(n_back, buf.buffer_length)
                            word_audio = seg[: len(seg) - n_drop]
                            if len(word_audio) / FREQUENCY > MAX_SEGMENT_SECONDS:    # :1114-1118
                                state = WAITING
                                t_state.append(state)
                                continue
                            ok, sim = (matcher.matches(word_audio, threshold=thr)    # :1121
                                       if matcher is not None else (False, float("nan")))
                            ev = {"tick": k, "seg_len": int(len(word_audio)), "score": float(sim),
                                  "matched": bool(ok), "n_back": n_back, "n_drop": n_drop}
                            if keep_audio:
                                ev["audio"] = word_audio.copy()
                            events.append(ev)
                            state = WAITING                                           # :1155
                    else:
                        state = WAITING                                               # :1157
                t_state.append(state)
            if not restart_on_timeout:
                break
    except _Exhausted:
        pass
    if timing is not None:
        import time as _time
        timing["t_end"] = _time.perf_counter()
        timing["steady_ticks"] = k - (full_tick or k)
    return {
        "full_tick": full_tick,
        "trace_tick": np.asarray(t_tick, dtype=np.int64),
        "trace_silent": np.asarray(t_silent, dtype=np.bool_),
        "trace_thr": np.asarray(t_thr, dtype=np.float64),
        "trace_rms": np.asarray(t_rms, dtype=np.float64),
        "trace_state": np.asarray(t_state, dtype=np.int8),
        "events": events,
        "timeouts": timeouts,
        "frame_size": int(buf.frame_size),
        "ticks_run": k,
    }


# ------------------------------------------------------------------ A9  dense per-hop scoring
def dense_window(n_template):
    """(n_hops_back, length): the dense window scored at hop h for a template of n_template
    samples is x[160*(h - n_hops_back) : 160*(h - n_hops_back) + n_template] — the latest
    template-length window that STARTS on the hop grid and is complete at hop h."""
    return -(-int(n_template) // 160), int(n_template)


def dense_scores(stream, templates, hops, preemphasis=0.0, n_mfcc=20):
    """A9 (SURVEY §8(a)): for every hop h in `hops` and template k, what
    WordMatcher.calculate_similarity (wakeword.py:591-625) returns when handed the dense
    window of dense_window(len(template_k)).  The usage shape is examples/tune_threshold.py:
    86-116 (consecutive chunks through calculate_similarity) at hop granularity.
    Returns float32 [len(hops), len(templates)]; NaN where the window is not yet available."""
    stream = np.asarray(stream, dtype=np.float32)
    out = np.full((len(hops), len(templates)), np.nan, dtype=np.float32)
    for ki, tpl in enumerate(templates):
        m = WordMatcherOracle(preemphasis=preemphasis, n_mfcc=n_mfcc)
        m.set_reference(np.asarray(tpl, dtype=np.float32))
        nb, ln = dense_window(len(tpl))
        for hi, h in enumerate(hops):
            s = 160 * (int(h) - nb)
            if s < 0 or s + ln > len(stream):
                continue
            out[hi, ki] = m.calculate_similarity(stream[s:s + ln])
    return out


# ------------------------------------------------------------------ N1  level-3 hand-off
def prepare_for_level3(audio_samples):
    """The pre-processing WakeWord._transcribe_audio applies before Whisper (wakeword.py:1020-1025)."""
    audio_samples = audio_samples - np.mean(audio_samples)
    max_val = np.max(np.abs(audio_samples))
    if max_val > 0:
        audio_samples = audio_samples / max_val
    audio_samples = audio_samples * 1.5
    return np.clip(audio_samples, -1.0, 1.0)


# ------------------------------------------------------------------ N2  template analysis
VOICE_ACTIVITY_THRESHOLD = 0.1   # wakeword.py:47
MIN_DETECTED_DURATION = 0.2      # wakeword.py:48


def analyze_reference_audio_duration(audio):
    """WakeWord._analyze_reference_audio_duration after loading (wakeword.py:872-893)."""
    frame_length = int(0.025 * FREQUENCY)
    hop_length = int(0.010 * FREQUENCY)
    rms = L.rms(y=audio, frame_length=frame_length, hop_length=hop_length)[0]
    threshold = np.max(rms) * VOICE_ACTIVITY_THRESHOLD
    voice_frames = rms > threshold
    if np.any(voice_frames):
        idx = np.where(voice_frames)[0]
        duration = (idx[-1] - idx[0]) * hop_length / FREQUENCY
        return max(duration, MIN_DETECTED_DURATION)
    return None


def auto_speech_durations(audio, user_min=None, user_max=None):
    """Contract of the (missing at HEAD, wakeword.py:786) `_auto_calculate_speech_durations`, as
    pinned by tests/test_wakeword_simulated.py:687-775 and README.md:254-289:
    min = VAD duration of the reference WAV (fallback 0.3), max = 2 * min (fallback 2.0);
    user-supplied values win."""
    dur = None
    if user_min is None or user_max is None:
        try:
            dur = analyze_reference_audio_duration(audio)
        except Exception:
            dur = None
    smin = user_min if user_min is not None else (float(dur) if dur is not None else 0.3)
    if user_max is not None:
        smax = user_max
    elif user_min is None and dur is None:
        smax = 2.0
    else:
        smax = 2.0 * smin
    return smin, smax
