"""Drop-in host surface: WakeWord / WordMatcher / SoundBuffer with the reference's names, defaults,
argument meaning and exceptions (/root/reference/easywakeword/wakeword.py:405-1240), backed by libewk.

The seam is the one the reference itself uses: WakeWord owns two duck-typed attributes,
``_sound_buffer`` and ``_matcher`` (wakeword.py:989-997).  Here both are thin facades over a device
context: the ring lives in HBM, ``is_silent`` is one K2 launch, ``matches`` is one K3 launch.  The
level-4 shell (threads, callback, timeout, level-3 text check) stays host Python, as in the reference.
There is no CPU fallback: constructing a facade without the CUDA library or a GPU raises.

For many streams use easywakeword_b200.bank.WakeWordBank, where the timing state machine itself
runs on the device.
"""
from __future__ import annotations

import inspect
import logging
import os
import threading
import time
import warnings
from typing import Callable, Dict, Optional, Union

import numpy as np

from . import _lib

logger = logging.getLogger(__name__)

# wakeword.py:31-48
DEFAULT_BUFFER_SECONDS = 10
DEFAULT_RETRY_COUNT = 3
DEFAULT_RETRY_BACKOFF = 0.5
DEFAULT_PRE_SPEECH_SILENCE = 0.8
DEFAULT_SPEECH_DURATION_MIN = 0.3
DEFAULT_SPEECH_DURATION_MAX = 2.0
DEFAULT_POST_SPEECH_SILENCE = 0.4
AUTO_CALCULATE = None
VOICE_ACTIVITY_THRESHOLD = 0.1
MIN_DETECTED_DURATION = 0.2

_shared_ctx = {}
_shared_lock = threading.Lock()


def shared_matcher_context(device: int = 0, preemphasis: float = 0.0, n_mfcc: int = 0):
    """One stream-less context per (CUDA device, front-end parameters) and process for WordMatcher facades
    (templates are per-facade slots)."""
    key = (int(device), float(preemphasis), int(n_mfcc) or 20)
    with _shared_lock:
        ctx = _shared_ctx.get(key)
        if ctx is None or not ctx.h:
            ctx = _lib.Context(device=device, n_streams=0, max_templates=64, preemphasis=preemphasis, n_mfcc=n_mfcc)
            ctx._slot_free = list(range(63, -1, -1))
            ctx._lock = threading.Lock()
            _shared_ctx[key] = ctx
        return ctx


def load_wav_16k(path: str, sample_rate: int = 16000, *, ctx=None) -> np.ndarray:
    """What ``librosa.load(path, sr=16000)`` yields (wakeword.py:588): float32 = PCM / full scale, mono
    mix-down, and — for files at another rate — conversion to 16 kHz on the device (resample.py, K7)."""
    if sample_rate != 16000:
        raise ValueError("easywakeword_b200 works at 16000 Hz (SoundBuffer.FREQUENCY)")
    from .resample import load_16k
    return load_16k(str(path), ctx=ctx)


class WordMatcher:
    """MFCC matcher (reference: wakeword.py:520-639); the arithmetic runs in the fused K3 kernel."""

    def __init__(self, sample_rate: int = 16000, *, context=None, device: int = 0, preemphasis: float = 0.0,
                 n_mfcc: int = 20) -> None:
        """preemphasis / n_mfcc: the front-end parameters the reference hard-codes (none / 20, wakeword.py:561-563) and
        lists as "expose" on its roadmap (LEARNINGS.md:87); the defaults are the reference's."""
        self.sample_rate: int = sample_rate
        self.reference_mfcc_mean: Optional[np.ndarray] = None
        self.reference_mfcc_std: Optional[np.ndarray] = None
        self.reference_word: Optional[str] = None
        self._ctx = context if context is not None else shared_matcher_context(device, preemphasis, n_mfcc)
        self._owns_slot = hasattr(self._ctx, "_slot_free")
        self._slot = self._ctx._slot_free.pop() if self._owns_slot else 0
        self._lock = getattr(self._ctx, "_lock", threading.Lock())

    def __del__(self):
        try:
            if self._owns_slot and self._ctx.h:
                self._ctx._slot_free.append(self._slot)
        except Exception:
            pass

    def extract_mfcc(self, audio: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
        """(mean[20], std[20]) of the MFCC frames of `audio` (wakeword.py:544-567)."""
        with self._lock:
            return self._ctx.extract_mfcc(np.asarray(audio))

    def mfcc(self, audio: np.ndarray) -> np.ndarray:
        """The [20, 1 + n//160] frame matrix extract_mfcc pools (librosa layout)."""
        with self._lock:
            return self._ctx.extract_mfcc(np.asarray(audio), want_frames=True)[2].T.copy()

    def set_reference(self, audio: np.ndarray, word_name: str = "target") -> None:
        """wakeword.py:569-578"""
        self.reference_word = word_name
        a = np.ascontiguousarray(audio, dtype=np.float32).reshape(-1)
        with self._lock:
            self._ctx.set_template(self._slot, a)
            self.reference_mfcc_mean, self.reference_mfcc_std, _ = self._ctx.get_template(self._slot)

    def load_reference_from_file(self, filepath: str, word_name: str = "target") -> None:
        """wakeword.py:580-589"""
        self.set_reference(load_wav_16k(filepath, self.sample_rate), word_name)

    def calculate_similarity(self, audio: np.ndarray) -> float:
        """0-100 similarity (wakeword.py:591-625); ValueError when no reference is set."""
        if self.reference_mfcc_mean is None:
            raise ValueError("No reference word set. Call set_reference() first.")
        a = np.ascontiguousarray(audio, dtype=np.float32).reshape(-1)
        with self._lock:
            scores, _ = self._ctx.similarity_batch(self._slot, a, [0], [len(a)])
        return scores[0]

    def matches(self, audio: np.ndarray, threshold: float = 75.0) -> tuple[bool, float]:
        """(similarity >= threshold, similarity)  (wakeword.py:627-639)"""
        similarity = self.calculate_similarity(audio)
        return bool(similarity >= threshold), similarity


class SoundBuffer:
    """Circular audio buffer with silence detection (reference: wakeword.py:405-517).

    The ring is a device ring of one stream in "live" mode: every `_add_sound_to_buffer` callback is
    one K1 push, every `is_silent()` one K2 tick that sees everything pushed so far.
    `source` replaces the PortAudio stream for tests and file playback (anything with start/stop)."""

    FREQUENCY = 16000
    MIN_THRESHOLD = 0.005
    MIN_FRAME_SIZE = 160     # libewk: smallest callback block the device gate chunks by (ewk_set_stream_params)
    MAX_CHUNKS = 2048        # libewk: storage-order chunks a gate warp holds in shared memory (ewk_tick)

    def __init__(self, seconds: int = DEFAULT_BUFFER_SECONDS, device: Optional[Union[int, str]] = None, *,
                 cuda_device: int = 0, source=None):
        self.buffer_seconds = seconds
        self.buffer_length = self.buffer_seconds * self.FREQUENCY
        self.frame_size = 0
        self.samples_collected = 0
        self._written = 0
        self._lock = threading.Lock()
        self._ctx = _lib.Context(device=cuda_device, n_streams=1, ring_samples=int(self.buffer_length),
                                 slack_samples=1600, pcm_format=_lib.PCM_F32, max_templates=1)
        self._ctx.set_stream_params(0, live=1, min_threshold=self.MIN_THRESHOLD, timeout=0.0)
        self._threshold_cache = 0.01
        self._dirty = False
        if source is not None:
            self.sd_stream = source
        else:
            try:
                import sounddevice as sd
            except Exception as e:  # the reference documents OSError for a missing device (wakeword.py:423-424)
                raise OSError(f"no audio input backend available: {e}") from e
            self.sd_stream = sd.InputStream(samplerate=self.FREQUENCY, channels=1,
                                            callback=self._add_sound_to_buffer, device=device)
        self.sd_stream.start()

    def stop(self) -> None:
        self.sd_stream.stop()

    def start(self) -> None:
        self.sd_stream.start()

    def _add_sound_to_buffer(self, indata, frames, time_info, status) -> None:
        """PortAudio callback (wakeword.py:454-470)."""
        new_data = np.ascontiguousarray(np.asarray(indata, dtype=np.float32).reshape(-1))
        if len(new_data) == 0:
            return
        with self._lock:
            if self.frame_size == 0:
                # the adaptive threshold works on ring_length // frame_size chunks of the FIRST callback's length
                # (wakeword.py:457-458, 477-478); the device gate keeps them in shared memory
                n = len(new_data)
                if n < self.MIN_FRAME_SIZE or self.buffer_length // n > self.MAX_CHUNKS:
                    raise ValueError(f"SoundBuffer: a first callback of {n} samples is not supported with a "
                                     f"{self.buffer_seconds} s ring: the block must hold at least {self.MIN_FRAME_SIZE} samples and "
                                     f"ring_length // block may not exceed {self.MAX_CHUNKS} (use a PortAudio blocksize "
                                     f">= {max(self.MIN_FRAME_SIZE, -(-self.buffer_length // self.MAX_CHUNKS))})")
                self.frame_size = n
            for p in range(0, len(new_data), self.buffer_length):
                self._ctx.push(new_data[p:p + self.buffer_length].reshape(1, -1))
            self._written += len(new_data)
            self.samples_collected = min(self.buffer_length, self.samples_collected + len(new_data))
            self._dirty = True

    @property
    def pointer(self) -> int:
        return self._written % self.buffer_length

    @property
    def silence_threshold(self) -> float:
        """Adaptive threshold max(1.5 * P25(chunk RMS), 0.005) once the ring is full (wakeword.py:472-486)."""
        with self._lock:
            self._refresh()
            return self._threshold_cache

    @property
    def data(self) -> np.ndarray:
        """The ring in the reference's storage order (float64 like wakeword.py:428)."""
        with self._lock:
            last = self._ctx.read_last(0, min(self._written, self.buffer_length)) if self._written else np.zeros(0, np.float32)
        out = np.zeros(self.buffer_length)
        n = len(last)
        idx = (self._written - n + np.arange(n)) % self.buffer_length
        out[idx] = last
        return out

    def _refresh(self):
        if self._dirty:
            self._ctx.tick(1)
            self._dirty = False
            st = self._ctx.status(0)
            self._threshold_cache = float(st.silence_threshold)
            self._silent_cache = bool(st.is_silent)

    def is_silent(self) -> bool:
        """RMS of the last 0.1 s below the adaptive threshold (wakeword.py:488-496)."""
        if self.buffer_length == 0 or self.frame_size == 0:
            return True
        with self._lock:
            self._refresh()
            return self._silent_cache

    def return_last_n_seconds(self, n: float) -> np.ndarray:
        """Last n seconds with wrap-around (wakeword.py:498-513); float64 copy like the reference."""
        n_samples = int(n * self.FREQUENCY)
        if n_samples > self.buffer_length:
            n_samples = self.buffer_length
        if n_samples == 0:
            return np.array([])
        with self._lock:
            return self._ctx.read_last(0, n_samples).astype(np.float64)

    def is_buffer_full(self) -> bool:
        return self.samples_collected >= self.buffer_length


def template_frame_rms(audio: np.ndarray) -> np.ndarray:
    """Frame RMS of the reference's voice-activity rule: 25 ms frames every 10 ms, zero-padded centring.
    The audio is taken as float32, as librosa.load returns it.  Each frame is a contiguous row, so its mean square is
    numpy's pairwise float32 sum over the row: the arithmetic of librosa.feature.rms, and of K6."""
    frame_length = int(0.025 * SoundBuffer.FREQUENCY)
    hop_length = int(0.010 * SoundBuffer.FREQUENCY)
    y = np.pad(np.asarray(audio, dtype=np.float32).reshape(-1), frame_length // 2)
    n_frames = 1 + (len(y) - frame_length) // hop_length
    idx = np.arange(frame_length)[None, :] + hop_length * np.arange(n_frames)[:, None]
    return np.sqrt(np.mean(np.abs(y[idx]) ** 2, axis=1))


def analyze_reference_audio_duration(audio: np.ndarray) -> Optional[float]:
    """Speech duration of a template by the reference's RMS voice-activity rule (wakeword.py:872-893):
    frames above 0.1 * max RMS (template_frame_rms), first-to-last span."""
    hop_length = int(0.010 * SoundBuffer.FREQUENCY)
    rms = template_frame_rms(audio)
    voiced = np.where(rms > np.max(rms) * VOICE_ACTIVITY_THRESHOLD)[0]
    if len(voiced) == 0:
        return None
    return max((voiced[-1] - voiced[0]) * hop_length / SoundBuffer.FREQUENCY, MIN_DETECTED_DURATION)


def _accepts_initial_prompt(t) -> bool:
    try:
        sig = inspect.signature(t.transcribe)
    except (TypeError, ValueError):
        return False
    return "initial_prompt" in sig.parameters or any(p.kind == p.VAR_KEYWORD for p in sig.parameters.values())


class _LocalWhisper:
    """The reference's bundled level-3 backend (transcriber.py:11-140: openai-whisper "tiny", language="en",
    fp16=False), loaded lazily.  Out of the accelerated path: this is the host-side hand-off only."""

    def __init__(self, model_name: str = "tiny"):
        self.model_name = model_name
        self._model = None

    @classmethod
    def if_available(cls):
        import importlib.util
        try:
            ok = importlib.util.find_spec("whisper") is not None
        except (ImportError, ValueError):
            ok = False
        return cls() if ok else None

    def load_model(self) -> bool:
        if self._model is None:
            import whisper
            self._model = whisper.load_model(self.model_name)
        return True

    def transcribe(self, audio: np.ndarray, initial_prompt: Optional[str] = None) -> Optional[str]:
        self.load_model()
        kw = {"initial_prompt": initial_prompt} if initial_prompt else {}
        result = self._model.transcribe(np.asarray(audio, dtype=np.float32), language="en", fp16=False, **kw)
        return result.get("text", "").strip()


class WakeWord:
    """Wake-word detector with the reference's public surface (wakeword.py:642-1240):
    ``WakeWord(textword, wavword, ...)``, ``waitforit()``, ``start()`` / ``stop()`` / ``callback``.

    Levels 1 and 2 run on the GPU through ``_sound_buffer`` / ``_matcher``; level 3 uses the object
    passed as ``transcriber`` (anything with ``transcribe(audio) -> str``), else openai-whisper if it
    is importable (the reference's bundled backend, transcriber.py:11-140), else no confirmation.
    """

    def __init__(self, textword: str, wavword: str, numberofwords: int = 2, timeout: int = 30,
                 callback: Optional[Callable[[str], None]] = None, device: Optional[Union[int, str]] = None,
                 similarity_threshold: float = 75.0, pre_speech_silence: float = DEFAULT_PRE_SPEECH_SILENCE,
                 speech_duration_min: Optional[float] = AUTO_CALCULATE,
                 speech_duration_max: Optional[float] = AUTO_CALCULATE,
                 post_speech_silence: float = DEFAULT_POST_SPEECH_SILENCE,
                 buffer_seconds: int = DEFAULT_BUFFER_SECONDS, verbose: bool = False,
                 retry_count: int = DEFAULT_RETRY_COUNT, retry_backoff: float = DEFAULT_RETRY_BACKOFF,
                 external_whisper_url: Optional[str] = None, stt_backend: str = "bundled",
                 session_headers: Optional[Dict[str, str]] = None, *, transcriber=None, cuda_device: int = 0):
        # same checks, same messages (wakeword.py:743-763; asserted by the reference's tests)
        if numberofwords < 1:
            raise ValueError("numberofwords must be at least 1")
        if buffer_seconds <= 0:
            raise ValueError("buffer_seconds must be positive")
        if retry_count < 0:
            raise ValueError("retry_count must be non-negative")
        if retry_backoff < 0:
            raise ValueError("retry_backoff must be non-negative")
        if pre_speech_silence <= 0:
            raise ValueError("pre_speech_silence must be positive")
        if speech_duration_min is not None and speech_duration_min <= 0:
            raise ValueError("speech_duration_min must be positive")
        if speech_duration_max is not None and speech_duration_max <= 0:
            raise ValueError("speech_duration_max must be positive")
        if (speech_duration_min is not None and speech_duration_max is not None
                and speech_duration_min > speech_duration_max):
            raise ValueError("speech_duration_min must be <= speech_duration_max")
        if post_speech_silence <= 0:
            raise ValueError("post_speech_silence must be positive")

        self.textword = textword.lower().strip()
        self.wavword = wavword
        self.numberofwords = numberofwords
        self.timeout = timeout
        self.callback = callback
        self.device = device
        self.similarity_threshold = similarity_threshold
        self.buffer_seconds = buffer_seconds
        self.verbose = verbose
        self.retry_count = retry_count
        self.retry_backoff = retry_backoff
        self.cuda_device = cuda_device
        self._user_speech_duration_min = speech_duration_min
        self._user_speech_duration_max = speech_duration_max
        self.pre_speech_silence = pre_speech_silence
        self.post_speech_silence = post_speech_silence
        self._auto_calculate_speech_durations()
        self._sound_buffer = None
        self._matcher = None
        self._listening = False
        self._listen_thread: Optional[threading.Thread] = None
        self._stop_event = threading.Event()
        # Level 3 stays on the host and on its existing backend (SURVEY §2 row 8: out of the accelerated path).  The
        # reference always builds its bundled WhisperTranscriber (wakeword.py:795); here an injected `transcriber` wins,
        # else openai-whisper is used when importable, else the caller is told — loudly — that no confirmation exists.
        self.external_whisper_url = external_whisper_url
        self.stt_backend = stt_backend
        self.session_headers = session_headers
        ignored = [n for n, v, d in (("external_whisper_url", external_whisper_url, None), ("stt_backend", stt_backend, "bundled"),
                                     ("session_headers", session_headers, None)) if v != d]
        if ignored:
            warnings.warn(f"easywakeword_b200.WakeWord ignores {', '.join(ignored)}: only the local level-3 backend "
                          "(an injected `transcriber` or openai-whisper) is supported; levels 1-2 run on the GPU",
                          RuntimeWarning, stacklevel=2)
        self._transcriber = transcriber if transcriber is not None else _LocalWhisper.if_available()
        if self._transcriber is None:
            warnings.warn("easywakeword_b200.WakeWord: no level-3 speech-to-text backend (no `transcriber` given and "
                          "openai-whisper is not importable): MFCC matches cannot be confirmed, so waitforit() will end "
                          "in TimeoutError and start() will never call the callback.  Pass transcriber=<object with "
                          "transcribe(audio) -> str> or install openai-whisper.", RuntimeWarning, stacklevel=2)
        self._log(f"Initialized WakeWord detector for '{self.textword}'")

    def _log(self, message: str, level: int = logging.DEBUG) -> None:
        if self.verbose:
            logger.log(level, message)

    def _auto_calculate_speech_durations(self) -> None:
        """min = VAD duration of the reference WAV (fallback 0.3 s), max = 2 x min (fallback 2.0 s);
        user values win.  HEAD of the reference calls this method without defining it (wakeword.py:786);
        the contract is the one its tests and README pin (tests/test_wakeword_simulated.py:687-775,
        README.md:254-289)."""
        duration = None
        if self._user_speech_duration_min is None:
            try:
                duration = analyze_reference_audio_duration(load_wav_16k(self.wavword, SoundBuffer.FREQUENCY))
            except Exception as e:
                self._log(f"Could not analyze reference audio duration: {e}", logging.WARNING)
        if self._user_speech_duration_min is not None:
            self.speech_duration_min = self._user_speech_duration_min
        else:
            self.speech_duration_min = float(duration) if duration is not None else DEFAULT_SPEECH_DURATION_MIN
        if self._user_speech_duration_max is not None:
            self.speech_duration_max = self._user_speech_duration_max
        elif self._user_speech_duration_min is None and duration is None:
            self.speech_duration_max = DEFAULT_SPEECH_DURATION_MAX
        else:
            self.speech_duration_max = 2.0 * self.speech_duration_min

    def check_transcriber_health(self) -> Dict[str, Union[bool, str, float]]:
        t = self._transcriber
        return {"healthy": True, "model_loaded": bool(t is not None and getattr(t, "_model", getattr(t, "model", None)) is not None),
                "backend": "internal_whisper"}

    def _initialize_audio(self) -> None:
        """wakeword.py:989-1000"""
        if self._sound_buffer is None:
            self._sound_buffer = SoundBuffer(seconds=self.buffer_seconds, device=self.device, cuda_device=self.cuda_device)
            self._log(f"Audio buffer initialized: {self.buffer_seconds}s")
        if self._matcher is None:
            self._matcher = WordMatcher(sample_rate=SoundBuffer.FREQUENCY, device=self.cuda_device)
            self._matcher.load_reference_from_file(self.wavword, self.textword)
            self._log(f"Word matcher initialized with reference: {self.wavword}")
        if self._transcriber is not None and hasattr(self._transcriber, "load_model"):
            self._transcriber.load_model()

    def _wait_for_buffer(self) -> None:
        while not self._sound_buffer.is_buffer_full():
            if self._stop_event.is_set():
                return
            time.sleep(0.1)

    @staticmethod
    def prepare_for_transcription(audio_samples: np.ndarray) -> np.ndarray:
        """DC removal, peak normalisation, x1.5, clip: what level 3 is handed (wakeword.py:1020-1025)."""
        audio_samples = audio_samples - np.mean(audio_samples)
        max_val = np.max(np.abs(audio_samples))
        if max_val > 0:
            audio_samples = audio_samples / max_val
        return np.clip(audio_samples * 1.5, -1.0, 1.0)

    def _transcribe_audio(self, audio_samples: np.ndarray) -> Optional[str]:
        if self._transcriber is None:
            self._log("No level-3 transcriber configured", logging.WARNING)
            return None
        try:
            audio = self.prepare_for_transcription(audio_samples)
            if _accepts_initial_prompt(self._transcriber):      # wakeword.py:1029 passes initial_prompt=f"Wake word: ..."
                text = self._transcriber.transcribe(audio, initial_prompt=f"Wake word: {self.textword}")
            else:
                text = self._transcriber.transcribe(audio)
            self._log(f"Transcription result: '{text}'")
            return text
        except Exception as e:
            self._log(f"Transcription failed: {e}", logging.ERROR)
            return None

    def _confirm(self, word_audio) -> Optional[str]:
        """Level 3: word-count and all-words check on the transcription (wakeword.py:1126-1153)."""
        transcription = self._transcribe_audio(word_audio)
        if not transcription:
            self._log("Transcription failed, cannot confirm detection")
            return None
        clean = transcription.strip().lower().rstrip(".,!?;:")
        heard = clean.split()
        if len(heard) != self.numberofwords:
            self._log(f"Word count mismatch: expected {self.numberofwords}, got {len(heard)} ('{clean}')")
            return None
        if all(w in heard for w in self.textword.split()):
            self._log(f"Wake word detected: '{transcription}'")
            return transcription
        self._log(f"Target words not found in transcription: '{clean}' vs '{self.textword}'")
        return None

    def _detect_word(self) -> Optional[str]:
        """One run of the three-level loop (wakeword.py:1036-1159), polling every 100 ms."""
        machine = TimingMachine(self.pre_speech_silence, self.speech_duration_min, self.speech_duration_max,
                                self.post_speech_silence)
        start_time = time.time()
        machine.enter(self._sound_buffer.is_silent(), time.time())
        while not self._stop_event.is_set():
            if time.time() - start_time > self.timeout:
                raise TimeoutError(f"Wake word detection timed out after {self.timeout} seconds")
            time.sleep(0.1)
            silent = self._sound_buffer.is_silent()
            now = time.time()
            cut = machine.step(silent, now)
            if cut is None:
                continue
            back_seconds, n_drop = cut
            samples = self._sound_buffer.return_last_n_seconds(back_seconds)
            word_audio = samples[: len(samples) - n_drop]
            if len(word_audio) / SoundBuffer.FREQUENCY > 3.0:
                self._log("Audio segment too long, skipping")
                continue
            matches, similarity = self._matcher.matches(word_audio, threshold=self.similarity_threshold)
            self._log(f"MFCC similarity: {similarity:.1f}%")
            if matches:
                text = self._confirm(word_audio)
                if text is not None:
                    return text
        return None

    def waitforit(self) -> str:
        """Blocking detection; TimeoutError after `timeout` seconds (wakeword.py:1161-1182)."""
        self._initialize_audio()
        self._stop_event.clear()
        self._listening = True
        try:
            self._wait_for_buffer()
            result = self._detect_word()
            if result is None:
                raise TimeoutError(f"Wake word detection timed out after {self.timeout} seconds")
            return result
        finally:
            self._listening = False

    def start(self) -> None:
        """Background listening; needs a callback (wakeword.py:1184-1216)."""
        if self.callback is None:
            raise ValueError("Callback must be set for async operation. Use waitforit() for synchronous operation.")
        if self._listening:
            return
        self._initialize_audio()
        self._stop_event.clear()
        self._listening = True

        def listen_loop():
            try:
                self._wait_for_buffer()
                while not self._stop_event.is_set():
                    try:
                        result = self._detect_word()
                        if result and self.callback:
                            self.callback(result)
                    except TimeoutError:
                        continue
            finally:
                self._listening = False

        self._listen_thread = threading.Thread(target=listen_loop, daemon=True)
        self._listen_thread.start()

    def stop(self) -> None:
        """wakeword.py:1218-1227 (safe on half-built objects)"""
        if getattr(self, "_stop_event", None):
            self._stop_event.set()
        t = getattr(self, "_listen_thread", None)
        if t and t.is_alive():
            t.join(timeout=2.0)
        if getattr(self, "_sound_buffer", None):
            self._sound_buffer.stop()
        if hasattr(self, "_listening"):
            self._listening = False

    def is_listening(self) -> bool:
        return self._listening

    def __del__(self):
        try:
            self.stop()
        except Exception:
            pass


class TimingMachine:
    """The level-1 timing rules of WakeWord._detect_word (wakeword.py:1048-1057, 1069-1111, 1155-1157)
    as an explicit state machine; K2 runs the same transitions on the device for the batched case.

    step(silent, now) returns None, or (seconds_back, n_drop) when a candidate word is complete:
    the word is the last `seconds_back` seconds of the ring minus its final `n_drop` samples."""

    WAITING, IN_SILENCE, IN_SOUND, AFTER_SOUND = range(4)

    def __init__(self, pre, dmin, dmax, post, padding=0.05, frequency=16000):
        self.pre, self.dmin, self.dmax, self.post = pre, dmin, dmax, post
        self.padding, self.frequency = padding, frequency
        self.state = self.WAITING
        self.t_silence = self.t_sound = self.t_end = None

    def enter(self, silent, now):
        self.state = self.WAITING
        if silent:
            self.state, self.t_silence = self.IN_SILENCE, now

    def step(self, silent, now):
        s = self.state
        if s == self.WAITING:
            if silent:
                self.state, self.t_silence = self.IN_SILENCE, now
        elif s == self.IN_SILENCE:
            if not silent:
                if now - self.t_silence >= self.pre:
                    self.state, self.t_sound = self.IN_SOUND, now
                else:
                    self.state = self.WAITING
        elif s == self.IN_SOUND:
            dur = now - self.t_sound
            if not silent:
                if dur > self.dmax:
                    self.state = self.WAITING
            elif self.dmin <= dur <= self.dmax:
                self.state, self.t_end = self.AFTER_SOUND, now
            else:
                self.state = self.WAITING
        elif s == self.AFTER_SOUND:
            if not silent:
                self.state = self.WAITING
            elif now - self.t_end >= self.post:
                back = abs(self.t_sound - now - self.padding)
                n_drop = int(abs(self.t_end - now + self.padding) * self.frequency)
                self.state = self.WAITING
                return back, n_drop
        return None
