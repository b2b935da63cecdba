"""ORACLE — TEST INFRASTRUCTURE ONLY.  Not shipped, not on the product path.

CPU restatement (numpy/scipy) of the third-party arithmetic the reference's hot
path calls but does not vendor:

    librosa == 0.11.0   (pinned in /root/reference/uv.lock:324-325; declared
                         ``librosa>=0.10.0`` at pyproject.toml:27)
    call sites:  easywakeword/wakeword.py:561-563  librosa.feature.mfcc
                 easywakeword/wakeword.py:588      librosa.load
                 easywakeword/wakeword.py:866-878  librosa.load / resample / feature.rms

librosa is not installable in this image (no network), so its *published*
algorithm is restated here and anchored on what the reference holds for this
path: the ``== 100.0`` self-similarity tests, the 89 %+/77 %+ scores of
LEARNINGS.md:92-93 and the reference's own classes run unmodified on top of
this module (oracle/ref_harness.py).  Independent cross-checks: torchaudio's
Slaney mel filterbank and ortho DCT (tests/test_oracle.py).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline
legs may import this file.

numpy / scipy are used directly for what the reference's dependency stack uses
them for (numpy.fft.rfft, scipy.fft.dct, scipy.signal.get_window).
"""
from __future__ import annotations

import functools

import numpy as np
import scipy.fft
import scipy.signal

SR = 16000
N_FFT = 512
HOP = 160
N_MELS = 128
N_MFCC = 20


# --------------------------------------------------------------------------- mel
def hz_to_mel(f):
    """librosa.core.convert.hz_to_mel(htk=False): Slaney auditory-toolbox scale."""
    f = np.asanyarray(f, dtype=np.float64)
    f_sp = 200.0 / 3
    mels = f / f_sp
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    if f.ndim:
        big = f >= min_log_hz
        mels[big] = min_log_mel + np.log(f[big] / min_log_hz) / logstep
    elif f >= min_log_hz:
        mels = min_log_mel + np.log(f / min_log_hz) / logstep
    return mels


def mel_to_hz(m):
    """librosa.core.convert.mel_to_hz(htk=False)."""
    m = np.asanyarray(m, dtype=np.float64)
    f_sp = 200.0 / 3
    freqs = f_sp * m
    min_log_hz = 1000.0
    min_log_mel = min_log_hz / f_sp
    logstep = np.log(6.4) / 27.0
    if m.ndim:
        big = m >= min_log_mel
        freqs[big] = min_log_hz * np.exp(logstep * (m[big] - min_log_mel))
    elif m >= min_log_mel:
        freqs = min_log_hz * np.exp(logstep * (m - min_log_mel))
    return freqs


def mel_frequencies(n_mels, fmin, fmax):
    lo = hz_to_mel(fmin)
    hi = hz_to_mel(fmax)
    return mel_to_hz(np.linspace(lo, hi, n_mels))


@functools.lru_cache(maxsize=8)
def mel_filterbank(sr=SR, n_fft=N_FFT, n_mels=N_MELS, fmin=0.0, fmax=None):
    """librosa.filters.mel(htk=False, norm='slaney', dtype=float32) -> [n_mels, 1+n_fft//2]."""
    if fmax is None:
        fmax = sr / 2.0
    weights = np.zeros((n_mels, 1 + n_fft // 2), dtype=np.float32)
    fftfreqs = np.fft.rfftfreq(n=n_fft, d=1.0 / sr)
    mel_f = mel_frequencies(n_mels + 2, fmin, fmax)
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fftfreqs)
    for i in range(n_mels):
        lower = -ramps[i] / fdiff[i]
        upper = ramps[i + 2] / fdiff[i + 1]
        weights[i] = np.maximum(0, np.minimum(lower, upper))
    enorm = 2.0 / (mel_f[2 : n_mels + 2] - mel_f[:n_mels])
    weights *= enorm[:, np.newaxis]
    weights.setflags(write=False)
    return weights


# -------------------------------------------------------------------------- stft
@functools.lru_cache(maxsize=8)
def hann_window(n=N_FFT):
    """scipy.signal.get_window('hann', n, fftbins=True): periodic Hann, float64."""
    w = scipy.signal.get_window("hann", n, fftbins=True)
    w.setflags(write=False)
    return w


def frame_signal(y, frame_length, hop_length):
    """librosa.util.frame on the last axis -> [frame_length, n_frames] (view)."""
    n_frames = 1 + (len(y) - frame_length) // hop_length
    idx = np.arange(frame_length)[:, None] + hop_length * np.arange(n_frames)[None, :]
    return y[idx]


def stft(y, n_fft=N_FFT, hop_length=HOP):
    """librosa.stft(center=True, pad_mode='constant', window='hann', win_length=n_fft).

    Frame t covers y[hop*t - n_fft//2 : hop*t + n_fft//2] with zeros outside the
    signal; n_frames = 1 + len(y)//hop.  The float64 window promotes the product
    to double, numpy.fft.rfft runs in double, the result is stored in
    complex64 for float32 input (librosa.util.dtype_r2c) / complex128 for float64.
    """
    y = np.asarray(y)
    if y.dtype not in (np.float32, np.float64):
        y = y.astype(np.float32)
    cdtype = np.complex64 if y.dtype == np.float32 else np.complex128
    ypad = np.pad(y, n_fft // 2, mode="constant")
    frames = frame_signal(ypad, n_fft, hop_length)
    win = hann_window(n_fft)[:, None]
    return np.fft.rfft(win * frames, axis=0).astype(cdtype)


def power_to_db(S, amin=1e-10, top_db=80.0):
    """librosa.power_to_db(ref=1.0): 10 log10(max(amin,S)), floor at global max - top_db."""
    S = np.asarray(S)
    log_spec = 10.0 * np.log10(np.maximum(amin, S))
    log_spec -= 10.0 * np.log10(np.maximum(amin, 1.0))
    if top_db is not None:
        log_spec = np.maximum(log_spec, log_spec.max() - top_db)
    return log_spec


def melspectrogram(y, sr=SR, n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS):
    S = np.abs(stft(y, n_fft=n_fft, hop_length=hop_length)) ** 2.0
    mel_basis = mel_filterbank(sr=sr, n_fft=n_fft, n_mels=n_mels)
    return np.einsum("ft,mf->mt", S, mel_basis, optimize=True)


def log_mel(y, sr=SR, n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS, top_db=80.0):
    return power_to_db(melspectrogram(y, sr, n_fft, hop_length, n_mels), top_db=top_db)


def mfcc(y, sr=SR, n_mfcc=N_MFCC, n_fft=N_FFT, hop_length=HOP, n_mels=N_MELS):
    """librosa.feature.mfcc(dct_type=2, norm='ortho', lifter=0) -> [n_mfcc, 1+len(y)//hop]."""
    S = log_mel(y, sr=sr, n_fft=n_fft, hop_length=hop_length, n_mels=n_mels)
    return scipy.fft.dct(S, axis=-2, type=2, norm="ortho")[..., :n_mfcc, :]


def preemphasis(y, coef=0.97):
    """librosa.effects.preemphasis(y, coef=coef, zi=None): ``scipy.signal.lfilter([1, -coef], [1], y, zi=2*y[0] - y[1])``
    in y's dtype — i.e. out[n] = y[n] - coef*y[n-1] for n >= 1 and out[0] = y[0] + (2*y[0] - y[1]): librosa hands its
    "linear extrapolation" value to lfilter as the filter STATE, unscaled (restated from librosa 0.11's effects.py from
    memory; the source is not available offline).  The reference never calls it (wakeword.py:561-563 passes the raw
    segment to librosa.feature.mfcc), so this is the definition of the build's `preemphasis` EXTENSION parameter:
    parity for coef != 0 is unpinned by anything the reference holds."""
    y = np.asarray(y)
    if y.dtype not in (np.float32, np.float64):
        y = y.astype(np.float32)
    b = np.asarray([1.0, -coef], dtype=y.dtype)
    a = np.asarray([1.0], dtype=y.dtype)
    x1 = y[..., 1:2] if y.shape[-1] > 1 else np.zeros_like(y[..., 0:1])
    zi = 2 * y[..., 0:1] - x1
    out, _ = scipy.signal.lfilter(b, a, y, zi=np.asarray(zi, dtype=y.dtype))
    return out.astype(y.dtype, copy=False)


def rms(y, frame_length=2048, hop_length=512):
    """librosa.feature.rms(center=True, pad_mode='constant', dtype=float32) -> [1, n_frames].

    Framed the way librosa.util.frame frames: a strided view [frame_length, n_frames] whose frame-sample axis (-2)
    is contiguous, squared in float32 (util.abs2) and averaged with np.mean over that axis.  Because the reduced axis
    is contiguous, numpy runs its pairwise float32 sum once per frame; oracle/vad_model.py states that sum's shape
    and tests/test_vad_model.py pins the two together.  (frame_signal's fancy-indexed [frame_length, n_frames] copy
    would reduce row by row instead and differs from librosa in the last bit of about half of all frames.)"""
    y = np.asarray(y)
    ypad = np.pad(y, frame_length // 2, mode="constant")
    n_frames = 1 + (len(ypad) - frame_length) // hop_length
    s = ypad.strides[-1]
    x = np.lib.stride_tricks.as_strided(ypad, shape=(frame_length, n_frames), strides=(s, hop_length * s),
                                        writeable=False)
    power = np.mean(np.square(x, dtype=np.float32), axis=-2, keepdims=True)
    return np.sqrt(power)


# -------------------------------------------------------------------- WAV (PCM16)
def wav_read_pcm16(path):
    """-> (int16 mono-or-multichannel array [n] or [n, ch], sample_rate). stdlib `wave`."""
    import wave

    with wave.open(str(path), "rb") as w:
        if w.getsampwidth() != 2:
            raise ValueError("only PCM16 WAV is supported by the oracle reader")
        sr = w.getframerate()
        ch = w.getnchannels()
        raw = w.readframes(w.getnframes())
    pcm = np.frombuffer(raw, dtype="<i2")
    if ch > 1:
        pcm = pcm.reshape(-1, ch)
    return pcm, sr


def wav_write_pcm16(path, audio, sr):
    """libsndfile semantics for float input to a PCM_16 WAV: lrint(x * 32767) (no clipping
    below full scale); integer input is written as is."""
    import wave

    a = np.asarray(audio)
    if a.dtype.kind == "f":
        a = np.clip(np.rint(a.astype(np.float64) * 32767.0), -32768, 32767).astype("<i2")
    else:
        a = a.astype("<i2")
    ch = 1 if a.ndim == 1 else a.shape[1]
    with wave.open(str(path), "wb") as w:
        w.setnchannels(ch)
        w.setsampwidth(2)
        w.setframerate(int(sr))
        w.writeframes(a.tobytes())


def load(path, sr=SR):
    """librosa.load(path, sr=sr, mono=True): float32 = int16/32768, mono mix-down.
    Resampling (soxr_hq in librosa) is outside the hot path: only native-rate files."""
    pcm, native = wav_read_pcm16(path)
    y = pcm.astype(np.float32) / np.float32(32768.0)
    if y.ndim > 1:
        y = np.mean(y, axis=1, dtype=np.float32)
    if sr is not None and native != sr:
        raise NotImplementedError(
            f"oracle: resampling {native}->{sr} Hz is not restated (SURVEY §8(f) N3)"
        )
    return y, native
