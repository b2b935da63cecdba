"""Ingest of audio that is not 16 kHz mono PCM16 (SURVEY §8(f) N3): WAV decoding on the host, sample-rate
conversion to 16 kHz on the device (K7, ``ewk_resample``).

The reference delegates both to ``librosa.load(path, sr=16000)`` / ``librosa.resample`` (soxr HQ;
/root/reference/easywakeword/wakeword.py:588, 866-870, examples/tune_threshold.py:33-47).  The framing is
librosa's (float32 = integer PCM / full scale, channel mean, output length ceil(n * 16000 / sr), sample n at input
time n * sr / 16000); the filter meets soxr HQ's published specification but is not soxr bit for bit — see
include/ewk.h and oracle/resample_restated.py.  There is no CPU fallback: without the CUDA library this raises."""
from __future__ import annotations

import struct
from typing import Optional

import numpy as np

from . import _lib

TARGET_SR = 16000


def _context(ctx=None, device: int = 0):
    if ctx is not None:
        return ctx
    from .wakeword import shared_matcher_context
    return shared_matcher_context(device)


def resample_to_16k(y, sr_native: int, sr_target: int = TARGET_SR, *, ctx=None, device: int = 0) -> np.ndarray:
    """``librosa.resample(y, orig_sr=sr_native, target_sr=16000)`` on the device.  y: [n] or [rows, n]."""
    if sr_target != TARGET_SR:
        raise ValueError("easywakeword_b200 works at 16000 Hz (SoundBuffer.FREQUENCY)")
    y = np.asarray(y)
    if sr_native == sr_target:
        return y.astype(np.float32, copy=False)
    if y.shape[-1] == 0:
        return np.zeros(y.shape, np.float32)
    c = _context(ctx, device)
    lock = getattr(c, "_lock", None)
    if lock is not None:
        with lock:
            return c.resample(y, sr_native)
    return c.resample(y, sr_native)


def ready_outputs(n_in: int, half_width: int, up: int, down: int) -> int:
    """16 kHz outputs computable from the first n_in input samples: output n needs input up to floor(n * down / up) + W
    (what ``StreamResampler.push`` emits, and what ``Context.push_resampled`` lands)."""
    a = n_in - half_width
    return (a * up + down - 1) // down if a > 0 else 0


def landed_counts(positions, n_in: int, sr_in: int) -> np.ndarray:
    """16 kHz samples a push of n_in inputs at sr_in lands on streams that had received `positions` inputs
    (ewk_push_resampled_each): ready(c + n_in) - ready(c) per stream."""
    from . import _lib
    W, L, M = _lib.resample_info(sr_in)
    return np.array([ready_outputs(int(c) + n_in, W, L, M) - ready_outputs(int(c), W, L, M) for c in positions],
                    dtype=np.int64)


def due_ticks(written, ticks, max_ticks=None) -> np.ndarray:
    """Ticks a stream may take under ewk_tick_ready: tick k is due once 1600 k samples have landed, so a stream that
    landed `written` 16 kHz samples and took `ticks` ticks has max(0, written // 1600 - ticks) due, at most max_ticks."""
    due = np.maximum(0, np.asarray(written, dtype=np.int64) // 1600 - np.asarray(ticks, dtype=np.int64))
    return due if max_ticks is None else np.minimum(due, int(max_ticks))


def due_hops(written, next_hop, max_hops=None) -> np.ndarray:
    """Hops ewk_dense_ready scores: hop h is due once 160 h samples have landed, so a stream that landed `written`
    16 kHz samples and whose dense cursor is at `next_hop` has max(0, written // 160 + 1 - next_hop) due (hops
    next_hop, next_hop + 1, ...), at most max_hops."""
    due = np.maximum(0, np.asarray(written, dtype=np.int64) // 160 + 1 - np.asarray(next_hop, dtype=np.int64))
    return due if max_hops is None else np.minimum(due, int(max_hops))


class StreamResampler:
    """Chunked conversion of [rows, n] feeds to 16 kHz whose concatenated output equals the one-shot result
    sample for sample: every call is given the filter's half-width of history and emits only the outputs whose
    look-ahead has arrived; ``flush()`` emits the rest (zeros beyond the end, like the one-shot form)."""

    def __init__(self, sr_in: int, rows: int, *, ctx=None, device: int = 0, dtype=np.int16):
        self.sr_in, self.rows = int(sr_in), int(rows)
        self.W, self.up, self.down = _lib.resample_info(sr_in)
        self.ctx = _context(ctx, device)
        self.dtype = np.dtype(dtype)
        self.hist = np.zeros((rows, 0), self.dtype)      # input samples [hist_first, n_in)
        self.hist_first = 0
        self.n_in = 0                                     # input samples received
        self.n_out = 0                                    # output samples emitted

    def _emit(self, upto_out: int) -> np.ndarray:
        n = upto_out - self.n_out
        if n <= 0:
            return np.zeros((self.rows, 0), np.float32)
        out = self.ctx.resample(self.hist, self.sr_in, in_first=self.hist_first, out_first=self.n_out, n_out=n)
        self.n_out = upto_out
        # keep what later outputs still need: taps start at floor(n_out * down / up) - W + 1
        keep_from = max(self.hist_first, self.n_out * self.down // self.up - self.W + 1, 0)
        self.hist = np.ascontiguousarray(self.hist[:, keep_from - self.hist_first:])
        self.hist_first = keep_from
        return out

    def push(self, chunk) -> np.ndarray:
        """chunk [rows, n] at sr_in -> the newly computable 16 kHz samples [rows, m]."""
        chunk = np.asarray(chunk, self.dtype).reshape(self.rows, -1)
        self.hist = np.concatenate([self.hist, chunk], axis=1)
        self.n_in += chunk.shape[1]
        return self._emit(max(ready_outputs(self.n_in, self.W, self.up, self.down), self.n_out))

    def flush(self) -> np.ndarray:
        total = int(_lib.load().ewk_resample_out_len(self.n_in, self.sr_in))
        return self._emit(max(total, self.n_out))


# ------------------------------------------------------------------------------------------------ WAV
def _g711_tables():
    """ITU-T G.711 expansion tables, code -> 16-bit linear sample (what libsndfile's ulaw / alaw readers produce)."""
    c = np.arange(256, dtype=np.int32)
    u = ~c & 0xFF
    mu = ((((u & 0x0F) << 3) + 0x84) << ((u >> 4) & 7)) - 0x84
    mu = np.where(u & 0x80, -mu, mu)
    a = c ^ 0x55
    e, m = (a >> 4) & 7, a & 0x0F
    al = np.where(e == 0, (m << 4) + 8, ((m << 4) + 0x108) << np.maximum(e - 1, 0))
    al = np.where(a & 0x80, al, -al)
    return mu.astype(np.int16), al.astype(np.int16)


ULAW_TABLE, ALAW_TABLE = _g711_tables()


def read_wav(path) -> tuple[np.ndarray, int]:
    """RIFF/WAVE reader with libsndfile's float conversion (what ``soundfile.read(dtype='float32')`` under
    ``librosa.load`` yields): PCM 8 (unsigned) / 16 / 24 / 32 bit -> x / full scale, IEEE float 32 / 64 as is,
    G.711 A-law / mu-law (format tags 6 / 7) expanded to 16 bit then / 32768, WAVE_FORMAT_EXTENSIBLE.
    -> (float32 [n] or [n, channels], sample_rate)."""
    with open(path, "rb") as f:
        data = f.read()
    if len(data) < 12 or data[:4] != b"RIFF" or data[8:12] != b"WAVE":
        raise ValueError(f"{path}: not a RIFF/WAVE file")
    pos, fmt, pcm = 12, None, None
    while pos + 8 <= len(data):
        cid, size = data[pos:pos + 4], struct.unpack_from("<I", data, pos + 4)[0]
        body = data[pos + 8:pos + 8 + size]
        if cid == b"fmt ":
            fmt = body
        elif cid == b"data":
            pcm = body
        pos += 8 + size + (size & 1)
    if fmt is None or pcm is None or len(fmt) < 16:
        raise ValueError(f"{path}: missing fmt / data chunk")
    tag, ch, sr, _, _, bits = struct.unpack_from("<HHIIHH", fmt, 0)
    if tag == 0xFFFE and len(fmt) >= 26:
        tag = struct.unpack_from("<H", fmt, 24)[0]
    if ch < 1:
        raise ValueError(f"{path}: no channels")
    if tag == 1 and bits == 16:
        y = np.frombuffer(pcm[:len(pcm) // 2 * 2], "<i2").astype(np.float32) / np.float32(32768.0)
    elif tag == 1 and bits == 8:
        y = (np.frombuffer(pcm, np.uint8).astype(np.float32) - np.float32(128.0)) / np.float32(128.0)
    elif tag == 1 and bits == 24:
        b = np.frombuffer(pcm[:len(pcm) // 3 * 3], np.uint8).reshape(-1, 3).astype(np.int32)
        v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
        v = np.where(v >= 1 << 23, v - (1 << 24), v)
        y = (v.astype(np.float64) / 8388608.0).astype(np.float32)
    elif tag == 1 and bits == 32:
        y = (np.frombuffer(pcm[:len(pcm) // 4 * 4], "<i4").astype(np.float64) / 2147483648.0).astype(np.float32)
    elif tag in (6, 7) and bits == 8:
        y = (ALAW_TABLE if tag == 6 else ULAW_TABLE)[np.frombuffer(pcm, np.uint8)].astype(np.float32) / np.float32(32768.0)
    elif tag == 3 and bits == 32:
        y = np.frombuffer(pcm[:len(pcm) // 4 * 4], "<f4").astype(np.float32)
    elif tag == 3 and bits == 64:
        y = np.frombuffer(pcm[:len(pcm) // 8 * 8], "<f8").astype(np.float32)
    else:
        raise ValueError(f"{path}: unsupported WAV encoding (format tag {tag}, {bits} bits)")
    if ch > 1:
        y = y[:len(y) // ch * ch].reshape(-1, ch)
    return y, int(sr)


def load_16k(path, *, ctx=None, device: int = 0) -> np.ndarray:
    """``librosa.load(path, sr=16000)``: decode, mix down to mono (channel mean), convert to 16 kHz (device)."""
    y, sr = read_wav(path)
    if y.ndim > 1:
        y = y.mean(axis=1, dtype=np.float32)
    if sr != TARGET_SR:
        y = resample_to_16k(y, sr, ctx=ctx, device=device)
    return y
