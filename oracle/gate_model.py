"""ORACLE — TEST INFRASTRUCTURE ONLY.  An exact model of what the level-1 gate (K2, tick_gate_kernel in
easywakeword_b200/csrc/ewk_streams.cuh) must produce, per stream, bit for bit: the per-tick is_silent flag, state,
adaptive threshold and RMS, the events and timeouts, the final ewk_stream_status and bits 1-4 and 8.. of the
ewk_stream_result flags (bit 0 and the score belong to K3).

It is written from the reference's semantics (oracle/ewk_oracle.py: SoundBuffer, WakeWord._detect_word under the audio
clock), not from K2's plan: nothing here knows of chunk pieces, GATE_MAXP, the aliased-window shortcut, sorted arrays or
cached order statistics.  Every tick is a pure function of the samples visible at it:

* Visible samples.  Tick k of an audio-clock stream sees
  V_k = max(V_{k-1}, min(floor(1600 k / fs) * fs, floor(written / fs) * fs)); a live stream sees everything pushed
  (V = written) (include/ewk.h: ewk_stream_params.live, a departure from the reference's clock on purpose).  A paced call
  (ewk_tick_ready) gives a stream min(n, written // 1600 - tick) ticks.  frame_size 0 latches the first push's length.
* Chunks.  Once V >= R the reference ring holds the last R samples: logical position p < V % R was written in the
  current lap, the others in the previous one.  Chunk c < R // fs holds logical positions [c fs, (c+1) fs); the tail
  R - (R // fs) fs is in no chunk.  Its mean square is (sum of squares) / fs, the sum taken over the current-lap part
  and then the previous-lap part, added.
* Threshold.  np.percentile(sqrt(ms), 25) * 1.5, then max(., min_threshold) (ewk_stream_params.min_threshold replaces
  the reference's constant 0.005).  It moves only when the chunks change; before the first full tick it is 0.01.
* is_silent.  The RMS of the last nrec = min(1600, R) samples, zeros before the stream began:
  sqrt(sum of squares / nrec); silent = rms < thr.  Before the first push: silent, rms 0.
* Timing machine and segment cut: WakeWord._detect_word with Python floats, which are the IEEE double operations of
  gate_state_step (no contraction there).  The timeout test uses the previous tick's time; n_back is clamped to R; a
  candidate becomes an event only when 1 <= len <= 48000 (the device drops len < 1, which the reference would hand to
  the matcher as an empty or wrapped slice; include/ewk.h: ewk_event).

Sums of squares, and why the sum source does not matter:

* int16 rings: the device sums integer squares exactly (64-bit integers), then scales by 2^-30.  The model does the
  same with prefix sums; the order is irrelevant.
* f32 rings: the order is fixed by warp_sumsq.  Lane l of the warp owns 16-byte word l + 32 m of a range; even m add
  into one double accumulator, odd m into a second, each word's four squares in order; the two are added, then the
  scalar tail (element i goes to lane i % 32), then a xor butterfly over the 32 lanes (offsets 16, 8, 4, 2, 1).  That
  vector path is taken only when the physical start a0 % P is a multiple of 4 and the range does not wrap; otherwise
  every element goes through the scalar loop (element i to lane i % 32).  A square of a float32 is exact in double,
  so fma(x, x, acc) is the double addition acc + x*x, which is what the model computes.
  For an aligned, non-wrapping 1600-sample block the four places that sum a block produce the very same additions:
  ring_push_sums_kernel (word lane + 32 u, u odd -> second accumulator, u < 13), ring_push_bulk_kernel through
  warp_sumsq_smem (same loop over the staged block), and warp_sumsq's vector path (k0 = 0, 256: word k0 + lane + 32 u
  with the parity of u equal to the parity of the word's m).  Each lane's sequence of additions into each
  accumulator, the final a0 + a1 and the xor tree coincide, and padding words add +0.0, which changes nothing.  So
  K1's block sums (the "presummed" gate), the TMA push form and the gate's own reads all give one value, and the model
  needs no knowledge of which source ran.
"""
from __future__ import annotations

import math

import numpy as np

TICK = 1600
MAX_SEG = 48000
INITIAL_THRESHOLD = 0.01
GATE_MAX_TICKS = 16                 # ticks per K2 launch: bit 4 of the flags covers the last launch of a call
WAITING, IN_SILENCE, IN_SOUND, AFTER_SOUND = 0, 1, 2, 3
EV_TIMEOUT, EV_SCORED = 1, 2
_LANE = np.arange(32)

DEFAULT_PARAMS = dict(frame_size=0, pre_speech_silence=0.8, speech_duration_min=0.3, speech_duration_max=2.0,
                      post_speech_silence=0.4, timeout=30.0, min_threshold=0.005, live=0)


def physical_ring(ring_samples, slack_samples):
    """P of a context: ring + slack rounded up to 64 samples (ewk_ctx::init_streams)."""
    return ((ring_samples + slack_samples + 63) // 64) * 64


def _xor_tree(acc):
    """acc: [..., 32] lane values -> the value every lane holds after the warp's xor butterfly."""
    v = acc.copy()
    for o in (16, 8, 4, 2, 1):
        v = v + v[..., _LANE ^ o]
    return v[..., 0]


def warp_sumsq_f32(x, p0, P):
    """Sum of squares of the float32 rows x [B, L] (or [L]) in warp_sumsq's order, for ranges whose physical start is
    p0 (same for every row) in a ring of P samples."""
    x = np.asarray(x, dtype=np.float32)
    one = x.ndim == 1
    X = x.reshape(1, -1) if one else x
    Bn, L = X.shape
    sq = X.astype(np.float64) ** 2                       # exact: 24-bit mantissas squared fit a double
    acc = np.zeros((Bn, 32))
    i = 0
    if L > 0 and p0 % 4 == 0 and p0 + L <= P:
        nv = L // 4
        a1 = np.zeros((Bn, 32))
        for m in range((nv + 31) // 32):
            w = 32 * m + _LANE
            ok = w < nv
            lanes, words = _LANE[ok], w[ok]
            t = acc if m % 2 == 0 else a1
            for c in range(4):
                t[:, lanes] = t[:, lanes] + sq[:, 4 * words + c]
        acc = acc + a1
        i = 4 * nv
    for r in range((L - i + 31) // 32):
        k = i + 32 * r + _LANE
        ok = k < L
        acc[:, _LANE[ok]] = acc[:, _LANE[ok]] + sq[:, k[ok]]
    s = _xor_tree(acc)
    return float(s[0]) if one else s


def block_sumsq_f32(x):
    """ring_push_sums_kernel's (and warp_sumsq_smem's) f32 block sum, restated from its own loop: word lane + 32 u,
    u < 13, odd u into the second accumulator.  For the tests that show the block sources agree with warp_sumsq."""
    sq = np.asarray(x, dtype=np.float32).astype(np.float64).reshape(-1) ** 2
    assert sq.size == TICK
    a0, a1 = np.zeros(32), np.zeros(32)
    for u in range(13):
        for lane in range(32):
            k = lane + 32 * u
            if k < TICK // 4:
                for c in range(4):
                    if u & 1:
                        a1[lane] += sq[4 * k + c]
                    else:
                        a0[lane] += sq[4 * k + c]
    return float(_xor_tree(a0 + a1))


class _Stream:
    def __init__(self, fmt, params):
        self.fmt = fmt
        self.p = dict(DEFAULT_PARAMS)
        self.p.update(params)
        self.data = np.zeros(0, np.int16 if fmt == "i16" else np.float32)
        self.csq = np.zeros(1, np.int64)                  # int16: prefix sums of integer squares
        self.memo = {}                                    # f32: (a0, len) -> sum of squares
        self.written = self.visible = self.tick = 0
        self.frame_size = 0
        self.thr = INITIAL_THRESHOLD
        self.ms = None                                    # chunk mean squares at `visible` (None before the first full tick)
        self.last_rms = 0.0
        self.state = WAITING
        self.started = 0
        self.last_silent = 0
        self.n_timeouts = self.n_events = 0
        self.silence_start = self.sound_start = self.sound_end = self.start_time = 0.0
        self.evflag = 0

    # ---- sums
    def sumsq(self, a0, n, P):
        """sum of squares of absolute samples [a0, a0 + n) as the device forms it (int16: scaled by 2^-30)"""
        if n <= 0:
            return 0.0
        if self.fmt == "i16":
            return float(int(self.csq[a0 + n] - self.csq[a0])) * (1.0 / 1073741824.0)
        key = (a0, n)
        v = self.memo.get(key)
        if v is None:
            v = self.memo[key] = warp_sumsq_f32(self.data[a0:a0 + n], a0 % P, P)
        return v

    def chunk_ms(self, V, R, P):
        fs = self.frame_size
        nc = R // fs
        lap, q = divmod(V, R)
        out = np.empty(nc)
        for c in range(nc):
            lo, hi = c * fs, c * fs + fs
            split = min(max(q, lo), hi)                    # [lo, split) current lap, [split, hi) previous lap
            ss = 0.0
            if split > lo:
                ss += self.sumsq(lap * R + lo, split - lo, P)
            if hi > split:
                ss += self.sumsq((lap - 1) * R + split, hi - split, P)
            out[c] = ss / fs                               # np.mean(frame ** 2)
        return out


class GateModel:
    """One context's streams: R ring samples, P physical samples, fmt "i16" or "f32".  params: one dict per stream
    (keys of DEFAULT_PARAMS; missing keys take the defaults).  max_events: the event queue's capacity (only the count
    events + dropped is meaningful when it overflows)."""

    def __init__(self, R, P, fmt, params):
        self.R, self.P, self.fmt = int(R), int(P), fmt
        self.params = [dict(p) for p in params]
        self.s = [_Stream(fmt, p) for p in self.params]
        self.events = []                                  # (stream, kind, tick, seg_start, seg_len)

    @property
    def n_streams(self):
        return len(self.s)

    def set_params(self, stream, **over):
        self.params[stream].update(over)
        self.s[stream].p.update(over)

    def reset(self, streams):
        for i in streams:
            self.s[i] = _Stream(self.fmt, self.params[i])

    def push(self, stream, x):
        st = self.s[stream]
        x = np.asarray(x, dtype=st.data.dtype).reshape(-1)
        if x.size == 0:
            return
        if st.frame_size == 0:
            st.frame_size = st.p["frame_size"] if st.p["frame_size"] > 0 else int(x.size)
        st.data = np.concatenate([st.data, x])
        if self.fmt == "i16":
            q = x.astype(np.int64)
            st.csq = np.concatenate([st.csq, st.csq[-1] + np.cumsum(q * q)])
        st.written += int(x.size)

    # ---- one tick of one stream
    def _tick(self, i, k):
        st, R, P = self.s[i], self.R, self.P
        fs = st.frame_size
        V = st.visible
        if fs > 0:
            V = st.written if st.p["live"] else min((k * TICK // fs) * fs, (st.written // fs) * fs)
            V = max(V, st.visible)
        full = fs > 0 and V >= R
        if full and R // fs > 0 and (st.ms is None or V != st.visible):
            ms = st.chunk_ms(V, R, P)
            if st.ms is None or not np.array_equal(ms, st.ms):
                new = np.percentile(np.sqrt(ms), 25) * 1.5
                st.thr = float(max(new, st.p["min_threshold"]))
            st.ms = ms
        silent, rms = 1, 0.0
        if fs > 0:
            nrec = min(TICK, R)
            a0 = V - nrec
            ss = st.sumsq(max(a0, 0), V if a0 < 0 else nrec, P)
            rms = math.sqrt(ss / nrec)
            silent = int(rms < st.thr)
        st.last_rms = rms
        self._state_step(i, st, k, V, full, silent)
        st.last_silent = silent
        st.tick, st.visible = k, V
        return silent, (st.state if st.started else 255), st.thr, rms

    def _state_step(self, i, st, k, V, full, silent):
        p = st.p
        now = k * 0.1
        if full and not st.started:                                   # _wait_for_buffer done: _detect_word entry
            st.started = 1
            st.state = IN_SILENCE if silent else WAITING
            st.start_time = now
            if silent:
                st.silence_start = now
            return
        if not st.started:
            return
        prev = (k - 1) * 0.1
        if p["timeout"] > 0.0 and prev - st.start_time > p["timeout"]:   # the listen loop re-enters at `prev`
            self.events.append((i, EV_TIMEOUT, k - 1, 0, 0))
            st.n_timeouts += 1
            st.state = IN_SILENCE if st.last_silent else WAITING
            st.start_time = prev
            if st.last_silent:
                st.silence_start = prev
        if st.state == WAITING:
            if silent:
                st.state, st.silence_start = IN_SILENCE, now
        elif st.state == IN_SILENCE:
            if not silent:
                if now - st.silence_start >= p["pre_speech_silence"]:
                    st.state, st.sound_start = IN_SOUND, now
                else:
                    st.state = WAITING
        elif st.state == IN_SOUND:
            dur = now - st.sound_start
            if not silent:
                if dur > p["speech_duration_max"]:
                    st.state = WAITING
            elif p["speech_duration_min"] <= dur <= p["speech_duration_max"]:
                st.state, st.sound_end = AFTER_SOUND, now
            else:
                st.state = WAITING
        elif st.state == AFTER_SOUND:
            if silent:
                if now - st.sound_end >= p["post_speech_silence"]:
                    es = st.sound_start - now - 0.05
                    ee = st.sound_end - now + 0.05
                    n_back = min(int(abs(es) * 16000), self.R)
                    n_drop = int(abs(ee) * 16000)
                    ln = n_back - n_drop
                    if 1 <= ln <= MAX_SEG:
                        self.events.append((i, EV_SCORED, k, V - n_back, ln))
                        st.n_events += 1
                        st.evflag = 16
                    st.state = WAITING
            else:
                st.state = WAITING

    def tick(self, n, paced=False):
        """ewk_tick_trace (paced=False) or ewk_tick_ready with a trace (paced=True) -> (taken int32 [n_streams],
        trace dict of [n_streams, n]: silent / state uint8, thr / rms float64; cells of ticks not taken: 255 and NaN
        with all bits set)."""
        ns = self.n_streams
        tr = {"silent": np.full((ns, n), 255, np.uint8), "state": np.full((ns, n), 255, np.uint8),
              "thr": np.full((ns, n), -1, np.int64).view(np.float64), "rms": np.full((ns, n), -1, np.int64).view(np.float64)}
        taken = np.zeros(ns, np.int32)
        for i, st in enumerate(self.s):
            taken[i] = max(0, min(n, st.written // TICK - st.tick)) if paced else n
        rounds = max(1, int(taken.max())) if paced else n
        last_launch0 = ((rounds - 1) // GATE_MAX_TICKS) * GATE_MAX_TICKS
        for i, st in enumerate(self.s):
            k0 = st.tick
            for j in range(int(taken[i])):
                if j == last_launch0:
                    st.evflag = 0
                cell = self._tick(i, k0 + j + 1)
                tr["silent"][i, j], tr["state"][i, j], tr["thr"][i, j], tr["rms"][i, j] = cell
            if int(taken[i]) <= last_launch0:
                st.evflag = 0
        return taken, tr

    # ---- what the host reads
    def status(self, i):
        st = self.s[i]
        return dict(written=st.written, visible=st.visible, tick=st.tick, silence_threshold=st.thr, last_rms=st.last_rms,
                    frame_size=st.frame_size, state=st.state, started=st.started, is_silent=st.last_silent,
                    n_timeouts=st.n_timeouts, n_events=st.n_events)

    def flags(self, i):
        """ewk_stream_result.flags without bit 0"""
        st = self.s[i]
        return (2 if st.last_silent else 0) | (st.state << 2) | st.evflag | (st.n_events << 8)

    def event_array(self):
        """events sorted by (stream, tick, kind): int64 [n, 5] of (stream, kind, tick, seg_start, seg_len)"""
        e = np.array(self.events, np.int64).reshape(-1, 5)
        return e[np.lexsort((e[:, 1], e[:, 2], e[:, 0]))] if len(e) else e
