"""Host model of the dense detector (K4D, include/ewk.h: ewk_dense_detect): the per-stream peak picker over per-hop
scores, in plain Python.  It uses only comparisons and integer arithmetic on the float32 scores, so the device must equal
it exactly.

    detect(scores[n_hops, T], hop0, state, thr, hold, refractory, slot0, tmpl_lens) -> (events, state)

scores are the call's rows for one stream (hops hop0 .. hop0 + n_hops - 1, templates slot0 .. slot0 + T - 1); state is
what the previous call returned (None: a new or reset stream); thr the stream's similarity_threshold (rounded to
float32, as the device holds it).  events is a structured array of DETECTION_DTYPE in emit order.
"""
from __future__ import annotations

import math

import numpy as np

DETECTION_DTYPE = np.dtype([("stream", "<i4"), ("template_slot", "<i4"), ("hop", "<i8"), ("run_start", "<i8"),
                            ("emit_hop", "<i8"), ("seg_start", "<i8"), ("seg_len", "<i4"), ("score", "<f4")])
IDLE, ARMED, SPENT = 0, 1, 2


def initial_state():
    return dict(mode=IDLE, quiet_until=0, peak=0, run_start=0, score=0.0, slot=0, seg_start=0, seg_len=0)


def best(row):
    """(b, k*): max of the row ignoring NaN (NaN when all are NaN), and the lowest k reaching it."""
    b, kb = math.nan, 0
    for k, v in enumerate(float(x) for x in row):
        if v > b or (math.isnan(b) and not math.isnan(v)):
            b, kb = v, k
    return b, kb


def detect(scores, hop0, state, thr, hold, refractory, slot0, tmpl_lens, stream=0):
    if hold < 1 or refractory < 0:
        raise ValueError("hold >= 1 and refractory >= 0")
    st = dict(initial_state() if state is None else state)
    thr = float(np.float32(thr))
    n_win = [(int(L) + 159) // 160 for L in tmpl_lens]
    scores = np.asarray(scores, np.float32).reshape(len(scores), -1) if len(scores) else np.zeros((0, 1), np.float32)
    ev = []

    def take_peak(h, b, k):
        st.update(peak=h, score=b, slot=slot0 + k, seg_start=160 * (h - n_win[k]), seg_len=int(tmpl_lens[k]))

    for i, row in enumerate(scores):
        h = int(hop0) + i
        b, k = best(row)
        above = b >= thr                                   # False for NaN
        if st["mode"] == IDLE:
            if above and h >= st["quiet_until"]:
                st.update(mode=ARMED, run_start=h)
                take_peak(h, b, k)
        elif st["mode"] == ARMED:
            if above:
                if b > st["score"]:                        # strictly: the first maximum wins
                    take_peak(h, b, k)
                if h - st["peak"] >= hold:
                    ev.append((stream, st["slot"], st["peak"], st["run_start"], h, st["seg_start"], st["seg_len"],
                               st["score"]))
                    st["mode"] = SPENT
            else:
                ev.append((stream, st["slot"], st["peak"], st["run_start"], h, st["seg_start"], st["seg_len"],
                           st["score"]))
                st.update(mode=IDLE, quiet_until=h + refractory)
        elif not above:                                    # SPENT
            st.update(mode=IDLE, quiet_until=h + refractory)
    return np.array(ev, DETECTION_DTYPE), st
