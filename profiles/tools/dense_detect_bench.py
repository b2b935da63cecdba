"""Dense detection on one GPU: ewk_dense_detect (K4 + K4D, scores left on the device) against ewk_dense_ready with host
scores and the same peak picker in numpy on the host.

    python profiles/tools/dense_detect_bench.py [--out profiles/r07_dense_detect.json] [--steps 8]

Bank: 4096 slots, 10 s int16 rings.  Every active slot plays one of 64 synth.stream feeds (known word inserts and
distractors); a step pushes U(0.5, 1.5) s of its feed to each active slot (push_streams), then
  (a) dense_ready until nothing is due, scores copied to the host, and the detector of oracle/dense_detect.py
      vectorised over streams in numpy;
  (b) dense_detect until nothing is due, out = NULL.
At 100 / 50 / 10 % occupancy, for one template (the bundled word) and bench.py's 4-template sweep set, the two legs run
alternated step by step in one process, each on its own context fed the same audio.  Step times are host clocks around
work that ends in a synchronise; K4 and K4D kernel times come from torch.profiler in passes of their own (kernel names
dense_score_kernel and dense_detect_kernel); D2H bytes per step are counted from the shapes (scores in (a); per-row
counts plus 48-byte records in (b), which K4D writes straight into mapped host memory).  Detections of the two legs must
be equal; hits / misses / extras are counted against the feeds' word inserts at hold 20, refractory 50 and the default
threshold.  The card's name and power limit are read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

TOOLS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(TOOLS))
sys.path.insert(0, REPO)
sys.path.insert(0, TOOLS)

from easywakeword_b200 import _lib, synth  # noqa: E402
from native_rate_bench import gpu_info, sm_clock_now  # noqa: E402
from bench import sweep_templates  # noqa: E402

SLOTS, RING, SLACK, POOL = 4096, 160000, 32000, 64
HOLD, REFR = 20, 50


def load_word():
    return np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))["pcm_i16"].astype(np.float32) / np.float32(32768)


def make_ctx(tpls):
    ctx = _lib.Context(device=0, n_streams=SLOTS, ring_samples=RING, slack_samples=SLACK, pcm_format=_lib.PCM_I16,
                       max_templates=len(tpls), max_events=8 * SLOTS)
    for i, t in enumerate(tpls):
        ctx.set_template(i, t)
    ctx.set_stream_params(-1, frame_size=1600, live=1)
    return ctx


class HostDetector:
    """oracle/dense_detect.py vectorised over streams (one numpy pass per hop column)."""

    def __init__(self, n, thr, slot0, lens):
        self.mode = np.zeros(n, np.int8)
        self.quiet = np.zeros(n, np.int64)
        self.peak = np.zeros(n, np.int64)
        self.run = np.zeros(n, np.int64)
        self.score = np.zeros(n, np.float32)
        self.k = np.zeros(n, np.int64)
        self.thr = np.float32(thr)
        self.slot0, self.lens = slot0, np.asarray(lens, np.int64)
        self.nwin = (self.lens + 159) // 160
        self.n_hops = self.n_above = 0

    def feed(self, streams, hop0, rows):
        """rows[i]: float32 [n_i, T] of stream streams[i] from hop hop0[i] -> records (DETECTION_DTYPE, list order)"""
        n = np.array([len(r) for r in rows])
        if n.max(initial=0) == 0:
            return np.zeros(0, _lib.DETECTION_DTYPE)
        T = rows[0].shape[1]
        X = np.full((len(rows), n.max(), T), np.nan, np.float32)
        for i, r in enumerate(rows):
            X[i, :len(r)] = r
        Xm = np.where(np.isnan(X), -np.inf, X)
        kb = np.argmax(Xm, axis=2)                               # lowest k reaching the max
        b = np.take_along_axis(X, kb[..., None], 2)[..., 0]      # NaN only where every score is NaN
        st = np.asarray(streams)
        ev = []
        for j in range(n.max()):
            live = j < n
            h = np.asarray(hop0) + j
            bj, kj = b[:, j], kb[:, j]
            above = live & (bj >= self.thr)
            self.n_hops += int(live.sum())
            self.n_above += int(above.sum())
            mode, S = self.mode[st], st
            arm = live & (mode == 0) & above & (h >= self.quiet[S])
            armed = live & (mode == 1)
            newpk = armed & above & (bj > self.score[S])
            set_pk = arm | newpk
            self.peak[S[set_pk]] = h[set_pk]
            self.score[S[set_pk]] = bj[set_pk]
            self.k[S[set_pk]] = kj[set_pk]
            self.run[S[arm]] = h[arm]
            emit_hold = armed & above & (h - self.peak[S] >= HOLD)
            emit_end = armed & ~above
            spent_end = live & (mode == 2) & ~above
            for m in np.flatnonzero(emit_hold | emit_end):
                s, k = int(S[m]), int(self.k[S[m]])
                ev.append((m, j, (s, self.slot0 + k, self.peak[s], self.run[s], h[m], 160 * (self.peak[s] - self.nwin[k]),
                                  self.lens[k], self.score[s])))
            self.mode[S[arm]] = 1
            self.mode[S[emit_hold]] = 2
            self.mode[S[emit_end | spent_end]] = 0
            self.quiet[S[emit_end | spent_end]] = h[emit_end | spent_end] + REFR
        ev.sort(key=lambda e: (e[0], e[1]))
        return np.array([e[2] for e in ev], _lib.DETECTION_DTYPE)


def run_case(tpls, occ, feeds, inserts, wlen, steps, warmup, prof_steps, rng):
    T = len(tpls)
    n_act = int(round(occ * SLOTS))
    active = np.sort(rng.choice(SLOTS, n_act, replace=False)).astype(np.int32)
    a, b = make_ctx(tpls), make_ctx(tpls)
    thr = float(_lib.default_stream_params().similarity_threshold)
    host = HostDetector(SLOTS, thr, 0, [len(t) for t in tpls])
    pos = np.zeros(SLOTS, np.int64)
    det_a, det_b = [], []
    ta, tb, bytes_a, bytes_b, hops = [], [], [], [], []

    def leg_a():
        nb, got = 0, []
        while True:
            h0, rows = a.dense_ready(active, 200, 0, T)
            nb += 4 * sum(r.size for r in rows)
            got.append(host.feed(active, h0, rows))
            if max(len(r) for r in rows) < 200:
                return np.concatenate(got), nb

    def leg_b():
        got, nh_all = [], 0
        while True:
            d, (_, nh) = b.dense_detect(active, 200, 0, T, HOLD, REFR, hops=True)
            got.append(d)
            nh_all += int(nh.sum())
            if nh.max() < 200:
                return np.concatenate(got), 4 * n_act + 48 * sum(len(g) for g in got), nh_all

    def push():
        lens = (rng.uniform(0.5, 1.5, n_act) * 16000).astype(np.int64)
        blocks = []
        for s, n in zip(active, lens):
            f = feeds[s % POOL]
            blocks.append(f[pos[s]:pos[s] + n])
            pos[s] += len(blocks[-1])
        for c in (a, b):
            c.push_streams(active, blocks)

    def step(record):
        push()
        a.synchronize()
        t0 = time.perf_counter()
        da, nba = leg_a()
        a.synchronize()
        t1 = time.perf_counter()
        db, nbb, nh = leg_b()
        b.synchronize()
        t2 = time.perf_counter()
        det_a.append(da)
        det_b.append(db)
        if record:
            ta.append(t1 - t0)
            tb.append(t2 - t1)
            bytes_a.append(nba)
            bytes_b.append(nbb)
            hops.append(nh)

    try:
        for i in range(warmup + steps):
            step(i >= warmup)
        da, db = np.concatenate(det_a), np.concatenate(det_b)
        key = lambda d: np.lexsort((d["emit_hop"], d["stream"]))   # noqa: E731
        equal = bool(np.array_equal(da[key(da)], db[key(db)]))
        hit = miss = extra = 0
        for s in active:
            d = db[db["stream"] == s]
            fed = pos[s]
            used = np.zeros(len(d), bool)
            for off, g in inserts[s % POOL]:
                if g < 0 or off + wlen > fed - HOLD * 160:
                    continue
                ov = np.minimum(d["seg_start"] + d["seg_len"], off + wlen) - np.maximum(d["seg_start"], off)
                m = ov >= wlen // 2
                if m.any():
                    hit += 1
                    used |= m
                else:
                    miss += 1
            extra += int((~used).sum())
        # kernel times in passes of their own (each context detects on every push it gets: leg b catches up on the
        # pushes of leg a's pass)
        kern = {}
        for leg, fn in (("a", leg_a), ("b", leg_b)):
            fn()                                                 # catch up on the other leg's profiled pushes first
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                for _ in range(prof_steps):
                    push()
                    fn()
                torch.cuda.synchronize()
            for e in prof.key_averages():
                for name in ("dense_score_kernel", "dense_detect_kernel"):
                    if name in e.key:
                        k = f"{leg}_{name}"
                        kern[k] = kern.get(k, 0.0) + e.device_time_total / 1e3 / prof_steps   # ms per step
    finally:
        a.close()
        b.close()
    return {"active_streams": n_act, "templates": T, "hops_per_step": float(np.mean(hops)),
            "a_step_ms_median": float(np.median(ta)) * 1e3, "b_step_ms_median": float(np.median(tb)) * 1e3,
            "a_step_ms_spread": [float(np.min(ta)) * 1e3, float(np.max(ta)) * 1e3],
            "b_step_ms_spread": [float(np.min(tb)) * 1e3, float(np.max(tb)) * 1e3],
            "a_d2h_bytes_per_step": float(np.mean(bytes_a)), "b_d2h_bytes_per_step": float(np.mean(bytes_b)),
            "kernel_ms_per_step": kern, "detections": int(len(db)), "legs_equal": equal,
            "hops_above_threshold_frac": host.n_above / max(1, host.n_hops),
            "detections_per_active_stream": np.bincount(np.searchsorted(active, db["stream"]), minlength=n_act).tolist()[:16],
            "hits": hit, "misses": miss, "extras": extra}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(REPO, "profiles", "r07_dense_detect.json"))
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--prof-steps", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    total_s = 1.5 * (a.warmup + a.steps + 2 * a.prof_steps) + 1
    res = {"gpu": gpu_info(), "slots": SLOTS, "ring_samples": RING, "steps": a.steps, "hold_hops": HOLD,
           "refractory_hops": REFR}
    word = load_word()
    feeds, inserts = [], []
    for i in range(POOL):
        x, ins = synth.stream(9000 + i, total_s, word, gain=(1.0, 4.0), inserts_per_10s=(2, 4))
        feeds.append(synth.to_int16(x))
        inserts.append(ins)
    sweep, _ = sweep_templates(word)
    rng = np.random.default_rng(2026)
    for name, tpls in (("T1", [word]), ("T4_sweep_set", sweep)):
        for occ in (1.0, 0.5, 0.1):
            k = f"{name}_occupancy{int(occ * 100)}"
            res[k] = run_case(tpls, occ, feeds, inserts, len(word), a.steps, a.warmup, a.prof_steps, rng)
            print(json.dumps({k: res[k]}), flush=True)
    res["gpu"]["sm_clock_mhz_at_end"] = sm_clock_now()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
