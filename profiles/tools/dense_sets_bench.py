"""Per-row template sets in dense detection on one GPU: one ewk_dense_detect_sets call for a bank of personal wake
words against one ewk_dense_detect call per distinct set, and against one shared set; and the set forms against the
single-set forms when every row has the same set.

    python profiles/tools/dense_sets_bench.py [--out profiles/r09_dense_sets.json] [--steps 6] [--warmup 2] [--shared-T 1]

Bank: 4096 slots, 10 s int16 rings; every slot plays one of 64 synth.stream feeds (word inserts and distractors),
rolled per slot; a step pushes 1 s to every slot (ewk_push), then runs one detector leg until nothing is due (100 hops,
scores left on the device).  Templates: 64 one-template slots of 0.6 .. 1.5 s (a context holds at most 64 template
slots, so 64 is the largest number of distinct one-template sets).  Legs, each on its own context fed the same audio,
alternated step by step:
  shared    ewk_dense_detect of every stream against slot 0;
  sets      ewk_dense_detect_sets, stream s against slot s % 64 (64 sets, 64 streams each), one call;
  grouped   the same work as one ewk_dense_detect call per set (64 calls);
  shared_sets  ewk_dense_detect_sets with every row given the shared set (what shared computes, through the set form);
  ready / ready_sets  ewk_dense_ready of every stream against the shared set, and ewk_dense_ready_sets with every row
            given it, until nothing is due (scores to a device buffer).
The shared set is slot 0 (the bundled word) with --shared-T 1, and bench.sweep_templates' four templates with 4.
Step time: a host clock around the detector call(s), which end in a synchronise (the push is not timed).  Launches per
step from ewk_launch_count.  The detections of `sets` and `grouped` must be equal, and so must those of `shared` and
`shared_sets`, and the scores of `ready` and `ready_sets`.  The card's name and power limit
are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

TOOLS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(TOOLS))
sys.path.insert(0, REPO)

from easywakeword_b200 import _lib, synth  # noqa: E402
from bench import sweep_templates  # noqa: E402

SLOTS, RING, SLACK, POOL, NT = 4096, 160000, 32000, 64, 64
HOLD, REFR = 20, 50


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--shared-T", type=int, default=1, choices=(1, 4))
    a = ap.parse_args()
    word = np.load(os.path.join(REPO, "tests", "golden", "reference_word.npz"))["pcm_i16"].astype(np.float32) / np.float32(32768)
    rng = np.random.default_rng(9)
    lens = rng.integers(9600, 24001, NT)
    tpls = [word.copy() if k == 0 else synth.synthetic_word(seed=300 + k, duration=1.5)[:int(lens[k])] for k in range(NT)]
    tpls += sweep_templates(word)[0]                     # slots NT .. NT + 3
    T = a.shared_T
    first = 0 if T == 1 else NT
    secs = a.warmup + a.steps + 1
    pool = [synth.to_int16(synth.stream(8100 + i, float(secs), word, gain=(1.5, 3.0))[0]) for i in range(POOL)]
    feed = np.stack([np.roll(pool[s % POOL], 37 * s) for s in range(SLOTS)])

    def make():
        ctx = _lib.Context(device=0, n_streams=SLOTS, ring_samples=RING, slack_samples=SLACK, pcm_format=_lib.PCM_I16,
                           max_templates=len(tpls), max_events=8 * SLOTS)
        for i, t in enumerate(tpls):
            ctx.set_template(i, t)
        ctx.set_stream_params(-1, frame_size=1600, live=1, similarity_threshold=62.0)
        return ctx

    legs = {k: make() for k in ("shared", "shared_sets", "sets", "grouped", "ready", "ready_sets")}
    slot_of = np.arange(SLOTS) % NT
    groups = [np.flatnonzero(slot_of == k).astype(np.int32) for k in range(NT)]
    all_first, all_count = np.full(SLOTS, first, np.int32), np.full(SLOTS, T, np.int32)
    ready_out = {k: torch.zeros(SLOTS * 100 * T, dtype=torch.float32, device="cuda:0") for k in ("ready", "ready_sets")}

    def run(name, ctx):
        d = []
        while True:
            if name == "shared":
                r, (_, nh) = ctx.dense_detect(None, 100, first, T, HOLD, REFR, hops=True)
                d.append(r)
            elif name == "shared_sets":
                r, (_, nh) = ctx.dense_detect_sets(None, 100, all_first, all_count, HOLD, REFR, hops=True)
                d.append(r)
            elif name == "ready":
                _, nh = ctx.dense_ready(None, 100, first, T, out_device_ptr=ready_out[name].data_ptr())
            elif name == "ready_sets":
                _, nh = ctx.dense_ready_sets(None, 100, all_first, all_count, out_device_ptr=ready_out[name].data_ptr())
            elif name == "sets":
                r, (_, nh) = ctx.dense_detect_sets(None, 100, slot_of, np.ones(SLOTS, np.int32), HOLD, REFR, hops=True)
                d.append(r)
            else:
                nh = np.zeros(0, np.int32)
                for k, g in enumerate(groups):
                    r, (_, n_) = ctx.dense_detect(g, 100, k, 1, HOLD, REFR, hops=True)
                    d.append(r)
                    nh = np.concatenate([nh, n_])
            if nh.size == 0 or nh.max() < 100:
                ctx.synchronize()                            # the ready legs' device output is asynchronous
                return np.concatenate(d) if d else np.zeros(0, _lib.DETECTION_DTYPE)

    times = {k: [] for k in legs}
    launches = {k: [] for k in legs}
    dets = {k: [] for k in legs}
    for step in range(a.warmup + a.steps):
        blk = np.ascontiguousarray(feed[:, step * 16000:(step + 1) * 16000])
        for name, ctx in legs.items():
            ctx.push(blk)
            n0 = ctx.launch_count()
            t0 = time.perf_counter()
            d = run(name, ctx)
            dt = time.perf_counter() - t0
            if step >= a.warmup:
                times[name].append(dt * 1e3)
                launches[name].append(ctx.launch_count() - n0)
            dets[name].append(d)
        bits = [ready_out[k].view(torch.int32) for k in ("ready", "ready_sets")]   # scores before a stream's start are NaN
        assert torch.equal(*bits), "ready and ready_sets scores differ"
    key = lambda d: np.sort(d, order=["stream", "emit_hop"])
    ds, dg = key(np.concatenate(dets["sets"])), key(np.concatenate(dets["grouped"]))
    assert ds.tobytes() == dg.tobytes(), "sets and grouped detections differ"
    assert np.concatenate(dets["shared"]).tobytes() == np.concatenate(dets["shared_sets"]).tobytes(), \
        "shared and shared_sets detections differ"
    res = {
        "gpu": gpu_info(),
        "streams": SLOTS, "step_s": 1.0, "shared_set": [first, T], "distinct_sets": NT, "template_s": [float(lens.min()) / 16000, float(lens.max()) / 16000],
        "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)), "all": v}
                        for k, v in times.items()},
        "launches_per_step": {k: float(np.median(v)) for k, v in launches.items()},
        "detections": {k: int(sum(len(x) for x in v)) for k, v in dets.items()},
        "sets_equal_grouped": True, "shared_sets_equal_shared": True, "ready_sets_equal_ready": True,
    }
    res["speedup_sets_over_grouped"] = res["ms_per_step"]["grouped"]["median"] / res["ms_per_step"]["sets"]["median"]
    res["cost_sets_over_shared"] = res["ms_per_step"]["sets"]["median"] / res["ms_per_step"]["shared"]["median"]
    for one, rows in (("shared", "shared_sets"), ("ready", "ready_sets")):
        res[f"cost_{rows}_over_{one}"] = res["ms_per_step"][rows]["median"] / res["ms_per_step"][one]["median"]
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    for c in legs.values():
        c.close()


if __name__ == "__main__":
    main()
