"""Template enrolment on one GPU: 4096 templates of 0.6 .. 1.5 s installed three ways.

    python profiles/tools/enroll_bench.py [--out profiles/r10_enroll.json] [--runs 7] [--warmup 2]

Legs, alternated run by run on one context (4096 streams, 4096 template slots, 3 s int16 rings):
  singles       4096 ewk_set_template calls (one K3 + one dense-feature launch, two synchronisations each);
  batch_host    one ewk_set_templates call from host audio (one K3 + one install launch, one synchronisation);
  from_streams  one ewk_set_templates_from_streams call: each stream's template is 0.6 .. 1.5 s of its own ring (gather +
                K3 + install, one synchronisation).
Time: a host clock around the call(s), each of which ends in a synchronise; median over the timed runs after warm-up.
Launches per leg from ewk_launch_count.  Every leg must install the same bytes in every slot (checked on the last run:
the rings hold the host audio exactly, as float32 of int16).  The card's name and power limit are read in the same
run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

TOOLS = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(TOOLS))
sys.path.insert(0, REPO)

from easywakeword_b200 import _lib, synth  # noqa: E402

N, SR = 4096, 16000


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30)
    return r.stdout.strip().splitlines()[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    a = ap.parse_args()
    rng = np.random.default_rng(10)
    lens = rng.integers(int(0.6 * SR), int(1.5 * SR) + 1, N)
    bases = [synth.synthetic_word(seed=100 + i, duration=1.5) for i in range(64)]
    q = np.stack([synth.to_int16(np.concatenate([bases[s % 64] * np.float32(1.0 + (s % 7) / 7),
                                                 np.zeros(SR * 2 - len(bases[0]), np.float32)])) for s in range(N)])
    audios = [synth.from_int16(q[s, :lens[s]]) for s in range(N)]
    ctx = _lib.Context(device=0, n_streams=N, ring_samples=3 * SR, slack_samples=2 * SR, pcm_format=_lib.PCM_I16,
                       max_templates=N, max_events=8192)
    ctx.set_stream_params(-1, frame_size=1600, live=1)
    ctx.push(q)
    slots = np.arange(N, dtype=np.int32)

    def singles():
        for s in range(N):
            ctx.set_template(s, audios[s])

    legs = {"singles": singles,
            "batch_host": lambda: ctx.set_templates(slots, audios),
            "from_streams": lambda: ctx.set_templates_from_streams(slots, slots, np.zeros(N, np.int64), lens)}
    times = {k: [] for k in legs}
    launches = {}
    snaps = {}
    for r in range(a.warmup + a.runs):
        for k, f in legs.items():
            l0 = ctx.launch_count()
            t0 = time.perf_counter()
            f()
            dt = time.perf_counter() - t0
            launches[k] = ctx.launch_count() - l0
            if r >= a.warmup:
                times[k].append(dt * 1e3)
            if r == a.warmup + a.runs - 1:
                snaps[k] = b"".join(b"".join(np.asarray(v).tobytes() for v in ctx.get_template(s)[:2]) for s in range(N))
    same = snaps["singles"] == snaps["batch_host"] == snaps["from_streams"]
    res = {"gpu": gpu_info(), "templates": N, "template_seconds": [0.6, 1.5],
           "total_template_seconds": round(float(lens.sum()) / SR, 1), "runs": a.runs, "warmup": a.warmup,
           "identical_templates": bool(same), "launches": launches,
           "ms_median": {k: round(float(np.median(v)), 3) for k, v in times.items()},
           "ms_min": {k: round(float(np.min(v)), 3) for k, v in times.items()},
           "ms_max": {k: round(float(np.max(v)), 3) for k, v in times.items()}}
    res["speedup_vs_singles"] = {k: round(res["ms_median"]["singles"] / res["ms_median"][k], 1)
                                 for k in ("batch_host", "from_streams")}
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
            f.write("\n")
    ctx.close()
    if not same:
        sys.exit("the legs installed different templates")


if __name__ == "__main__":
    main()
