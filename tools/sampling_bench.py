#!/usr/bin/env python
"""Cost of seeded sampling on the bench configuration: 64 utterances x 128 synthetic ids, forced 5 frames per id, the
`single_speaker_fast` architecture with seeded random weights (bench.py's workload; durations are forced, so the weights do
not change the shapes).  stts_batch_run is timed with sampling off and on (noise_scale 0.667, noise_scale_w 0.8, seed = the
utterance index), alternating after warm-up; each mode is staged before its run, outside the timed region.  Reports per-stage
GPU milliseconds from stts_last_timing (CUDA events on the engine's stream; the text encoder gains the `logs` conv, the length
regulator gains the RNG), the kernel launches per run, and the card's name and power limit read in the same process.

    python tools/sampling_bench.py [--steps 30] [--warmup 5] [--out profiles/sampling_bench.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

STAGES = ("enc", "dp", "regulate", "flow", "dec", "total")


def card():
    q = "name,power.limit,clocks.max.sm,driver_version"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().split(",")])) if r.returncode == 0 else {"error": r.stderr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from parity_util import synth_ids

    from summertts_b200 import binfmt, build, engine

    build.build_native()
    B, N, FR = 64, 128, 5
    E = engine.SynthesizerTrn(binfmt.synthetic_model(seed=11, **binfmt.ARCH["single_speaker_fast"]))
    utts = [synth_ids(np.random.default_rng(1234 + i), N) for i in range(B)]
    E.set_forced_durations(np.full(B * N, float(FR), np.float32))
    modes = {"off": {}, "on": dict(noise_scale=0.667, noise_scale_w=0.8, seed=np.arange(B, dtype=np.uint64))}
    rec = {m: {s: [] for s in STAGES} for m in modes}
    launches = {}
    for step in range(a.warmup + a.steps):
        for m, kw in modes.items():
            E.stage(utts, **kw)
            n0 = E.kernel_launches()
            total = E.run()
            launches[m] = E.kernel_launches() - n0
            assert total == B * N * FR * 256
            if step >= a.warmup:
                t = E.last_timing()
                for s in STAGES:
                    rec[m][s].append(t[s])
    res = {"workload": "%d x %d ids, forced %d frames/id, single_speaker_fast architecture, random weights" % (B, N, FR),
           "card": card(), "steps": a.steps, "warmup": a.warmup, "launches_per_run": launches,
           "note": "GPU ms per stage from CUDA events (stts_last_timing); modes alternate; no L2 flush (the 64 x 640-frame "
                   "working set is several times the 126 MB L2)"}
    for m in modes:
        res[m] = {s: dict(median=float(np.median(v)), min=float(np.min(v)), mean=float(np.mean(v))) for s, v in rec[m].items()}
    res["delta_median_ms"] = {s: res["on"][s]["median"] - res["off"][s]["median"] for s in STAGES}
    res["overhead_total_pct"] = 100.0 * res["delta_median_ms"]["total"] / res["off"]["total"]["median"]
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    E.close()


if __name__ == "__main__":
    main()
