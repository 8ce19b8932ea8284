#!/usr/bin/env python
"""Whole-frame bench of HeterModelBaseline -- intermediate fusion of full BEV features without GenComm -- from raw LiDAR
points to decoded, NMS-filtered boxes, next to the stage-1 GenComm detector measured the same way in the same run.

    python scripts/bench_baseline.py [--frames 15] [--agents 4] [--points 100000] [--steps 30] [--warmup 5] [--out FILE]

Both detectors run through pipeline.DetectorPipeline at the OPV2V-H shape (m1_att.yaml model arguments, att fusion; the
baseline drops the message extractor, sampler and Enhancer blocks) on pipeline.synthetic_detector_inputs, the inputs
bench.py uses.  Three distinct input sets are cycled, so a step never finds its inputs in L2 (each step also streams the
> 1 GB canvas and backbone activations of its 60 agents).  Per detector: warm-up steps, then ``--steps`` steps between two
CUDA events (no per-stage events in that window: ``ms_per_step`` / ``frames_per_s``), then the same steps again with CUDA
events around every stage (``stage_ms``; ``heads_and_glue`` is that window's step time minus the stages).
"""
import argparse
import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from bench_eval import card  # noqa: E402
from gencomm_b200 import pipeline, synth  # noqa: E402

N_SETS = 3


def measure(detector, sets, F, N, P, steps, warmup):
    pipe = pipeline.DetectorPipeline(F, N, P, detector=detector)
    pipe.enable_stage_timing()
    pipe._marks = None                 # hooks registered, no events until the stage window

    def run(n):
        det = None
        for k in range(n):
            det = pipe.step(*sets[k % N_SETS])
        return det

    run(warmup)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    det = run(steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps

    pipe._marks = []
    e0.record()
    run(steps)
    e1.record()
    torch.cuda.synchronize()
    ms_marked = e0.elapsed_time(e1) / steps
    stage = pipe.stage_ms(steps)
    stage["heads_and_glue"] = ms_marked - sum(stage.values())
    return {"ms_per_step": round(ms, 3), "frames_per_s": round(F / ms * 1e3, 1),
            "stage_ms": {k: round(v, 3) for k, v in stage.items()}, "ms_per_step_with_stage_events": round(ms_marked, 3),
            "detections_per_frame": det[2].tolist()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=15)
    ap.add_argument("--agents", type=int, default=4)
    ap.add_argument("--points", type=int, default=100_000)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_baseline: needs a CUDA device")
    F, N, P = args.frames, args.agents, args.points
    name, limit = card()
    sets = []
    for s in range(N_SETS):
        p, pw = pipeline.synthetic_detector_inputs(1 + s, F, N, P, synth.OPV2V_H_RANGE)
        sets.append((torch.from_numpy(p).cuda(), torch.from_numpy(pw).cuda()))
    results = {}
    for detector in ("baseline", "gencomm"):
        results[detector] = measure(detector, sets, F, N, P, args.steps, args.warmup)
        torch.cuda.empty_cache()
    out = {"workload": f"raw points -> NMS'd boxes, {F} frames x {N} agents x {P} points per step, OPV2V-H grid, att fusion; "
                       f"{N_SETS} input sets cycled, {args.warmup} warm-up + {args.steps} timed steps, CUDA events",
           "gpu": name, "power_limit": limit,
           "baseline": dict(results["baseline"], model="HeterModelBaseline (full 128-channel BEV features)"),
           "gencomm": dict(results["gencomm"], model="HeterModelBaselineWGenComm (stage 1, default sampler precision)")}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
