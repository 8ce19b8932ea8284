#!/usr/bin/env python
"""Microbench of the GPU evaluation matching (DetectionEvaluator.update -> gc_eval_match) on synthetic frames.

    python scripts/bench_eval.py [--iters 200] [--warmup 20] [--out FILE]

Two shapes, three IoU thresholds (0.3 / 0.5 / 0.7): 15 frames x K = 100 detections x G = 60 ground truths, and 15 frames x
K = 1000 x G = 200.  CUDA-event time of update() per call (inputs already on the device; the whole working set stays in
L2, as it does after the NMS that produces it).  The only host figure is the in-repo CPU oracle (tests/eval_oracle.py:
Python loop + the C IoU of oracle/nms_ref.c), labelled as such -- it is not the reference's shapely path.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from gencomm_b200 import DetectionEvaluator, synth  # noqa: E402

THRESH = (0.3, 0.5, 0.7)
SHAPES = {"15x100x60": (15, 100, 60), "15x1000x200": (15, 1000, 200)}


def card():
    name = torch.cuda.get_device_name()
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def aabb_pairs(f):
    """IoU pairs per frame that pass the axis-aligned box test (the ones k_eval_iou clips), mean over frames."""
    n = []
    for b in range(f["det_counts"].shape[0]):
        k, g = int(f["det_counts"][b]), int(f["gt_counts"][b])
        d, t = f["det_boxes"][b, :k, :4, :2].double().numpy(), f["gt_boxes"][b, :g, :4, :2].double().numpy()
        dlo, dhi, tlo, thi = d.min(1), d.max(1), t.min(1), t.max(1)
        apart = (tlo[None, :, 0] > dhi[:, None, 0]) | (thi[None, :, 0] < dlo[:, None, 0]) | \
                (tlo[None, :, 1] > dhi[:, None, 1]) | (thi[None, :, 1] < dlo[:, None, 1])
        n.append(int((~apart).sum()))
    return float(np.mean(n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--oracle-frames", type=int, default=1, help="frames of the CPU oracle timing per shape (0: skip)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval: needs a CUDA device")
    name, limit = card()
    rows = []
    for label, (B, K, G) in SHAPES.items():
        f = synth.eval_frames(31, B, k_max=K, g_max=G, n_gt=(G, G), full=range(B))
        d = {k: v.cuda() for k, v in f.items()}
        ev = DetectionEvaluator(THRESH)
        for _ in range(args.warmup):
            ev.update(d["det_boxes"], d["det_scores"], d["det_counts"], d["gt_boxes"], d["gt_counts"])
        torch.cuda.synchronize()
        ev.reset()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            ev.update(d["det_boxes"], d["det_scores"], d["det_counts"], d["gt_boxes"], d["gt_counts"])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.iters
        ev.reset()
        row = {"shape": f"{B} frames x K {K} x G {G}, thresholds {list(THRESH)}", "ms_per_update": round(ms, 4),
               "frames_per_s": round(B / ms * 1e3, 1), "iou_pairs_per_frame": K * G,
               "iou_pairs_per_frame_after_aabb_reject": aabb_pairs(f), "iters": args.iters}
        if args.oracle_frames > 0:
            import eval_oracle as E
            st = {t: {'tp': [], 'fp': [], 'gt': 0, 'score': []} for t in THRESH}
            t0 = time.perf_counter()
            for b in range(args.oracle_frames):
                for t in THRESH:
                    E.caluclate_tp_fp(f["det_boxes"][b], f["det_scores"][b], f["gt_boxes"][b], st, t)
            row["cpu_oracle_ms_per_frame_not_reference"] = round((time.perf_counter() - t0) * 1e3 / args.oracle_frames, 2)
        rows.append(row)
    out = {"workload": "DetectionEvaluator.update (gc_eval_match: prep + IoU + match), CUDA events",
           "gpu": name, "power_limit": limit, "results": rows}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
