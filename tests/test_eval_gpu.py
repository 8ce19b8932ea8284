"""GPU evaluation matching (csrc/eval.cu) against the oracle's literal caluclate_tp_fp (tests/eval_oracle.py).

Bar: identical.  The IoU is bit-matched to the oracle's (the same float64 clipping), the sort and the greedy match are
integer work, so sorted scores, TP / FP flags, GT counts and the AP computed from them must all be equal.
"""
import copy

import numpy as np
import pytest
import torch

from gencomm_b200 import DetectionEvaluator, VoxelPostprocessor, caluclate_tp_fp, ops, synth
import eval_oracle as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
THRESH = (0.3, 0.5, 0.7)
# 8 frames, G up to 200, frame 3 at K = 1000, frame 1 without detections, frame 5 without ground truths; and a batch
# with many equal scores
BATCHES = {"mixed": dict(seed=7, n_frames=8, k_max=1000, g_max=200, n_gt=(1, 200), no_det=(1,), no_gt=(5,), full=(3,)),
           "ties": dict(seed=8, n_frames=4, k_max=400, g_max=120, n_gt=(40, 120), score_step=0.05)}


def _stat():
    return {t: {'tp': [], 'fp': [], 'gt': 0, 'score': []} for t in THRESH}


def _frame(f, b):
    k, g = int(f["det_counts"][b]), int(f["gt_counts"][b])
    return f["det_boxes"][b, :k], f["det_scores"][b, :k], f["gt_boxes"][b, :g]


@pytest.fixture(scope="module")
def batches():
    """name -> (frames, per-frame oracle result_stat)"""
    out = {}
    for name, kw in BATCHES.items():
        kw = dict(kw)
        f = synth.eval_frames(kw.pop("seed"), kw.pop("n_frames"), **kw)
        per_frame = []
        for b in range(f["det_counts"].shape[0]):
            det, sc, gt = _frame(f, b)
            st = _stat()
            for t in THRESH:
                R.caluclate_tp_fp(det if det.shape[0] else None, sc, gt, st, t)
            per_frame.append(st)
        out[name] = (f, per_frame)
    return out


def _merged(per_frame):
    st = _stat()
    for fr in per_frame:
        for t in THRESH:
            for key in ('tp', 'fp', 'gt', 'score'):
                st[t][key] += fr[t][key]
    return st


@pytest.mark.parametrize("name", list(BATCHES))
def test_kernel_matches_oracle(batches, name):
    f, per_frame = batches[name]
    d = {k: v.to(DEV) for k, v in f.items()}
    scores, tp = ops.eval_match(d["det_boxes"], d["det_scores"], d["det_counts"], d["gt_boxes"], d["gt_counts"], THRESH)
    scores, tp = scores.cpu().numpy(), tp.cpu().numpy()
    for b, ref in enumerate(per_frame):
        k = int(f["det_counts"][b])
        assert not scores[b, k:].any() and not tp[b, :, k:].any(), b
        for ti, t in enumerate(THRESH):
            assert scores[b, :k].tolist() == ref[t]['score'], (b, t)
            assert tp[b, ti, :k].tolist() == ref[t]['tp'], (b, t)
    if name == "mixed":   # the batch exercises what it is meant to
        ref = _merged(per_frame)
        assert sum(ref[0.3]['tp']) > sum(ref[0.7]['tp']) > 0 and sum(ref[0.7]['fp']) > 0


def test_counts_out_of_range_are_clamped(batches):
    f, _ = batches["ties"]
    d = {k: v.to(DEV) for k, v in f.items()}
    K, G = d["det_boxes"].shape[1], d["gt_boxes"].shape[1]
    dc = torch.tensor([-5, 10 ** 6, 3, 2], dtype=torch.int32, device=DEV)
    gc = torch.tensor([7, -1, 10 ** 6, 5], dtype=torch.int32, device=DEV)
    scores, tp = ops.eval_match(d["det_boxes"], d["det_scores"], dc, d["gt_boxes"], gc, THRESH)
    c = {"det_counts": torch.tensor([0, K, 3, 2], dtype=torch.int32), "gt_counts": torch.tensor([7, 0, G, 5], dtype=torch.int32)}
    want = dict(f, **c)
    s2, tp2 = ops.eval_match(*(want[k].to(DEV) for k in ("det_boxes", "det_scores", "det_counts", "gt_boxes", "gt_counts")),
                             THRESH)
    assert torch.equal(scores, s2) and torch.equal(tp, tp2)


@pytest.mark.parametrize("name", list(BATCHES))
def test_drop_in_fills_result_stat_like_the_oracle(batches, name):
    f, per_frame = batches[name]
    st = _stat()
    for b in range(f["det_counts"].shape[0]):
        det, sc, gt = _frame(f, b)
        for t in THRESH:
            caluclate_tp_fp(det.to(DEV) if det.shape[0] else None, sc.to(DEV), gt.to(DEV), st, t)
    ref = _merged(per_frame)
    assert st == ref
    for t in THRESH:
        for glob in (False, True):
            assert R.calculate_ap(copy.deepcopy(st), t, glob) == R.calculate_ap(copy.deepcopy(ref), t, glob)


def test_evaluator_end_to_end_on_post_process_batch():
    """post_process_batch output of synthetic head maps (one frame without detections), ground truths made from
    jittered detections plus extra cars, over two updates: result_stat() equals the per-frame drop-in calls and the
    oracle."""
    pp = VoxelPostprocessor(synth.postprocess_params(), train=False)
    anchors = torch.from_numpy(pp.generate_anchor_box()).float().to(DEV)
    ev = DetectionEvaluator(THRESH)
    st, ref = _stat(), _stat()
    g_max = 96
    for part, (seeds, biases) in enumerate([((1, 2, 3), (-3.0, -1.0, -9.0)), ((4, 5), (-4.5, -3.0))]):
        heads = [synth.head_outputs(s, bias=bb) for s, bb in zip(seeds, biases)]
        cls, reg, dr = (torch.cat([h[i] for h in heads]).to(DEV) for i in range(3))
        boxes, scores, counts = pp.post_process_batch(cls, reg, dr, anchors)
        B = boxes.shape[0]
        hb, hc = boxes.cpu().numpy(), counts.cpu().numpy()
        assert part or hc[2] == 0
        gt = np.zeros((B, g_max, 8, 3), np.float32)
        gcount = np.zeros(B, np.int32)
        for b in range(B):
            g = np.random.default_rng(100 * part + b)
            pick = hb[b, :hc[b]][g.random(hc[b]) < 0.6]
            moved = pick + np.concatenate([g.normal(0, 0.4, (len(pick), 1, 2)), np.zeros((len(pick), 1, 1))], 2).astype(np.float32)
            extra = synth.box_corners(np.stack([g.uniform(-90, 90, 5), g.uniform(-45, 45, 5), np.full(5, -1.5),
                                                np.full(5, 4.0), np.full(5, 1.8), np.full(5, 1.6), g.uniform(-3, 3, 5)], 1))
            both = np.concatenate([moved, extra])[:g_max]
            gt[b, :len(both)], gcount[b] = both, len(both)
        gt_d, gc_d = torch.from_numpy(gt).to(DEV), torch.from_numpy(gcount).to(DEV)
        ev.update(boxes, scores, counts, gt_d, gc_d)
        for b in range(B):
            k, g = int(hc[b]), int(gcount[b])
            for t in THRESH:
                caluclate_tp_fp(boxes[b, :k] if k else None, scores[b, :k], gt_d[b, :g], st, t)
                R.caluclate_tp_fp(hb[b, :k] if k else None, scores[b, :k].cpu(), gt[b, :g], ref, t)
    out = ev.result_stat()
    assert out == st == ref
    assert sum(out[0.5]['tp']) > 0 and sum(out[0.5]['fp']) > 0
    assert ev.result_stat() == out     # nothing is counted twice


def _car(x, y, l, w):
    return synth.box_corners(np.array([[x, y, -1.5, l, w, 1.5, 0.0]]))[0]


def test_nan_rule_and_float32_threshold_on_the_gpu():
    """Hand-built frames for the two rules synth.eval_frames never reaches.  Frames 0 and 1: zero-area detections against
    zero-area ground truths give IoU 0 / 0 = NaN, through the disjoint-AABB branch of k_eval_iou (frame 0) and through the
    clipping (frame 1, same place); numpy's max / argmax make each a TP matched to the first NaN.  Frame 2: IoU exactly
    float32(0.7) (overlap 7 x 2 over union 10 x 2), which the float32-widened-to-double comparison makes a FP at 0.7."""
    frames = [([_car(60, -20, 0, 2)] * 3, [_car(0, 0, 4, 2), _car(50, 20, 0, 2), _car(-50, 20, 0, 2)]),
              ([_car(50, 20, 0, 2)] * 2, [_car(0, 0, 4, 2), _car(50, 20, 0, 2)]),
              ([_car(4.25, 0, 8.5, 2)], [_car(5.75, 0, 8.5, 2)])]
    K, G = 3, 3
    det, gt = np.zeros((3, K, 8, 3), np.float32), np.zeros((3, G, 8, 3), np.float32)
    sc = np.zeros((3, K), np.float32)
    dc, gc = np.zeros(3, np.int32), np.zeros(3, np.int32)
    for b, (d, g) in enumerate(frames):
        det[b, :len(d)], gt[b, :len(g)] = d, g
        sc[b, :len(d)] = [0.9, 0.8, 0.7][:len(d)]
        dc[b], gc[b] = len(d), len(g)
    assert R.compute_iou(R.convert_format(det[2, :1])[0], R.convert_format(gt[2, :1]))[0] == np.float32(0.7)
    scores, tp = ops.eval_match(*(torch.from_numpy(a).to(DEV) for a in (det, sc, dc, gt, gc)), THRESH)
    tp = tp.cpu().numpy()
    st = _stat()
    for b in range(3):
        k, g = int(dc[b]), int(gc[b])
        ref = _stat()
        for ti, t in enumerate(THRESH):
            R.caluclate_tp_fp(det[b, :k], sc[b, :k], gt[b, :g], ref, t)
            caluclate_tp_fp(torch.from_numpy(det[b, :k]).to(DEV), torch.from_numpy(sc[b, :k]).to(DEV),
                            torch.from_numpy(gt[b, :g]).to(DEV), st, t)
            assert tp[b, ti, :k].tolist() == ref[t]['tp'], (b, t)
    assert tp[0, :, :3].tolist() == [[1, 1, 0]] * 3 and tp[1, :, :2].tolist() == [[1, 0]] * 3
    assert tp[2, :, 0].tolist() == [1, 1, 0]
    assert st[0.7]['tp'] == [1, 1, 0, 1, 0, 0] and st[0.5]['tp'][-1] == 1
