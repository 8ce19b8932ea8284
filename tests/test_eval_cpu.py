"""Evaluation matching without a GPU: known answers of the oracle's caluclate_tp_fp / calculate_ap / voc_ap
(tests/eval_oracle.py: the reference's eval_utils with the polygon IoU of oracle/nms_ref.c), the argument errors of
gc_eval_match and the synthetic frame generator."""
import copy
import ctypes

import numpy as np
import pytest
import torch

from gencomm_b200 import _lib, ops, synth
import eval_oracle as R


def _boxes(*specs):
    """(x, y, l, w[, yaw]) -> [N,8,3] f32 corners (z centre -1.5, h 1.5)."""
    rows = [(s[0], s[1], -1.5, s[2], s[3], 1.5, s[4] if len(s) > 4 else 0.0) for s in specs]
    return synth.box_corners(np.array(rows, dtype=np.float64))


def _stat(*thresholds):
    return {t: {'tp': [], 'fp': [], 'gt': 0, 'score': []} for t in thresholds}


def _quads(b):
    return R.convert_format(b)


def _run(det, scores, gt, thr=0.5):
    st = _stat(thr)
    R.caluclate_tp_fp(det, None if det is None else np.asarray(scores, np.float32), gt, st, thr)
    return st[thr]


def test_iou_known_answers():
    a, far, half = _quads(_boxes((0, 0, 4, 2), (30, 30, 4, 2), (2, 0, 4, 2)))
    assert R.compute_iou(a, [a])[0] == np.float32(1.0)
    assert R.compute_iou(a, [far])[0] == np.float32(0.0)
    assert R.compute_iou(a, [half])[0] == np.float32(1.0 / 3.0)      # 4 / (8 + 8 - 4)
    rot = _quads(_boxes((0, 0, 4, 2, np.pi)))[0]                        # same rectangle, corners in another order
    assert abs(float(R.compute_iou(a, [rot])[0]) - 1.0) < 1e-6
    assert R.compute_iou(a, []).shape == (0,)


def test_higher_score_takes_the_gt_a_later_detection_wanted():
    gt = _boxes((0, 0, 4, 2))
    det = _boxes((0.6, 0, 4, 2), (0, 0, 4, 2))                          # IoU 0.74 (score 0.9), IoU 1 (score 0.8)
    assert 0.5 < float(R.compute_iou(_quads(det)[0], _quads(gt))[0]) < 1.0
    r = _run(det, [0.9, 0.8], gt)
    assert r == {'tp': [1, 0], 'fp': [0, 1], 'gt': 1, 'score': [np.float32(0.9).item(), np.float32(0.8).item()]}


def test_equal_ious_match_the_lower_gt_index():
    gt = _boxes((1, 0, 4, 2), (-1, 0, 4, 2))                            # symmetric about the first detection
    det = _boxes((0, 0, 4, 2), (-1, 0, 4, 2))
    ious = R.compute_iou(_quads(det)[0], _quads(gt))
    assert ious[0] == ious[1] and ious[0] > 0.5
    # the first detection takes gt 0, so the second (identical to gt 1) still finds its box; had the first taken gt 1,
    # the second would be left with gt 0 at IoU 1/3
    assert _run(det, [0.9, 0.8], gt)['tp'] == [1, 1]


def test_equal_scores_keep_input_order():
    gt = _boxes((0, 0, 4, 2))
    det = _boxes((2.2, 0, 4, 2), (0, 0, 4, 2))                          # IoU 0.29, then IoU 1, equal scores
    assert _run(det, [0.7, 0.7], gt)['tp'] == [0, 1]
    assert _run(det[::-1].copy(), [0.7, 0.7], gt)['tp'] == [1, 0]
    r = _run(det, [0.6, 0.7], gt)                                       # a strictly larger score goes first
    assert r['tp'] == [1, 0] and r['score'] == [np.float32(0.7).item(), np.float32(0.6).item()]


def test_empty_detections_and_empty_gts():
    gt = _boxes((0, 0, 4, 2), (10, 0, 4, 2))
    assert _run(None, None, gt) == {'tp': [], 'fp': [], 'gt': 2, 'score': []}
    r = _run(_boxes((0, 0, 4, 2), (5, 5, 4, 2)), [0.3, 0.4], np.zeros((0, 8, 3), np.float32))
    assert r['tp'] == [0, 0] and r['fp'] == [1, 1] and r['gt'] == 0 and len(r['score']) == 2


def test_nan_iou_is_a_tp_matched_to_the_first_nan():
    """A zero-area detection against a zero-area ground truth gives 0 / 0: numpy's max is NaN (not < threshold, so a TP)
    and argmax picks the first NaN."""
    gt = _boxes((0, 0, 4, 2), (50, 20, 0, 2), (-50, 20, 0, 2))         # a real box, then two zero-area ones
    det = _boxes((60, -20, 0, 2), (60, -20, 0, 2), (60, -20, 0, 2))
    ious = R.compute_iou(_quads(det)[0], _quads(gt))
    assert ious[0] == 0 and np.isnan(ious[1]) and np.isnan(ious[2])
    # 1st takes gt 1, 2nd takes gt 2, 3rd only sees the real box (IoU 0)
    assert _run(det, [0.9, 0.8, 0.7], gt)['tp'] == [1, 1, 0]


def test_voc_ap_and_calculate_ap_against_hand_computed_lists():
    ap, mrec, mpre = R.voc_ap([0.5, 0.5, 1.0], [1.0, 0.5, 2.0 / 3.0])
    assert mrec == [0.0, 0.5, 0.5, 1.0, 1.0]
    assert mpre == [1.0, 1.0, 2.0 / 3.0, 2.0 / 3.0, 0.0]
    assert ap == 0.5 * 1.0 + 0.5 * (2.0 / 3.0)
    st = {0.5: {'tp': [1, 0, 1], 'fp': [0, 1, 0], 'gt': 2, 'score': [0.9, 0.8, 0.7]}}
    ap2, _, _ = R.calculate_ap(copy.deepcopy(st), 0.5)
    assert ap2 == ap
    # global sorting reorders by score first: scores 0.7 / 0.9 / 0.8 -> tp [0, 1, 1] -> rec [0, .5, 1], prec [0, .5, 2/3]
    st = {0.5: {'tp': [1, 0, 1], 'fp': [0, 1, 0], 'gt': 2, 'score': [0.8, 0.9, 0.7]}}
    ap3, _, _ = R.calculate_ap(copy.deepcopy(st), 0.5, True)
    assert ap3 == 0.5 * (2.0 / 3.0) + 0.5 * (2.0 / 3.0)
    # the reference writes the cumulative sums back into result_stat when it does not sort globally
    R.calculate_ap(st, 0.5)
    assert st[0.5]['tp'] == [1, 1, 2] and st[0.5]['fp'] == [0, 1, 1]


def test_eval_match_argument_errors_are_reported_without_a_gpu():
    lib = _lib.load()
    p = ctypes.c_void_p(16)                        # never dereferenced: every call below fails its argument check
    th = (ctypes.c_double * 3)(0.3, 0.5, 0.7)

    def call(k_max=10, g_max=10, n_frames=2, n_thresh=3, null=None):
        args = [p, p, p, k_max, p, p, g_max, n_frames, th, n_thresh, p, p, p, None]
        if null is not None:
            args[null] = None
        return lib.gc_eval_match(*args)

    for null in (0, 1, 2, 4, 5, 8, 10, 11, 12):
        assert call(null=null) == -1 and b"null" in lib.gc_last_error()
    for kw, word in [({"n_frames": 0}, b"n_frames"), ({"k_max": 0}, b"k_max"), ({"k_max": 1025}, b"k_max"),
                     ({"g_max": 0}, b"g_max"), ({"g_max": 1025}, b"g_max"), ({"n_thresh": 0}, b"n_thresh"),
                     ({"n_thresh": 9}, b"n_thresh")]:
        assert call(**kw) == -1 and word in lib.gc_last_error(), kw
    assert lib.gc_eval_workspace_bytes(0, 10, 10) == 0 and lib.gc_eval_workspace_bytes(1, 1025, 10) == 0
    assert lib.gc_eval_workspace_bytes(2, 1000, 200) > lib.gc_eval_workspace_bytes(1, 1000, 200) > 1000 * 200 * 4


def test_ops_eval_match_refuses_cpu_tensors():
    f = synth.eval_frames(1, 1, k_max=4, g_max=4, n_gt=(2, 2))
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.eval_match(f["det_boxes"], f["det_scores"], f["det_counts"], f["gt_boxes"], f["gt_counts"], (0.5,))


def test_eval_frames_generator():
    f = synth.eval_frames(3, 6, k_max=1000, g_max=200, n_gt=(1, 200), no_det=(1,), no_gt=(2,), full=(3,))
    assert f["det_boxes"].shape == (6, 1000, 8, 3) and f["gt_boxes"].shape == (6, 200, 8, 3)
    assert f["det_scores"].dtype == torch.float32 and f["det_counts"].dtype == torch.int32
    dc, gc = f["det_counts"].tolist(), f["gt_counts"].tolist()
    assert dc[1] == 0 and gc[2] == 0 and dc[2] > 0 and dc[3] == 1000 and max(gc) <= 200
    for b in range(6):
        s = f["det_scores"][b, :dc[b]]
        assert bool(((s >= 0.2) & (s <= 1.0)).all()) and not f["det_scores"][b, dc[b]:].any()
        g = f["gt_boxes"][b, :gc[b]].numpy()
        assert (g[..., 0] > -102.4).all() and (g[..., 0] < 102.4).all() and (g[..., 1] > -51.2).all() and (g[..., 1] < 51.2).all()
        length = np.linalg.norm(g[:, 0, :2] - g[:, 3, :2], axis=1)                  # corners 0 -> 3 span l
        width = np.linalg.norm(g[:, 0, :2] - g[:, 1, :2], axis=1)
        assert (length > 3.49).all() and (length < 5.01).all() and (width > 1.59).all() and (width < 2.11).all()
    again = synth.eval_frames(3, 6, k_max=1000, g_max=200, n_gt=(1, 200), no_det=(1,), no_gt=(2,), full=(3,))
    assert all(torch.equal(f[k], again[k]) for k in f)
    ties = synth.eval_frames(3, 2, k_max=300, g_max=100, n_gt=(50, 100), score_step=0.05)
    s = ties["det_scores"][0, :int(ties["det_counts"][0])]
    assert len(torch.unique(s)) < len(s)
