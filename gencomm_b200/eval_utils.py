"""Detection evaluation on the GPU: the matching step of ``opencood/utils/eval_utils.py``.

``caluclate_tp_fp(det_boxes, det_score, gt_boxes, result_stat, iou_thresh)`` keeps the reference's name (misspelling
included), signature and in-place update of ``result_stat``; ``tools/inference.py`` calls it once per frame and IoU
threshold.  The reference copies the boxes to the host and, in score order, intersects each detection's shapely polygon
with every still-unmatched ground-truth polygon in Python; here one ``gc_eval_match`` launch (csrc/eval.cu) sorts,
intersects and matches on the device (the two counts go up in one small host-to-device copy) and one device-to-host
copy brings back the sorted scores and TP flags.

``DetectionEvaluator`` is the batched form: ``update`` takes ``VoxelPostprocessor.post_process_batch``'s padded output
plus padded ground truths, matches all frames at all thresholds in one launch and keeps the results on the device (no
host synchronisation); ``result_stat()`` returns the reference-format dict for every frame so far after one
synchronisation.  ``calculate_ap`` / ``eval_final_results`` stay with the reference: they read ``result_stat`` as is.

Pinned where the reference is unspecified: equal scores keep their input order (``np.argsort(-score)`` is a quicksort).
The polygon IoU is float64 convex clipping (DESIGN §5i); parity with shapely's polygon area is unpinned.  No CPU path.
"""
import numpy as np
import torch

from . import ops


def _at_least_one(t, shape):
    """Zero-row inputs get one unused row: the kernels take K, G >= 1 and read no row at or beyond the count."""
    return t if t.shape[1] > 0 else torch.empty(shape, dtype=t.dtype, device=t.device)


def _tail_offset(B, K, T):
    return (B * K * (4 + T) + 3) // 4 * 4


def _out_buffer(B, K, T, extra, dev):
    """One byte buffer holding sorted_scores [B,K] f32, tp [B,T,K] u8 and, from _tail_offset on, `extra` more bytes, so
    that a single copy brings everything to the host."""
    buf = torch.empty(_tail_offset(B, K, T) + extra, dtype=torch.uint8, device=dev)
    scores = buf[:B * K * 4].view(torch.float32).view(B, K)
    tp = buf[B * K * 4:B * K * (4 + T)].view(B, T, K)
    return buf, scores, tp


def caluclate_tp_fp(det_boxes, det_score, gt_boxes, result_stat, iou_thresh):
    """Drop-in for ``opencood.utils.eval_utils.caluclate_tp_fp``: det_boxes [K,8,3] f32 (or None), det_score [K] f32,
    gt_boxes [G,8,3] f32, CUDA tensors.  Appends the sorted scores, TP and FP flags to ``result_stat[iou_thresh]`` and
    adds G to its ``'gt'``, exactly as the reference does.  One ``gc_eval_match`` call, one 8-byte host-to-device copy of
    the counts (K, G) and one device-to-host copy of the results."""
    fp, tp = [], []
    gt = gt_boxes.shape[0]
    if det_boxes is not None:
        K = int(det_boxes.shape[0])
        scores = []
        if K > 0:
            dev = det_boxes.device
            boxes = ops._chk(det_boxes.contiguous(), "det_boxes", torch.float32, 3).view(1, K, 8, 3)
            score = ops._chk(det_score.contiguous(), "det_score", torch.float32, 1).view(1, K)
            gts = ops._chk(gt_boxes.contiguous(), "gt_boxes", torch.float32, 3).reshape(1, gt, 8, 3)
            gts = _at_least_one(gts, (1, 1, 8, 3))
            counts = torch.tensor([K, gt], dtype=torch.int32).to(dev)
            buf, s_out, tp_out = _out_buffer(1, K, 1, 0, dev)
            ops.eval_match(boxes, score, counts[0:1], gts, counts[1:2], [iou_thresh], out=(s_out, tp_out))
            host = buf.cpu()
            scores = host[:4 * K].view(torch.float32).tolist()
            tp = host[4 * K:5 * K].tolist()
            fp = [1 - v for v in tp]
        result_stat[iou_thresh]['score'] += scores
    result_stat[iou_thresh]['fp'] += fp
    result_stat[iou_thresh]['tp'] += tp
    result_stat[iou_thresh]['gt'] += gt


class DetectionEvaluator:
    """Sync-free, batched ``caluclate_tp_fp`` over frames and thresholds.

        ev = DetectionEvaluator((0.3, 0.5, 0.7))
        boxes, scores, counts = post_processor.post_process_batch(...)      # [B,1000,8,3], [B,1000], [B]
        ev.update(boxes, scores, counts, gt_boxes, gt_counts)              # [B,G,8,3], [B]
        ...
        result_stat = ev.result_stat()                                     # one synchronisation
    """

    def __init__(self, iou_thresholds=(0.3, 0.5, 0.7)):
        self.iou_thresholds = tuple(iou_thresholds)
        if not 1 <= len(self.iou_thresholds) <= ops.EVAL_MAX_THRESHOLDS:
            raise ValueError(f"DetectionEvaluator: 1..{ops.EVAL_MAX_THRESHOLDS} thresholds")
        self._pending = []   # (device buffer, B, K, G) of updates not yet copied to the host
        self._frames = []    # per frame: (sorted scores [k] f32, tp [T,k] u8, n_gt)

    def update(self, boxes, scores, counts, gt_boxes, gt_counts):
        """boxes [B,K,8,3] f32, scores [B,K] f32, counts [B] i32, gt_boxes [B,G,8,3] f32, gt_counts [B] i32 (cuda).
        Rows at or beyond a frame's count are ignored; counts outside [0, K] / [0, G] are clamped.  Asynchronous."""
        B, K = int(boxes.shape[0]), int(boxes.shape[1])
        T = len(self.iou_thresholds)
        dev = boxes.device
        G = int(gt_boxes.shape[1])
        ops._chk(counts, "counts", torch.int32, 1)
        ops._chk(gt_counts, "gt_counts", torch.int32, 1)
        if K == 0:   # nothing to match: every frame adds its ground truths only
            counts = torch.zeros_like(counts)
        if G == 0:
            gt_counts = torch.zeros_like(gt_counts)
        boxes = _at_least_one(boxes.contiguous(), (B, 1, 8, 3))
        scores = _at_least_one(scores.contiguous(), (B, 1))
        gt_boxes = _at_least_one(gt_boxes.contiguous(), (B, 1, 8, 3))
        Kp = int(boxes.shape[1])
        buf, s_out, tp_out = _out_buffer(B, Kp, T, 8 * B, dev)
        ops.eval_match(boxes, scores, counts, gt_boxes, gt_counts, self.iou_thresholds, out=(s_out, tp_out))
        # the counts travel with the results (the host applies the kernel's clamping to them)
        tail = buf[_tail_offset(B, Kp, T):].view(torch.int32).view(2, B)
        tail[0].copy_(counts)
        tail[1].copy_(gt_counts)
        self._pending.append((buf, B, Kp, G))

    def _drain(self):
        if not self._pending:
            return
        host = [(b.to("cpu", non_blocking=True), B, Kp, G) for b, B, Kp, G in self._pending]
        torch.cuda.current_stream().synchronize()
        self._pending = []
        T = len(self.iou_thresholds)
        for h, B, Kp, G in host:
            a = h.numpy()
            sc = a[:B * Kp * 4].view(np.float32).reshape(B, Kp)
            tp = a[B * Kp * 4:B * Kp * (4 + T)].reshape(B, T, Kp)
            cnt = a[_tail_offset(B, Kp, T):].view(np.int32).reshape(2, B)
            for b in range(B):
                k = min(max(int(cnt[0, b]), 0), Kp)
                g = min(max(int(cnt[1, b]), 0), G)
                self._frames.append((sc[b, :k], tp[b, :, :k], g))

    def result_stat(self):
        """{iou_thresh: {'tp': [...], 'fp': [...], 'gt': int, 'score': [...]}} over every frame passed to ``update``, in
        update order -- what the reference's per-frame ``caluclate_tp_fp`` calls accumulate.  A frame with no detection
        adds its ground truths only (the reference's ``det_boxes is None``).  Synchronises once."""
        self._drain()
        out = {t: {'tp': [], 'fp': [], 'gt': 0, 'score': []} for t in self.iou_thresholds}
        for sc, tp, g in self._frames:
            for ti, t in enumerate(self.iou_thresholds):
                r = out[t]
                r['gt'] += g
                if sc.shape[0] == 0:
                    continue
                flags = tp[ti].tolist()
                r['score'] += sc.tolist()
                r['tp'] += flags
                r['fp'] += [1 - v for v in flags]
        return out

    def reset(self):
        self._pending, self._frames = [], []
