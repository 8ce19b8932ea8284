"""TEST INFRASTRUCTURE ONLY -- CPU oracle of the evaluation matching: eval_utils.caluclate_tp_fp / calculate_ap / voc_ap
(opencood/utils/eval_utils.py) with common_utils.convert_format and compute_iou (utils/common_utils.py:230-270).

A literal transcription (Python lists, list.pop, np.argmax), except:
  - shapely's Polygon IoU is gc_ref_quad_iou (oracle/nms_ref.c, through oracle/ref_ops.py) over the bottom-face quads:
    parity with shapely's area is unpinned, as for the NMS (DESIGN §5g);
  - np.argsort(-det_score) is pinned stable: equal scores keep their input order (the reference's quicksort leaves it
    unspecified);
  - `np.max(ious) < iou_thresh` is evaluated as numpy 1 does for a float32 scalar against a Python float: the float32
    widened to double (numpy 2 would compare in float32).
Imported by the evaluation tests and by scripts/bench_eval.py's labelled host comparison; gencomm_b200 never imports it.
"""
import numpy as np
import torch

from oracle import ref_ops as R


def _host(a):
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)


def convert_format(boxes_array):
    """[N,8,3] corners -> list of bottom-face quads [4,2] float64 (the vertices of convert_format's Polygons)."""
    quads = np.ascontiguousarray(np.asarray(boxes_array)[:, :4, :2], dtype=np.float64)
    return [quads[i] for i in range(quads.shape[0])]


def compute_iou(box, boxes):
    iou = [R._lib().gc_ref_quad_iou(R._p(box), R._p(b)) for b in boxes]
    return np.array(iou, dtype=np.float32)


def caluclate_tp_fp(det_boxes, det_score, gt_boxes, result_stat, iou_thresh):
    fp = []
    tp = []
    gt = gt_boxes.shape[0]
    if det_boxes is not None:
        det_boxes = _host(det_boxes)
        det_score = _host(det_score)
        gt_boxes = _host(gt_boxes)

        score_order_descend = np.argsort(-det_score, kind="stable")
        det_score = det_score[score_order_descend]
        det_polygon_list = list(convert_format(det_boxes))
        gt_polygon_list = list(convert_format(gt_boxes))

        for i in range(score_order_descend.shape[0]):
            det_polygon = det_polygon_list[score_order_descend[i]]
            ious = compute_iou(det_polygon, gt_polygon_list)

            if len(gt_polygon_list) == 0 or float(np.max(ious)) < iou_thresh:
                fp.append(1)
                tp.append(0)
                continue

            fp.append(0)
            tp.append(1)

            gt_index = np.argmax(ious)
            gt_polygon_list.pop(gt_index)
        result_stat[iou_thresh]['score'] += det_score.tolist()

    result_stat[iou_thresh]['fp'] += fp
    result_stat[iou_thresh]['tp'] += tp
    result_stat[iou_thresh]['gt'] += gt


def calculate_ap(result_stat, iou, global_sort_detections=False):
    """As the reference, including its side effect: without global sorting the cumulative sums are written into
    result_stat[iou]['tp'] / ['fp'] themselves."""
    iou_5 = result_stat[iou]

    if global_sort_detections:
        fp = np.array(iou_5['fp'])
        tp = np.array(iou_5['tp'])
        score = np.array(iou_5['score'])

        assert len(fp) == len(tp) and len(tp) == len(score)
        sorted_index = np.argsort(-score)
        fp = fp[sorted_index].tolist()
        tp = tp[sorted_index].tolist()
    else:
        fp = iou_5['fp']
        tp = iou_5['tp']
        assert len(fp) == len(tp)

    gt_total = iou_5['gt']

    cumsum = 0
    for idx, val in enumerate(fp):
        fp[idx] += cumsum
        cumsum += val

    cumsum = 0
    for idx, val in enumerate(tp):
        tp[idx] += cumsum
        cumsum += val

    rec = tp[:]
    for idx, val in enumerate(tp):
        rec[idx] = float(tp[idx]) / gt_total

    prec = tp[:]
    for idx, val in enumerate(tp):
        prec[idx] = float(tp[idx]) / (fp[idx] + tp[idx])

    ap, mrec, mprec = voc_ap(rec[:], prec[:])

    return ap, mrec, mprec


def voc_ap(rec, prec):
    rec.insert(0, 0.0)
    rec.append(1.0)
    mrec = rec[:]

    prec.insert(0, 0.0)
    prec.append(0.0)
    mpre = prec[:]

    for i in range(len(mpre) - 2, -1, -1):
        mpre[i] = max(mpre[i], mpre[i + 1])

    i_list = []
    for i in range(1, len(mrec)):
        if mrec[i] != mrec[i - 1]:
            i_list.append(i)

    ap = 0.0
    for i in i_list:
        ap += ((mrec[i] - mrec[i - 1]) * mpre[i])
    return ap, mrec, mpre
