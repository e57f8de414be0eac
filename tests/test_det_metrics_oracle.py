"""CPU: the detection-metric specification (oracle/det_metrics_oracle.py) -- the restated ultralytics matching and
ap_per_class that the metric kernels are compared against."""
import numpy as np
import pytest

from oracle import det_metrics_oracle as S


def _records(tp_rows, conf, cls):
    return np.array(tp_rows, bool).reshape(-1, 10), np.array(conf, np.float32), np.array(cls, np.int64)


def test_matcher_equals_unique_chain_on_tie_heavy_cases():
    rng = np.random.default_rng(0)
    for it in range(4000):
        ng, npd = int(rng.integers(0, 7)), int(rng.integers(0, 10))
        if it % 2:
            # IoU matrices on a coarse grid: many exact ties within and across rows / columns
            iou = (np.round(rng.random((ng, npd)) * 5) / 10 + 0.45).astype(np.float32) * (rng.random((ng, npd)) < 0.8)
        else:
            # boxes on an integer grid, duplicated predictions: ties from identical geometry
            gt = rng.integers(0, 8, (ng, 2)).astype(np.float32)
            gt = np.concatenate((gt, gt + rng.integers(1, 4, (ng, 2))), 1)
            src = gt[rng.integers(0, max(ng, 1), npd)] if ng else np.zeros((npd, 4), np.float32)
            pr = (src + rng.integers(-1, 2, (npd, 4)) * (rng.random((npd, 1)) < 0.5)).astype(np.float32)
            pr[:, 2:] = np.maximum(pr[:, 2:], pr[:, :2] + 1)
            iou = S.box_iou(gt, pr)
        gc = rng.integers(0, 2, ng).astype(np.float32)
        pc = rng.integers(0, 2, npd).astype(np.float32)
        np.testing.assert_array_equal(S.match_predictions(pc, gc, iou), S.match_predictions_unique_chain(pc, gc, iou))


def test_perfect_detections_give_0995_at_every_threshold():
    rows = np.zeros((1, 5, 6), np.float32)
    gt_box = np.array([[[0.1, 0.1, 0.1, 0.1], [0.3, 0.3, 0.2, 0.2], [0.5, 0.6, 0.1, 0.3], [0.8, 0.2, 0.2, 0.2],
                        [0.7, 0.7, 0.3, 0.1]]], np.float32)
    rows[0, :, :4] = S.gt_boxes_xyxy(gt_box[0], 64, 32)
    rows[0, :, 4] = [0.9, 0.8, 0.7, 0.6, 0.5]
    rows[0, :, 5] = [0, 1, 0, 1, 1]
    m = S.SpecMetrics()
    m.update(rows, [5], np.array([[0, 1, 0, 1, 1]]), gt_box, np.ones((1, 5), bool), 64, 32)
    r = m.compute()
    np.testing.assert_allclose(r["ap"], 0.995, atol=1e-12)
    assert r["metrics/precision(B)"] == 1.0 and r["metrics/recall(B)"] == 1.0
    assert abs(r["metrics/mAP50-95(B)"] - 0.995) < 1e-12 and abs(r["fitness"] - 0.995) < 1e-12


def test_duplicate_detection_is_a_false_positive():
    gt = np.array([[0, 0, 10, 10]], np.float32)
    pred = np.array([[0, 0, 10, 10], [0, 0, 10, 10]], np.float32)
    tp = S.match_predictions(np.zeros(2, np.float32), np.zeros(1, np.float32), S.box_iou(gt, pred))
    assert tp[0].all() and not tp[1].any()


def test_best_gt_already_taken_is_a_false_positive():
    # row 1's best gt is gt 0 (taken by row 0); it also overlaps the free gt 1 at IoU 0.54 -- still an FP
    gt = np.array([[0, 0, 10, 10], [4, 0, 14, 10]], np.float32)
    pred = np.array([[0, 0, 10, 10], [1, 0, 11, 10]], np.float32)
    iou = S.box_iou(gt, pred)
    assert iou[1, 1] >= 0.5 and iou[0, 1] > iou[1, 1]
    tp = S.match_predictions(np.zeros(2, np.float32), np.zeros(2, np.float32), iou)
    np.testing.assert_array_equal(tp, S.match_predictions_unique_chain(np.zeros(2, np.float32), np.zeros(2, np.float32), iou))
    assert tp[0].all() and not tp[1].any()


def test_classes_without_gts_are_ignored_and_classes_without_predictions_score_zero():
    tp, conf, cls = _records([[1] * 10, [0] * 10], [0.9, 0.8], [0, 2])
    alone = S.results_dict(tp[:1], conf[:1], cls[:1], np.array([0]))
    with_extra_pred = S.results_dict(tp, conf, cls, np.array([0]))            # class 2 has a prediction but no gt
    assert with_extra_pred["metrics/mAP50(B)"] == alone["metrics/mAP50(B)"] == pytest.approx(0.995)
    assert list(with_extra_pred["ap_class_index"]) == [0]
    missed = S.results_dict(tp[:1], conf[:1], cls[:1], np.array([0, 1]))       # class 1 has a gt but no prediction
    assert list(missed["ap_class_index"]) == [0, 1] and missed["ap"][1].max() == 0.0
    assert missed["metrics/mAP50(B)"] == pytest.approx(0.995 / 2)


def test_iou_of_exactly_one_half_counts_at_050():
    gt = np.array([[0, 0, 10, 10]], np.float32)
    pred = np.array([[0, 0, 10, 5]], np.float32)
    iou = S.box_iou(gt, pred)
    assert iou[0, 0] == np.float32(0.5)                       # the +1e-7 vanishes next to an area of 100 px^2
    tp = S.match_predictions(np.zeros(1, np.float32), np.zeros(1, np.float32), iou)
    assert tp[0, 0] and not tp[0, 1:].any()


def test_equal_confidences_keep_record_order():
    tp_first = S.results_dict(*_records([[1] * 10, [0] * 10], [0.5, 0.5], [0, 0]), np.array([0, 0]))
    fp_first = S.results_dict(*_records([[0] * 10, [1] * 10], [0.5, 0.5], [0, 0]), np.array([0, 0]))
    # a TP ranked first keeps precision 1 up to recall 0.5; ranked second it does not
    assert tp_first["metrics/mAP50(B)"] > fp_first["metrics/mAP50(B)"]
    decreasing = S.results_dict(*_records([[1] * 10, [0] * 10], [0.5, 0.49], [0, 0]), np.array([0, 0]))
    assert tp_first["metrics/mAP50(B)"] == decreasing["metrics/mAP50(B)"]


def test_hand_computed_two_class_example():
    # class 0: 2 gts, detections TP / FP / TP by falling confidence -> recall .5 .5 1, precision 1 .5 2/3;
    #   the envelope is 1 up to recall .5 (x < .5), 2/3 from .5 to 1 (exclusive), 0 at x = 1
    # class 1: 1 gt, one TP -> 0.995
    tp, conf, cls = _records([[1] * 10, [0] * 10, [1] * 10, [1] * 10], [0.9, 0.8, 0.7, 0.6], [0, 0, 0, 1])
    r = S.results_dict(tp, conf, cls, np.array([0, 0, 1]))
    ap0 = 49 * 0.01 + 0.01 * (1 + 2 / 3) / 2 + 49 * 0.01 * 2 / 3 + 0.01 * (2 / 3) / 2
    np.testing.assert_allclose(r["ap"][0], ap0, atol=1e-12)
    np.testing.assert_allclose(r["ap"][1], 0.995, atol=1e-12)
    assert r["metrics/mAP50(B)"] == pytest.approx((ap0 + 0.995) / 2, abs=1e-12)
    assert r["fitness"] == pytest.approx(0.1 * r["metrics/mAP50(B)"] + 0.9 * r["metrics/mAP50-95(B)"], abs=1e-15)
