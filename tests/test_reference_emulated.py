"""The oracle against outputs of the reference's OWN source files (imported unmodified from /root/reference and run
under the NumPy stand-in for TensorFlow, tests/golden/make_golden_emulated.py -> tests/golden/ref_emulated.npz).

Integer results (NMS indices, class ids, masks, one-hot rows) must be identical; floating-point results agree to a few
ulp (the stand-in uses libm exp/log/atan/pow, the oracle the deterministic detmath).  This pins the oracle's
restatement of the reference's control flow, operation order, broadcasting and index conventions."""
import os

import numpy as np
import pytest

from oracle import effdet as oe
from oracle import yolo as oy

F = np.float32
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_emulated.npz"))


def close(a, b, rtol=3e-6, atol=3e-6):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    np.testing.assert_allclose(np.nan_to_num(a, nan=0.0), np.nan_to_num(b, nan=0.0), rtol=rtol, atol=atol)


def test_yolo_iou_family():
    for t in ("iou", "diou", "ciou"):
        close(oy.get_iou(G["iou_b1"][:, None, :], G["iou_b2"][None, :, :], t), G["iou_" + t])


def test_yolo_nms_indices_identical():
    b, s, c = G["nms_boxes"], G["nms_scores"], G["nms_classes"]
    for t in ("iou", "diou", "ciou"):
        assert oy.get_iou_nms(b, s, 500, 0.5, t).tolist() == G["nms_plain_" + t].tolist()
        assert oy.get_iou_nms_by_classes(b, s, c, 500, 0.45, t).tolist() == G["nms_class_" + t].tolist()
        assert 20 < len(G["nms_plain_" + t]) < 300          # suppression really happened
    assert oy.get_iou_nms(b, s, 25, 0.5, "iou").tolist() == G["nms_plain_cap"].tolist() and len(G["nms_plain_cap"]) == 25


def test_yolo_get_boxes_and_get_nms_boxes():
    anc, C, image = G["y_anchors"], 6, 96
    got = oy.get_boxes(G["y_heads1"].reshape(1, 6, 6, 3, 5 + C), anc[1] / F(image), C)
    close(got[0], G["y_getboxes_boxes"]); close(got[1], G["y_getboxes_conf"]); close(got[2], G["y_getboxes_classes"])
    r = oy.get_nms_boxes(G["y_heads0"], G["y_heads1"], G["y_heads2"], anc, (image, image), C, 0.5, 0.3, 0.5, "diou")
    assert r[1].tolist() == G["y_nms_classes_id"].tolist() and len(r[1]) > 10
    close(r[0], G["y_nms_boxes"]); close(r[2], G["y_nms_scores"]); close(r[3], G["y_nms_classes"]); close(r[4], G["y_nms_confidence"])


def test_yolo_losses():
    y_true = [G["yl_true%d" % l] for l in range(3)]
    y_pred = [G["yl_pred%d" % l] for l in range(3)]
    for t in ("iou", "diou", "ciou"):
        want = float(G["yl_loss_" + t])
        got, _, ign = oy.get_loss(y_true, y_pred, (96, 96), G["y_anchors"], 0.5, t, return_ignore=True)
        assert abs(float(got) - want) <= 2e-5 * abs(want), t
        assert 0 < int((ign == 0).sum())                     # the ignore mask had zeros: the metric mattered
    want = float(G["yl_yolov4loss"])
    got = float(oy.yolov4_loss(G["yl_anchors9"], 6, y_true, y_pred))
    assert abs(got - want) <= 2e-5 * abs(want)


def test_effdet_iou_family_and_nms():
    for t in ("iou", "giou", "diou", "ciou"):
        close(oe.get_iou(G["e_b1"][:, None, :], G["e_b2"][None, :, :], t), G["e_iou_" + t])
        assert oe.get_nms(G["e_nms_boxes"], G["e_nms_scores"], 200, 0.5, 0.0001, t).tolist() == G["e_nms_" + t].tolist()
        assert 20 < len(G["e_nms_" + t]) <= 200
    assert oe.get_nms(G["e_nms_boxes"], G["e_nms_scores"], 7, 0.5, float("-inf"), "diou").tolist() == G["e_nms_cap"].tolist()


def test_effdet_anchors_targets_decode_postprocess():
    a = oe.Anchors(3, 5, (64, 96), 2, [(1.0, 1.0), (1.4, 0.7)], 3.0)
    L = len(a.boxes)
    for l in range(L):
        assert np.array_equal(a.boxes[l], G["ea_boxes%d" % l])          # anchors: no transcendental, bit-exact
    tb, tc, tm = a.generate_targets(G["ea_gt_boxes"], G["ea_gt_classes"], 5, 0.5)
    pos = 0
    for l in range(L):
        close(tb[l], G["ea_tb%d" % l])
        assert np.array_equal(tc[l], G["ea_tc%d" % l]) and np.array_equal(tm[l], G["ea_tm%d" % l])
        pos += int(tm[l].sum())
    assert pos > 0
    rel = [G["ea_rel%d" % l] for l in range(L)]
    cls = [G["ea_cls%d" % l] for l in range(L)]
    dec = a.convert_outputs_boxes(rel)
    for l in range(L):
        close(dec[l], G["ea_dec%d" % l], rtol=3e-6, atol=3e-5)
    for b in range(2):
        bx, ci, sc = a.convert_outputs_one(b, dec, cls)
        assert ci.tolist() == G["ea_one%d_ids" % b].tolist() and len(ci) > 0
        close(bx, G["ea_one%d_boxes" % b], rtol=3e-6, atol=3e-5); close(sc, G["ea_one%d_scores" % b])


def test_focal_and_box_loss():
    close(oe.focal_loss_elements(3.0, G["fl_true"], G["fl_pred"]), G["fl_elem"], rtol=1e-5, atol=1e-7)
    assert abs(float(oe.focal_loss(3.0, G["fl_true"], G["fl_pred"])) - float(G["fl_mean"])) <= 1e-5 * abs(float(G["fl_mean"]))
    assert abs(float(oe.box_loss(7.0, G["bl_true"], G["bl_pred"])) - float(G["bl_loss"])) <= 1e-5 * abs(float(G["bl_loss"]))


def test_get_targets_identical():
    used = 0
    for tag in ("px", "norm"):
        got = oy.get_targets(G["gt_%s_boxes" % tag], G["gt_%s_classes" % tag], G["gt_%s_anchors" % tag], (416, 416), 20)
        for l in range(3):
            want = G["gt_%s_t%d" % (tag, l)]
            assert got[l].dtype == np.float32 and np.array_equal(got[l], want), (tag, l)   # no transcendental: bit-exact
            used += int(want[..., 4].sum() > 0)
        assert G["gt_%s_t2" % tag][..., 4].sum() < 30                                     # the triple collision was zeroed
    assert used >= 4   # pixel anchors put everything on one layer (quirk Q8); normalised anchors use all three


def test_effdet_get_loss_class_focal_loss_and_ground_truth_rows():
    tb = [G["gl_tb%d" % l] for l in range(3)]; tc = [G["gl_tc%d" % l] for l in range(3)]; tm = [G["gl_tm%d" % l] for l in range(3)]
    pb = [G["gl_pb%d" % l] for l in range(3)]; pc = [G["gl_pc%d" % l] for l in range(3)]
    want = float(G["gl_loss"])                                   # EfficientDetNetTrain._get_loss with the L2 term at 0
    assert abs(float(oe.get_loss(tb, tc, tm, pb, pc)) - want) <= 1e-5 * abs(want) and want > 0
    tm2 = [m.copy() for m in tm]; tm2[2][:] = False
    want = float(G["cfl_loss"])
    assert abs(float(oe.class_focal_loss(tc, pc, tm2)) - want) <= 1e-5 * abs(want)
    for l in range(3):                                            # yolo_v4/model.py GetGroudTruth: no transcendental
        got = oy.get_ground_truth(G["yl_true%d" % l])
        assert got.shape == G["ggt%d" % l].shape and np.array_equal(got, G["ggt%d" % l])


def test_reference_test_anchors_main():
    """ai_models/tests/test_anchors.py main(), run unmodified: generate_targets -> convert_outputs_boxes -> convert_outputs_one
    round-trips the two boxes; the oracle does the same."""
    a = oe.Anchors(0, 0, (10, 10), 3, [(1.0, 1.0)], 3.0)
    boxes, classes = np.array([[3, 3, 6, 6], [5, 5, 9, 9]], F), np.array([1, 2])
    tb, tc, tm = a.generate_targets(boxes, classes, 3, iou_threshold=0.5)
    dec = a.convert_outputs_boxes([t[None] for t in tb])
    bx, ci, sc = a.convert_outputs_one(0, dec, [t[None] for t in tc])
    assert ci.tolist() == G["rt_convert_classes_id"].tolist() == [1, 2]
    close(bx, G["rt_convert_boxes"], atol=2e-5); close(sc, G["rt_convert_scores"])


# the AIServer directory of a checkout of the original tensorflow2-machine-vision project, which this repository does not
# contain; the two relations these unit tests assert are also checked on the oracle by tests/test_oracle_pins.py
REF = os.environ.get("TFMV_REFERENCE_DIR", "")


@pytest.mark.skipif(not os.path.isdir(REF), reason="set TFMV_REFERENCE_DIR to the original project's AIServer directory")
@pytest.mark.parametrize("name", ["grid_test", "loss_test"])
def test_reference_unit_tests_pass_under_the_stand_in(name):
    """The reference's only two unit tests (yolo_v3/unit_test/grid_test.py: grid layout equality; loss_test.py:
    GetLoss-copy == Yolov4Loss, exact), executed unmodified with the NumPy stand-in as `tensorflow`: they pass, which
    checks the stand-in itself against the reference's own expectations."""
    import subprocess
    import sys
    env = dict(os.environ)
    env["PYTHONPATH"] = os.path.join(os.path.dirname(__file__), "golden", "fake_tf") + os.pathsep + REF
    r = subprocess.run([sys.executable, os.path.join(REF, "ai_api/ai_models/yolo_v3/unit_test", name + ".py")], cwd=REF, env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0 and "OK" in r.stdout.splitlines()[-1], r.stdout[-2000:]


def test_baseline_config1_through_the_reference_get_nms_boxes():
    """BASELINE config 1 (YOLOv3 416x416, 80 classes, N(0,1) heads, cap 500): the reference's own GetNMSBoxes vs the oracle."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import emulated_inputs as ei
    heads = ei.yolo_416_heads()
    for t, thr in (("iou", 0.5), ("diou", 0.45)):
        r = oy.get_nms_boxes(heads[0], heads[1], heads[2], ei.COCO_ANCHORS, (416, 416), 80, 0.5, 0.3, thr, t)
        assert len(G["c1_%s_ids" % t]) == 500                                  # the cap was reached
        assert r[1].tolist() == G["c1_%s_ids" % t].tolist()
        close(r[0], G["c1_%s_boxes" % t]); close(r[2], G["c1_%s_scores" % t]); close(r[4], G["c1_%s_conf" % t])
        np.testing.assert_allclose(r[3].sum(-1, dtype=np.float64), G["c1_%s_classes_rowsum" % t], rtol=1e-5)


def test_baseline_config3_image_through_the_reference_anchors():
    """One EfficientDet-D0 image (49 104 anchors, 81 classes, cap 200) through the reference's own Anchors code vs the oracle."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import emulated_inputs as ei
    a = oe.Anchors(**ei.D0)
    np.testing.assert_array_equal(np.array([b.astype(np.float64).sum() for b in a.boxes]), G["c3_anchor_checksum"])
    rel, cls = ei.effdet_d0_heads([b.shape[:3] for b in a.boxes])
    dec = a.convert_outputs_boxes(rel)
    bx, ci, sc = a.convert_outputs_one(0, dec, cls)
    assert len(G["c3_ids"]) == 200 and ci.tolist() == G["c3_ids"].tolist()
    close(bx, G["c3_boxes"], rtol=3e-6, atol=1e-4); close(sc, G["c3_scores"])


def test_ciou_v_custom_gradient_matches_reference_source():
    """efficientnet/utils/iou.py:5-24: _get_v and the hand-written gradient its tf.custom_gradient returns, evaluated by
    the reference's own code under the stand-in.  atan(w1/h1) - atan(w2/h2) cancels, so the comparison is absolute on the
    scale of the operands (libm vs detmath atan differ by an ulp of a value near 1)."""
    from oracle import effdet as oe
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_emulated.npz"))
    v, gdh, gdw = oe.get_v_grad(g["cv_h1"], g["cv_w1"], g["cv_h2"], g["cv_w2"], g["cv_dv"])
    np.testing.assert_allclose(v, g["cv_v"], rtol=1e-5, atol=2e-7)
    scale_h = np.abs(g["cv_dv"]) * 8 * g["cv_w2"] / np.pi ** 2
    scale_w = np.abs(g["cv_dv"]) * 8 * g["cv_h2"] / np.pi ** 2
    assert np.all(np.abs(gdh - g["cv_gdh"]) <= 4e-7 * scale_h + 1e-12)
    assert np.all(np.abs(gdw - g["cv_gdw"]) <= 4e-7 * scale_w + 1e-12)
    # sign convention and the divide_no_nan branches (h2 == 0 -> atan(0)); the gradient is NOT the true derivative: no 1/(w^2+h^2)
    assert np.sign(gdh[0]) == -np.sign(gdw[0]) or gdh[0] == 0
