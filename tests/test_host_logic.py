"""CPU: host mirrors - parameter packing, API surface, error behaviour, no silent CPU path."""
import inspect

import numpy as np
import pytest
import torch

import tf2_yolo_b200
from tf2_yolo_b200 import dist as ydist
from tf2_yolo_b200 import engine, synth
from tf2_yolo_b200._native import YoloB200Error
from tf2_yolo_b200.utils import kmeans as km
from tf2_yolo_b200.utils import measurement as meas
from tf2_yolo_b200.utils import tools

REF_SIGNATURES = {  # keyword lists of the reference (SURVEY 8b), kept verbatim
    ("yolov4", "wrap_yolo_loss"): ["grid_shape", "bbox_num", "class_num", "anchors", "binary_weight", "loss_weight",
                                   "wh_reg_weight", "ignore_thresh", "truth_thresh", "label_smooth", "focal_loss_gamma"],
    ("yolov3", "wrap_yolo_loss"): ["grid_shape", "bbox_num", "class_num", "anchors", "binary_weight", "loss_weight",
                                   "ignore_thresh", "use_focal_loss", "focal_loss_gamma", "use_scale"],
    ("yolov2", "wrap_yolo_loss"): ["grid_shape", "bbox_num", "class_num", "anchors", "binary_weight", "loss_weight",
                                   "ignore_thresh"],
    ("yolov1_5", "wrap_yolo_loss"): ["grid_shape", "bbox_num", "class_num", "binary_weight", "loss_weight"],
}


def test_loss_signatures_match_the_reference():
    import importlib
    for (pkg, fn), names in REF_SIGNATURES.items():
        mod = importlib.import_module(f"tf2_yolo_b200.{pkg}.losses")
        assert list(inspect.signature(getattr(mod, fn)).parameters) == names
        assert hasattr(mod, "cal_iou")
    assert list(inspect.signature(tools.decode).parameters) == ["label_datas", "class_num", "threshold", "version"]
    assert list(inspect.signature(tools.nms).parameters) == ["xywhcp", "class_num", "nms_threshold", "iou_mode"]
    assert list(inspect.signature(tools.cal_iou).parameters) == ["xywh_true", "xywh_pred", "mode"]
    assert list(inspect.signature(km.kmeans).parameters)[:6] == ["data", "n_cluster", "dist_func", "stop_dist",
                                                                 "max_iternum", "verbose"]
    assert list(inspect.signature(meas.PRfunc.__init__).parameters)[1:12] == [
        "y_trues", "y_preds", "class_names", "conf_threshold", "nms_mode", "nms_threshold", "nms_sigma",
        "iou_threshold", "precision_mode", "max_per_img", "version"]


def test_loss_param_packing():
    from tf2_yolo_b200.yolov4.losses import wrap_yolo_loss
    f = wrap_yolo_loss((19, 38), 3, 80, anchors=[[.1, .2], [.3, .4], [.5, .6]], binary_weight=np.array([0.25]),
                       loss_weight=[1, 5, 1], truth_thresh=0.7, label_smooth=0.1, focal_loss_gamma=1.5)
    p = f.params
    assert (p.version, p.grid_h, p.grid_w, p.bbox_num, p.class_num, p.has_anchors) == (4, 19, 38, 3, 80, 1)
    assert np.allclose(list(p.anchors)[:6], [.1, .2, .3, .4, .5, .6])
    assert p.binary_weight == 0.25 and f.out_shape == (1,)
    assert list(p.loss_weight) == [1, 5, 1, 0]
    assert abs(p.truth_thresh - 0.7) < 1e-6 and abs(p.label_smooth - 0.1) < 1e-6 and p.focal_gamma == 1.5
    from tf2_yolo_b200.yolov3.losses import wrap_yolo_loss as w3
    p3 = w3((13, 13), 3, 80, use_focal_loss=True, use_scale=False).params
    assert (p3.version, p3.use_focal, p3.use_scale, p3.has_anchors) == (3, 1, 0, 0)
    with pytest.raises(ValueError):
        wrap_yolo_loss((19, 19), 3, 80, anchors=[[.1, .2]])
    with pytest.raises(ValueError):
        wrap_yolo_loss((19, 19), 40, 80)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks behaviour without a GPU")
def test_no_cpu_fallback_anywhere():
    from tf2_yolo_b200.yolov4.losses import wrap_yolo_loss
    f = wrap_yolo_loss((4, 4), 3, 2)
    yt, yp = np.zeros((1, 4, 4, 7), np.float32), np.full((1, 4, 4, 21), 0.5, np.float32)
    with pytest.raises(YoloB200Error):
        f(yt, yp)
    with pytest.raises(YoloB200Error):
        engine.loss_fwd_bwd([f.params], [torch.from_numpy(yt)], [torch.from_numpy(yp)])
    with pytest.raises(YoloB200Error):
        tools.decode(yp[0], class_num=2, version=3)
    with pytest.raises(YoloB200Error):
        tools.nms(np.zeros((3, 7)), 2)
    with pytest.raises(YoloB200Error):
        tools.soft_nms(np.zeros((3, 7)), 2)
    with pytest.raises(YoloB200Error):
        km.kmeans(np.random.rand(10, 2), 2, km.iou_dist, 1e-3, verbose=False)
    with pytest.raises(YoloB200Error):
        meas.PRfunc(np.zeros((1, 4, 4, 7)), yp, class_names=["a", "b"])


def test_error_behaviour_matches_the_reference():
    with pytest.raises(ValueError, match="Invalid version"):
        tools.decode(np.zeros((2, 2, 14), np.float32), class_num=2, version=7)
    with pytest.raises(IndexError):
        tools.soft_nms(np.zeros(0))
    with pytest.raises(YoloB200Error):
        km.kmeans(np.random.rand(10, 2), 2, lambda a, b: a, 1e-3)     # arbitrary Python distance
    centre, data = np.array([[[0.3, 0.5]]]), np.random.default_rng(0).uniform(0.1, 1.0, (1, 1 << 17, 2))
    if torch.cuda.is_available():      # a data-sized call runs on the device and gives the host formula
        ca, da = 0.3 * 0.5, data[..., 0] * data[..., 1]
        assert np.allclose(km.iou_dist(centre, data), 1 - np.minimum(ca, da) / np.maximum(ca, da), rtol=0, atol=1e-12)
    else:                              # without a device it is refused, not run on the host
        with pytest.raises(YoloB200Error):
            km.iou_dist(centre, data)
    c = np.array([[[0.2, 0.4]], [[0.5, 0.5]]])
    assert np.allclose(km.iou_dist(c, c), 0) and np.allclose(km.euclidean_dist(c, c), 0)
    assert km.iou(c[0], c[1])[0] == (0.2 * 0.4) / (0.5 * 0.5)


def test_install_rebinds_reference_modules():
    import types
    fake_tools = types.ModuleType("utils.tools")
    fake_tools.decode = fake_tools.nms = fake_tools.cal_iou = lambda *a, **k: "reference"
    fake_meas = types.ModuleType("utils.measurement")
    fake_meas.decode = fake_meas.PRfunc = fake_meas.nms = lambda *a, **k: "reference"
    fake_pkg = types.ModuleType("yolov4")
    fake_pkg.wrap_yolo_loss = lambda *a, **k: "reference"
    fake_losses = types.ModuleType("yolov4.losses")
    fake_losses.wrap_yolo_loss = fake_losses.cal_iou = lambda *a, **k: "reference"
    done = tf2_yolo_b200.install({"utils.tools": fake_tools, "utils.measurement": fake_meas, "yolov4": fake_pkg,
                                  "yolov4.losses": fake_losses})
    assert fake_tools.decode is tools.decode and fake_tools.nms is tools.nms
    assert fake_meas.PRfunc is meas.PRfunc and fake_meas.decode is tools.decode
    from tf2_yolo_b200.yolov4.losses import wrap_yolo_loss
    assert fake_pkg.wrap_yolo_loss is wrap_yolo_loss and fake_losses.wrap_yolo_loss is wrap_yolo_loss
    assert "utils.tools.decode" in done and "yolov4.wrap_yolo_loss" in done
    # the in-training metric wrappers follow the same rule (facade global + metrics module)
    fake_pkg3 = types.ModuleType("yolov3")
    fake_metrics3 = types.ModuleType("yolov3.metrics")
    for m in (fake_pkg3, fake_metrics3):
        m.wrap_obj_acc = m.wrap_mean_iou = m.wrap_class_acc = m.wrap_recall = lambda *a, **k: "reference"
    done = tf2_yolo_b200.install({"yolov3": fake_pkg3, "yolov3.metrics": fake_metrics3})
    from tf2_yolo_b200.yolov3.metrics import wrap_recall
    assert fake_pkg3.wrap_recall is wrap_recall and fake_metrics3.wrap_recall is wrap_recall
    assert "yolov3.metrics.wrap_obj_acc" in done and "yolov3.wrap_class_acc" in done


def test_synth_shapes_and_invariants():
    cfg = synth.make_config("v4-608", batch=2, seed=3)
    assert [a.shape for a in cfg["y_preds"]] == [(2, 19, 19, 255), (2, 38, 38, 255), (2, 76, 76, 255)]
    assert [a.shape for a in cfg["y_trues"]] == [(2, 19, 19, 85), (2, 38, 38, 85), (2, 76, 76, 85)]
    for yt in cfg["y_trues"]:
        obj = yt[..., 4]
        assert set(np.unique(obj)) <= {0.0, 1.0} and obj.sum() >= 2
        assert np.all(yt[obj == 1][:, 5:].sum(axis=1) == 1)
    for yp in cfg["y_preds"]:
        assert yp.dtype == np.float32 and yp.min() > 0 and yp.max() <= 1
    again = synth.make_config("v4-608", batch=2, seed=3)
    assert all(np.array_equal(a, b) for a, b in zip(cfg["y_preds"], again["y_preds"]))
    assert ydist.shard_range(10, 3, 4) == (8, 10) and ydist.shard_range(7, 0, 8) == (0, 1)
    assert sum(b - a for a, b in (ydist.shard_range(1001, r, 8) for r in range(8))) == 1001


def test_prfunc_call_fast_path_equals_the_reference_expression():
    """PRfunc.__call__: binary search + suffix maxima == `(recalls > r).sum()` / `precisions[-k:].max()`
    (utils/measurement.py:333-337) on sorted recalls; unsorted or NaN inputs take the literal form."""
    rng = np.random.default_rng(4)
    pr = meas.PRfunc.__new__(meas.PRfunc)
    pr.class_num = 3
    tp = np.cumsum(rng.integers(0, 2, 500))
    rec = np.append(tp / 200.0, tp[-1] / 200.0)                  # non-decreasing + the sentinel
    prec = np.append(tp / np.arange(1, 501), 0)
    pr.recalls = [rec, rng.permutation(rec), np.array([0.5])]
    pr.precisions = [prec, prec, np.array([0.0])]
    for c in range(3):
        for r in [0, 0.14, 0.29, 0.43, 0.57, 0.71, 1, -1.0, 2.0, float(rec[10]), float(rec[-1]), 0.5]:
            k = (pr.recalls[c] > r).sum()
            want = 0 if k == 0 else pr.precisions[c][-k:].max()
            got = pr(r, c)
            assert got == want and type(got) is type(want), (c, r)
    assert pr._suffix_max[1] is None and pr._suffix_max[0] is not None
