"""CPU: host-side validation of raw-logit heads in the decoding entry points and of yb_activate_head.
Every call here is rejected before any CUDA call, so it runs without a GPU (pointers are dummies)."""
import ctypes
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "tf2_yolo_b200", "libyolo_b200.so")
YB_E_NULL, YB_E_PARAM = -1, -3
FAKE = ctypes.c_void_p(1 << 20)        # never dereferenced: the calls must fail on the host


@pytest.fixture(scope="module")
def N():
    if not os.path.exists(LIB):
        import __graft_entry__ as g
        g.build()
    from tf2_yolo_b200 import _native
    return _native


def v4_params(N, from_logits=True, grid=19):
    from tf2_yolo_b200 import engine
    return engine.make_loss_params(4, (grid, grid), 3, 80, anchors=[[0.1, 0.1]] * 3, from_logits=from_logits)


def scales(N, params):
    sc = (N.LossScale * len(params))()
    for i, p in enumerate(params):
        sc[i].y_true = sc[i].y_pred = sc[i].dpred = FAKE.value
        sc[i].n_cells = 2 * p.grid_h * p.grid_w
        sc[i].p = p
    return sc


def test_activate_head_is_declared_and_bound(N):
    header = open(os.path.join(ROOT, "include", "yolo_b200.h")).read()
    assert "int yb_activate_head(const yb_loss_params* p, const float* raw, float* out, int64_t n_cells" in header
    assert "yb_activate_head" in N.SIGNATURES


def test_activate_head_validates_on_the_host(N):
    p = v4_params(N)
    act = N.lib.yb_activate_head
    assert act(None, FAKE, FAKE, 1, None) == YB_E_NULL
    assert act(ctypes.byref(p), None, FAKE, 1, None) == YB_E_NULL
    assert act(ctypes.byref(p), FAKE, None, 1, None) == YB_E_NULL
    q = N.LossParams.from_buffer_copy(p)
    q.version = 2                                        # softmax heads
    assert act(ctypes.byref(q), FAKE, FAKE, 1, None) == YB_E_PARAM
    q = N.LossParams.from_buffer_copy(p)
    q.has_anchors = 0                                    # w, h need the anchors
    assert act(ctypes.byref(q), FAKE, FAKE, 1, None) == YB_E_PARAM
    q = N.LossParams.from_buffer_copy(p)
    q.bbox_num = 0
    assert act(ctypes.byref(q), FAKE, FAKE, 1, None) == -2     # YB_E_SHAPE
    assert act(ctypes.byref(p), ctypes.c_void_p(FAKE.value + 2), FAKE, 1, None) == -5    # YB_E_ALIGN
    assert act(ctypes.byref(p), FAKE, FAKE, 0, None) == 0      # nothing to do: no launch


def test_decode_fused_rejects_raw_heads(N):
    """yb_loss_decode_fused re-reads the head tensors to emit rows: raw heads are refused up front."""
    for ps in ([v4_params(N)] * 3, [v4_params(N, False), v4_params(N, True)]):
        sc = scales(N, ps)
        rc = N.lib.yb_loss_decode_fused(sc, len(ps), FAKE, None, 0.5, None, 0, FAKE, FAKE, 1 << 20, FAKE, 1 << 20, None)
        assert rc == YB_E_PARAM


def test_step_rejects_softmax_and_mixed_raw_heads(N):
    from tf2_yolo_b200 import engine
    v2 = engine.make_loss_params(2, (13, 13), 5, 20, anchors=[[1.0, 1.0]] * 5)
    v2.from_logits = 1
    mixed = [v4_params(N, True), v4_params(N, False)]
    for ps in ([v2], mixed):
        sc = scales(N, ps)
        for fn in (N.lib.yb_loss_decode_nms_fused, N.lib.yb_loss_decode_nms_fused_clean):
            rc = fn(sc, len(ps), FAKE, None, 0.5, 0.45, 2, 1024, FAKE, 1024, FAKE, None, FAKE, 1 << 20, FAKE, 1 << 20,
                    None)
            assert rc == YB_E_PARAM
    with pytest.raises(ValueError):
        engine.make_loss_params(2, (13, 13), 5, 20, anchors=[[1.0, 1.0]] * 5, from_logits=True)
