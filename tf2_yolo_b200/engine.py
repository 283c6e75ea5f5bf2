"""Device-side entry points: thin wrappers that hand torch CUDA tensors' device
pointers (torch is only the tensor carrier / allocator here) and the current
CUDA stream to the C ABI in libyolo_b200.so.  Everything is asynchronous on the
current stream; nothing here computes on the host and nothing falls back to
PyTorch ops.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _native as N

_I64 = torch.int64
_F64 = torch.float64


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def require_cuda(*tensors):
    for t in tensors:
        if t is None:
            continue
        if not torch.is_tensor(t) or not t.is_cuda:
            raise N.YoloB200Error("tf2_yolo_b200 ops need CUDA tensors (no CPU fallback)")
        if not t.is_contiguous():
            raise N.YoloB200Error("tf2_yolo_b200 ops need contiguous tensors")


class _WorkspacePool:
    """Grow-only scratch buffers, one per (device, stream, tag).  Host-side
    convenience only: the C library itself owns no memory."""

    def __init__(self):
        self._bufs = {}

    def get(self, tag, nbytes, device):
        key = (device.index, torch.cuda.current_stream(device).cuda_stream, tag)
        nbytes = int(nbytes)
        buf = self._bufs.get(key)
        # usable capacity = what is left after aligning the base to 256 bytes
        if buf is None or buf.numel() - ((-buf.data_ptr()) % 256) < nbytes:
            buf = torch.empty(max(nbytes, 4096) + 256, dtype=torch.uint8, device=device)
            self._bufs[key] = buf
        off = (-buf.data_ptr()) % 256
        out = buf[off:off + nbytes]
        assert out.numel() == nbytes
        return out

    def clear(self):
        self._bufs.clear()


workspaces = _WorkspacePool()


# --------------------------------------------------------------------------
# losses
# --------------------------------------------------------------------------
def make_loss_params(version, grid_shape, bbox_num, class_num, anchors=None, binary_weight=1.0,
                     loss_weight=(1, 1, 1, 1), wh_reg_weight=0.01, ignore_thresh=0.6,
                     truth_thresh=1.0, label_smooth=0.0, focal_loss_gamma=2.0,
                     use_focal_loss=False, use_scale=True, from_logits=False):
    if version not in (1, 2, 3, 4):
        raise ValueError(f"Invalid version: {version}")
    if bbox_num > N.YB_MAX_BOXES:
        raise ValueError(f"bbox_num {bbox_num} exceeds {N.YB_MAX_BOXES}")
    p = N.LossParams()
    p.version = version
    p.grid_h, p.grid_w = int(grid_shape[0]), int(grid_shape[1])
    p.bbox_num, p.class_num = int(bbox_num), int(class_num)
    if anchors is not None and version != 1:
        a = np.asarray(anchors, dtype=np.float32).reshape(-1)
        if a.size != 2 * bbox_num:
            raise ValueError("anchors must hold bbox_num (w, h) pairs")
        p.has_anchors = 1
        for i, v in enumerate(a):
            p.anchors[i] = float(v)
    else:
        p.has_anchors = 0
    p.binary_weight = float(np.asarray(binary_weight, dtype=np.float64).reshape(-1)[0])
    lw = list(loss_weight) + [0.0] * 4
    for i in range(4):
        p.loss_weight[i] = float(lw[i])
    p.wh_reg_weight = float(wh_reg_weight)
    p.ignore_thresh = float(ignore_thresh)
    p.truth_thresh = float(truth_thresh)
    p.label_smooth = float(label_smooth)
    p.focal_gamma = float(focal_loss_gamma)
    p.use_focal = int(bool(use_focal_loss))
    p.use_scale = int(bool(use_scale))
    if from_logits and version not in (3, 4):
        raise ValueError("from_logits is available for the v3/v4 heads (sigmoid scores); v1/v2 end in a softmax")
    p.from_logits = int(bool(from_logits))
    p.inv_batch = 1.0
    return p


def floats_per_cell(p):
    """Floats of one y_pred cell: v1 heads share one row of class scores between the boxes of a cell."""
    return (5 * p.bbox_num + p.class_num) if p.version == 1 else p.bbox_num * (5 + p.class_num)


def bind_loss_scales(params, y_trues, y_preds, global_batch=None, dpreds=None, want_grad=True, same_images=True,
                     images=None):
    """The yb_loss_scale array of one launch over the scales in ``params``.

    y_trues[i]: (N, gh, gw, 5+C) fp32 CUDA; y_preds[i]: (N, gh, gw, info) fp32 CUDA.  ``same_images``:
    every scale holds the N = y_preds[0].shape[0] images the decoding entry points need; without it each
    scale's N follows from its own size.  ``images=(a, b)`` binds images a..b-1 of every tensor.
    ``global_batch`` = divisor of reduce_mean(axis=0) (defaults to the scale's N).  The gradient goes to
    ``dpreds`` (fresh tensors when None).  Returns (scales, dpreds list or None, number of images bound).
    """
    n = len(params)
    if not (1 <= n <= N.YB_MAX_SCALES) or len(y_trues) != n or len(y_preds) != n:
        raise ValueError("between 1 and 4 scales, one y_true / y_pred each")
    require_cuda(*y_trues, *y_preds)
    n_img = y_preds[0].shape[0]
    a, b = images if images is not None else (0, None)
    scales = (N.LossScale * n)()
    outs = []
    for i, (p, yt, yp) in enumerate(zip(params, y_trues, y_preds)):
        if yt.dtype != torch.float32 or yp.dtype != torch.float32:
            raise N.YoloB200Error("loss tensors must be float32 (Keras casts y_true to y_pred.dtype)")
        cells_per_img, pcf, tcf = p.grid_h * p.grid_w, floats_per_cell(p), 5 + p.class_num
        if yp.numel() % (cells_per_img * pcf) != 0:
            raise ValueError(f"y_pred with {yp.numel()} elements does not reshape to (-1,{p.grid_h},{p.grid_w},{pcf})")
        m = yp.numel() // (cells_per_img * pcf)
        if yt.numel() != m * cells_per_img * tcf:
            raise ValueError(f"y_true with {yt.numel()} elements does not reshape to ({m},{p.grid_h},{p.grid_w},{tcf})")
        if same_images and m != n_img:
            raise ValueError("every scale must hold the same images")
        q = N.LossParams.from_buffer_copy(p)
        q.inv_batch = 1.0 / float(global_batch if global_batch is not None else max(m, 1))
        d = None
        if want_grad:
            d = dpreds[i] if dpreds is not None else torch.empty_like(yp)
            require_cuda(d)
        outs.append(d)
        scales[i].y_true = yt.data_ptr() + 4 * a * cells_per_img * tcf
        scales[i].y_pred = yp.data_ptr() + 4 * a * cells_per_img * pcf
        scales[i].dpred = d.data_ptr() + 4 * a * cells_per_img * pcf if d is not None else None
        scales[i].n_cells = ((b if b is not None else m) - a) * cells_per_img
        scales[i].p = q
    return scales, (outs if want_grad else None), (b - a if images is not None else n_img)


def loss_decode_params(params, threshold):
    """DecodeParams of the float32 heads ``params`` describe: the decode that the loss entry points
    with a counting pass derive from their scales (yb_loss_decode_fused, yb_loss_decode_nms_fused)."""
    p = N.DecodeParams()
    p.version, p.class_num, p.n_scales, p.is_f64 = params[0].version, params[0].class_num, len(params), 0
    for i, q in enumerate(params):
        p.grid_h[i], p.grid_w[i], p.bbox_num[i] = q.grid_h, q.grid_w, q.bbox_num
    p.threshold = float(threshold)
    return p


def loss_fwd_bwd(params, y_trues, y_preds, global_batch=None, want_grad=True, want_terms=False,
                 dpreds=None, want_metrics=False, recall_iou_threshold=0.5):
    """One fused launch over the scales in ``params``.

    y_trues[i]: (N, gh, gw, 5+C) fp32 CUDA; y_preds[i]: (N, gh, gw, B*(5+C)) fp32 CUDA.
    Returns (loss [n_scales] fp32 CUDA, dpreds list or None, terms [n_scales, 8] f64 or None).
    ``global_batch`` = divisor of reduce_mean(axis=0) (defaults to the local N).
    """
    n = len(params)
    scales, outs, _ = bind_loss_scales(params, y_trues, y_preds, global_batch, dpreds, want_grad, same_images=False)
    dev = y_preds[0].device
    with torch.cuda.device(dev):
        loss = torch.empty(n, dtype=torch.float32, device=dev)
        terms = torch.empty((n, N.YB_LOSS_TERMS), dtype=_F64, device=dev) if want_terms else None
        ws_bytes = N.lib.yb_loss_workspace_bytes(n)
        ws = workspaces.get("loss", ws_bytes, dev)
        if want_metrics:
            metrics = torch.empty((n, N.YB_LOSS_METRICS), dtype=_F64, device=dev)
            N.check(N.lib.yb_loss_fwd_bwd_metrics(scales, n, _ptr(loss), _ptr(terms), _ptr(metrics),
                                                  float(recall_iou_threshold), _ptr(ws), ws_bytes, _stream()),
                    "yb_loss_fwd_bwd_metrics")
            return loss, outs, terms, metrics
        N.check(N.lib.yb_loss_fwd_bwd(scales, n, _ptr(loss), _ptr(terms), _ptr(ws), ws_bytes, _stream()),
                "yb_loss_fwd_bwd")
    return loss, outs, terms


def loss_decode_fused(params, y_trues, y_preds, threshold=0.5, global_batch=None, dpreds=None,
                      capacity=None, rows=None, want_terms=False, split_hook=None):
    """Loss forward+gradient and decode of the same head outputs, y_pred read from HBM once
    (yb_loss_decode_fused).  Returns (loss [n], dpreds, terms, rows (capacity,7) f64, row_offsets).
    Activated heads only: the rows are read back from y_pred (raw heads: loss_decode_nms_fused, or
    activate_head first)."""
    n = len(params)
    scales, outs, n_img = bind_loss_scales(params, y_trues, y_preds, global_batch, dpreds)
    dev = y_preds[0].device
    dparams = loss_decode_params(params, threshold)
    if rows is not None:
        capacity = rows.shape[0]
    if capacity is None:
        capacity = max(1024, 512 * n_img)
    with torch.cuda.device(dev):
        if rows is None:
            rows = torch.empty((capacity, 7), dtype=_F64, device=dev)
        offsets = torch.empty(n_img + 1, dtype=_I64, device=dev)
        loss = torch.empty(n, dtype=torch.float32, device=dev)
        terms = torch.empty((n, N.YB_LOSS_TERMS), dtype=_F64, device=dev) if want_terms else None
        lws_bytes = N.lib.yb_loss_workspace_bytes(n)
        lws = workspaces.get("loss", lws_bytes, dev)
        dws_bytes = N.lib.yb_decode_workspace_bytes(C.byref(dparams), n_img)
        dws = workspaces.get("decode", dws_bytes, dev)
        if split_hook is None:
            N.check(N.lib.yb_loss_decode_fused(scales, n, _ptr(loss), _ptr(terms), float(threshold), _ptr(rows),
                                               capacity, _ptr(offsets), _ptr(lws), lws_bytes, _ptr(dws), dws_bytes,
                                               _stream()), "yb_loss_decode_fused")
        else:   # two calls so that a timer can bracket the fused kernel alone (bench.py roofline)
            N.check(N.lib.yb_loss_decode_fused(scales, n, _ptr(loss), _ptr(terms), float(threshold), None, 0, None,
                                               _ptr(lws), lws_bytes, _ptr(dws), dws_bytes, _stream()),
                    "yb_loss_decode_fused(count)")
            split_hook()
            ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in y_preds])
            N.check(N.lib.yb_decode_finish(ptrs, n_img, C.byref(dparams), _ptr(rows), capacity, _ptr(offsets),
                                           _ptr(dws), dws_bytes, _stream()), "yb_decode_finish")
    return loss, outs, terms, rows, offsets


def activate_head(params, raw, out=None):
    """The head transform of one v3/v4 scale on the device (yb_activate_head): sigmoid on x, y,
    objectness and class scores, anchor * exp on w, h of the raw head outputs ``raw`` (N, gh, gw,
    B*(5+C)) fp32 CUDA, with the anchors of ``params`` (the scale's LossParams).  The same float32
    arithmetic as the from-logits loss kernel, so decoding the result gives the rows the two-launch
    step gives for ``raw``.  ``out`` may be ``raw`` (in place).  Returns the activated tensor."""
    require_cuda(raw, out)
    if raw.dtype != torch.float32 or (out is not None and out.dtype != torch.float32):
        raise N.YoloB200Error("activate_head: float32 heads")
    pcf = floats_per_cell(params)
    if raw.numel() % pcf != 0:
        raise ValueError(f"a head of {raw.numel()} floats does not reshape to (-1, {pcf})")
    if out is None:
        out = torch.empty_like(raw)
    elif out.numel() != raw.numel():
        raise ValueError("out must have the size of raw")
    with torch.cuda.device(raw.device):
        N.check(N.lib.yb_activate_head(C.byref(params), _ptr(raw), _ptr(out), raw.numel() // pcf, _stream()),
                "yb_activate_head")
    return out


def grid_iou(box_true, box_pred, grid_shape, want_ciou=False):
    """box_true (..., 1, >=4), box_pred (..., B, >=4) fp32 CUDA, last-dim strides kept."""
    require_cuda(box_true, box_pred)
    B = box_pred.shape[-2]
    n_cells = box_pred.numel() // (B * box_pred.shape[-1])
    iou = torch.empty(box_pred.shape[:-1], dtype=torch.float32, device=box_pred.device)
    ciou = torch.empty_like(iou) if want_ciou else None
    with torch.cuda.device(box_pred.device):
        N.check(N.lib.yb_grid_iou(_ptr(box_true), box_true.shape[-1], _ptr(box_pred), box_pred.shape[-1],
                                  n_cells, B, int(grid_shape[0]), int(grid_shape[1]), _ptr(iou), _ptr(ciou),
                                  _stream()), "yb_grid_iou")
    return (iou, ciou) if want_ciou else iou


# --------------------------------------------------------------------------
# decode / NMS
# --------------------------------------------------------------------------
def make_decode_params(preds, class_num, threshold, version):
    n = len(preds)
    if not (1 <= n <= N.YB_MAX_SCALES):
        raise ValueError("between 1 and 4 scales")
    p = N.DecodeParams()
    p.version, p.class_num, p.n_scales = int(version), int(class_num), n
    if version not in (1, 2, 3, 4):
        raise ValueError(f"Invalid version: {version}")
    dt = preds[0].dtype
    if dt not in (torch.float32, torch.float64):
        raise N.YoloB200Error("decode inputs must be float32 or float64")
    p.is_f64 = int(dt == torch.float64)
    n_img = preds[0].shape[0]
    for i, t in enumerate(preds):
        if t.dim() != 4 or t.shape[0] != n_img or t.dtype != dt:
            raise ValueError("decode inputs must be (n_img, gh, gw, info) tensors of one dtype")
        p.grid_h[i], p.grid_w[i] = t.shape[1], t.shape[2]
        info = t.shape[3]
        if version == 1:
            p.bbox_num[i] = (info - class_num) // 5
            ok = p.bbox_num[i] * 5 + class_num == info
        else:
            p.bbox_num[i] = info // (5 + class_num)
            ok = p.bbox_num[i] * (5 + class_num) == info
        if not ok or p.bbox_num[i] < 1:
            raise ValueError(f"cannot reshape info axis {info} for class_num={class_num}, version={version}")
    p.threshold = float(threshold)
    return p, n_img


def decode_batch(preds, class_num=1, threshold=0.5, version=1, capacity=None, rows=None):
    """Batched decode.  Returns (rows (capacity,7) f64, row_offsets (n_img+1) i64), both
    CUDA; rows beyond row_offsets[-1] are unspecified.  If the true count exceeds the
    capacity the caller must retry (see decode_batch_exact)."""
    require_cuda(*preds)
    p, n_img = make_decode_params(preds, class_num, threshold, version)
    dev = preds[0].device
    if rows is not None:
        capacity = rows.shape[0]
    if capacity is None:
        capacity = max(1024, 512 * n_img)
    with torch.cuda.device(dev):
        if rows is None:
            rows = torch.empty((capacity, 7), dtype=_F64, device=dev)
        offsets = torch.empty(n_img + 1, dtype=_I64, device=dev)
        ws_bytes = N.lib.yb_decode_workspace_bytes(C.byref(p), n_img)
        ws = workspaces.get("decode", ws_bytes, dev)
        ptrs = (C.c_void_p * len(preds))(*[t.data_ptr() for t in preds])
        N.check(N.lib.yb_decode(ptrs, n_img, C.byref(p), _ptr(rows), capacity, _ptr(offsets), _ptr(ws),
                                ws_bytes, _stream()), "yb_decode")
    return rows, offsets


def decode_batch_exact(preds, class_num=1, threshold=0.5, version=1, capacity=None):
    """decode_batch + overflow check (one host sync); grows the buffer when needed."""
    rows, offsets = decode_batch(preds, class_num, threshold, version, capacity)
    total = int(offsets[-1].item())
    if total > rows.shape[0]:
        rows, offsets = decode_batch(preds, class_num, threshold, version, capacity=total)
    return rows[:total], offsets


def nms_batch(rows, row_offsets, class_num=1, nms_threshold=0.45, iou_mode=1, want_rows=True,
              want_seg_offsets=False, soft=None):
    """Batched per-class NMS.  rows (R,7) f64 CUDA (R = capacity), row_offsets (n_img+1) i64
    CUDA.  Returns dict(keep u8[R], out_rows (R,7), out_offsets (n_img+1), seg_offsets)."""
    require_cuda(rows, row_offsets)
    if rows.dtype != _F64 or row_offsets.dtype != _I64:
        raise N.YoloB200Error("nms needs float64 rows and int64 offsets")
    dev = rows.device
    R = rows.shape[0]
    n_img = row_offsets.numel() - 1
    with torch.cuda.device(dev):
        keep = torch.empty(max(R, 1), dtype=torch.uint8, device=dev)
        out_rows = torch.empty((max(R, 1), 7), dtype=_F64, device=dev) if want_rows else None
        out_offsets = torch.empty(n_img + 1, dtype=_I64, device=dev)
        seg = torch.empty(n_img * class_num + 1, dtype=_I64, device=dev) if want_seg_offsets else None
        ws_bytes = N.lib.yb_nms_workspace_bytes(R, n_img, class_num)
        ws = workspaces.get("nms", ws_bytes, dev)
        if soft is not None:   # (conf_threshold, sigma): Gaussian soft-NMS
            N.check(N.lib.yb_soft_nms(_ptr(rows), _ptr(row_offsets), R, n_img, class_num, float(nms_threshold),
                                      float(soft[0]), float(soft[1]), _ptr(keep), _ptr(out_rows),
                                      _ptr(out_offsets), _ptr(seg), _ptr(ws), ws_bytes, _stream()), "yb_soft_nms")
        else:
            N.check(N.lib.yb_nms(_ptr(rows), _ptr(row_offsets), R, n_img, class_num, float(nms_threshold),
                                 int(iou_mode), _ptr(keep), _ptr(out_rows), _ptr(out_offsets), _ptr(seg),
                                 _ptr(ws), ws_bytes, _stream()), "yb_nms")
    return dict(keep=keep[:R], out_rows=out_rows, out_offsets=out_offsets, seg_offsets=seg)


def _fused_outputs(dev, n_img, out_capacity, out):
    if out is not None:
        return out["out_rows"], out["out_offsets"], out["n_overflow"]
    return (torch.empty((max(out_capacity, 1), 7), dtype=_F64, device=dev),
            torch.empty(n_img + 1, dtype=_I64, device=dev), torch.empty(1, dtype=torch.int32, device=dev))


def decode_nms_batch(preds, class_num=1, threshold=0.5, version=1, nms_threshold=0.45, iou_mode=1,
                     rows_per_img_cap=1024, out_capacity=None, out=None):
    """Decode + per-class NMS of a batch in one launch after the counting pass (yb_decode_nms), for
    images of at most ``rows_per_img_cap`` decode rows.  Returns dict(out_rows (cap,7) f64,
    out_offsets (n_img+1) i64, n_overflow i32[1]) - all CUDA; images that exceed the cap produce no
    rows and are counted in n_overflow (see decode_nms_batch_exact for the checked form)."""
    require_cuda(*preds)
    p, n_img = make_decode_params(preds, class_num, threshold, version)
    dev = preds[0].device
    if out_capacity is None:
        out_capacity = rows_per_img_cap * max(n_img, 1)
    with torch.cuda.device(dev):
        out_rows, out_offsets, n_overflow = _fused_outputs(dev, n_img, out_capacity, out)
        ws_bytes = N.lib.yb_decode_nms_workspace_bytes(C.byref(p), n_img, int(rows_per_img_cap))
        if ws_bytes == 0:
            raise ValueError("yb_decode_nms: float32 heads, class_num <= 256, 32 <= rows_per_img_cap <= "
                             f"{N.YB_FUSED_MAX_ROWS}")
        ws = workspaces.get("decode_nms", ws_bytes, dev)
        ptrs = (C.c_void_p * len(preds))(*[t.data_ptr() for t in preds])
        N.check(N.lib.yb_decode_nms(ptrs, n_img, C.byref(p), float(nms_threshold), int(iou_mode),
                                    int(rows_per_img_cap), _ptr(out_rows), out_rows.shape[0], _ptr(out_offsets),
                                    _ptr(n_overflow), _ptr(ws), ws_bytes, _stream()), "yb_decode_nms")
    return dict(out_rows=out_rows, out_offsets=out_offsets, n_overflow=n_overflow)


def decode_nms_batch_exact(preds, class_num=1, threshold=0.5, version=1, nms_threshold=0.45, iou_mode=1,
                           rows_per_img_cap=1024):
    """decode_nms_batch with the overflow check (one host sync): falls back to the general chain
    (yb_decode + yb_nms, any size) when an image exceeds the cap.  Returns (rows (K,7), offsets)."""
    p, n_img = make_decode_params(preds, class_num, threshold, version)
    supported = (not p.is_f64) and N.lib.yb_decode_nms_workspace_bytes(C.byref(p), n_img, int(rows_per_img_cap)) > 0
    if supported:   # float32 heads, class_num <= 256, grids below 2^19 cells per image
        r = decode_nms_batch(preds, class_num, threshold, version, nms_threshold, iou_mode, rows_per_img_cap)
        if int(r["n_overflow"].item()) == 0:
            total = int(r["out_offsets"][-1].item())
            if total <= r["out_rows"].shape[0]:
                return r["out_rows"][:total], r["out_offsets"]
    rows, offs = decode_batch_exact(preds, class_num, threshold, version)
    g = nms_batch(rows, offs, class_num, nms_threshold, iou_mode)
    return g["out_rows"][:int(g["out_offsets"][-1].item())], g["out_offsets"]


def loss_decode_nms_fused(params, y_trues, y_preds, threshold=0.5, nms_threshold=0.45, iou_mode=1,
                          rows_per_img_cap=1024, global_batch=None, dpreds=None, want_terms=False, out=None,
                          out_capacity=None, split_hook=None, loss_out=None, loss_box=None):
    """The train-and-evaluate step in two launches (yb_loss_decode_nms_fused): loss forward +
    gradient with the decode counting pass riding on its read of y_pred, then decode + NMS with one
    CTA per image.  Returns (loss [n], dpreds, terms, dict(out_rows, out_offsets, n_overflow)).
    ``params`` with from_logits (grid_loss.wrap_yolo_loss_from_logits): y_preds hold the RAW v3/v4
    head outputs, the gradient is d/d(raw) and the survivors are those of the activated heads
    (activate_head).  An image over ``rows_per_img_cap`` rows has no survivors and is counted in
    n_overflow: take it from decode_nms_batch_exact on the activated heads."""
    n = len(params)
    scales, outs, n_img = bind_loss_scales(params, y_trues, y_preds, global_batch, dpreds)
    dev = y_preds[0].device
    dparams = loss_decode_params(params, threshold)
    if out_capacity is None:
        out_capacity = rows_per_img_cap * max(n_img, 1)
    with torch.cuda.device(dev):
        out_rows, out_offsets, n_overflow = _fused_outputs(dev, n_img, out_capacity, out)
        loss = loss_out if loss_out is not None else torch.empty(n, dtype=torch.float32, device=dev)
        if loss_box is not None:
            loss_box[0] = loss      # lets a split_hook see the tensor the loss kernel has just written
        terms = torch.empty((n, N.YB_LOSS_TERMS), dtype=_F64, device=dev) if want_terms else None
        lws_bytes = N.lib.yb_loss_workspace_bytes(n)
        lws = workspaces.get("loss", lws_bytes, dev)
        fws_bytes = N.lib.yb_decode_nms_workspace_bytes(C.byref(dparams), n_img, int(rows_per_img_cap))
        if fws_bytes == 0:
            raise ValueError("yb_loss_decode_nms_fused: class_num <= 256, 32 <= rows_per_img_cap <= "
                             f"{N.YB_FUSED_MAX_ROWS}")
        fws = workspaces.get("decode_nms", fws_bytes, dev)
        if split_hook is None:
            N.check(N.lib.yb_loss_decode_nms_fused(scales, n, _ptr(loss), _ptr(terms), float(threshold),
                                                   float(nms_threshold), int(iou_mode), int(rows_per_img_cap),
                                                   _ptr(out_rows), out_rows.shape[0], _ptr(out_offsets),
                                                   _ptr(n_overflow), _ptr(lws), lws_bytes, _ptr(fws), fws_bytes,
                                                   _stream()), "yb_loss_decode_nms_fused")
        else:   # two calls so that a timer can bracket the loss kernel alone (bench.py roofline)
            N.check(N.lib.yb_loss_decode_nms_fused(scales, n, _ptr(loss), _ptr(terms), float(threshold),
                                                   float(nms_threshold), int(iou_mode), int(rows_per_img_cap),
                                                   None, 0, None, None, _ptr(lws), lws_bytes, _ptr(fws), fws_bytes,
                                                   _stream()), "yb_loss_decode_nms_fused(loss)")
            split_hook()
            ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in y_preds])
            N.check(N.lib.yb_decode_nms_finish(ptrs, n_img, C.byref(dparams), float(nms_threshold), int(iou_mode),
                                               int(rows_per_img_cap), _ptr(out_rows), out_rows.shape[0],
                                               _ptr(out_offsets), _ptr(n_overflow), _ptr(fws), fws_bytes, _stream()),
                    "yb_decode_nms_finish")
    return loss, outs, terms, dict(out_rows=out_rows, out_offsets=out_offsets, n_overflow=n_overflow)


class TrainEvalStep:
    """The two-launch train-and-evaluate step over STATIC buffers, replayed from a CUDA graph.

    What a training loop with fixed shapes does with loss_decode_nms_fused: the tensors handed in
    are the buffers every step reads (refill them in place), the workspaces belong to this object
    and are zeroed once - both kernels leave them zeroed (yb_loss_decode_nms_fused_clean) - so a
    step is exactly two kernel nodes, plus whatever `tail` enqueues on the capturing stream, captured
    once and replayed by run().  graph=False launches the same two kernels eagerly.
    A collective is better issued after run() than captured through `tail`: bench.py alternates two
    steps and all-reduces each one's loss asynchronously (a graph that holds NCCL kernels has to be
    destroyed before the process group, or the teardown can hang).
    ``params`` may be from-logits params (raw v3/v4 heads, see loss_decode_nms_fused); a step that
    reports n_overflow takes its survivors from fallback_survivors()."""

    def __init__(self, params, y_trues, y_preds, threshold=0.5, nms_threshold=0.45, iou_mode=1,
                 rows_per_img_cap=1024, global_batch=None, dpreds=None, want_terms=False, out=None,
                 out_capacity=None, tail=None, graph=True):
        n = len(params)
        self.scales, self.dpreds, n_img = bind_loss_scales(params, y_trues, y_preds, global_batch, dpreds)
        self.params = [N.LossParams.from_buffer_copy(p) for p in params]
        self.dev = dev = y_preds[0].device
        self.n = n
        self.n_img = n_img
        self._keep = (list(y_trues), list(y_preds))
        dparams = loss_decode_params(params, threshold)
        self.args = (float(threshold), float(nms_threshold), int(iou_mode), int(rows_per_img_cap))
        if out_capacity is None:
            out_capacity = rows_per_img_cap * max(n_img, 1)
        with torch.cuda.device(dev):
            self.out_rows, self.out_offsets, self.n_overflow = _fused_outputs(dev, n_img, out_capacity, out)
            self.loss = torch.empty(n, dtype=torch.float32, device=dev)
            self.terms = torch.empty((n, N.YB_LOSS_TERMS), dtype=_F64, device=dev) if want_terms else None
            self.lws_bytes = N.lib.yb_loss_workspace_bytes(n)
            self.fws_bytes = N.lib.yb_decode_nms_workspace_bytes(C.byref(dparams), n_img, int(rows_per_img_cap))
            if self.fws_bytes == 0:
                raise ValueError("TrainEvalStep: class_num <= 256, 32 <= rows_per_img_cap <= "
                                 f"{N.YB_FUSED_MAX_ROWS}")
            # private, zeroed once: nothing but the clean entry point ever touches them
            self.lws = torch.zeros(self.lws_bytes + 256, dtype=torch.uint8, device=dev)
            self.fws = torch.zeros(self.fws_bytes + 256, dtype=torch.uint8, device=dev)
        self.tail = tail
        self.graph = None
        if graph:
            self._capture()

    def _aligned(self, t):
        return (t.data_ptr() + 255) // 256 * 256

    def _launch(self):
        thr, nms_thr, mode, cap = self.args
        rc = N.lib.yb_loss_decode_nms_fused_clean(self.scales, self.n, _ptr(self.loss), _ptr(self.terms), thr,
                                                  nms_thr, mode, cap, _ptr(self.out_rows), self.out_rows.shape[0],
                                                  _ptr(self.out_offsets), _ptr(self.n_overflow),
                                                  self._aligned(self.lws), self.lws_bytes,
                                                  self._aligned(self.fws), self.fws_bytes, _stream())
        if rc != 0:     # the kernels may not have run to their self-cleaning end
            self.lws.zero_()
            self.fws.zero_()
        N.check(rc, "yb_loss_decode_nms_fused_clean")
        if self.tail is not None:
            self.tail(self)

    def _capture(self):
        with torch.cuda.device(self.dev):
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):      # warm-up outside the capture (lazy module load, smem opt-in)
                self._launch()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                self._launch()
            self.graph = g

    def run(self):
        """One step on the current stream.  Returns (loss [n], dpreds, terms, dict(out_rows, ...))
        - the same static tensors every time."""
        with torch.cuda.device(self.dev):
            if self.graph is not None:
                self.graph.replay()
            else:
                self._launch()
        return self.loss, self.dpreds, self.terms, dict(out_rows=self.out_rows, out_offsets=self.out_offsets,
                                                        n_overflow=self.n_overflow)

    def fallback_survivors(self):
        """The survivors of the current inputs from the checked decode + NMS (decode_nms_batch_exact,
        any number of rows per image): what a step that reported n_overflow > 0 falls back to.  Raw
        heads (from-logits params) are activated first, into fresh tensors.  Returns (rows (K,7) f64,
        offsets (n_img+1) i64), both CUDA."""
        thr, nms_thr, mode, cap = self.args
        p0 = self.params[0]
        preds = self._keep[1]
        if p0.from_logits:
            preds = [activate_head(p, t) for p, t in zip(self.params, preds)]
        with torch.cuda.device(self.dev):
            return decode_nms_batch_exact(preds, p0.class_num, thr, p0.version, nms_thr, mode, cap)


def pairwise_iou(a, b, mode=1):
    """(na, >=4) x (nb, >=4) f64 CUDA -> (na, nb) f64; a plays xywh_true."""
    require_cuda(a, b)
    if a.dtype != _F64 or b.dtype != _F64:
        raise N.YoloB200Error("pairwise_iou needs float64")
    out = torch.empty((a.shape[0], b.shape[0]), dtype=_F64, device=a.device)
    with torch.cuda.device(a.device):
        N.check(N.lib.yb_pairwise_iou(_ptr(a), a.shape[0], a.shape[1], _ptr(b), b.shape[0], b.shape[1],
                                      int(mode), _ptr(out), _stream()), "yb_pairwise_iou")
    return out


def elementwise_iou(a, b, mode=1):
    """(n, >=4) vs (n, >=4) f64 CUDA -> (n,) f64."""
    require_cuda(a, b)
    out = torch.empty(a.shape[0], dtype=_F64, device=a.device)
    with torch.cuda.device(a.device):
        N.check(N.lib.yb_elementwise_iou(_ptr(a), a.shape[1], _ptr(b), b.shape[1], a.shape[0], int(mode),
                                         _ptr(out), _stream()), "yb_elementwise_iou")
    return out


# --------------------------------------------------------------------------
# k-means
# --------------------------------------------------------------------------
def kmeans_assign(data, centers, dist_kind=N.YB_DIST_IOU, want_assign=False):
    """data (M,d) f64 CUDA, centers (k,d) f64 CUDA -> (assign i32[M] | None, sums (k,d), counts i64[k])."""
    require_cuda(data, centers)
    if data.dtype != _F64 or centers.dtype != _F64:
        raise N.YoloB200Error("kmeans needs float64")
    M, d = data.shape
    k = centers.shape[0]
    dev = data.device
    with torch.cuda.device(dev):
        assign = torch.empty(M, dtype=torch.int32, device=dev) if want_assign else None
        sums = torch.empty((k, d), dtype=_F64, device=dev)
        counts = torch.empty(k, dtype=_I64, device=dev)
        ws_bytes = N.lib.yb_kmeans_workspace_bytes(M, k, d)
        if ws_bytes == 0:
            raise ValueError("unsupported k / n_dim")
        ws = workspaces.get("kmeans", ws_bytes, dev)
        N.check(N.lib.yb_kmeans_assign(_ptr(data), M, d, _ptr(centers), k, int(dist_kind), _ptr(assign),
                                       _ptr(sums), _ptr(counts), _ptr(ws), ws_bytes, _stream()),
                "yb_kmeans_assign")
    return assign, sums, counts


def kmeans_dist(a, b, what, outer):
    """utils/kmeans.py:9-40 on CUDA tensors: a (na,d), b (nb,d) f64 -> (na,nb) if outer else (nb,).
    what: 0 iou, 1 iou_dist, 2 euclidean_dist."""
    require_cuda(a, b)
    if a.dtype != _F64 or b.dtype != _F64:
        raise N.YoloB200Error("kmeans distances need float64")
    dev = a.device
    with torch.cuda.device(dev):
        out = torch.empty((a.shape[0], b.shape[0]) if outer else (b.shape[0],), dtype=_F64, device=dev)
        N.check(N.lib.yb_kmeans_dist(_ptr(a), a.shape[0], _ptr(b), b.shape[0], a.shape[1], int(what), int(bool(outer)),
                                     _ptr(out), _stream()), "yb_kmeans_dist")
    return out


class KMeansLloyd:
    """Device-resident Lloyd loop (yb_kmeans_lloyd_init / _step / _update): the boxes, the centres and
    the loop state stay on the GPU; ``step()`` queues one iteration without touching the host."""

    def __init__(self, data, centers, dist_kind, stop_dist, max_iternum, sharded=False, peer_group=None):
        require_cuda(data, centers)
        if data.dtype != _F64 or centers.dtype != _F64:
            raise N.YoloB200Error("kmeans needs float64")
        self.data, self.centers = data, centers
        self.k, self.d = centers.shape
        self.kind, self.stop, self.max_iter = int(dist_kind), float(stop_dist), int(max_iternum)
        dev = data.device
        with torch.cuda.device(dev):
            sb = N.lib.yb_kmeans_state_bytes(self.k, self.d)
            if sb == 0:
                raise ValueError("unsupported k / n_dim (k <= 16, n_dim <= 4)")
            self.state = torch.empty(sb // 8, dtype=_I64, device=dev)
            self.ws_bytes = N.lib.yb_kmeans_workspace_bytes(data.shape[0], self.k, self.d)
            self.ws = torch.empty(self.ws_bytes + 256, dtype=torch.uint8, device=dev)
            self.ws_ptr = self.ws.data_ptr() + ((-self.ws.data_ptr()) % 256)
            self.packed = torch.zeros(self.k * (self.d + 1), dtype=_F64, device=dev) if (sharded and peer_group is None) else None
            N.check(N.lib.yb_kmeans_lloyd_init(_ptr(self.state), self.k, self.d, C.c_void_p(self.ws_ptr), self.ws_bytes,
                                               _stream()), "yb_kmeans_lloyd_init")
            self.peers = None
            self._graphs = {}      # step_many: one captured batch per length
            if peer_group is not None:
                self._open_peers(peer_group)

    def _open_peers(self, group):
        """Mailboxes for the in-kernel all-reduce: allocate + export ours, open every peer's
        (handles travel through the process group once)."""
        import torch.distributed as dist
        alone = isinstance(group, str) and group == "self"     # a single rank exchanging with itself (tests)
        self.world, self.rank = (1, 0) if alone else (dist.get_world_size(group), dist.get_rank(group))
        nbytes = N.lib.yb_peer_mailbox_bytes(self.world)
        if nbytes == 0:
            raise ValueError(f"peer exchange supports up to {N.YB_MAX_PEERS} ranks")
        own, handle = C.c_void_p(), (C.c_char * 64)()
        N.check(N.lib.yb_peer_alloc(nbytes, C.byref(own), handle), "yb_peer_alloc")
        handles = [None] * self.world
        if alone:
            handles[0] = bytes(handle.raw)
        else:
            dist.all_gather_object(handles, bytes(handle.raw), group=group)
        ptrs = (C.c_void_p * self.world)()
        self._opened = []
        for r, h in enumerate(handles):
            if r == self.rank:
                ptrs[r] = own.value
            else:
                p = C.c_void_p()
                N.check(N.lib.yb_peer_open((C.c_char * 64).from_buffer_copy(h), C.byref(p)), "yb_peer_open")
                ptrs[r] = p.value
                self._opened.append(p.value)
        self._own_mailbox = own.value
        self.peers = ptrs
        if not alone:
            dist.barrier(group=group)  # every mailbox is mapped everywhere before the first exchange

    def close(self):
        """Release the peer mappings and the mailbox (after a barrier: nobody may still write to it)."""
        if self.peers is not None:
            torch.cuda.synchronize()
            self._graphs.clear()
            for p in self._opened:
                N.lib.yb_peer_close(C.c_void_p(p))
            N.lib.yb_peer_free(C.c_void_p(self._own_mailbox))
            self.peers = None

    def step(self, assign=None):
        """The assignment pass (+ the update when not sharded, + the peer all-reduce and the update
        when sharded over peer memory) of one iteration."""
        if self.peers is not None:
            N.check(N.lib.yb_kmeans_lloyd_step_peers(_ptr(self.data), self.data.shape[0], self.d, _ptr(self.centers),
                                                     self.k, self.kind, self.stop, self.max_iter, _ptr(self.state),
                                                     _ptr(assign), C.c_void_p(self.ws_ptr), self.ws_bytes, self.peers,
                                                     self.rank, self.world, _stream()), "yb_kmeans_lloyd_step_peers")
            return
        N.check(N.lib.yb_kmeans_lloyd_step(_ptr(self.data), self.data.shape[0], self.d, _ptr(self.centers), self.k,
                                           self.kind, self.stop, self.max_iter, _ptr(self.state), _ptr(self.packed),
                                           _ptr(assign), C.c_void_p(self.ws_ptr), self.ws_bytes, _stream()),
                "yb_kmeans_lloyd_step")

    def step_many(self, n):
        """n iterations of the loop whose exchange (if any) happens inside the launch - unsharded, or
        sharded over peer memory - replayed from a CUDA graph captured once per n: the host's launch
        cost (one ctypes call per iteration) is out of the loop.  Every rank must ask for the same n."""
        if self.packed is not None:
            raise N.YoloB200Error("step_many: the NCCL-exchanged loop queues step() / all-reduce / update() itself")
        g = self._graphs.get(n)
        if g is None:
            with torch.cuda.device(self.data.device):
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=side):   # capture runs nothing: the loop state is untouched
                    for _ in range(n):
                        self.step()
                torch.cuda.current_stream().wait_stream(side)
            self._graphs[n] = g
        g.replay()

    def update(self):
        """Sharded loop: the update on the all-reduced ``packed`` sums / counts."""
        N.check(N.lib.yb_kmeans_lloyd_update(_ptr(self.packed), _ptr(self.centers), self.k, self.d, self.kind,
                                             self.stop, self.max_iter, _ptr(self.state), _stream()),
                "yb_kmeans_lloyd_update")

    def read_state(self):
        """(status, completed updates, loss history array, saved sums (k,d), saved counts (k,)) - one sync."""
        host = self.state.cpu().numpy()
        hist = host[4:4 + N.YB_KMEANS_HIST].view(np.float64)
        saved = host[4 + N.YB_KMEANS_HIST:].view(np.float64).reshape(self.k, self.d + 1)
        return int(host[0]), int(host[1]), hist, saved[:, :self.d].copy(), saved[:, self.d].copy()

    def resume(self, status, completed):
        """Host finished an update itself (empty-cluster redraw): write status / counter back."""
        self.state[0:2].copy_(torch.tensor([status, completed], dtype=_I64), non_blocking=False)


def minmax(data):
    require_cuda(data)
    if data.dtype != _F64:
        raise N.YoloB200Error("minmax needs float64")
    dev = data.device
    with torch.cuda.device(dev):
        out = torch.empty(2, dtype=_F64, device=dev)
        ws = workspaces.get("minmax", 64 * 1024, dev)
        N.check(N.lib.yb_minmax_f64(_ptr(data), data.numel(), _ptr(out), _ptr(ws), 64 * 1024, _stream()),
                "yb_minmax_f64")
    return out


# --------------------------------------------------------------------------
# mAP matching
# --------------------------------------------------------------------------
def map_match(gt_rows, gt_offsets, det_rows, det_offsets, class_num):
    require_cuda(gt_rows, gt_offsets, det_rows, det_offsets)
    dev = det_offsets.device
    n_img = det_offsets.numel() - 1
    with torch.cuda.device(dev):
        best_iou = torch.empty(max(det_rows.shape[0], 1), dtype=_F64, device=dev)
        best_gt = torch.empty(max(det_rows.shape[0], 1), dtype=torch.int32, device=dev)
        counts = torch.empty((n_img, class_num), dtype=torch.int32, device=dev)
        N.check(N.lib.yb_map_match(_ptr(gt_rows), _ptr(gt_offsets), _ptr(det_rows), _ptr(det_offsets), n_img,
                                   class_num, gt_rows.shape[0], det_rows.shape[0], _ptr(best_iou),
                                   _ptr(best_gt), _ptr(counts), _stream()), "yb_map_match")
    return best_iou[:det_rows.shape[0]], best_gt[:det_rows.shape[0]], counts


def map_accumulate(det_rows, seg_offsets, best_iou, best_gt, gt_counts, class_num, iou_threshold,
                   max_per_img, gt_base, score_acc):
    """Triples of one image batch grouped by class (see yb_map_accumulate).  Returns
    (conf f64[D], gt_id i64[D], flag u8[D], cls i32[D], class_offsets i64[C+1]); entries past
    class_offsets[-1] are unspecified.  ``score_acc`` (3*C int64 CUDA) is added to."""
    require_cuda(det_rows, seg_offsets, best_iou, best_gt, gt_counts, gt_base, score_acc)
    dev = seg_offsets.device
    n_img = gt_counts.shape[0]
    D = max(det_rows.shape[0], 1)
    with torch.cuda.device(dev):
        conf = torch.empty(D, dtype=_F64, device=dev)
        gid = torch.empty(D, dtype=_I64, device=dev)
        flag = torch.empty(D, dtype=torch.uint8, device=dev)
        cls = torch.empty(D, dtype=torch.int32, device=dev)
        coff = torch.empty(class_num + 1, dtype=_I64, device=dev)
        ws_bytes = N.lib.yb_map_accumulate_workspace_bytes(n_img, class_num)
        ws = workspaces.get("map_acc", ws_bytes, dev)
        N.check(N.lib.yb_map_accumulate(_ptr(det_rows), _ptr(seg_offsets), _ptr(best_iou), _ptr(best_gt),
                                        _ptr(gt_counts), n_img, class_num, float(iou_threshold),
                                        int(max_per_img) if max_per_img else 0, _ptr(gt_base), _ptr(conf),
                                        _ptr(gid), _ptr(flag), _ptr(cls), _ptr(coff), _ptr(score_acc), _ptr(ws),
                                        ws_bytes, _stream()), "yb_map_accumulate")
    return conf, gid, flag, cls, coff


def map_append(chunk, n_src, dst, total, counter):
    """Append the first ``*n_src`` records of ``chunk`` = (conf, gid, flag, cls) to ``dst`` (same
    four arrays, larger) at the device-side running ``total`` and advance it (yb_map_append)."""
    conf, gid, flag, cls = chunk
    dconf, dgid, dflag, dcls = dst
    with torch.cuda.device(conf.device):
        N.check(N.lib.yb_map_append(_ptr(conf), _ptr(gid), _ptr(flag), _ptr(cls), _ptr(n_src), conf.shape[0],
                                    _ptr(dconf), _ptr(dgid), _ptr(dflag), _ptr(dcls), dconf.shape[0], _ptr(total),
                                    _ptr(counter), _stream()), "yb_map_append")


def pr_curve(conf, cls, gt_id, flag, gt_table_base, n_gt_total):
    """Sort by (class, confidence desc, later position first) and count distinct true positives.
    Returns (order i64[D], tp_cum i64[D+1], tpp_cum i64[D+1])."""
    require_cuda(conf, cls, gt_id, flag, gt_table_base)
    dev = conf.device
    D = conf.shape[0]
    with torch.cuda.device(dev):
        order = torch.empty(max(D, 1), dtype=_I64, device=dev)
        tp = torch.empty(D + 1, dtype=_I64, device=dev)
        tpp = torch.empty(D + 1, dtype=_I64, device=dev)
        ws_bytes = N.lib.yb_pr_curve_workspace_bytes(D, int(n_gt_total))
        ws = workspaces.get("pr_curve", ws_bytes, dev)
        N.check(N.lib.yb_pr_curve(_ptr(conf), _ptr(cls), _ptr(gt_id), _ptr(flag), D, _ptr(gt_table_base),
                                  int(n_gt_total), _ptr(order), _ptr(tp), _ptr(tpp), _ptr(ws), ws_bytes,
                                  _stream()), "yb_pr_curve")
    return order[:D], tp, tpp


def pr_points(tp_cum, tpp_cum, class_start, gts, precision_mode):
    """precision / recall of every sorted record (yb_pr_points): two f64[D] CUDA tensors."""
    require_cuda(tp_cum, tpp_cum, class_start, gts)
    D = tp_cum.shape[0] - 1
    dev = tp_cum.device
    with torch.cuda.device(dev):
        precision = torch.empty(max(D, 1), dtype=_F64, device=dev)
        recall = torch.empty(max(D, 1), dtype=_F64, device=dev)
        N.check(N.lib.yb_pr_points(_ptr(tp_cum), _ptr(tpp_cum), _ptr(class_start), _ptr(gts), gts.shape[0], D,
                                   int(precision_mode), _ptr(precision), _ptr(recall), _stream()), "yb_pr_points")
    return precision[:D], recall[:D]


# --------------------------------------------------------------------------
# label-side helpers
# --------------------------------------------------------------------------
def encode_labels(boxes, box_offsets, img_size, grid_shape, class_num, n_levels=1, dtype=torch.float32,
                  max_boxes_per_img=None, outs=None, n_bad=None):
    """Box lists -> label grids on the device (yb_encode_labels; utils/tools.py:179-209 plus
    down2xlabel :342-367 per extra level).  boxes (n_boxes, 5) f64 CUDA [x1, y1, x2, y2, class],
    box_offsets (n_img+1) i64 CUDA; grid_shape = the FINEST grid.  Returns (list of n_levels
    label tensors coarse grid first, n_bad u64[1] CUDA = boxes the reference would have raised on).
    ``max_boxes_per_img`` bounds the boxes of one image (host knowledge; one sync to read it from
    the offsets when omitted)."""
    require_cuda(boxes, box_offsets)
    if boxes.dtype != _F64 or box_offsets.dtype != _I64:
        raise N.YoloB200Error("encode_labels needs float64 boxes and int64 offsets")
    if boxes.dim() != 2 or boxes.shape[1] != 5:
        raise ValueError("boxes must be (n_boxes, 5): x1, y1, x2, y2, class index")
    if dtype not in (torch.float32, _F64):
        raise N.YoloB200Error("label grids are float32 or float64")
    dev = boxes.device
    n_img = box_offsets.numel() - 1
    gh, gw = int(grid_shape[0]), int(grid_shape[1])
    if max_boxes_per_img is None:
        max_boxes_per_img = int((box_offsets[1:] - box_offsets[:-1]).max().item()) if n_img > 0 else 0
    if max_boxes_per_img > N.YB_ENCODE_MAX_BOXES:
        raise ValueError(f"more than {N.YB_ENCODE_MAX_BOXES} boxes in one image")
    with torch.cuda.device(dev):
        if outs is None:
            outs = [torch.empty((n_img, gh >> (n_levels - 1 - l), gw >> (n_levels - 1 - l), 5 + class_num),
                                dtype=dtype, device=dev) for l in range(n_levels)]
        else:
            require_cuda(*outs)
        if n_bad is None:
            n_bad = torch.zeros(1, dtype=torch.int64, device=dev)
        ptrs = (C.c_void_p * n_levels)(*[t.data_ptr() for t in outs])
        N.check(N.lib.yb_encode_labels(_ptr(boxes), _ptr(box_offsets), n_img, int(max_boxes_per_img),
                                       float(img_size[0]), float(img_size[1]), gh, gw, int(class_num),
                                       int(n_levels), ptrs, int(dtype == _F64), _ptr(n_bad), _stream()),
                "yb_encode_labels")
    return outs, n_bad


def down2x_labels(labels):
    """(N, gh, gw, ch) f32/f64 CUDA -> (N, gh/2, gw/2, ch) f64 CUDA (utils/tools.py:342-367)."""
    require_cuda(labels)
    if labels.dtype not in (torch.float32, _F64) or labels.dim() != 4:
        raise N.YoloB200Error("labels must be a (N, gh, gw, ch) float32/float64 tensor")
    n, gh, gw, ch = labels.shape
    if gh % 2 or gw % 2:
        raise IndexError("index out of bounds: down2xlabel needs even grid sizes (the reference raises here too)")
    out = torch.empty((n, gh // 2, gw // 2, ch), dtype=_F64, device=labels.device)
    with torch.cuda.device(labels.device):
        N.check(N.lib.yb_down2x_labels(_ptr(labels), int(labels.dtype == _F64), n, gh, gw, ch, _ptr(out), _stream()),
                "yb_down2x_labels")
    return out


def column_sums(data2d):
    """(rows, cols) f32/f64 CUDA -> (cols,) f64 CUDA."""
    require_cuda(data2d)
    rows, cols = data2d.shape
    dev = data2d.device
    with torch.cuda.device(dev):
        out = torch.empty(cols, dtype=_F64, device=dev)
        ws_bytes = N.lib.yb_column_sums_workspace_bytes(cols)
        ws = workspaces.get("colsum", ws_bytes, dev)
        N.check(N.lib.yb_column_sums(_ptr(data2d), int(data2d.dtype == _F64), rows, cols, _ptr(out), _ptr(ws),
                                     ws_bytes, _stream()), "yb_column_sums")
    return out
