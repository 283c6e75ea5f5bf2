"""A whole train-and-evaluate step on HOST buffers, pipelined.

``HostBatchStep`` is the end-to-end form of the hot path: the caller holds the batch where the
reference holds it - head outputs as (pinned) host arrays and the labels as the box lists its
reader parsed (utils/tools.py:230-297) - and gets back the loss per scale, dL/dy_pred on the
device (for the backbone's backward pass) and the NMS survivors in host memory.

What crosses PCIe per step: the head outputs (H2D, unavoidable), the box lists (a few KB instead
of the dense label grids: they are encoded on the device by ``yb_encode_labels``,
utils/tools.py:179-209 + down2xlabel :342-367) and the survivors + loss scalars (written by the
kernels straight into mapped host memory, so no sized D2H copy and no mid-step round trip).
The batch is cut into chunks of images: the H2D copy of chunk k+1 runs on a copy stream under
the kernels of chunk k, and the host synchronises ONCE per step.

Per chunk (all through the C ABI, include/yolo_b200.h): yb_encode_labels ->
yb_loss_decode_nms_fused (loss fwd+grad with the decode counting pass riding on its read of
y_pred, then decode + NMS with one CTA per image): three launches.  A chunk in which an image
exceeds ``rows_per_img`` decode rows is redone after the step's sync with the general chain
(yb_decode + yb_nms).  Chunk losses are partial sums with the divisor of the whole (global) batch,
so their sum is the reference's ``reduce_mean(axis=0)`` loss (yolov4/losses/loss.py:117).
"""
import ctypes as C

import numpy as np
import torch

from . import _native as N
from . import engine


def _mapped(t):
    """Device alias of a pinned host tensor."""
    out = C.c_void_p()
    N.check(N.lib.yb_mapped_host_pointer(C.c_void_p(t.data_ptr()), C.byref(out)), "yb_mapped_host_pointer")
    return out.value


class HostBatchStep:
    def __init__(self, loss_fns, img_size, batch, conf_threshold=0.5, nms_threshold=0.45, nms_mode=2,
                 n_chunks=8, rows_per_img=1024, max_boxes_per_img=64, max_boxes=None, global_batch=None,
                 device=None):
        if not torch.cuda.is_available():
            raise N.YoloB200Error("no CUDA device: tf2_yolo_b200 has no CPU fallback")
        self.dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.params = [f.params for f in loss_fns]
        p0 = self.params[0]
        self.n_scales = len(self.params)
        self.version, self.C = p0.version, p0.class_num
        self.batch = int(batch)
        self.global_batch = int(global_batch if global_batch is not None else batch)
        self.img_size = (float(img_size[0]), float(img_size[1]))
        self.thr, self.nms_thr, self.nms_mode = float(conf_threshold), float(nms_threshold), int(nms_mode)
        self.max_boxes_per_img = int(max_boxes_per_img)
        n_chunks = max(1, min(int(n_chunks), self.batch))
        # chunk edges on multiples of 4 images where the batch allows: keeps every chunk's tensors
        # 16-byte aligned (bulk-async copies) whatever the per-image size is
        q = 4 if self.batch >= 4 * n_chunks else 1
        edges = [self.batch // q * c // n_chunks * q for c in range(n_chunks)] + [self.batch]
        self.chunks = [(a, b) for a, b in zip(edges[:-1], edges[1:]) if b > a]
        self.rows_per_img = int(rows_per_img)
        # the finest grid is the last scale (reference order: coarse first, yolov4/__init__.py:518-528)
        fine = self.params[-1]
        self.fine_grid = (fine.grid_h, fine.grid_w)
        for l, p in enumerate(self.params):
            sh = self.n_scales - 1 - l
            if (p.grid_h << sh, p.grid_w << sh) != self.fine_grid:
                raise ValueError("scales must halve from the last (finest) grid, coarse first")
        dev = self.dev
        with torch.cuda.device(dev):
            self.copy_stream = torch.cuda.Stream(dev)
            self.compute_stream = torch.cuda.Stream(dev)
            f32 = torch.float32
            self.y_pred = [torch.empty((self.batch, p.grid_h, p.grid_w, engine.floats_per_cell(p)), dtype=f32,
                                       device=dev) for p in self.params]
            self.dpred = [torch.empty_like(t) for t in self.y_pred]
            self.y_true = [torch.empty((self.batch, p.grid_h, p.grid_w, 5 + self.C), dtype=f32, device=dev)
                           for p in self.params]
            max_boxes = int(max_boxes if max_boxes is not None else self.batch * self.max_boxes_per_img)
            self.boxes = torch.empty((max(max_boxes, 1), 5), dtype=torch.float64, device=dev)
            self.box_offsets = torch.zeros(self.batch + 1, dtype=torch.int64, device=dev)
            self.n_bad = torch.zeros(1, dtype=torch.int64, device=dev)
            most = max(b - a for a, b in self.chunks)
            cap = self.rows_per_img * most
            self.row_cap = cap
            self.rows = torch.empty((cap, 7), dtype=torch.float64, device=dev)          # decode rows of one chunk
            self.row_offsets = torch.empty(most + 1, dtype=torch.int64, device=dev)
            self.keep = torch.empty(cap, dtype=torch.uint8, device=dev)
            lws = N.lib.yb_loss_workspace_bytes(self.n_scales)
            self.dparams = engine.loss_decode_params(self.params, self.thr)
            dws = N.lib.yb_decode_workspace_bytes(C.byref(self.dparams), most)
            nws = N.lib.yb_nms_workspace_bytes(cap, most, self.C)
            fws = N.lib.yb_decode_nms_workspace_bytes(C.byref(self.dparams), most, self.rows_per_img)
            if fws == 0:
                raise ValueError(f"rows_per_img must be in [32, {N.YB_FUSED_MAX_ROWS}] and class_num <= 256")
            self.ws = [torch.empty(int(b) + 256, dtype=torch.uint8, device=dev) for b in (lws, dws, nws, fws)]
            self.ws_bytes = (lws, dws, nws, fws)
        # results, written by the kernels into mapped pinned host memory
        nc = len(self.chunks)
        self.loss_host = torch.zeros((nc, self.n_scales), dtype=torch.float32).pin_memory()
        self.out_offsets_host = torch.zeros((nc, most + 1), dtype=torch.int64).pin_memory()
        self.out_rows_host = torch.zeros((nc, cap, 7), dtype=torch.float64).pin_memory()
        self.n_bad_host = torch.zeros(1, dtype=torch.int64).pin_memory()
        self.overflow_host = torch.zeros(nc, dtype=torch.int32).pin_memory()  # images over rows_per_img, per chunk
        self._calls = [self._bind_chunk(ci, a, b) for ci, (a, b) in enumerate(self.chunks)]
        self.launches_per_step = 3 * nc   # encode, loss + count, decode + NMS

    # -- argument binding (once) ---------------------------------------------------------------
    @staticmethod
    def _al(t):
        return t.data_ptr() + ((-t.data_ptr()) % 256)

    def _bind_chunk(self, ci, a, b):
        scales, _, n = engine.bind_loss_scales(self.params, self.y_true, self.y_pred, self.global_batch, self.dpred,
                                               images=(a, b))
        label_ptrs = (C.c_void_p * self.n_scales)(*[scales[s].y_true for s in range(self.n_scales)])
        vp = C.c_void_p
        lws, dws, nws, fws = (vp(self._al(w)) for w in self.ws)
        pred_ptrs = (C.c_void_p * self.n_scales)(*[scales[s].y_pred for s in range(self.n_scales)])
        return dict(
            n=n, scales=scales, label_ptrs=label_ptrs, lws=lws, dws=dws, nws=nws, fws=fws, pred_ptrs=pred_ptrs,
            overflow=vp(_mapped(self.overflow_host) + 4 * ci),
            offs=vp(self.box_offsets.data_ptr() + 8 * a),
            loss=vp(_mapped(self.loss_host) + 4 * self.n_scales * ci),
            out_offsets=vp(_mapped(self.out_offsets_host) + 8 * self.out_offsets_host.shape[1] * ci),
            out_rows=vp(_mapped(self.out_rows_host) + 56 * self.row_cap * ci))

    # -- one step ----------------------------------------------------------------------------------
    def run(self, host_preds, host_boxes, host_box_offsets):
        """host_preds: per scale a pinned (batch, gh, gw, info) float32 tensor; host_boxes: pinned
        (n_boxes, 5) float64 [x1, y1, x2, y2, class] in pixels; host_box_offsets: pinned (batch+1,)
        int64.  Returns dict(loss (n_scales,) float32 ndarray, dpred (device tensors), rows: list
        of per-chunk (rows ndarray view (k,7), offsets ndarray view) in image order, n_rows)."""
        lib, vp = N.lib, C.c_void_p
        cs, ks = self.copy_stream, self.compute_stream
        nb = host_boxes.shape[0]
        if nb > self.boxes.shape[0]:
            raise ValueError("more boxes than the step was sized for (max_boxes)")
        with torch.cuda.device(self.dev):
            cs.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(cs):
                self.boxes[:nb].copy_(host_boxes, non_blocking=True)
                self.box_offsets.copy_(host_box_offsets, non_blocking=True)
                events = []
                for (a, b) in self.chunks:
                    for s in range(self.n_scales):
                        self.y_pred[s][a:b].copy_(host_preds[s][a:b], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(cs)
                    events.append(ev)
            k = vp(ks.cuda_stream)
            lws_b, dws_b, nws_b, fws_b = self.ws_bytes
            boxes_p = vp(self.boxes.data_ptr())
            gh, gw = self.fine_grid
            for call, ev in zip(self._calls, events):
                ks.wait_event(ev)
                n = call["n"]
                N.check(lib.yb_encode_labels(boxes_p, call["offs"], n, self.max_boxes_per_img, self.img_size[0],
                                             self.img_size[1], gh, gw, self.C, self.n_scales, call["label_ptrs"], 0,
                                             vp(self.n_bad.data_ptr()), k), "yb_encode_labels")
                N.check(lib.yb_loss_decode_nms_fused(call["scales"], self.n_scales, call["loss"], None, self.thr,
                                                     self.nms_thr, self.nms_mode, self.rows_per_img, call["out_rows"],
                                                     self.row_cap, call["out_offsets"], call["overflow"],
                                                     call["lws"], lws_b, call["fws"], fws_b, k),
                        "yb_loss_decode_nms_fused")
            with torch.cuda.stream(ks):
                self.n_bad_host.copy_(self.n_bad, non_blocking=True)
            ks.synchronize()                                   # the ONE host sync of the step
            for ci, call in enumerate(self._calls):
                if int(self.overflow_host[ci]):                # an image beyond rows_per_img: general chain
                    self._redo_chunk(call, k)
        if int(self.n_bad_host[0]):
            raise IndexError(f"{int(self.n_bad_host[0])} boxes the reference's label encoder raises on")
        loss = self.loss_host.numpy().sum(axis=0, dtype=np.float32)
        offs = self.out_offsets_host.numpy()
        rows = self.out_rows_host.numpy()
        out, total = [], 0
        for ci, (a, b) in enumerate(self.chunks):
            o = offs[ci, :b - a + 1]
            out.append((rows[ci, :o[-1]], o))
            total += int(o[-1])
        return dict(loss=loss, dpred=self.dpred, rows=out, n_rows=total)

    def _redo_chunk(self, call, k):
        """Decode + NMS of one chunk with the general chain (any number of rows per image)."""
        lib, vp = N.lib, C.c_void_p
        n = call["n"]
        cap = self.row_cap
        while True:
            rows = torch.empty((cap, 7), dtype=torch.float64, device=self.dev)
            roff = torch.empty(n + 1, dtype=torch.int64, device=self.dev)
            keep = torch.empty(cap, dtype=torch.uint8, device=self.dev)
            N.check(lib.yb_decode(call["pred_ptrs"], n, C.byref(self.dparams), vp(rows.data_ptr()), cap,
                                  vp(roff.data_ptr()), call["dws"], self.ws_bytes[1], k), "yb_decode")
            self.compute_stream.synchronize()
            total = int(roff[-1].item())
            if total <= cap:
                break
            cap = total
        if total > self.row_cap:
            raise N.YoloB200Error("more survivors than the host result buffer holds; raise rows_per_img")
        nws_bytes = N.lib.yb_nms_workspace_bytes(cap, n, self.C)
        nws = torch.empty(int(nws_bytes) + 256, dtype=torch.uint8, device=self.dev)
        N.check(lib.yb_nms(vp(rows.data_ptr()), vp(roff.data_ptr()), cap, n, self.C, self.nms_thr, self.nms_mode,
                           vp(keep.data_ptr()), call["out_rows"], call["out_offsets"], None, vp(self._al(nws)),
                           nws_bytes, k), "yb_nms")
        self.compute_stream.synchronize()

    def d2h_bytes(self, n_rows):
        """Bytes the kernels wrote into host memory for a step with ``n_rows`` survivors."""
        return (4 * self.loss_host.numel() + 8 * sum(b - a + 1 for a, b in self.chunks) + 56 * n_rows + 8 +
                4 * len(self.chunks))
