#!/usr/bin/env python
"""Benchmark of the anchor-grid hot path on the BASELINE.json headline config.

    python bench.py --gpus N --steps K --warmup W          # this repo (CUDA)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm

Workload (one "step"): YOLOv4-608, 3 FPN scales x 3 anchors, 80 classes, batch 128
per GPU of synthetic head outputs + labels:
    fused CIoU loss forward+gradient (all scales, one launch)
    -> decode at joint-confidence 0.5 -> per-class DIoU-NMS at 0.45.
`value`  : images/s over exactly --steps steps, inputs resident in HBM, timed with CUDA events (max
           over ranks); the step is two launches over static buffers replayed from a CUDA graph
           (--no-graph: eager).
`--dump-outputs DIR`: after the timed steps, what the last one returned (see dump_outputs) as
           DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output.
`e2e`    : same step through the reference-facing Python API with HOST buffers
           (pinned H2D of labels + head outputs inside the timed region, D2H of the
           loss scalars and the NMS survivors; the gradient stays on the device for
           the backbone's backward pass, as in the reference's train step).
`roofline`: the loss kernel (dominant) - algorithmic bytes / its CUDA-event time.
`cpu_baseline` / `--impl reference`: the oracle port of the reference's path
           (torch-CPU fp32 loss fwd+bwd on all host threads; NumPy decode/NMS) on a
           bounded sample of the same workload.  TensorFlow is not installable here.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec YOLOv4-608 loss+grad+decode+NMS"
UNIT = "images/s"
CONFIG_NAME = "v4-608"
IMG_SIZE = (608, 608)
DUMP_SAMPLE = 1 << 21                # gradient elements per scale that --dump-outputs keeps (8 MB each)
# both arms print this string (the driver compares the arms' configs)
WORKLOAD = ("YOLOv4-608 (BASELINE configs[2]): 3 scales (19/38/76) x 3 anchors, 80 classes, batch 128 per GPU; "
            "CIoU loss fwd+grad + decode(thr 0.5) + per-class DIoU-NMS(thr 0.45)")
CONF_THR, NMS_THR, NMS_MODE = 0.5, 0.45, 2
ROW_CAPACITY_PER_IMG = 4096          # decode rows per image, general chain (--chain / --unfused)
ROWS_PER_IMG_FUSED = 1024            # rows per image the one-CTA-per-image decode + NMS holds in shared memory
# my kernels per step: loss fwd+grad with the decode counting pass | decode + NMS, one CTA per image
#   --chain : loss + count 1 | decode: look-back scan, emit | nms: classify, scatter, sweep, emit
#   --unfused: one more (separate decode counting pass)
LAUNCHES_PER_STEP = {"fused": 2, "chain": 7, "unfused": 8}


def loss_algorithmic_bytes(cfg, batch):
    B, ch = cfg["bbox_num"], 5 + cfg["class_num"]
    return sum(4 * batch * s * s * (2 * B * ch + ch) for s in cfg["grids"])


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def profiled_traffic():
    p = os.path.join(ROOT, "profiles", "loss_kernel_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch")
        except Exception:
            return None
    return None


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)     # the sampler never outlives the benchmark, however it ends
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def wait_first_sample(self, keep_busy, timeout=5.0):
        """Run `keep_busy()` (untimed work) until nvidia-smi has delivered its first line."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t0 < timeout:
            keep_busy()

    def stop(self, t_begin=None, t_end=None):
        """Summary of the samples that arrived inside [t_begin, t_end] (host clock), i.e. under load."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, power = [], None, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lines = [ln for t, ln in self.lines if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end)]
        if not lines:   # region shorter than one sampling period: the nearest sample
            lines = [ln for _, ln in self.lines[-1:]]
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(sm),
                "power_w_median": float(np.median(power)) if power else None}


# ---------------------------------------------------------------------------
# CPU arm: oracle port of the reference path
# ---------------------------------------------------------------------------
def cpu_step(cfg, y_trues, y_preds, n_threads):
    """loss fwd+bwd (torch-CPU fp32, all threads) + decode + DIoU-NMS (NumPy) on the given images."""
    import torch
    from oracle import losses as ol
    from oracle import tools as ot
    B, C = cfg["bbox_num"], cfg["class_num"]
    torch.set_num_threads(n_threads)
    for si, S in enumerate(cfg["grids"]):
        spec = ol.GridLossSpec(version=4, grid_shape=(S, S), bbox_num=B, class_num=C,
                               anchors=cfg["anchors"][si * B:(si + 1) * B], loss_weight=[1, 5, 1])
        ol.loss_and_grad(spec, y_trues[si], y_preds[si], dtype=torch.float32)
    for i in range(y_preds[0].shape[0]):
        rows = ot.decode(*[p[i] for p in y_preds], class_num=C, threshold=CONF_THR, version=4)
        if len(rows):
            ot.nms(rows, C, NMS_THR, NMS_MODE)


def cpu_baseline(cfg, budget_s=12.0):
    from tf2_yolo_b200 import synth
    cores = os.cpu_count() or 1
    small = synth.make_config(CONFIG_NAME, batch=4, seed=2, rank=999)
    yt, yp = small["y_trues"], small["y_preds"]
    cpu_step(small, [a[:1] for a in yt], [a[:1] for a in yp], cores)      # warm
    t0 = time.perf_counter()
    n = 0
    while True:
        cpu_step(small, yt, yp, cores)
        n += 4
        if time.perf_counter() - t0 > budget_s or n >= 4096:
            break
    dt = time.perf_counter() - t0
    return {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} images of the v4-608 workload in batches of 4 ({dt:.1f} s): oracle port of the "
                      "reference path - loss fwd+bwd on torch-CPU fp32 (all threads), decode + DIoU-NMS in NumPy; "
                      "TensorFlow not installable"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tf2_yolo_b200 import synth
    cores = os.cpu_count() or 1
    probe = synth.make_config(CONFIG_NAME, batch=1, seed=2, rank=998)
    cpu_step(probe, probe["y_trues"], probe["y_preds"], cores)
    t0 = time.perf_counter()
    cpu_step(probe, probe["y_trues"], probe["y_preds"], cores)
    t_img = max(time.perf_counter() - t0, 1e-3)
    per_step = int(max(1, min(128, 150.0 / ((args.steps + args.warmup) * t_img))))
    cfg = synth.make_config(CONFIG_NAME, batch=per_step, seed=2, rank=0)
    for _ in range(args.warmup):
        cpu_step(cfg, cfg["y_trues"], cfg["y_preds"], cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_step(cfg, cfg["y_trues"], cfg["y_preds"], cores)
    dt = time.perf_counter() - t0
    value = per_step * args.steps / dt
    sample = (f"{per_step} images/step of the v4-608 workload, oracle port of the reference path "
              f"(torch-CPU fp32 loss fwd+bwd on {cores} threads; NumPy decode + DIoU-NMS); TensorFlow not installable")
    emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "images_per_step": per_step,
                   "sample": "the CPU arm processes a bounded sample of the workload per step"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------
def h2d_ceiling(host_tensors, dev_tensors, barrier, reps=4):
    """Plain pinned cudaMemcpyAsync of the step's head outputs, nothing else on the GPU, every rank
    at once: the fabric's ceiling for the e2e step (GB/s per GPU, slowest rank decides)."""
    import torch
    nbytes = sum(t.numel() * t.element_size() for t in host_tensors)
    for d, h in zip(dev_tensors, host_tensors):
        d.copy_(h, non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for d, h in zip(dev_tensors, host_tensors):
            d.copy_(h, non_blocking=True)
    e1.record()
    barrier()
    return nbytes * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9


def dump_outputs(out_dir, loss, dpreds, res):
    """Write what one step returned to its caller as out_dir/<name>.npy (at most 33 MB in all):
    loss.npy          float32 [n_scales], the loss per scale
    dpred<s>.npy      float32, DUMP_SAMPLE elements of scale s's gradient at the flat indices
                      np.sort(np.random.default_rng(s).choice(numel, DUMP_SAMPLE, replace=False))
    out_rows.npy      float64 [kept, 7], the NMS survivors of all images
    out_offsets.npy   float64 [n_img + 1], where each image's survivors start in out_rows"""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n_kept = int(res["out_offsets"][-1].item())
    arrays = {"loss": loss.cpu().numpy().astype(np.float32),
              "out_rows": res["out_rows"][:n_kept].cpu().numpy().astype(np.float64),
              "out_offsets": res["out_offsets"].cpu().numpy().astype(np.float64)}
    for si, d in enumerate(dpreds):
        flat = d.reshape(-1)
        idx = np.random.default_rng(si).choice(flat.numel(), min(DUMP_SAMPLE, flat.numel()), replace=False)
        arrays[f"dpred{si}"] = flat[torch.from_numpy(np.sort(idx)).to(flat.device)].cpu().numpy().astype(np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from tf2_yolo_b200 import engine, synth
    from tf2_yolo_b200.grid_loss import fused_losses
    from tf2_yolo_b200.pipeline import HostBatchStep
    from tf2_yolo_b200.yolov4.losses import wrap_yolo_loss

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    strong = args.scaling == "strong"
    if strong and args.batch % world:
        raise SystemExit("--scaling strong needs a batch divisible by the number of GPUs")
    batch = args.batch // world if strong else args.batch     # images on this GPU
    global_batch = batch * world
    cfg = synth.make_config(CONFIG_NAME, batch=batch, seed=2, rank=rank)
    B, C = cfg["bbox_num"], cfg["class_num"]
    fns = [wrap_yolo_loss((S, S), B, C, anchors=cfg["anchors"][si * B:(si + 1) * B], loss_weight=[1, 5, 1],
                          wh_reg_weight=0.01, ignore_thresh=0.6)
           for si, S in enumerate(cfg["grids"])]
    params = [f.params for f in fns]
    # the labels as the reference's reader holds them: box lists in pixels of the 608x608 image
    boxes_np, offs_np = synth.boxes_from_labels(cfg["y_trues"][-1], IMG_SIZE)
    host_boxes = torch.from_numpy(boxes_np).pin_memory()
    host_offs = torch.from_numpy(offs_np).pin_memory()
    max_per_img = int(np.diff(offs_np).max())
    host_p = [torch.from_numpy(a).pin_memory() for a in cfg["y_preds"]]
    dev_p = [a.to(dev) for a in host_p]
    # device-resident labels = the same box lists through yb_encode_labels (coarse grid first)
    dev_t, n_bad = engine.encode_labels(host_boxes.to(dev), host_offs.to(dev), IMG_SIZE, (cfg["grids"][-1],) * 2, C,
                                        n_levels=len(cfg["grids"]), max_boxes_per_img=max_per_img)
    assert int(n_bad.item()) == 0
    dpreds = [torch.empty_like(a) for a in dev_p]
    cap = ROW_CAPACITY_PER_IMG * batch
    rows = torch.empty((cap, 7), dtype=torch.float64, device=dev)
    loss_ev = []

    mode = "unfused" if args.unfused else ("chain" if args.chain else "fused")
    step_loss = [torch.empty(3, dtype=torch.float32, device=dev) for _ in range(2)]   # double-buffered
    in_flight = [None, None]     # the asynchronous loss all-reduce of each buffer
    step_no = [0]

    def join_collectives():      # every rank's loss scalars are global after this
        for pending in (in_flight, static_pending):
            for i in range(2):
                if pending[i] is not None:
                    pending[i].wait()
                    pending[i] = None
    fused_out = dict(out_rows=torch.empty((ROWS_PER_IMG_FUSED * batch, 7), dtype=torch.float64, device=dev),
                     out_offsets=torch.empty(batch + 1, dtype=torch.int64, device=dev),
                     n_overflow=torch.zeros(1, dtype=torch.int32, device=dev))

    def step(y_t, y_p, record=False):
        slot = step_no[0] & 1
        step_no[0] += 1
        if mode == "fused" and in_flight[slot] is not None:   # the all-reduce that last used this loss buffer
            in_flight[slot].wait()                            # (two steps ago)
            in_flight[slot] = None
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        if mode == "fused":   # two launches: loss + counting pass, then decode + NMS with one CTA per image

            def after_loss():   # between the two launches: the loss scalars are final
                if record:
                    e1.record()
                    loss_ev.append((e0, e1))
                if world > 1:   # the only collective (3 scalars): runs beside the decode + NMS kernel and
                    # the next step's loss kernel; it is joined when its buffer comes round again
                    in_flight[slot] = dist.all_reduce(step_loss[slot], async_op=True)
            loss, _, _, res = engine.loss_decode_nms_fused(params, y_t, y_p, CONF_THR, NMS_THR, NMS_MODE,
                                                           rows_per_img_cap=ROWS_PER_IMG_FUSED,
                                                           global_batch=global_batch, dpreds=dpreds, out=fused_out,
                                                           split_hook=after_loss, loss_out=step_loss[slot])
            return loss, None, res
        if args.unfused:
            loss, _, _ = fused_losses(fns, y_t, y_p, global_batch=global_batch, dpreds=dpreds)
        else:   # loss fwd+grad and the decode counting pass share one read of y_pred
            def mark():
                if record:
                    e1.record()
                    loss_ev.append((e0, e1))
            loss, _, _, _, offs = engine.loss_decode_fused(params, y_t, y_p, CONF_THR, global_batch=global_batch,
                                                           dpreds=dpreds, rows=rows, split_hook=mark)
        if record and args.unfused:
            e1.record()
            loss_ev.append((e0, e1))
        work = dist.all_reduce(loss, async_op=True) if world > 1 else None   # the only collective: 3 scalars
        if args.unfused:
            _, offs = engine.decode_batch(y_p, C, CONF_THR, 4, rows=rows)
        res = engine.nms_batch(rows, offs, C, NMS_THR, NMS_MODE)
        if work is not None:
            work.wait()                       # NCCL ran beside decode/NMS; join it to this stream
        return loss, offs, res

    # The timed step of the default mode: the same two launches over static buffers, replayed from a
    # CUDA graph (engine.TrainEvalStep, workspaces zeroed once - no memsets).  For N > 1 two such
    # graphs alternate, each with its own loss scalars: their all-reduce (the only collective) is
    # issued asynchronously after the replay and joined when that graph comes round again.
    # --no-graph times the eager calls.
    static_steps = None
    if mode == "fused" and not args.no_graph:
        static_steps = [engine.TrainEvalStep(params, dev_t, dev_p, CONF_THR, NMS_THR, NMS_MODE,
                                             rows_per_img_cap=ROWS_PER_IMG_FUSED, global_batch=global_batch,
                                             dpreds=dpreds, graph=True) for _ in range(1 if world == 1 else 2)]
    static_pending = [None, None]

    def static_step(k):
        i = k % len(static_steps)
        if static_pending[i] is not None:
            static_pending[i].wait()
            static_pending[i] = None
        res = static_steps[i].run()
        if world > 1:
            static_pending[i] = dist.all_reduce(static_steps[i].loss, async_op=True)
        return res

    def barrier():
        join_collectives()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def agree(x, op):   # one number every rank uses
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=op)
        return float(t.item())

    # ---- device-resident timing ---------------------------------------------------
    for _ in range(args.warmup):
        out = step(dev_t, dev_p)
    barrier()
    if mode == "fused":
        if int(out[2]["n_overflow"].item()):
            raise SystemExit("an image exceeds ROWS_PER_IMG_FUSED decode rows: run with --chain")
        # untimed: the general six-launch chain must give the same survivors, bit for bit
        rows_c, offs_c = engine.decode_batch_exact(dev_p, C, CONF_THR, 4)
        total_rows = int(offs_c[-1].item())
        chain = engine.nms_batch(rows_c, offs_c, C, NMS_THR, NMS_MODE)
        n_c = int(chain["out_offsets"][-1].item())
        if not (torch.equal(chain["out_offsets"], out[2]["out_offsets"]) and
                torch.equal(chain["out_rows"][:n_c], out[2]["out_rows"][:n_c])):
            raise SystemExit("one-CTA-per-image decode+NMS differs from the general chain")
    else:
        total_rows = int(out[1][-1].item())
        if total_rows > cap:
            raise SystemExit(f"decode produced {total_rows} rows > capacity {cap}")
    kept_rows = int(out[2]["out_offsets"][-1].item())
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        # untimed local work (no collective) until nvidia-smi delivers its first line
        clocks.wait_first_sample(lambda: (fused_losses(fns, dev_t, dev_p, global_batch=global_batch, dpreds=dpreds),
                                          torch.cuda.synchronize()))
    barrier()
    # the timed region: exactly `steps` steps (every rank runs the same number)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = time.perf_counter()
    ev0.record()
    if static_steps is not None:
        for k in range(args.steps):
            g_out = static_step(k)
        out = (g_out[0], None, g_out[3])
    else:
        for _ in range(args.steps):
            out = step(dev_t, dev_p, record=True)
    join_collectives()              # the timed steps end when every step's collective has completed
    ev1.record()
    barrier()
    ms = agree(ev0.elapsed_time(ev1), dist.ReduceOp.MAX if world > 1 else None) / args.steps
    if args.dump_outputs and rank == 0:     # before anything else writes the gradient buffers
        dump_outputs(args.dump_outputs, out[0], dpreds, out[2])
    eager_rounds = 0
    if static_steps is not None:
        # the loss kernel alone cannot be bracketed inside a graph: after the timed steps the same
        # step runs as two eager launches with an event between them (not counted in ms)
        for _ in range(args.steps):
            eager_out = step(dev_t, dev_p, record=True)
        barrier()                       # its events are read next
        eager_rounds = 1
    loss_ms = float(np.median([a.elapsed_time(b) for a, b in loss_ev]))
    loss_vals = out[0].cpu().numpy().tolist()
    if static_steps is not None:   # the replayed step returns what the eager step returned
        barrier()
        if not torch.equal(out[0], eager_out[0]):
            raise SystemExit("graph replay: loss differs from the eager step's")
        if not (torch.equal(out[2]["out_offsets"], eager_out[2]["out_offsets"]) and
                torch.equal(out[2]["out_rows"][:kept_rows], eager_out[2]["out_rows"][:kept_rows])) or \
                int(out[2]["n_overflow"].item()):
            raise SystemExit("graph replay: survivors differ from the eager step's")

    # ---- end to end through the host-buffer API -----------------------------------
    pipe = HostBatchStep(fns, IMG_SIZE, batch, CONF_THR, NMS_THR, NMS_MODE, n_chunks=args.chunks,
                         rows_per_img=ROWS_PER_IMG_FUSED, max_boxes_per_img=max_per_img,
                         max_boxes=boxes_np.shape[0], global_batch=global_batch)
    h2d = sum(a.numel() * 4 for a in host_p) + boxes_np.nbytes + offs_np.nbytes
    res = None
    for _ in range(max(1, min(args.warmup, 3))):
        res = pipe.run(host_p, host_boxes, host_offs)
    # untimed check: the pipelined host-buffer step returns what the device-resident step computes
    loss_e2e = torch.tensor(res["loss"], device=dev)
    if world > 1:
        dist.all_reduce(loss_e2e)
    if not np.allclose(loss_e2e.cpu().numpy(), np.asarray(loss_vals), rtol=2e-6):
        raise SystemExit(f"e2e loss {loss_e2e.tolist()} != device-resident loss {loss_vals}")
    if res["n_rows"] != kept_rows:
        raise SystemExit(f"e2e survivors {res['n_rows']} != device-resident survivors {kept_rows}")
    kept_ref = out[2]["out_rows"][:kept_rows].cpu().numpy()
    if not np.array_equal(np.concatenate([r for r, _ in res["rows"]], axis=0), kept_ref):
        raise SystemExit("e2e survivors differ from the device-resident step's")
    barrier()
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        res = pipe.run(host_p, host_boxes, host_offs)
    ev1.record(pipe.compute_stream)
    barrier()
    e2e_wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    e2e_ms = agree(ev0.elapsed_time(ev1), dist.ReduceOp.MAX if world > 1 else None) / args.steps
    t_end = time.perf_counter()
    clock_info = clocks.stop(t_begin, t_end) if rank == 0 else None   # samples inside both timed regions
    ceiling = agree(h2d_ceiling(host_p, pipe.y_pred, barrier), dist.ReduceOp.MIN if world > 1 else None)

    if rank == 0:
        algo = loss_algorithmic_bytes(cfg, batch)
        peak, peak_src = peak_hbm()
        achieved = algo / (loss_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": global_batch / (ms * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": WORKLOAD,
                "per_gpu_batch": batch, "global_batch": global_batch,
                "fusion": {"fused": "2 launches per step (yb_loss_decode_nms_fused%s): loss fwd+grad with the decode "
                                    "counting pass riding on its read of y_pred, then decode + NMS with one CTA per "
                                    "image; roofline counts only the loss's algorithmic bytes"
                                    % ("_clean, replayed from a CUDA graph by engine.TrainEvalStep; the loss kernel's "
                                       "own duration is taken from the same steps run eagerly after the timed "
                                       "ones" if static_steps is not None else ""),
                           "chain": "7 launches per step: loss fwd+grad + decode counting pass (yb_loss_decode_fused), "
                                    "scan, emit, NMS classify / scatter / sweep / emit",
                           "unfused": "separate loss and decode launches"}[mode],
                "timing": f"{args.steps} steps (CUDA events, max over ranks)",
                "l2_policy": f"inputs larger than L2: {sum(a.numel() * 4 for a in dev_p + dev_t) / 1e6:.0f} MB read + "
                             f"{sum(d.numel() * 4 for d in dpreds) / 1e6:.0f} MB written per step vs 126 MB L2",
                "decode_rows_per_image": total_rows / batch, "nms_kept_per_image": kept_rows / batch,
                "loss_per_scale": loss_vals, "sharding": "batch split across ranks; all-reduce of 3 loss scalars",
                "precision_note": "loss/decode fp32 (objectness, class, box terms of responsible boxes in fp64), "
                                  "NMS fp64 bit-exact",
            },
            "clocks": clock_info,
            "e2e": {"value": global_batch / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": pipe.d2h_bytes(res["n_rows"]), "ms_per_step": e2e_ms,
                    "wall_ms_per_step": e2e_wall_ms,
                    "h2d_gbs": h2d / (e2e_ms * 1e-3) / 1e9, "h2d_ceiling_gbs": ceiling,
                    "frac_of_h2d_ceiling": (h2d / (e2e_ms * 1e-3) / 1e9) / ceiling,
                    "chunks": len(pipe.chunks), "steps": args.steps,
                    "note": "HostBatchStep: pinned head outputs + box lists in (labels encoded on the device), "
                            "loss scalars + NMS survivors written to mapped host memory; H2D of chunk k+1 under the "
                            "kernels of chunk k, one host sync per step; gradient stays on the device. "
                            "h2d_ceiling_gbs = the same head outputs copied with plain pinned cudaMemcpyAsync, "
                            "all ranks at once, nothing else running"},
            "gpu_launches": LAUNCHES_PER_STEP[mode] * args.steps * (1 + eager_rounds)
                            + pipe.launches_per_step * args.steps,
            "gpu_launches_per_step": LAUNCHES_PER_STEP[mode],
            "roofline": {"bound": "hbm",
                         "kernel": "loss_fwd_bwd_kernel<4,false,%s>" % ("false" if args.unfused else "true"),
                         "tail_ms_per_step": ms - loss_ms,
                         "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": profiled_traffic(),
                         "traffic_source": "ncu --set full capture of this kernel (profiles/loss_kernel_traffic.json)",
                         "algorithmic_bytes_per_launch": algo, "ms_per_launch": loss_ms, "peak_source": peak_src,
                         "kernel_share_of_step": loss_ms / ms,
                         "step_frac": algo / (ms * 1e-3) / 1e9 / peak},
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(cfg)
        emit(json.dumps(line))
    if world > 1:
        # nothing of the measurement is left to do: a stuck NCCL teardown must not hold the launcher
        import threading
        dog = threading.Timer(60.0, os._exit, (0,))
        dog.daemon = True
        dog.start()
        static_steps = None          # graphs go before the communicator
        torch.cuda.synchronize()
        dist.destroy_process_group()
        dog.cancel()


class _StdoutGuard:
    """Keep fd 1 clean for the ONE JSON line: native libraries (NCCL prints its version banner on
    stdout) write to stderr while the benchmark runs; emit() writes the line to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.write(self.real, (line + "\n").encode())


GUARD = None


def emit(line):
    if GUARD is not None:
        GUARD.emit(line)
    else:
        print(line)


def main():
    global GUARD
    GUARD = _StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=128, help="images per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the CUDA-graph replay")
    ap.add_argument("--unfused", action="store_true", help="separate loss and decode launches (y_pred read twice)")
    ap.add_argument("--chain", action="store_true",
                    help="decode and NMS as the general six-launch chain instead of the one-CTA-per-image kernel")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch images per GPU (default); strong: --batch images in total, split over the GPUs")
    ap.add_argument("--chunks", type=int, default=8, help="image chunks of the pipelined end-to-end step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA arm's outputs (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
