#!/usr/bin/env python
"""The two-launch train-and-evaluate step on raw-logit heads against what the other heads cost.

    python benchmarks/logits_step.py --out DIR [--rounds 7] [--round-s 0.5] [--warmup 5]

Workload: YOLOv4-608, 3 scales (19/38/76) x 3 anchors, 80 classes, batch 128, decode at 0.5,
per-class DIoU-NMS at 0.45 - bench.py's step.  The raw heads are the synthetic heads of
synth.make_config through the inverse head transform (logit of x, y, objectness and class scores,
log(w / anchor)).  The heads alone are ~1 GB, far beyond the 126 MB L2, so every step reads them
from HBM.  Arms, all in this process, one round of each in turn:

  (a) activated : engine.TrainEvalStep on activated heads, graph replay (bench.py's timed step)
  (b) logits    : engine.TrainEvalStep on raw heads (from-logits params), graph replay
  (c) unfused   : what raw heads needed before the step took them: the from-logits loss
                  (yb_loss_fwd_bwd), the head transform in torch ops (sigmoid, anchor * exp - what
                  tf_ops.head.activate_head does in TensorFlow), then decode_nms_batch
  (d) loss only : the from-logits loss kernel alone (yb_loss_fwd_bwd): (b) - (d) is the share of the
                  counting pass and the per-image decode + NMS kernel

Every round is timed with CUDA events and lasts at least --round-s seconds; the reported time per
step is the median round.  Writes DIR/logits_step.json with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BATCH, CONF_THR, NMS_THR, NMS_MODE, ROWS_PER_IMG = 128, 0.5, 0.45, 2, 1024


def card():
    import torch
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power, sm_clock = [s.strip() for s in out.stdout.strip().split(",")]
    except Exception as e:  # the number is still labelled with the card's name
        power, sm_clock = f"unavailable ({e.__class__.__name__})", "unavailable"
    return dict(name=name, power_limit=power, max_sm_clock=sm_clock)


def to_raw(act, anchors):
    """Inverse head transform on the device, in float64: act (N, S, S, B*(5+C)) activated fp32."""
    import torch
    B = anchors.shape[0]
    a = act.double().reshape(act.shape[0], -1, B, act.shape[-1] // B)
    raw = torch.log(a / (1 - a))
    raw[..., 2:4] = torch.log(a[..., 2:4] / anchors.double())
    return raw.float().reshape(act.shape).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for logits_step.json")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--round-s", type=float, default=0.5)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()

    import torch
    from tf2_yolo_b200 import engine, synth
    from tf2_yolo_b200.grid_loss import wrap_yolo_loss_from_logits
    from tf2_yolo_b200.yolov4.losses import wrap_yolo_loss
    if not torch.cuda.is_available():
        raise SystemExit("logits_step.py needs a CUDA device")
    dev = torch.device("cuda")

    cfg = synth.make_config("v4-608", batch=BATCH, seed=2)
    B, C = cfg["bbox_num"], cfg["class_num"]
    kw = [dict(anchors=cfg["anchors"][si * B:(si + 1) * B], loss_weight=[1, 5, 1], wh_reg_weight=0.01,
               ignore_thresh=0.6) for si in range(len(cfg["grids"]))]
    p_act = [wrap_yolo_loss((S, S), B, C, **k).params for S, k in zip(cfg["grids"], kw)]
    p_raw = [wrap_yolo_loss_from_logits(4, (S, S), B, C, **k).params for S, k in zip(cfg["grids"], kw)]
    anchors = [torch.tensor(np.asarray(k["anchors"], dtype=np.float32), device=dev) for k in kw]
    yts = [torch.from_numpy(a).to(dev) for a in cfg["y_trues"]]
    acts = [torch.from_numpy(a).to(dev) for a in cfg["y_preds"]]
    raws = [to_raw(a, anc) for a, anc in zip(acts, anchors)]
    del cfg
    dpreds = [torch.empty_like(a) for a in acts]
    head_bytes = sum(a.numel() * 4 for a in acts)

    step_a = engine.TrainEvalStep(p_act, yts, acts, CONF_THR, NMS_THR, NMS_MODE, rows_per_img_cap=ROWS_PER_IMG,
                                  dpreds=dpreds)
    step_b = engine.TrainEvalStep(p_raw, yts, raws, CONF_THR, NMS_THR, NMS_MODE, rows_per_img_cap=ROWS_PER_IMG,
                                  dpreds=dpreds)
    scratch = [torch.empty_like(a) for a in raws]
    out_c = dict(out_rows=torch.empty((ROWS_PER_IMG * BATCH, 7), dtype=torch.float64, device=dev),
                 out_offsets=torch.empty(BATCH + 1, dtype=torch.int64, device=dev),
                 n_overflow=torch.zeros(1, dtype=torch.int32, device=dev))

    def unfused():
        engine.loss_fwd_bwd(p_raw, yts, raws, dpreds=dpreds)
        for r, o, anc in zip(raws, scratch, anchors):
            torch.sigmoid(r, out=o)
            ov = o.view(o.shape[0], -1, B, 5 + C)
            ov[..., 2:4] = anc * torch.exp(r.view(ov.shape)[..., 2:4])
        return engine.decode_nms_batch(scratch, C, CONF_THR, 4, NMS_THR, NMS_MODE, rows_per_img_cap=ROWS_PER_IMG,
                                       out=out_c)

    arms = {
        "a_activated_step": lambda: step_a.run(),
        "b_logits_step": lambda: step_b.run(),
        "c_logits_loss_torch_activation_decode_nms": unfused,
        "d_logits_loss_kernel": lambda: engine.loss_fwd_bwd(p_raw, yts, raws, dpreds=dpreds),
    }

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3

    steps = {}
    for name, fn in arms.items():       # warm-up, then the steps one round of --round-s needs
        timed(fn, args.warmup)
        t = timed(fn, 20) / 20
        steps[name] = max(20, int(np.ceil(args.round_s / t)))
    rounds = {name: [] for name in arms}
    t0 = time.time()
    for _ in range(args.rounds):
        for name, fn in arms.items():
            rounds[name].append(timed(fn, steps[name]) / steps[name] * 1e3)
    wall = time.time() - t0

    # outputs of the last steps: survivors per arm (a and b: the same synthetic heads, two head kinds)
    def n_rows(r):
        return int(r["out_offsets"][-1].item()), int(r["n_overflow"].item())
    a_rows, a_ovf = n_rows(step_a.run()[3])
    b_rows, b_ovf = n_rows(step_b.run()[3])
    c_rows, c_ovf = n_rows(unfused())
    b_res = step_b.run()[3]
    c_res = unfused()
    same_bc = bool(b_rows == c_rows and torch.equal(b_res["out_rows"][:b_rows], c_res["out_rows"][:c_rows]))

    ms = {k: float(np.median(v)) for k, v in rounds.items()}
    result = dict(
        benchmark="logits_step",
        workload=f"YOLOv4-608, 3 scales (19/38/76) x 3 anchors, 80 classes, batch {BATCH}; loss fwd+grad + decode "
                 f"(thr {CONF_THR}) + per-class DIoU-NMS ({NMS_THR}); synthetic heads, raw = inverse head transform",
        gpu=card(), torch=torch.__version__, cuda=torch.version.cuda,
        head_bytes=head_bytes, rounds=args.rounds, steps_per_round=steps,
        ms_per_step_median=ms, ms_per_step_rounds=rounds,
        logits_over_activated=ms["b_logits_step"] / ms["a_activated_step"],
        logits_over_unfused=ms["b_logits_step"] / ms["c_logits_loss_torch_activation_decode_nms"],
        survivors=dict(a=a_rows, b=b_rows, c=c_rows), n_overflow=dict(a=a_ovf, b=b_ovf, c=c_ovf),
        b_equals_c_survivors=same_bc, timed_wall_s=wall)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "logits_step.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
