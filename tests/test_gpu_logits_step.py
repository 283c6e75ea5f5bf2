"""GPU: raw-logit heads in the two-launch train-and-evaluate step (yb_loss_decode_nms_fused with
from_logits) and the device-side head transform (yb_activate_head).  The step on raw heads must give
the loss and d/d(raw) of the from-logits loss, and the survivors of the chain (yb_decode + yb_nms) on
the heads yb_activate_head activates - bit for bit."""
import numpy as np
import pytest
import torch

from oracle import tools as ot
from tf2_yolo_b200 import _native as N
from tf2_yolo_b200 import engine, synth
from tf2_yolo_b200.grid_loss import fused_losses, wrap_yolo_loss_from_logits
from tf2_yolo_b200.pipeline import HostBatchStep

pytestmark = pytest.mark.gpu


def to_raw(act, anchors, B, C):
    """The inverse head transform of synthetic (activated) head outputs, as in test_gpu_loss.py."""
    a = act.astype(np.float64).reshape(-1, B, 5 + C)
    raw = a.copy()
    raw[..., 0:2] = np.log(a[..., 0:2] / (1 - a[..., 0:2]))
    raw[..., 4:] = np.log(a[..., 4:] / (1 - a[..., 4:]))
    raw[..., 2:4] = np.log(a[..., 2:4] / np.asarray(anchors, dtype=np.float64).reshape(B, 2)[None])
    return raw.reshape(act.shape).astype(np.float32)


def logits_config(name, batch, seed):
    cfg = synth.make_config(name, batch=batch, seed=seed)
    ver = int(name[1])
    B, C = cfg["bbox_num"], cfg["class_num"]
    anchors = [cfg["anchors"][si * B:(si + 1) * B] for si in range(len(cfg["grids"]))]
    fns = [wrap_yolo_loss_from_logits(ver, (S, S), B, C, anchors=anchors[si],
                                      loss_weight=[1, 5, 1] if ver == 4 else [1, 1, 5, 1])
           for si, S in enumerate(cfg["grids"])]
    raws = [to_raw(a, anchors[si], B, C) for si, a in enumerate(cfg["y_preds"])]
    return cfg, ver, fns, raws


def chain(preds, C, thr, version, nms_thr, mode):
    rows, offs = engine.decode_batch_exact(preds, C, thr, version)
    g = engine.nms_batch(rows, offs, C, nms_thr, mode)
    n = int(g["out_offsets"][-1].item())
    return g["out_rows"][:n].cpu().numpy(), g["out_offsets"].cpu().numpy()


def survivors(r):
    offs = r["out_offsets"].cpu().numpy()
    return r["out_rows"][:offs[-1]].cpu().numpy(), offs


def ulps(a, b):
    ia = a.view(np.int32).astype(np.int64)
    ib = b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7fffffff), ia)
    ib = np.where(ib < 0, -(ib & 0x7fffffff), ib)
    return np.abs(ia - ib)


# ---- yb_activate_head ------------------------------------------------------------------------------
def test_activate_head_is_the_float32_head_transform():
    rng = np.random.default_rng(1)
    for ver, B, C, n_img, S in ((4, 3, 80, 2, 19), (3, 3, 1, 3, 7), (3, 2, 33, 1, 5)):
        anc = rng.uniform(0.02, 0.6, (B, 2)).astype(np.float32)
        p = engine.make_loss_params(ver, (S, S), B, C, anchors=anc, from_logits=True)
        raw = rng.normal(0.0, 4.0, (n_img, S, S, B * (5 + C))).astype(np.float32)
        r = raw.reshape(-1, B, 5 + C).astype(np.float64)
        want = 1.0 / (1.0 + np.exp(-r))                  # the transform in float64, rounded once
        want[..., 2:4] = anc[None].astype(np.float64) * np.exp(r[..., 2:4])
        want = want.astype(np.float32)
        t = torch.from_numpy(raw).cuda()
        got = engine.activate_head(p, t).cpu().numpy().reshape(want.shape)
        # CUDA's expf is within 2 ulp; the sum, the quotient and the anchor product round once more each
        d = ulps(got, want)
        assert d.max() <= 4 and d.mean() < 0.5, (ver, C, int(d.max()), float(d.mean()))
        # in place: the same bits
        engine.activate_head(p, t, out=t)
        assert np.array_equal(t.cpu().numpy().reshape(want.shape), got)
        # unaligned tensors (scalar path) and a tail of fewer than 4 floats: the same bits
        flat = torch.from_numpy(raw).cuda().reshape(-1)
        off = torch.empty(flat.numel() + 1, device="cuda")[1:]
        off.copy_(flat)
        g2 = engine.activate_head(p, off).cpu().numpy().reshape(want.shape)
        assert np.array_equal(g2, got)


def test_activate_head_rejects_heads_it_does_not_define():
    t = torch.zeros((1, 4, 4, 3 * 9), device="cuda")
    p = engine.make_loss_params(3, (4, 4), 3, 4, anchors=np.full((3, 2), 0.1))
    p2 = N.LossParams.from_buffer_copy(p)
    p2.version = 2
    with pytest.raises(N.YoloB200Error):
        engine.activate_head(p2, t)
    p3 = N.LossParams.from_buffer_copy(p)
    p3.has_anchors = 0
    with pytest.raises(N.YoloB200Error):
        engine.activate_head(p3, t)


# ---- the step on raw heads -------------------------------------------------------------------------
@pytest.mark.parametrize("name,batch", [("v4-608", 6), ("v3-416", 9)])
@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("thr", [0.5, 0.3])
def test_step_on_raw_heads_equals_the_chain_on_activated_heads(name, batch, mode, thr):
    cfg, ver, fns, raws = logits_config(name, batch, 40 + batch)
    C = cfg["class_num"]
    params = [f.params for f in fns]
    yts = [torch.from_numpy(a).cuda() for a in cfg["y_trues"]]
    yps = [torch.from_numpy(a).cuda() for a in raws]
    acts = [engine.activate_head(p, t) for p, t in zip(params, yps)]
    loss0, d0, _ = fused_losses(fns, yts, yps)
    loss, d, _, r = engine.loss_decode_nms_fused(params, yts, yps, thr, 0.45, mode, rows_per_img_cap=2048)
    assert torch.equal(loss, loss0) and all(torch.equal(a, b) for a, b in zip(d, d0))
    assert int(r["n_overflow"].item()) == 0
    rows, offs = survivors(r)
    ref_rows, ref_offs = chain(acts, C, thr, ver, 0.45, mode)
    assert offs[-1] > 0
    assert np.array_equal(offs, ref_offs) and np.array_equal(rows, ref_rows)
    rows2, offs2 = survivors(engine.decode_nms_batch(acts, C, thr, ver, 0.45, mode, rows_per_img_cap=2048))
    assert np.array_equal(offs2, offs) and np.array_equal(rows2, rows)
    per = [a[0].cpu().numpy() for a in acts]
    o = ot.nms(ot.decode(*per, class_num=C, threshold=thr, version=ver).reshape(-1, 7), C, 0.45, mode)
    assert np.array_equal(rows[offs[0]:offs[1]], o)
    for _ in range(3):      # the same bits on every run
        loss3, d3, _, r3 = engine.loss_decode_nms_fused(params, yts, yps, thr, 0.45, mode, rows_per_img_cap=2048)
        rows3, offs3 = survivors(r3)
        assert torch.equal(loss3, loss0) and all(torch.equal(a, b) for a, b in zip(d3, d0))
        assert np.array_equal(offs3, offs) and np.array_equal(rows3, rows)


def edge_heads(C, rng, S=8, B=3, n_img=4):
    """Raw v3 heads around every corner of the logits counting pass.  Image 3 has no candidates."""
    raw = np.zeros((n_img, S, S, B, 5 + C), dtype=np.float32)
    raw[..., 0:2] = rng.normal(0, 2, (n_img, S, S, B, 2))
    raw[..., 2:4] = rng.normal(-1.5, 0.5, (n_img, S, S, B, 2))
    raw[..., 4] = rng.normal(-3, 2.5, (n_img, S, S, B))
    raw[..., 5:] = rng.normal(-1, 3, (n_img, S, S, B, C))
    raw[0, 0, 0, 0, 4] = 10.0
    raw[0, 0, 0, 0, 5:] = 10.0                           # every class a hit
    for x, z in ((1, -1e-6), (2, 0.0), (3, 1e-6)):       # objectness just below / at / above 0.5 after sigmoidf_
        raw[1, 0, x, 1, 4] = z
        raw[1, 0, x, 1, 5:] = 30.0                       # sigmoidf_(30) == 1: c * p == c
    raw[1, 1, 0, 0, 4:] = 30.0                           # saturating logits
    raw[1, 1, 1, 0, 4] = 100.0
    raw[1, 1, 1, 0, 5:] = np.where(np.arange(C) % 2 == 0, 100.0, -100.0)
    raw[1, 1, 2, 0, 5:] = -30.0
    raw[1, 1, 3, 2, 4:] = 30.0
    raw[1, 1, 3, 2, 2] = 100.0                           # expf overflows: w = inf
    raw[2, 2, 0, 0, 4:] = 20.0
    raw[2, 2, 0, 0, 0] = np.nan                          # NaN x in a hot box
    raw[2, 2, 1, 0, 4] = np.nan                          # NaN objectness: no hits
    raw[2, 2, 1, 0, 5:] = 20.0
    raw[2, 2, 2, 1, 4:] = 20.0
    raw[2, 2, 2, 1, 5] = np.nan                          # NaN class score: that class is no hit
    raw[3, ..., 4] = -10.0                               # no candidates at all
    return raw.reshape(n_img, S, S, B * (5 + C))


@pytest.mark.parametrize("C", [1, 33, 80])
def test_logits_counting_pass_edge_cases(C):
    rng = np.random.default_rng(C)
    S, B = 8, 3
    anc = rng.uniform(0.05, 0.4, (B, 2)).astype(np.float32)
    fn = wrap_yolo_loss_from_logits(3, (S, S), B, C, anchors=anc)
    raw = torch.from_numpy(edge_heads(C, rng, S, B)).cuda()
    yt = torch.zeros((4, S, S, 5 + C), device="cuda")
    act = engine.activate_head(fn.params, raw)
    for mode in (1, 2):
        _, _, _, r = engine.loss_decode_nms_fused([fn.params], [yt], [raw], 0.5, 0.45, mode, rows_per_img_cap=1024)
        assert int(r["n_overflow"].item()) == 0
        rows, offs = survivors(r)
        ref_rows, ref_offs = chain([act], C, 0.5, 3, 0.45, mode)
        assert np.array_equal(offs, ref_offs)
        assert np.array_equal(rows, ref_rows, equal_nan=True)
        assert offs[4] == offs[3]                        # image 3: no survivors
    # the counted rows, before NMS: the pass files what the chain decodes
    rows_all, _ = engine.decode_batch_exact([act], C, 0.5, 3)
    rows_all = rows_all.cpu().numpy()
    a = act.cpu().numpy().reshape(4, S, S, B, 5 + C)
    assert a[1, 0, 1, 1, 4] < 0.5 and a[1, 0, 2, 1, 4] == 0.5 and a[1, 0, 3, 1, 4] > 0.5
    assert np.isinf(a[1, 1, 3, 2, 2])
    assert rows_all.shape[0] >= C                        # the all-hit box alone


# ---- TrainEvalStep on raw heads --------------------------------------------------------------------
@pytest.mark.parametrize("graph", [False, True])
def test_static_step_on_raw_heads(graph):
    cfgs = [logits_config("v4-608", 5, s) for s in (5, 6)]
    _, ver, fns, _ = cfgs[0]
    params = [f.params for f in fns]
    C = cfgs[0][0]["class_num"]
    yts = [torch.from_numpy(a).cuda() for a in cfgs[0][0]["y_trues"]]
    yps = [torch.from_numpy(a).cuda() for a in cfgs[0][3]]
    step = engine.TrainEvalStep(params, yts, yps, 0.5, 0.45, 2, rows_per_img_cap=1024, graph=graph)
    assert (step.graph is not None) == graph
    for rep in range(4):
        cfg, _, _, raws = cfgs[rep & 1]
        for dst, src in zip(yts + yps, cfg["y_trues"] + raws):
            dst.copy_(torch.from_numpy(src))
        loss, d, _, r = step.run()
        loss0, d0, _, r0 = engine.loss_decode_nms_fused(params, yts, yps, 0.5, 0.45, 2, rows_per_img_cap=1024)
        n = int(r0["out_offsets"][-1].item())
        assert n > 0 and int(r["n_overflow"].item()) == 0
        assert torch.equal(loss, loss0) and all(torch.equal(a, b) for a, b in zip(d, d0))
        assert torch.equal(r["out_offsets"], r0["out_offsets"]) and torch.equal(r["out_rows"][:n], r0["out_rows"][:n])
        torch.cuda.synchronize()
        assert int(step.lws.count_nonzero().item()) == 0
        head = step._aligned(step.fws) - step.fws.data_ptr()
        assert int(step.fws[head:head + 768].count_nonzero().item()) == 0
        fr, fo = step.fallback_survivors()
        assert torch.equal(fo, r["out_offsets"]) and torch.equal(fr, r["out_rows"][:n])
    # every image overflows a 32-row cap; the control block stays clean and the fallback has the survivors
    acts = [engine.activate_head(p, t) for p, t in zip(params, yps)]
    ref_rows, ref_offs = chain(acts, C, 0.5, ver, 0.45, 2)
    small = engine.TrainEvalStep(params, yts, yps, 0.5, 0.45, 2, rows_per_img_cap=32, graph=graph)
    for _ in range(2):
        _, _, _, r = small.run()
        assert int(r["n_overflow"].item()) == 5 and int(r["out_offsets"][-1].item()) == 0
    torch.cuda.synchronize()
    head = small._aligned(small.fws) - small.fws.data_ptr()
    assert int(small.fws[head:head + 768].count_nonzero().item()) == 0
    fr, fo = small.fallback_survivors()
    assert np.array_equal(fo.cpu().numpy(), ref_offs) and np.array_equal(fr.cpu().numpy(), ref_rows)


# ---- HostBatchStep on raw heads --------------------------------------------------------------------
def test_host_batch_step_on_raw_heads():
    cfg, ver, fns, raws = logits_config("v4-608", 8, 32)
    params = [f.params for f in fns]
    boxes, offs = synth.boxes_from_labels(cfg["y_trues"][-1], (608, 608))
    labels = ot.encode_label_pyramid(boxes, offs, (608, 608), (76, 76), 80, 3, dtype=np.float32)
    yts = [torch.from_numpy(a).cuda() for a in labels]
    yps = [torch.from_numpy(a).cuda() for a in raws]
    loss0, d0, _, r0 = engine.loss_decode_nms_fused(params, yts, yps, 0.5, 0.45, 2, rows_per_img_cap=1024)
    rows0, offs0 = survivors(r0)
    acts = [engine.activate_head(p, t) for p, t in zip(params, yps)]
    ref_rows, ref_offs = chain(acts, 80, 0.5, ver, 0.45, 2)
    assert np.array_equal(rows0, ref_rows) and rows0.shape[0] > 0
    host_p = [torch.from_numpy(a).pin_memory() for a in raws]
    hb, ho = torch.from_numpy(boxes).pin_memory(), torch.from_numpy(offs).pin_memory()
    mb = int(np.diff(offs).max())
    pipe = HostBatchStep(fns, (608, 608), 8, 0.5, 0.45, 2, n_chunks=1, rows_per_img=1024, max_boxes_per_img=mb,
                         max_boxes=len(boxes))
    res = pipe.run(host_p, hb, ho)
    assert np.array_equal(res["loss"], loss0.cpu().numpy())
    assert all(torch.equal(a, b) for a, b in zip(res["dpred"], d0))
    got = np.concatenate([r for r, _ in res["rows"]], axis=0)
    assert np.array_equal(got, rows0)
    # the most crowded image overflows: the chunk is redone on the ACTIVATED heads
    per_img = np.diff(engine.decode_batch_exact(acts, 80, 0.5, 4)[1].cpu().numpy())
    cap = int(max(32, np.sort(per_img)[-2]))
    assert per_img.max() > cap
    pipe = HostBatchStep(fns, (608, 608), 8, 0.5, 0.45, 2, n_chunks=2, rows_per_img=cap, max_boxes_per_img=mb,
                         max_boxes=len(boxes))
    res = pipe.run(host_p, hb, ho)
    assert int(pipe.overflow_host.sum()) >= 1
    got = np.concatenate([r for r, _ in res["rows"]], axis=0)
    assert np.array_equal(got, ref_rows)
