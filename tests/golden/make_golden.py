"""Generate the golden fixtures in tests/golden/ by running the UNMODIFIED reference (/root/reference).

Runs only in the build container (the GPU box has no /root/reference):
    python tests/golden/make_golden.py
The reference is imported through tests/golden/refshim.py (stand-ins for the absent ultralytics / matplotlib
packages).  All inputs are regenerated from seeds by oracle/* helpers (numpy RandomState: portable), so the
fixtures only hold the reference's OUTPUTS.  While generating, every oracle function is checked against the
reference output (hard assert) -- this is what pins the oracle.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import refshim  # noqa: E402

refshim.install()

import torch  # noqa: E402
import torchvision  # noqa: E402
import yaml  # noqa: E402

from oracle import loss_ref, model_ref, nms_ref  # noqa: E402
from yolov5_b200.cfg import HYP_SCRATCH_LOW, model_cfg, model_names  # noqa: E402

torch.set_num_threads(8)
REF = refshim.REFERENCE_ROOT


def synth_image(shape, seed):
    return torch.from_numpy(np.random.RandomState(seed).uniform(0, 1, shape).astype(np.float32))


def cfg_digest(cfg):
    return hashlib.sha256(json.dumps(cfg, sort_keys=True).encode()).hexdigest()


def gen_cfg():
    out = {}
    for name in model_names():
        sub = "models/segment/" if name.endswith("-seg") else "models/"
        with open(f"{REF}/{sub}{name}.yaml", encoding="ascii", errors="ignore") as f:
            ref = yaml.safe_load(f)
        assert ref == model_cfg(name), name
        out[name] = cfg_digest(ref)
    with open(f"{REF}/data/hyps/hyp.scratch-low.yaml") as f:
        hyp = yaml.safe_load(f)
    for k, v in HYP_SCRATCH_LOW.items():
        if k != "label_smoothing":
            assert hyp[k] == v, k
    json.dump(out, open(f"{HERE}/cfg_digest.json", "w"), indent=1)
    print("cfg tables == reference YAML for", list(out))


def ref_model(name, sd):
    from models.yolo import DetectionModel, SegmentationModel

    sub = "models/segment/" if name.endswith("-seg") else "models/"
    cls = SegmentationModel if name.endswith("-seg") else DetectionModel
    m = cls(f"{REF}/{sub}{name}.yaml")
    missing = m.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    # the reference divides its anchors by the probed stride at construction; our synthetic sd already holds them
    return m.eval()


def gen_model():
    cases = [("yolov5n", (2, 3, 96, 128), 10), ("yolov5s", (1, 3, 64, 64), 11), ("yolov5n-seg", (1, 3, 64, 96), 12)]
    store = {}
    for name, shape, seed in cases:
        cfg = model_cfg(name)
        sd = model_ref.synth_state_dict(cfg, seed=seed)
        m = ref_model(name, sd)
        assert [float(s) for s in m.stride] == model_ref.model_strides(cfg)
        x = synth_image(shape, seed + 100)
        with torch.no_grad():
            y_ref = m(x)
            y_orc = model_ref.forward(cfg, sd, x)
            mf = ref_model(name, sd).fuse()
            yf_ref = mf(x)
            yf_orc = model_ref.forward(cfg, sd, x, fused=True)
            m.train()
            yt_ref = m(x)  # NB train mode also updates BN running stats; outputs use batch stats -> not compared
            yt_orc = None
        seg = name.endswith("-seg")
        for tag, r, o in (("bn", y_ref, y_orc), ("fused", yf_ref, yf_orc)):
            z_r, z_o = r[0], o[0]
            raw_r, raw_o = (r[2], o[2]) if seg else (r[1], o[1])
            d = (z_r - z_o).abs().max().item()
            print(f"{name} {tag}: z max|ref-oracle| = {d:.3e}  (|z|max {z_r.abs().max():.1f})")
            assert torch.allclose(z_r, z_o, rtol=1e-4, atol=1e-4), (name, tag, d)
            for a, b in zip(raw_r, raw_o):
                assert torch.allclose(a, b, rtol=1e-4, atol=1e-4)
            store[f"{name}.{tag}.z"] = z_r.numpy()
            for l, a in enumerate(raw_r):
                store[f"{name}.{tag}.raw{l}"] = a.numpy()
            if seg:
                assert torch.allclose(r[1], o[1], rtol=1e-4, atol=1e-4)
                store[f"{name}.{tag}.proto"] = r[1].numpy()
        store[f"{name}.shape"] = np.array(shape)
        store[f"{name}.seed"] = np.array([seed, seed + 100])
    # config 1 of BASELINE.json: yolov5n, 1x3x640x640, CPU fp32 -- keep a strided sample + checksum only
    cfg = model_cfg("yolov5n")
    sd = model_ref.synth_state_dict(cfg, seed=20, head_bias="hot")
    m = ref_model("yolov5n", sd).fuse()
    x = synth_image((1, 3, 640, 640), 120)
    with torch.no_grad():
        z = m(x)[0]
        zo = model_ref.forward(cfg, sd, x, fused=True)[0]
    assert z.shape == (1, 25200, 85)
    assert torch.allclose(z, zo, rtol=1e-4, atol=1e-4), (z - zo).abs().max()
    store["yolov5n.640.z_sample"] = z[0, ::97].numpy()
    store["yolov5n.640.z_sum"] = np.array([z.double().sum().item(), z.double().abs().sum().item()])
    store["yolov5n.640.seed"] = np.array([20, 120])
    print("yolov5n 640 max|ref-oracle| =", (z - zo).abs().max().item(), " obj>0.25 rows:", int((z[0, :, 4] > 0.25).sum()))
    np.savez_compressed(f"{HERE}/model_forward.npz", **store)


def run_ref_nms(pred_np, dtype, **kw):
    from utils.general import non_max_suppression

    tdt = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}[dtype]
    outs = []
    for b in range(pred_np.shape[0]):  # one image per call so the reference's wall-clock abort cannot drop images
        out = non_max_suppression(torch.from_numpy(pred_np[b : b + 1]).to(tdt), **kw)
        assert out[0].dtype == torch.float32
        outs.append(out[0].numpy())
    return outs


def canon_ties(d):
    """Sort rows by (-score, then all columns) so rows with equal score are in a canonical order."""
    keys = [d[:, k] for k in range(d.shape[1] - 1, -1, -1) if k != 4] + [-d[:, 4]]
    return d[np.lexsort(keys)]


def gen_nms():
    rs = np.random.RandomState(7)
    # (1) the greedy core vs the installed torchvision op, including ties / zero-area / identical boxes
    for trial in range(40):
        n = int(rs.randint(1, 400))
        xy = rs.uniform(0, 100, (n, 2)).astype(np.float32)
        wh = rs.uniform(0, 40, (n, 2)).astype(np.float32)
        if trial % 4 == 0:
            xy, wh = np.round(xy / 8) * 8, np.round(wh / 8) * 8  # many exact ties and zero areas
        boxes = np.concatenate((xy, xy + wh), 1).astype(np.float32)
        scores = np.sort(rs.uniform(0, 1, n).astype(np.float32))[::-1].copy()
        thr = float(rs.choice([0.3, 0.45, 0.6]))
        ref = torchvision.ops.nms(torch.from_numpy(boxes), torch.from_numpy(scores), thr).numpy()
        got = nms_ref.nms_greedy(boxes, thr)
        assert np.array_equal(ref, got), trial
    print("nms_greedy == torchvision.ops.nms on 40 random cases")
    # box_iou vs the shim's torch expression
    a = np.concatenate((xy[:50], xy[:50] + wh[:50]), 1)
    b = np.concatenate((xy[50:90], xy[50:90] + wh[50:90]), 1) if n > 90 else a
    ref_iou = refshim.box_iou(torch.from_numpy(a), torch.from_numpy(b)).numpy()
    assert np.allclose(ref_iou, nms_ref.box_iou(a, b), rtol=1e-6, atol=1e-7)

    # (2) whole function vs the reference, several regimes
    store, meta = {}, []
    cases = [
        dict(tag="detect_fp32", bs=3, n=25200, nc=80, nm=0, seed=2, dtype="fp32", kw=dict(conf_thres=0.25, iou_thres=0.45, max_det=1000)),
        dict(tag="detect_fp16", bs=3, n=25200, nc=80, nm=0, seed=3, dtype="fp16", kw=dict(conf_thres=0.25, iou_thres=0.45, max_det=1000)),
        dict(tag="detect_bf16", bs=2, n=25200, nc=80, nm=0, seed=4, dtype="bf16", kw=dict(conf_thres=0.25, iou_thres=0.45, max_det=1000)),
        dict(tag="val_fp32", bs=2, n=25200, nc=80, nm=0, seed=5, dtype="fp32", kw=dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)),
        dict(tag="val_fp16", bs=2, n=25200, nc=80, nm=0, seed=6, dtype="fp16", kw=dict(conf_thres=0.001, iou_thres=0.6, multi_label=True, max_det=300)),
        dict(tag="agnostic_cls", bs=2, n=6300, nc=80, nm=0, seed=7, dtype="fp16", kw=dict(conf_thres=0.25, iou_thres=0.45, agnostic=True, classes=[0, 3, 17, 40, 79], max_det=300)),
        dict(tag="seg_fp16", bs=2, n=6300, nc=80, nm=32, seed=8, dtype="fp16", kw=dict(conf_thres=0.25, iou_thres=0.45, max_det=300, nm=32)),
        dict(tag="small_nc1", bs=2, n=1000, nc=1, nm=0, seed=9, dtype="fp32", kw=dict(conf_thres=0.1, iou_thres=0.5, multi_label=True, max_det=50)),
        dict(tag="empty", bs=2, n=500, nc=80, nm=0, seed=10, dtype="fp16", kw=dict(conf_thres=0.9999, iou_thres=0.45)),
    ]
    for c in cases:
        pred = nms_ref.synth_predictions(c["bs"], c["n"], c["nc"], c["nm"], c["seed"], c["dtype"])
        ref = run_ref_nms(pred, c["dtype"], **c["kw"])
        orc = nms_ref.non_max_suppression(pred, dtype=c["dtype"], **c["kw"])
        how = "bit-exact"
        for b, (r, o) in enumerate(zip(ref, orc)):
            assert r.shape == o.shape, (c["tag"], b, r.shape, o.shape)
            if not np.array_equal(r, o):
                # equal scores: the reference's argsort(descending=True) (utils/general.py:745) is not a stable sort,
                # so the order inside an equal-score run is implementation-defined there; the oracle (and the CUDA
                # path) define it as candidate order.  Compare with each equal-score run put in a canonical order.
                assert np.array_equal(canon_ties(r), canon_ties(o)), (c["tag"], b)
                how = "exact up to the order inside equal-score runs"
            store[f"{c['tag']}.{b}"] = o
        c["pinned"] = how
        meta.append({k: v for k, v in c.items()})
        print(f"NMS {c['tag']}: oracle == reference {how}; dets/img {[r.shape[0] for r in ref]}")
    # (3) apriori labels (val.py --save-hybrid, utils/general.py:706-712): the reference vs the oracle
    from utils.general import non_max_suppression as ref_nms

    for tag, dt in (("hybrid_fp16", "fp16"), ("hybrid_fp32", "fp32")):
        pred = nms_ref.synth_predictions(3, 6300, 80, 0, 11, dt)
        lrs = np.random.RandomState(12)
        labels = []
        for b in range(3):
            m = [4, 0, 7][b]
            cxy = lrs.uniform(60, 580, (m, 2))
            wh = lrs.uniform(20, 200, (m, 2))
            labels.append(np.concatenate((lrs.randint(0, 80, (m, 1)), cxy, wh), 1).astype(np.float32))
        kw = dict(conf_thres=0.25, iou_thres=0.45, multi_label=True, max_det=300)
        tdt = {"fp32": torch.float32, "fp16": torch.float16}[dt]
        ref = []
        for b in range(3):  # one image per call (wall-clock abort), labels list aligned with the single image
            ref.append(ref_nms(torch.from_numpy(pred[b : b + 1]).to(tdt), labels=[torch.from_numpy(labels[b])], **kw)[0].numpy())
        orc = nms_ref.non_max_suppression(pred, dtype=dt, labels=labels, **kw)
        for b, (r, o) in enumerate(zip(ref, orc)):
            assert r.shape == o.shape and np.array_equal(canon_ties(r), canon_ties(o)), (tag, b, r.shape, o.shape)
            store[f"{tag}.{b}"] = o
            store[f"{tag}.labels{b}"] = labels[b]
        meta.append(dict(tag=tag, bs=3, n=6300, nc=80, nm=0, seed=11, dtype=dt, kw=kw, labels=True, pinned="exact up to the order inside equal-score runs"))
        print(f"NMS {tag}: oracle == reference with apriori labels; dets/img {[r.shape[0] for r in ref]}")
    store["meta"] = np.array(json.dumps(meta))
    np.savez_compressed(f"{HERE}/nms.npz", **store)


def gen_loss():
    from models.yolo import DetectionModel
    from utils.loss import ComputeLoss

    cfg = model_cfg("yolov5n")
    sd = model_ref.synth_state_dict(cfg, seed=30)
    m = DetectionModel(f"{REF}/models/yolov5n.yaml")
    m.load_state_dict(sd)
    m.hyp = dict(HYP_SCRATCH_LOW)
    crit = ComputeLoss(m)
    anchors = sd["model.24.anchors"].numpy()
    store = {}
    for tag, bs, hw, seed in (("a", 4, (128, 160), 31), ("b", 16, (64, 64), 32), ("none", 2, (64, 64), 33)):
        rs = np.random.RandomState(seed)
        p = [torch.from_numpy(rs.normal(0, 1.5, (bs, 3, hw[0] // s, hw[1] // s, 85)).astype(np.float32)).requires_grad_(True) for s in (8, 16, 32)]
        tg = loss_ref.synth_targets(bs, seed) if tag != "none" else np.zeros((0, 6), np.float32)
        loss, items = crit(p, torch.from_numpy(tg))
        loss.backward()
        tcls, tbox, indices, anch = crit.build_targets(p, torch.from_numpy(tg))
        bt = loss_ref.build_targets(tg, anchors, [tuple(pi.shape[2:4]) for pi in p], 4.0)
        for i in range(3):
            assert np.array_equal(tcls[i].numpy(), bt[i]["tcls"])
            assert np.array_equal(tbox[i].numpy(), bt[i]["tbox"]), np.abs(tbox[i].numpy() - bt[i]["tbox"]).max()
            for q, k in enumerate(("b", "a", "gj", "gi")):
                assert np.array_equal(indices[i][q].numpy(), bt[i][k]), (tag, i, k)
            assert np.array_equal(anch[i].numpy(), bt[i]["anch"])
            store[f"{tag}.idx{i}"] = np.stack([indices[i][q].numpy() for q in range(4)] + [tcls[i].numpy()])
            store[f"{tag}.tbox{i}"] = tbox[i].numpy()
        p2 = [t.detach().clone().requires_grad_(True) for t in p]
        lo, it = loss_ref.compute_loss(p2, tg, anchors, HYP_SCRATCH_LOW)
        lo.backward()
        assert torch.allclose(loss, lo, rtol=1e-5, atol=1e-6), (loss, lo)
        assert torch.allclose(items, it, rtol=1e-5, atol=1e-6)
        for a, b in zip(p, p2):
            assert torch.allclose(a.grad, b.grad, rtol=1e-4, atol=1e-7), (a.grad - b.grad).abs().max()
        store[f"{tag}.loss"] = np.concatenate((loss.detach().numpy(), items.numpy()))
        store[f"{tag}.gradsum"] = np.array([[t.grad.double().sum().item(), t.grad.double().abs().sum().item()] for t in p])
        store[f"{tag}.grad_sample0"] = p[0].grad.numpy().reshape(-1)[::1009]
        store[f"{tag}.meta"] = np.array([bs, hw[0], hw[1], seed])
        print(f"loss {tag}: {loss.item():.6f} items {items.tolist()} matches {[len(d['b']) for d in bt]}; oracle == reference")
    np.savez_compressed(f"{HERE}/loss.npz", **store)
def gen_train():
    """Training-mode pin: the real reference in model.train() -- forward with batch-statistics BatchNorm (models/common.py:
    86-88), ComputeLoss, backward -- against the oracle's bn_batch_stats forward + loss_ref on the same seeded weights,
    images and labels: raw head maps, loss, BN running-statistic updates and parameter gradients."""
    from utils.loss import ComputeLoss

    from oracle import loss_ref
    from yolov5_b200.cfg import HYP_SCRATCH_LOW

    name, shape, seed = "yolov5n", (4, 3, 128, 128), 30
    cfg = model_cfg(name)
    sd = model_ref.synth_state_dict(cfg, seed=seed)
    m = ref_model(name, sd).train()
    m.hyp = dict(HYP_SCRATCH_LOW)
    x = synth_image(shape, seed + 100)
    targets = torch.from_numpy(loss_ref.synth_targets(shape[0], seed=seed + 200))
    p_ref = m(x)
    loss_r, items_r = ComputeLoss(m)(p_ref, targets)
    loss_r.backward()
    params = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k and "anchors" not in k) for k, v in sd.items()}
    p_orc = model_ref.forward(cfg, params, x, training=True, bn_batch_stats=True)
    loss_o, items_o = loss_ref.compute_loss(p_orc, targets, sd["model.24.anchors"], HYP_SCRATCH_LOW)
    loss_o.backward()
    store = {"shape": np.array(shape), "seed": np.array([seed, seed + 100, seed + 200])}
    for l, (a, b) in enumerate(zip(p_ref, p_orc)):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-4), (l, (a - b).abs().max())
        store[f"raw{l}"] = a.detach().numpy()
    assert torch.allclose(loss_r, loss_o, rtol=1e-5, atol=1e-6), (loss_r, loss_o)
    store["loss"] = loss_r.detach().numpy()
    store["items"] = items_r.detach().numpy()
    worst = 0.0
    for k, q in m.named_parameters():
        g_r, g_o = q.grad, params[k].grad
        assert g_o is not None, k
        err = float((g_r - g_o).abs().max() / (g_r.abs().max() + 1e-12))
        worst = max(worst, err)
        assert err < 1e-3, (k, err)
        store[f"gnorm.{k}"] = np.array([float(g_r.norm()), float(g_r.abs().max())])
    for k in ("model.0.conv.weight", "model.0.bn.weight", "model.9.cv2.conv.weight", "model.24.m.0.weight", "model.24.m.2.bias"):
        store[f"grad.{k}"] = dict(m.named_parameters())[k].grad.numpy()
    # running statistics after one training forward (momentum 0.03, unbiased variance)
    for k in ("model.0.bn.running_mean", "model.0.bn.running_var", "model.8.cv3.bn.running_var"):
        store[f"stat.{k}"] = m.state_dict()[k].numpy()
    print(f"train: loss {float(loss_r):.6f}, max rel grad diff ref-oracle {worst:.2e} over {len(list(m.parameters()))} tensors")
    np.savez_compressed(f"{HERE}/train_step.npz", **store)


def gen_post():
    """Post-NMS steps that SURVEY.md section 8(f) ranks next (mask post-processing, metric matching): the real reference's
    process_mask / crop_mask / scale_boxes / process_batch on seeded inputs, asserted equal to oracle/post_ref.py."""
    from utils.general import scale_boxes
    from utils.metrics import process_batch
    from utils.segment.general import process_mask

    from oracle import post_ref

    rs = np.random.RandomState(7)
    store = {}
    # process_mask: 32 prototypes at 40x56 for a 160x224 input, 9 detections
    protos = rs.randn(32, 40, 56).astype(np.float32)
    coef = (rs.randn(9, 32) * 0.5).astype(np.float32)
    xy = rs.uniform(0, 1, (9, 2)) * np.array([224, 160]) * 0.6
    wh = rs.uniform(0.1, 0.4, (9, 2)) * np.array([224, 160])
    boxes = np.concatenate((xy, xy + wh), 1).astype(np.float32)
    for up in (False, True):
        ref = process_mask(torch.from_numpy(protos), torch.from_numpy(coef), torch.from_numpy(boxes), (160, 224), upsample=up).numpy()
        got, val = post_ref.process_mask(protos, coef, boxes, (160, 224), upsample=up)
        off = (ref != got)
        assert ref.shape == got.shape and (not off.any() or np.abs(val[off] - 0.5).max() < 1e-5), (up, int(off.sum()))
        store[f"mask.up{int(up)}"] = np.packbits(ref.astype(bool), axis=None)
        store[f"mask.up{int(up)}.shape"] = np.array(ref.shape)
    from utils.segment.general import process_mask_native

    ref = process_mask_native(torch.from_numpy(protos), torch.from_numpy(coef), torch.from_numpy(boxes), (160, 224)).numpy()
    got, val = post_ref.process_mask_native(protos, coef, boxes, (160, 224))
    off = ref != got
    assert ref.shape == got.shape and (not off.any() or np.abs(val[off] - 0.5).max() < 1e-5), int(off.sum())
    store["mask.native"] = np.packbits(ref.astype(bool), axis=None)
    store["mask.native.shape"] = np.array(ref.shape)
    # a letterboxed (padded) prototype map: 40x56 prototypes for a 128x224 input -> the un-padded window is rows 4..36
    ref = process_mask_native(torch.from_numpy(protos), torch.from_numpy(coef), torch.from_numpy(boxes), (128, 224)).numpy()
    got, val = post_ref.process_mask_native(protos, coef, boxes, (128, 224))
    off = ref != got
    assert ref.shape == got.shape and (not off.any() or np.abs(val[off] - 0.5).max() < 1e-5), int(off.sum())
    store["mask.native_pad"] = np.packbits(ref.astype(bool), axis=None)
    store["mask.native_pad.shape"] = np.array(ref.shape)
    store.update({"mask.protos": protos, "mask.coef": coef, "mask.boxes": boxes, "mask.input_hw": np.array([160, 224])})
    # scale_boxes: letterboxed 640x640 -> 480x640 original, with and without an explicit ratio_pad
    b = (rs.uniform(-20, 660, (50, 4))).astype(np.float32)
    for tag, rp in (("auto", None), ("given", ((0.75, 0.75), (10.0, 80.0)))):
        ref = scale_boxes((640, 640), torch.from_numpy(b.copy()), (480, 640), rp).numpy()
        got = post_ref.scale_boxes((640, 640), b, (480, 640), rp)
        assert np.allclose(ref, got, rtol=0, atol=1e-4), tag
        store[f"scale.{tag}"] = ref
    store["scale.in"] = b
    # process_batch: 3 cases (dense matches with shared labels, no labels, no detections)
    iouv = np.linspace(0.5, 0.95, 10).astype(np.float32)
    for case, (nd, nl) in enumerate(((120, 14), (30, 0), (0, 6), (200, 40))):
        lab_xy = rs.uniform(50, 500, (nl, 2))
        lab_wh = rs.uniform(30, 120, (nl, 2))
        labels = np.concatenate((rs.randint(0, 3, (nl, 1)), lab_xy, lab_xy + lab_wh), 1).astype(np.float32)
        if nl and nd:
            src = rs.randint(0, nl, nd)
            jit = rs.normal(0, 6, (nd, 4))
            det_box = labels[src, 1:] + jit
            cls = np.where(rs.uniform(size=nd) < 0.85, labels[src, 0], rs.randint(0, 3, nd))
        else:
            det_box = np.concatenate((rs.uniform(0, 300, (nd, 2)), rs.uniform(310, 600, (nd, 2))), 1)
            cls = rs.randint(0, 3, nd)
        det = np.concatenate((det_box, rs.uniform(0.1, 1, (nd, 1)), cls[:, None]), 1).astype(np.float32)
        ref = process_batch(torch.from_numpy(det), torch.from_numpy(labels), torch.from_numpy(iouv)).numpy()
        got = post_ref.process_batch(det, labels, iouv)
        assert ref.shape == got.shape and np.array_equal(ref, got), (case, int((ref != got).sum()))
        store[f"match{case}.det"], store[f"match{case}.labels"], store[f"match{case}.correct"] = det, labels, ref
        print(f"process_batch case {case}: {nd} detections, {nl} labels, true positives per threshold {ref.sum(0).tolist()}")
    store["match.iouv"] = iouv
    np.savez_compressed(f"{HERE}/post.npz", **store)


from make_golden_cases import PRE_CASES  # noqa: E402


def gen_pre():
    """Step before the hot path: the reference's letterbox (cv2.resize INTER_LINEAR + copyMakeBorder) and the dataloader's
    HWC BGR -> CHW RGB on seeded images, asserted equal -- byte for byte -- to oracle/pre_ref.py."""
    import cv2
    from utils.augmentations import letterbox

    from oracle import pre_ref

    rs = np.random.RandomState(0)
    for t in range(200):  # the fixed-point bilinear restatement vs the installed OpenCV on random shapes
        h, w, dh, dw = rs.randint(5, 500), rs.randint(5, 700), rs.randint(4, 500), rs.randint(4, 700)
        img = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        assert np.array_equal(cv2.resize(img, (dw, dh), interpolation=cv2.INTER_LINEAR), pre_ref.resize_linear_u8(img, (dw, dh))), (t, h, w, dh, dw)
    store = {}
    for i, (h, w, seed, kw) in enumerate(PRE_CASES):
        im = pre_ref.synth_image(h, w, seed)
        ref, r_ratio, r_pad = letterbox(im, **kw)
        got, g_ratio, g_pad = pre_ref.letterbox(im, **kw)
        assert np.array_equal(ref, got) and tuple(r_ratio) == tuple(g_ratio) and tuple(r_pad) == tuple(g_pad), i
        chw = np.ascontiguousarray(ref.transpose((2, 0, 1))[::-1])  # utils/dataloaders.py:356
        assert np.array_equal(chw, pre_ref.to_chw_rgb(got))
        store[f"lb{i}"] = chw
        store[f"lb{i}.ratio_pad"] = np.array([*r_ratio, *r_pad], np.float64)
    np.savez_compressed(f"{HERE}/pre.npz", **store)
    print(f"letterbox: oracle == reference (cv2 {cv2.__version__}) byte for byte on {len(PRE_CASES)} cases + 200 random resizes")


def gen_optim():
    """Step after backward (train.py:413-421): torch.optim.SGD(nesterov) over the reference's 3-group layout + clip_grad_norm_
    + the reference's ModelEMA, vs oracle/optim_ref.py."""
    from utils.torch_utils import ModelEMA

    from oracle import optim_ref

    store = {}
    hyper = [dict(lr=0.01, momentum=0.937, weight_decay=0.0, nesterov=True), dict(lr=0.01, momentum=0.937, weight_decay=5e-4, nesterov=True),
             dict(lr=0.1, momentum=0.8, weight_decay=0.0, nesterov=True)]
    for case, (inv_scale, max_norm, poison) in enumerate(((1.0, 10.0, False), (1.0 / 1024, 10.0, False), (1.0, 1e9, False), (1.0 / 8, 10.0, True))):
        params, grads, moms, emas, groups = optim_ref.synth_problem(40 + case)
        if poison:
            grads[3].flat[5] = np.inf
        tp = [torch.nn.Parameter(torch.from_numpy(p.copy())) for p in params]

        class Holder(torch.nn.Module):
            def __init__(self):
                super().__init__()
                self.ps = torch.nn.ParameterList(tp)
                self.register_buffer("stat", torch.from_numpy(np.linspace(0, 1, 33, dtype=np.float32)))

        model = Holder()
        opt = torch.optim.SGD([dict(params=[tp[i] for i in range(len(tp)) if groups[i] == g], **{k: v for k, v in hyper[g].items()}) for g in range(3)],
                              lr=0.01)
        for i, p in enumerate(tp):  # momentum buffers as if a few steps had run
            opt.state[p]["momentum_buffer"] = torch.from_numpy(moms[i].copy())
            p.grad = torch.from_numpy(grads[i].copy())
        ema = ModelEMA(model, decay=0.9999, tau=2000, updates=37)
        with torch.no_grad():
            for e, v in zip(ema.ema.ps, emas):
                e.copy_(torch.from_numpy(v))
            ema.ema.stat.copy_(torch.from_numpy(np.linspace(1, 2, 33, dtype=np.float32)))
        # train.py:413-421
        for p in tp:
            p.grad.mul_(inv_scale)                                   # scaler.unscale_
        found_inf = not all(bool(torch.isfinite(p.grad).all()) for p in tp)
        norm = torch.nn.utils.clip_grad_norm_(tp, max_norm=max_norm)
        if not found_inf:                                            # scaler.step skips on overflow
            opt.step()
        ema.update(model)
        p_o, m_o, e_o, eb_o, gn, skipped = optim_ref.sgd_ema_step(params, grads, moms, emas, groups, hyper, inv_scale, max_norm, 0.9999, 2000.0, 37,
                                                                 buffers=[np.linspace(0, 1, 33, dtype=np.float32)],
                                                                 ema_buffers=[np.linspace(1, 2, 33, dtype=np.float32)])
        assert skipped == found_inf
        if not found_inf:
            assert abs(gn - float(norm)) <= 1e-5 * float(norm), (gn, float(norm))
        for i in range(len(tp)):
            assert np.allclose(tp[i].detach().numpy(), p_o[i], rtol=2e-6, atol=1e-7), (case, i)
            assert np.allclose(opt.state[tp[i]]["momentum_buffer"].numpy(), m_o[i], rtol=2e-6, atol=1e-7), (case, i)
            assert np.allclose(ema.ema.ps[i].detach().numpy(), e_o[i], rtol=2e-6, atol=1e-7), (case, i)
            sub = lambda a: a.reshape(-1)[:: optim_ref.FIXTURE_STRIDE].copy()  # noqa: E731
            store[f"c{case}.p{i}"], store[f"c{case}.m{i}"], store[f"c{case}.e{i}"] = (sub(tp[i].detach().numpy()), sub(opt.state[tp[i]]["momentum_buffer"].numpy()),
                                                                                      sub(ema.ema.ps[i].detach().numpy()))
        assert np.allclose(ema.ema.stat.numpy(), eb_o[0], rtol=2e-6, atol=1e-7)
        store[f"c{case}.ebuf"] = ema.ema.stat.numpy()
        store[f"c{case}.cfg"] = np.array([inv_scale, max_norm, float(poison), float(norm) if not found_inf else -1.0])
    store["hyper"] = np.array(json.dumps(hyper))
    np.savez_compressed(f"{HERE}/optim.npz", **store)
    print("optimizer step: oracle == torch.optim.SGD + clip_grad_norm_ + reference ModelEMA on 4 cases (one with an overflow skip)")


def tiny_cfg():
    """yolov5 v6 topology with narrow layers (the reference's YAML grammar): small enough to commit a pickled checkpoint."""
    cfg = json.loads(json.dumps(model_cfg("yolov5s")))
    cm = {64: 16, 128: 16, 256: 32, 512: 64, 1024: 64}
    for part in ("backbone", "head"):
        for row in cfg[part]:
            if row[2] in ("Conv", "C3", "SPPF") and isinstance(row[3][0], int):
                row[3][0] = cm[row[3][0]]
    cfg.update(nc=3, depth_multiple=0.33, width_multiple=1.0)
    return cfg


def gen_ckpt():
    """A checkpoint pickled BY THE REFERENCE (whole-module pickle naming models.yolo.DetectionModel, models.common.Conv ...,
    as train.py:469-482 writes them) + its forward on a seeded image: what yolov5_b200.compat / attempt_load must load."""
    from models.yolo import DetectionModel

    cfg = tiny_cfg()
    torch.manual_seed(3)
    m = DetectionModel(cfg, ch=3)
    g = torch.Generator().manual_seed(4)
    for mod in m.modules():  # non-trivial BatchNorm statistics so the fold matters
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.weight.data = torch.rand(mod.weight.shape, generator=g) + 0.5
            mod.bias.data = torch.randn(mod.bias.shape, generator=g) * 0.1
            mod.running_mean = torch.randn(mod.running_mean.shape, generator=g) * 0.1
            mod.running_var = torch.rand(mod.running_var.shape, generator=g) + 0.5
    m.names = {0: "a", 1: "b", 2: "c"}
    m.eval()
    x = synth_image((1, 3, 64, 96), 5)
    with torch.no_grad():
        z = m(x)[0].numpy()
    from copy import deepcopy

    torch.save({"epoch": -1, "best_fitness": None, "model": deepcopy(m).half(), "ema": None, "updates": 0, "optimizer": None, "opt": {},
                "date": "fixture"}, f"{HERE}/ref_tiny.pt")
    np.savez_compressed(f"{HERE}/ref_tiny_forward.npz", z=z, keys=np.array(json.dumps(list(m.state_dict().keys()))),
                        cfg=np.array(json.dumps(cfg)))
    print(f"reference-pickled checkpoint: {sum(p.numel() for p in m.parameters())} parameters, "
          f"{os.path.getsize(f'{HERE}/ref_tiny.pt') / 1e6:.2f} MB")


def gen_signatures():
    """The reference's call signatures on the drop-in surface (parameter name, repr of the default, kind), which
    tests/test_compat_cpu.py holds this package's callables against."""
    import importlib
    import inspect

    from make_golden_cases import SIGNATURE_SURFACE

    out = {}
    for mod, qual in SIGNATURE_SURFACE:
        obj = importlib.import_module(mod)
        assert obj.__file__.startswith(REF), obj.__file__
        for part in qual.split("."):
            obj = getattr(obj, part)
        out[f"{mod}:{qual}"] = [(n, repr(p.default) if p.default is not inspect.Parameter.empty else None, str(p.kind))
                                for n, p in inspect.signature(obj).parameters.items()]
    json.dump(out, open(f"{HERE}/ref_signatures.json", "w"), indent=1)


if __name__ == "__main__":
    which = sys.argv[1:] or ["cfg", "model", "nms", "loss", "train", "post", "pre", "optim", "ckpt", "signatures"]
    for w in which:
        {"cfg": gen_cfg, "model": gen_model, "nms": gen_nms, "loss": gen_loss, "train": gen_train, "post": gen_post, "pre": gen_pre,
         "optim": gen_optim, "ckpt": gen_ckpt, "signatures": gen_signatures}[w]()
    print("golden fixtures written to", HERE)
