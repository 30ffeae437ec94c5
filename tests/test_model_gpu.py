"""GPU: layers and whole models through the engine vs the oracle (oracle/model_ref.py, itself pinned to the
reference by tests/golden/model_forward.npz).

Tolerance (stated per north_star "within 1e-3 fp16 tolerance"): the reference's own fp16 pipeline rounds every
activation to fp16 (twice per Conv: after conv+bias and after SiLU); the engine rounds once per Conv.  Neither can be
closer to the fp32 oracle than accumulated fp16 rounding allows, so the test measures BOTH against the fp32 oracle
on the same weights/inputs:   err(engine) <= 1e-3 * max|oracle| + 1.5 * err(torch fp16 expression of the reference).
"""
import os

import numpy as np
import pytest
import torch

from oracle import model_ref
from yolov5_b200.cfg import model_cfg
from yolov5_b200.models.common import C3, SPPF, Bottleneck, Conv
from yolov5_b200.models.yolo import DetectionModel, SegmentationModel

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def _image(shape, seed):
    return torch.from_numpy(np.random.RandomState(seed).uniform(0, 1, shape).astype(np.float32))


def _randomize_bn(m, seed):
    g = torch.Generator().manual_seed(seed)
    for mod in m.modules():
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.weight.data = torch.rand(mod.weight.shape, generator=g) + 0.5
            mod.bias.data = torch.randn(mod.bias.shape, generator=g) * 0.1
            mod.running_mean = torch.randn(mod.running_mean.shape, generator=g) * 0.1
            mod.running_var = torch.rand(mod.running_var.shape, generator=g) + 0.5
            mod.eps = 1e-3


def _sd_of(layer, prefix="model.0"):
    return {f"{prefix}.{k}": v.detach().float().cpu() for k, v in layer.state_dict().items()}


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_single_layers_vs_oracle(cuda, dtype):
    torch.manual_seed(0)
    tol = 3e-3 if dtype == torch.float16 else 2.5e-2
    x = torch.rand(2, 64, 20, 20) * 2 - 1
    xq = x.to(dtype).float()
    cases = [
        (Conv(64, 128, 3, 2), lambda sd, t: model_ref.conv_block(sd, "model.0", t, 3, 2)),
        (Bottleneck(64, 64, True, e=1.0), lambda sd, t: model_ref.bottleneck(sd, "model.0", t, True, False)),
        (C3(64, 64, 2), lambda sd, t: model_ref.c3(sd, "model.0", t, 2, True, False)),
        (C3(64, 128, 1, False), lambda sd, t: model_ref.c3(sd, "model.0", t, 1, False, False)),
        (SPPF(64, 64, 5), lambda sd, t: model_ref.sppf(sd, "model.0", t, 5, False)),
    ]
    for i, (layer, ref_fn) in enumerate(cases):
        _randomize_bn(layer, i)
        layer.eval()
        with torch.no_grad():
            ref = ref_fn(_sd_of(layer), xq)
        got = layer.to(cuda, dtype)(x.to(cuda, dtype)).float().cpu()
        err = float((got - ref).abs().max() / ref.abs().max())
        assert got.shape == ref.shape and err < tol, (type(layer).__name__, err)


def _torch_lowp_reference(cfg, sd, x, dtype, dev):
    """The reference's own expressions evaluated in fp16/bf16 by torch on the GPU (what `model.half()` computes)."""
    sd_d = {k: (v.to(dev, dtype) if v.is_floating_point() else v.to(dev)) for k, v in sd.items()}
    with torch.no_grad():
        return model_ref.forward(cfg, sd_d, x.to(dev, dtype), fused=True)


def _check_model(name, shape, seed_w, seed_x, dtype, dev, head_bias="init"):
    cfg = model_cfg(name)
    sd = model_ref.synth_state_dict(cfg, seed=seed_w, head_bias=head_bias)
    x = _image(shape, seed_x)
    with torch.no_grad():
        ref = model_ref.forward(cfg, sd, x.to(dtype).float(), fused=True)
    cls = SegmentationModel if name.endswith("-seg") else DetectionModel
    m = cls(name)
    m.load_state_dict(sd)
    m = m.to(dev, dtype).eval()
    out = m(x.to(dev, dtype))
    low = _torch_lowp_reference(cfg, sd, x, dtype, dev)
    seg = name.endswith("-seg")
    pairs = [("z", out[0], ref[0], low[0])]
    raws, rraws, lraws = (out[2], ref[2], low[2]) if seg else (out[1], ref[1], low[1])
    pairs += [(f"raw{l}", a, b, c) for l, (a, b, c) in enumerate(zip(raws, rraws, lraws))]
    if seg:
        pairs.append(("proto", out[1], ref[1], low[1]))
    report = {}
    for tag, got, r, lo in pairs:
        got, lo = got.float().cpu(), lo.float().cpu()
        assert got.shape == r.shape, (tag, got.shape, r.shape)
        scale = float(r.abs().max())
        e_eng, e_low = float((got - r).abs().max()), float((lo - r).abs().max())
        report[tag] = (e_eng / scale, e_low / scale)
        assert e_eng <= 1e-3 * scale + 1.5 * e_low, (name, tag, e_eng / scale, e_low / scale)
    return report, out, ref


@pytest.mark.parametrize("name,shape,sw,sx", [("yolov5n", (2, 3, 96, 128), 10, 110), ("yolov5s", (1, 3, 64, 64), 11, 111),
                                               ("yolov5n-seg", (1, 3, 64, 96), 12, 112)])
def test_model_fp16_vs_oracle_and_golden(cuda, name, shape, sw, sx):
    report, out, ref = _check_model(name, shape, sw, sx, torch.float16, cuda)
    g = np.load(os.path.join(G, "model_forward.npz"))
    gz = g[f"{name}.fused.z"]  # output of the real reference on the same seeded weights / input
    z = out[0].float().cpu().numpy()
    assert np.abs(z - gz).max() <= 2e-2 * np.abs(gz).max(), report


def test_model_yolov5s_640_bf16(cuda):
    _check_model("yolov5s", (2, 3, 640, 640), 3, 103, torch.bfloat16, cuda)


def test_model_yolov5n_640_config1_golden(cuda):
    """BASELINE.json configs[0] (yolov5n, 1x3x640x640): engine fp16 vs the reference's CPU fp32 output sample."""
    report, out, _ = _check_model("yolov5n", (1, 3, 640, 640), 20, 120, torch.float16, cuda, head_bias="hot")
    g = np.load(os.path.join(G, "model_forward.npz"))
    z = out[0][0, ::97].float().cpu().numpy()
    ref = g["yolov5n.640.z_sample"]
    assert z.shape == ref.shape
    assert np.abs(z - ref).max() <= 2e-2 * np.abs(ref).max(), report


def test_model_yolov5l_bs2(cuda):
    _check_model("yolov5l", (2, 3, 320, 320), 4, 104, torch.float16, cuda)


@pytest.mark.parametrize("name,shape", [("yolov5m", (2, 3, 128, 160)), ("yolov5x-seg", (1, 3, 128, 128)), ("yolov5x", (1, 3, 96, 96))])
def test_model_widths_not_multiple_of_16(cuda, name, shape):
    """yolov5m / yolov5x channel counts (48, 96, 192 / 80, 160, 320 ...) are not multiples of the 64-channel K block:
    the K tail is zero-filled by TMA (out-of-bounds box) and the weights are zero padded.  x-seg adds Proto + no=117."""
    _check_model(name, shape, 7, 107, torch.float16, cuda)


def test_uint8_input_and_graph_replay_is_deterministic(cuda):
    m = DetectionModel("yolov5n")
    m.load_state_dict(model_ref.synth_state_dict(model_cfg("yolov5n"), seed=5))
    m = m.to(cuda).half().eval()
    u8 = torch.from_numpy(np.random.RandomState(0).randint(0, 256, (2, 3, 128, 128)).astype(np.uint8)).to(cuda)
    z1 = m(u8)[0].clone()
    z2 = m(u8)[0]
    z3 = m((u8.float() / 255).half())[0]
    assert torch.equal(z1, z2)
    assert float((z1.float() - z3.float()).abs().max()) <= 2e-3 * float(z1.float().abs().max())


def test_fused_checkpoint_equals_unfused(cuda):
    cfg = model_cfg("yolov5n")
    sd = model_ref.synth_state_dict(cfg, seed=6)
    a = DetectionModel("yolov5n"); a.load_state_dict(sd)
    b = DetectionModel("yolov5n"); b.load_state_dict(sd); b.fuse()
    x = _image((1, 3, 64, 64), 7).to(cuda).half()
    za = a.to(cuda).half().eval()(x)[0].float()
    zb = b.to(cuda).half().eval()(x)[0].float()
    assert float((za - zb).abs().max()) <= 2e-3 * float(za.abs().max())


def _check_model_batch_subset(name, batch, size, dtype, dev, seed_w, seed_x, check=(0, -1), head_bias="init"):
    """Engine on the WHOLE bench batch (tile choices depend on B*H*W); oracle and torch low-precision reference on the images
    `check` only (images are independent in eval mode), same criterion as _check_model."""
    cfg = model_cfg(name)
    sd = model_ref.synth_state_dict(cfg, seed=seed_w, head_bias=head_bias)
    x = torch.from_numpy(np.random.RandomState(seed_x).uniform(0, 1, (batch, 3, size, size)).astype(np.float32))
    seg = name.endswith("-seg")
    m = (SegmentationModel if seg else DetectionModel)(name)
    m.load_state_dict(sd)
    m = m.to(dev, dtype).eval()
    out = m(x.to(dev, dtype))
    sel = [i % batch for i in check]
    xs = x[sel]
    with torch.no_grad():
        ref = model_ref.forward(cfg, sd, xs.to(dtype).float(), fused=True)
    low = _torch_lowp_reference(cfg, sd, xs, dtype, dev)
    pairs = [("z", out[0][sel], ref[0], low[0])]
    raws, rraws, lraws = (out[2], ref[2], low[2]) if seg else (out[1], ref[1], low[1])
    pairs += [(f"raw{l}", a[sel], b, c) for l, (a, b, c) in enumerate(zip(raws, rraws, lraws))]
    if seg:
        pairs.append(("proto", out[1][sel], ref[1], low[1]))
    report = {}
    for tag, got, r, lo in pairs:
        got, lo = got.float().cpu(), lo.float().cpu()
        assert got.shape == r.shape, (tag, got.shape, r.shape)
        scale = float(r.abs().max())
        e_eng, e_low = float((got - r).abs().max()), float((lo - r).abs().max())
        report[tag] = (e_eng / scale, e_low / scale)
        assert e_eng <= 1e-3 * scale + 1.5 * e_low, (name, tag, e_eng / scale, e_low / scale)
    print("bench-shape parity", name, batch, size, dtype, {k: (f"{a:.2e}", f"{b:.2e}") for k, (a, b) in report.items()})
    return m, out


def test_bench_shape_config3_yolov5l_bs64_bf16(cuda):
    """BASELINE config 3 (the headline): yolov5l, 64 x 3 x 640 x 640, bf16 -- the exact shapes the benchmark times."""
    _check_model_batch_subset("yolov5l", 64, 640, torch.bfloat16, cuda, 31, 131)


@pytest.mark.parametrize("batch", [32, 16, 8])
def test_bench_shape_config3_shards(cuda, batch):
    """The per-GPU shards of config 3 when bench.py runs on 2 / 4 / 8 GPUs (64 images split over the ranks): other M extents,
    other tile / CTA-pair choices in the planner than the 64-image program."""
    _check_model_batch_subset("yolov5l", batch, 640, torch.bfloat16, cuda, 34, 134)


def test_bench_shape_config2_yolov5s_bs32_fp16(cuda):
    """BASELINE config 2: yolov5s, 32 x 3 x 640 x 640, fp16, then NMS bit-exact vs the oracle on the engine's own predictions."""
    from oracle import nms_ref
    from yolov5_b200.utils.general import non_max_suppression

    m, out = _check_model_batch_subset("yolov5s", 32, 640, torch.float16, cuda, 32, 132, head_bias="hot")
    z = out[0]
    dets, idx = non_max_suppression(z, 0.25, 0.45, max_det=300, return_indices=True)
    for b in (0, 13, 31):
        ref, ridx = nms_ref.non_max_suppression(z[b : b + 1].float().cpu().numpy(), 0.25, 0.45, max_det=300, dtype="fp16", return_index=True)
        assert np.array_equal(idx[b].cpu().numpy(), ridx[0]) and np.array_equal(dets[b].cpu().numpy(), ref[0]), b


def test_bench_shape_config5_yolov5x_seg_1280(cuda):
    """BASELINE config 5 per-GPU shard: yolov5x-seg, 2 x 3 x 1280 x 1280, fp16 (Proto at 320x320, z (2, 100800, 117));
    one image checked against the fp32 oracle."""
    _check_model_batch_subset("yolov5x-seg", 2, 1280, torch.float16, cuda, 33, 133, check=(1,))


def test_reference_pickled_checkpoint_runs_on_the_engine(cuda):
    """tests/golden/ref_tiny.pt was pickled by the unmodified reference; attempt_load (compat aliases) + the val.py call
    expressions `model(im, augment=augment)` (val.py:267) and `non_max_suppression(preds, conf, iou, labels=lb,
    multi_label=True, agnostic=single_cls, max_det=max_det)` (val.py:277-279) against the reference's stored forward."""
    from yolov5_b200 import compat
    from yolov5_b200.models.experimental import attempt_load
    from yolov5_b200.utils.general import non_max_suppression

    ref = np.load(os.path.join(G, "ref_tiny_forward.npz"))
    try:
        model = attempt_load(os.path.join(G, "ref_tiny.pt"), device=cuda)
    finally:
        compat.uninstall()
    model = model.half()
    im = _image((1, 3, 64, 96), 5).to(cuda).half()
    augment, compute_loss, single_cls, lb, conf_thres, iou_thres, max_det = False, None, False, [], 0.001, 0.6, 300
    preds, train_out = model(im) if compute_loss else (model(im, augment=augment), None)   # val.py:267 verbatim
    z = preds[0]
    rz = ref["z"]
    assert tuple(z.shape) == rz.shape
    assert float(np.abs(z.float().cpu().numpy() - rz).max()) <= 2e-2 * float(np.abs(rz).max())  # checkpoint stored in fp16, engine fp16
    out = non_max_suppression(preds, conf_thres, iou_thres, labels=lb, multi_label=True, agnostic=single_cls, max_det=max_det)  # val.py:277
    assert len(out) == 1 and out[0].shape[1] == 6
    # test-time augmentation (models/yolo.py:269-283): 3 scales + flip, tails clipped
    ya, none = model(im, augment=True)
    assert none is None and ya.shape[0] == 1 and ya.shape[2] == z.shape[2]
    n_full = z.shape[1]
    assert n_full < ya.shape[1] < 3 * n_full
    # the un-flipped full-scale copy leads the TTA output (minus its largest-stride tail): same numbers as the plain forward
    keep = n_full - n_full // 21
    assert torch.allclose(ya[0, :keep].float(), z[0, :keep].float(), rtol=1e-3, atol=1e-3)


def test_program_build_launches_are_library_kernels(cuda):
    """Building a Program folds BatchNorm and packs weights through y5_fold_pack (one launch per GEMM operand), not through
    ATen arithmetic: the library's launch counter accounts for (almost) every kernel of the first forward."""
    from yolov5_b200 import _lib

    m = DetectionModel("yolov5s")
    m.load_state_dict(model_ref.synth_state_dict(model_cfg("yolov5s"), seed=9))
    m = m.half().to(cuda).eval()
    x = _image((1, 3, 64, 64), 9).to(cuda).half()
    n0 = _lib.launch_count()
    m(x)
    torch.cuda.synchronize()
    built = _lib.launch_count() - n0
    n_convs = sum(1 for mod in m.modules() if isinstance(mod, torch.nn.Conv2d))
    assert built >= n_convs + 60  # >= one fold_pack per conv (+ stacked C3 halves, per-anchor head rows) + the forward itself
