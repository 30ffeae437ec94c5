"""CPU half of tests/test_train_kernels_gpu.py: its layer table, its restatement of the BN passes' block geometry and its
float64 convolution references, checked without a GPU."""
import pytest
import torch
import torch.nn.functional as F

from .test_train_kernels_gpu import (bn_classes, conv_ref, dgrad_ref, geometry_coverage, layer_table, row_geom, ulp,
                                     wgrad_ref)


def test_yolov5m_layer_table():
    """26 distinct (cin, cout, k, s) classes, from the 3 -> 48 6x6/s2 stem to SPPF's 1536 -> 768; BN rows 6 400 .. 1 638 400."""
    t = layer_table()
    classes = {l[:4] for l in t}
    assert len(classes) == 26, sorted(classes)
    assert (3, 48, 6, 2, 640, 640) in t and (1536, 768, 1, 1, 20, 20) in t
    rows = [r for c, r in bn_classes() if c not in (8, 16, 256)]
    assert min(rows) == 16 * 20 * 20 and max(rows) == 16 * 320 * 320


def test_bn_geometry_at_148_sms():
    """The geometry rule at the B200's 148 SMs: the yolov5m shapes of the 16 x 640^2 step, and every cgx
    from 1 to 32 reached by the BN cases in both reduce passes."""
    assert row_geom(48, 1638400, True, 4, 148)[0] == 4
    assert row_geom(96, 409600, True, 4, 148)[0] == 8 and row_geom(96, 409600, True, 2, 148)[0] == 8
    assert row_geom(192, 102400, True, 4, 148)[0] == 16
    assert row_geom(384, 25600, True, 4, 148)[0] == 4 and row_geom(384, 25600, True, 2, 148)[0] == 8
    assert row_geom(256, 409600, True, 4, 148)[0] == 32
    stats, bwd = geometry_coverage(148)
    assert stats == bwd == {1, 2, 4, 8, 16, 32}


@pytest.mark.parametrize("B,cin,cout,H,W,kh,kw,s,ph,pw", [
    (2, 3, 5, 11, 13, 3, 3, 1, 1, 1), (2, 4, 6, 10, 12, 3, 3, 2, 1, 1), (1, 3, 4, 12, 14, 6, 6, 2, 2, 2),
    (2, 5, 3, 9, 8, 1, 1, 1, 0, 0), (1, 4, 4, 9, 11, 5, 3, 1, 2, 1), (1, 4, 4, 9, 11, 1, 3, 1, 0, 1),
])
def test_float64_conv_references_match_torch(B, cin, cout, H, W, kh, kw, s, ph, pw):
    g = torch.Generator().manual_seed(kh * 10 + kw + s)
    x = torch.randn(B, cin, H, W, generator=g, dtype=torch.float64)
    w = torch.randn(cout, cin, kh, kw, generator=g, dtype=torch.float64)
    y = F.conv2d(x, w, stride=s, padding=(ph, pw))
    assert torch.allclose(conv_ref(x, w, s, ph, pw), y, rtol=1e-12, atol=1e-12)
    dy = torch.randn(y.shape, generator=g, dtype=torch.float64)
    assert torch.allclose(wgrad_ref(x, dy, kh, kw, s, ph, pw),
                          torch.nn.grad.conv2d_weight(x, w.shape, dy, stride=s, padding=(ph, pw)), rtol=1e-12, atol=1e-12)
    if kh == kw and ph == pw:
        assert torch.allclose(dgrad_ref(dy, w, s, ph, H, W), torch.nn.grad.conv2d_input(x.shape, w, dy, stride=s, padding=ph),
                              rtol=1e-12, atol=1e-12)


def test_ulp():
    x = torch.tensor([1.0, 1.5, 2.0, -3.0, 0.0, 1e-9], dtype=torch.float64)
    assert ulp(x, torch.float16).tolist() == [2 ** -10, 2 ** -10, 2 ** -9, 2 ** -9, 2 ** -24, 2 ** -24]
    assert ulp(x, torch.bfloat16)[:4].tolist() == [2 ** -7, 2 ** -7, 2 ** -6, 2 ** -6]
