"""-m gpu: the training kernels at the layer shapes of the yolov5m 16 x 640^2 training step, in the views the training step
passes them, against plain float64 restatements of each operation built from the same rounded inputs.

Layer table: every Conv of yolov5m, recorded from the oracle's forward at 64^2 and scaled to 640^2 (26 distinct
(cin, cout, k, s) classes), plus yolov5n's 16-channel stem, a 256-channel layer at yolov5l width and an 8-channel view.
Together these reach every block geometry of the BatchNorm reduce passes (`row_geom` in csrc/train_kernels.cu, restated
below): 1 to 32 channel groups of 8 per block.

Bounds (u = the dtype's spacing at 1: 2^-10 fp16, 2^-7 bf16; ulp(x) = its spacing at |x|):
  * BN statistics: |mean - ref| <= 1e-6 (sigma + |mean|), invstd relative error <= 1e-6 + 4e-7 (mean/sigma)^2.  The
    kernel forms E[y^2] - E[y]^2 from fp32 partial sums, so its error grows with the square of the channel's offset.
  * normalise + SiLU, given the kernel's statistics: within 1 ulp of float64 SiLU of the rounded BN output.
  * BN backward apply pass: within 2 u of the per-element scale |du a| + |y c1| + |c0| (floored at the smallest subnormal
    spacing); dgamma / dbeta relative to the L1 sums sum|du xhat| and sum|du| (random dz makes the plain sums small).
    du = dz * silu'(t) is evaluated by the kernel in fp32 with fast exp / divide, so where it lies within ~1e-6 of a
    rounding boundary either neighbour is correct: those elements add the distance between the two to the bounds.
  * weight gradient: <= 1e-5 of the L1 scale (the same op on |x| and |dy|), element by element.
  * data gradient: within 1 ulp of its L1 scale.
Every family also checks a negative control: the reference perturbed like a plausible kernel bug (one row block or one
64-pixel K block lost, one filter column or channel block dropped) must be rejected by the same bound.

The per-case error ratios (error / bound, and control / bound) are printed: run with -s to see them."""
import ctypes as C
import functools
import math
import os

import pytest
import torch
import torch.nn.functional as F

from yolov5_b200 import _lib, train_ops
from yolov5_b200.engine import pack_weight

pytestmark = pytest.mark.gpu

BATCH = 16  # config 4: yolov5m, 16 x 3 x 640 x 640
BN_EPS, BN_MOM = 1e-3, 0.03
EPS = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}
_MANT = {torch.float16: 10, torch.bfloat16: 7}
_MIN_ULP = {torch.float16: 2.0 ** -24, torch.bfloat16: 2.0 ** -133}
SENTINEL = 7.0  # guard value around output slices


# ---------------------------------------------------------------------------------------------------------------------
# layer table and block geometry
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def layer_table(name: str = "yolov5m", scale: int = 10):
    """Distinct (cin, cout, k, s, H, W) of every Conv of `name` at (64 * scale)^2 input: the F.conv2d calls of the oracle's
    forward at 64^2, spatial sizes multiplied by `scale` (input sizes of the layers; the stem is the 6x6/s2 conv)."""
    from oracle import model_ref
    from yolov5_b200.cfg import model_cfg

    calls = []
    orig = F.conv2d

    def record(x, w, b=None, stride=1, padding=0, *a, **kw):
        s = stride if isinstance(stride, int) else stride[0]
        calls.append((w.shape[1], w.shape[0], w.shape[2], s, x.shape[2] * scale, x.shape[3] * scale))
        return orig(x, w, b, stride, padding, *a, **kw)

    cfg = model_cfg(name)
    sd = model_ref.synth_state_dict(cfg, seed=0)
    F.conv2d = record
    try:
        with torch.no_grad():
            model_ref.forward(cfg, sd, torch.zeros(1, 3, 64, 64))
    finally:
        F.conv2d = orig
    return sorted(set(calls))


def out_hw(H, W, k, s):
    p = 2 if k == 6 else k // 2
    return (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1


def bn_classes():
    """(channels, rows) of every BatchNorm of the table (Detect's biased 1x1 convs have none), plus yolov5n's 16-channel stem,
    a 256-channel layer at 409 600 rows (yolov5l width) and an 8-channel view."""
    out = set()
    for cin, cout, k, s, H, W in layer_table():
        if cout == 255:
            continue
        ho, wo = out_hw(H, W, k, s)
        out.add((cout, BATCH * ho * wo))
    out |= {(16, BATCH * 320 * 320), (256, BATCH * 160 * 160), (8, 4096)}
    return sorted(out)


def row_geom(channels, nrows, reduce, resident, sms, red_min_rows=512, elt_waves=2):
    """(cgx, rpb) of csrc/train_kernels.cu's row_geom: channel groups of 8 per block and rows per block."""
    cg = channels // 8
    target = sms * (resident if reduce else elt_waves * resident)
    cgx = next(v for v in (32, 16, 8, 4, 2, 1) if cg >= v)
    while True:
        quantum = (256 // cgx) * 4
        gx = -(-cg // cgx)
        rpb = max(-(-nrows * gx // target), max(red_min_rows, quantum) if reduce else 2 * quantum)
        rpb = -(-rpb // quantum) * quantum
        if not reduce or cgx <= 4 or gx * -(-nrows // rpb) * 5 >= target * 3:
            return cgx, rpb
        cgx >>= 1


STATS_RESIDENT, BWD_RESIDENT = 4, 2  # y5_bn_stats / the reduce pass of y5_bn_act_bwd (Y5_BN_RED_U = 4)


def geometry_coverage(sms):
    """cgx values the BN cases reach in the statistics pass and the backward reduce pass."""
    return ({row_geom(c, r, True, STATS_RESIDENT, sms)[0] for c, r in bn_classes()},
            {row_geom(c, r, True, BWD_RESIDENT, sms)[0] for c, r in bn_classes()})


# ---------------------------------------------------------------------------------------------------------------------
# float64 references: per-tap GEMMs (an implicit GEMM restated; tests/test_train_geometry_cpu.py checks them against
# torch's conv2d / conv2d_weight / conv2d_input)
# ---------------------------------------------------------------------------------------------------------------------
def _taps(x, kh, kw, s, ph, pw):
    """yields (r, c, X): X[(n, oy, ox), ci] = x[n, ci, oy*s - ph + r, ox*s - pw + c] (zero outside)"""
    B, Cc, H, W = x.shape
    Ho, Wo = (H + 2 * ph - kh) // s + 1, (W + 2 * pw - kw) // s + 1
    xp = F.pad(x, (pw, pw, ph, ph))
    for r in range(kh):
        for c in range(kw):
            v = xp[:, :, r : r + s * (Ho - 1) + 1 : s, c : c + s * (Wo - 1) + 1 : s]
            yield r, c, v.permute(0, 2, 3, 1).reshape(-1, Cc)


def conv_ref(x, w, s, ph, pw, taps=None):
    """float64 conv2d(x, w) (no bias); `taps` restricts the sum to a subset of filter taps."""
    B, _, H, W = x.shape
    O, _, kh, kw = w.shape
    Ho, Wo = (H + 2 * ph - kh) // s + 1, (W + 2 * pw - kw) // s + 1
    y = torch.zeros(B * Ho * Wo, O, dtype=torch.float64, device=x.device)
    for r, c, X in _taps(x, kh, kw, s, ph, pw):
        if taps is None or (r, c) in taps:
            y += X @ w[:, :, r, c].T
    return y.view(B, Ho, Wo, O).permute(0, 3, 1, 2)


def wgrad_ref(x, dy, kh, kw, s, ph, pw, pixels=None):
    """float64 dL/dW (O, I, kh, kw) of y = conv2d(x, W); `pixels` (a slice of output pixels n*Ho*Wo + oy*Wo + ox) restricts
    the reduction."""
    O = dy.shape[1]
    d = dy.permute(0, 2, 3, 1).reshape(-1, O)
    pix = slice(None) if pixels is None else pixels
    out = torch.empty(O, x.shape[1], kh, kw, dtype=torch.float64, device=x.device)
    for r, c, X in _taps(x, kh, kw, s, ph, pw):
        out[:, :, r, c] = d[pix].T @ X[pix]
    return out


def dgrad_ref(dy, w, s, p, H, W, taps=None, out_ch=None):
    """float64 dL/dx (B, I, H, W) of y = conv2d(x, w, stride s, padding p); `taps` / `out_ch` restrict the reduction."""
    B, O, Ho, Wo = dy.shape
    _, I, k, _ = w.shape
    d = dy.permute(0, 2, 3, 1).reshape(-1, O)
    oc = slice(None) if out_ch is None else out_ch
    dxp = torch.zeros(B, I, H + 2 * p, W + 2 * p, dtype=torch.float64, device=dy.device)
    for r in range(k):
        for c in range(k):
            if taps is not None and (r, c) not in taps:
                continue
            part = (d[:, oc] @ w[oc, :, r, c]).view(B, Ho, Wo, I).permute(0, 3, 1, 2)
            dxp[:, :, r : r + s * (Ho - 1) + 1 : s, c : c + s * (Wo - 1) + 1 : s] += part
    return dxp[:, :, p : p + H, p : p + W]


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def ulp(x, dtype):
    """spacing of `dtype` at |x| (x float64)"""
    a = x.abs()
    _, e = torch.frexp(a)
    u = torch.ldexp(torch.ones_like(a), e - 1 - _MANT[dtype])
    return torch.where(a > 0, u, torch.zeros_like(u)).clamp_min(_MIN_ULP[dtype])


def _judge(tag, err, bound):
    """max(err / bound) must be <= 1"""
    r = float((err / bound.clamp_min(1e-300)).max())
    print(f"[ratio] {tag}: {r:.3g}")
    assert r <= 1.0, (tag, r)
    return r


def _reject(tag, err, bound):
    """negative control: the bound must reject the perturbed reference"""
    r = float((err / bound.clamp_min(1e-300)).max())
    print(f"[control] {tag}: {r:.3g}")
    assert r > 1.0, (tag, "the bound accepts a perturbed reference", r)
    return r


def _gen(dev, seed):
    return torch.Generator(device=dev).manual_seed(seed)


def _urand(shape, g, dev, lo=-1.0, hi=1.0):
    return torch.rand(*shape, generator=g, device=dev) * (hi - lo) + lo


def _st(dev):
    return C.c_void_p(_lib.stream_ptr(dev))


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last)


def _in_view(data, sliced, fill=float("nan")):
    """(buffer, view, pitch): `data` (rows, C) itself, or a copy at channel offset 8 of a wider buffer (pitch C + 24)
    whose other channels hold `fill`"""
    if not sliced:
        return data, data, data.shape[1]
    rows, c = data.shape
    buf = torch.full((rows, c + 24), fill, dtype=data.dtype, device=data.device)
    buf[:, 8 : 8 + c] = data
    return buf, buf[:, 8 : 8 + c], c + 24


def _out_view(rows, c, dtype, dev, sliced):
    buf = torch.full((rows, c + 24 if sliced else c), SENTINEL, dtype=dtype, device=dev)
    return buf, (buf[:, 8 : 8 + c] if sliced else buf), buf.shape[1]


def _guards_intact(buf, c, sliced):
    return not sliced or bool((buf[:, :8] == SENTINEL).all() and (buf[:, 8 + c :] == SENTINEL).all())


def _fma_round(y64, a32, b32, dtype):
    """round_to_dtype(fmaf(y, a, b)) of the BN kernels: y has <= 11 significant bits, so y*a is exact in float64"""
    return (y64 * a32.double() + b32.double()).float().to(dtype).double()


def _bn_affine(mean, invstd, gamma, beta):
    """a = invstd * gamma, b = beta - mean * a as the kernels form them (fp32, b one fused multiply-add)"""
    a = invstd * gamma
    b = (beta.double() - mean.double() * a.double()).float()
    return a, b


# ---------------------------------------------------------------------------------------------------------------------
# 0. geometry coverage
# ---------------------------------------------------------------------------------------------------------------------
def test_bn_cases_cover_every_reduce_block_geometry(cuda):
    """The BN cases below run the statistics pass and the backward reduce at cgx = 1, 2, 4, 8, 16 and 32 on this GPU.
    (Skipped when a Y5_BN_* tuning variable changes the geometry rule.)"""
    tuned = sorted(k for k in os.environ if k.startswith("Y5_BN_"))
    if tuned:
        pytest.skip(f"BN tuning variables set: {tuned}")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    stats, bwd = geometry_coverage(sms)
    print(f"[geometry] {sms} SMs: statistics cgx {sorted(stats)}, backward reduce cgx {sorted(bwd)}")
    assert stats >= {1, 2, 4, 8, 16, 32} and bwd >= {1, 2, 4, 8, 16, 32}, (stats, bwd)


# ---------------------------------------------------------------------------------------------------------------------
# 1. BatchNorm passes
# ---------------------------------------------------------------------------------------------------------------------
def _bn_case(dev, C_, rows, dtype, seed, sliced=False, alias=False, act=1, residual=False, eval_form=False):
    """y5_bn_stats + y5_bn_act_fwd (training form) + y5_bn_act_bwd on [rows][C_] data whose channels have mean/sigma in
    {0, 4, 16}, checked against float64."""
    lib, st, code = _lib.lib(), _st(dev), _lib.dtype_code(dtype)
    tag = f"C{C_} rows{rows} {str(dtype)[6:]}{' sliced' if sliced else ''}{' alias' if alias else ''}{' act=none' if not act else ''}" \
          f"{' residual' if residual else ''}{' eval' if eval_form else ''}"
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    g = _gen(dev, seed)
    ch = torch.arange(C_, device=dev)
    ratio = torch.tensor([0.0, 4.0, 16.0], device=dev)[ch % 3] * torch.where(ch % 2 == 0, 1.0, -1.0)
    sigma = 0.5 + 1.5 * torch.rand(C_, generator=g, device=dev)
    ydat = (torch.randn(rows, C_, generator=g, device=dev) * sigma + ratio * sigma).to(dtype)
    gamma = 0.5 + torch.rand(C_, generator=g, device=dev)
    beta = torch.rand(C_, generator=g, device=dev) - 0.5
    rm0 = 0.1 * torch.randn(C_, generator=g, device=dev)
    rv0 = 0.5 + torch.rand(C_, generator=g, device=dev)

    # ---- statistics + training forward
    _, y, yp = _in_view(ydat, sliced)
    ws = torch.zeros(2 * C_, dtype=torch.float64, device=dev)
    _lib.check(lib.y5_bn_stats(y.data_ptr(), yp, rows, C_, code, ws.data_ptr(), st), "bn_stats")
    zbuf, z, zp = _out_view(rows, C_, dtype, dev, sliced)
    q = qp = None
    if residual:
        qdat = _urand((rows, C_), g, dev, -2, 2).to(dtype)
        _, q, qp = _in_view(qdat, sliced)
    mean, invstd = torch.empty(C_, device=dev), torch.empty(C_, device=dev)
    rm, rv = rm0.clone(), rv0.clone()
    _lib.check(lib.y5_bn_act_fwd(y.data_ptr(), yp, z.data_ptr(), zp, rows, C_, code, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                 beta.data_ptr(), act, ws.data_ptr(), BN_EPS, BN_MOM, rm.data_ptr(), rv.data_ptr(),
                                 q.data_ptr() if residual else None, qp or 0, st), "bn_act_fwd")
    assert _guards_intact(zbuf, C_, sliced), (tag, "bn_act_fwd wrote outside its channel slice")
    y64 = ydat.double()
    m_ref = y64.mean(0)
    v_ref = y64.var(0, unbiased=False)
    sd = v_ref.sqrt()
    r = m_ref.abs() / sd
    is_ref = 1 / torch.sqrt(v_ref + BN_EPS)
    b_mean = 1e-6 * (sd + m_ref.abs())
    b_is_rel = 1e-6 + 4e-7 * r * r
    _judge(f"stats mean {tag}", (mean.double() - m_ref).abs(), b_mean)
    _judge(f"stats invstd {tag}", (invstd.double() - is_ref).abs() / is_ref, b_is_rel)
    mom = float(torch.tensor(BN_MOM, dtype=torch.float32))
    keep = float(torch.tensor(1.0) - torch.tensor(BN_MOM))
    v_unb = v_ref * rows / (rows - 1)
    rm_ref = keep * rm0.double() + mom * m_ref
    rv_ref = keep * rv0.double() + mom * v_unb
    _judge(f"running_mean {tag}", (rm.double() - rm_ref).abs(), 2.0 ** -22 * (rm0.double().abs() + m_ref.abs()) + mom * b_mean)
    _judge(f"running_var {tag}", (rv.double() - rv_ref).abs(), 2.0 ** -22 * (rv0.double().abs() + v_unb) + mom * v_unb * 2 * b_is_rel)
    # control: one row block of the statistics pass lost (its atomics never landed)
    _, rpb = row_geom(C_, rows, True, STATS_RESIDENT, sms)
    blk = slice(rpb, 2 * rpb) if rows > 2 * rpb else slice(0, rpb)
    s1 = y64.sum(0) - y64[blk].sum(0)
    s2 = (y64 * y64).sum(0) - (y64[blk] ** 2).sum(0)
    m_c = s1 / rows
    is_c = 1 / torch.sqrt((s2 / rows - m_c * m_c).clamp_min(0) + BN_EPS)
    _reject(f"stats lost row block {tag}", torch.maximum((m_c - m_ref).abs() / b_mean, (is_c - is_ref).abs() / is_ref / b_is_rel),
            torch.ones_like(b_mean))
    del s1, s2

    # ---- normalise + activate, given the kernel's statistics
    a32, b32 = _bn_affine(mean, invstd, gamma, beta)
    t = _fma_round(y64, a32, b32, dtype)
    s = t * torch.sigmoid(t) if act else t
    if residual:
        z_ref = s + qdat.double()
        bound = ulp(s.to(dtype).double(), dtype) + ulp(z_ref.to(dtype).double(), dtype)
    else:
        z_ref = s
        bound = ulp(s.to(dtype).double(), dtype)
    _judge(f"bn_act_fwd z {tag}", (z.double() - z_ref).abs(), bound)
    del z_ref, bound, s
    if eval_form:  # statistics given: the same z, running statistics untouched
        rm_e, rv_e = rm.clone(), rv.clone()
        zbuf2, z2, zp2 = _out_view(rows, C_, dtype, dev, sliced)
        _lib.check(lib.y5_bn_act_fwd(y.data_ptr(), yp, z2.data_ptr(), zp2, rows, C_, code, mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(),
                                     beta.data_ptr(), act, None, BN_EPS, BN_MOM, rm_e.data_ptr(), rv_e.data_ptr(),
                                     q.data_ptr() if residual else None, qp or 0, st), "bn_act_fwd eval")
        assert torch.equal(z2, z) and torch.equal(rm_e, rm) and torch.equal(rv_e, rv), tag
        assert _guards_intact(zbuf2, C_, sliced), tag
        del zbuf2, z2
    del zbuf, z

    # ---- backward
    dzdat = _urand((rows, C_), g, dev).to(dtype)
    dz_keep = dzdat.double()
    if alias:  # dy is dz: same pointer, same pitch
        dzbuf, dz, dzp = _in_view(dzdat.clone(), sliced, SENTINEL)
        dybuf, dy, dyp = dzbuf, dz, dzp
    else:
        _, dz, dzp = _in_view(dzdat, sliced)
        dybuf, dy, dyp = _out_view(rows, C_, dtype, dev, sliced)
    dg, db = torch.empty(C_, device=dev), torch.empty(C_, device=dev)
    ws = torch.zeros(2 * C_, dtype=torch.float64, device=dev)
    _lib.check(lib.y5_bn_act_bwd(y.data_ptr(), yp, dz.data_ptr(), dzp, dy.data_ptr(), dyp, rows, C_, code, mean.data_ptr(), invstd.data_ptr(),
                                 gamma.data_ptr(), beta.data_ptr(), act, dg.data_ptr(), db.data_ptr(), ws.data_ptr(), st), "bn_act_bwd")
    assert _guards_intact(dybuf, C_, sliced), (tag, "bn_act_bwd wrote outside its channel slice")
    if act:
        sg = torch.sigmoid(t)
        du_x = dz_keep * sg * (1 + t * (1 - sg))
        du = du_x.to(dtype).double()
        # the kernel evaluates dz * silu'(t) in fp32 with fast exp / divide (~1e-6 of the magnitude of its terms): where that
        # lands within reach of a rounding boundary of the dtype, either neighbour is a correct result.  `flip` is the
        # distance between the two (0 elsewhere).
        reach = 2.0 ** -19 * dz_keep.abs() * sg * (1 + t.abs() * (1 - sg))
        flip = ((du_x + reach).to(dtype).double() - (du_x - reach).to(dtype).double()).abs()
        del sg, du_x, reach
    else:
        du, flip = dz_keep, torch.zeros_like(dz_keep)
    del t, dz_keep
    m64, is64 = mean.double(), invstd.double()
    xh = (y64 - m64) * is64
    dg_ref, db_ref = (du * xh).sum(0), du.sum(0)
    l1_dg, l1_db = (du * xh).abs().sum(0), du.abs().sum(0)
    b_dg = 2e-6 * l1_dg + 2.0 ** -21 * (m64 * is64).abs() * l1_db + (flip * xh.abs()).sum(0)
    b_db = 2e-6 * l1_db + flip.sum(0)
    _judge(f"dgamma {tag}", (dg.double() - dg_ref).abs(), b_dg)
    _judge(f"dbeta {tag}", (db.double() - db_ref).abs(), b_db)
    # control: one row block of the reduce pass lost
    _, rpb = row_geom(C_, rows, True, BWD_RESIDENT, sms)
    blk = slice(rpb, 2 * rpb) if rows > 2 * rpb else slice(0, rpb)
    _reject(f"bwd reduce lost row block {tag}",
            torch.maximum((du[blk] * xh[blk]).sum(0).abs() / b_dg, du[blk].sum(0).abs() / b_db), torch.ones_like(b_dg))
    del xh
    a64 = is64 * gamma.double()
    dgn, dbn = dg.double() / rows, db.double() / rows
    c1 = -is64 * dgn * a64
    c0 = -(dbn - m64 * is64 * dgn) * a64
    dy_ref = du * a64 + y64 * c1 + c0
    scale = (du * a64).abs() + (y64 * c1).abs() + c0.abs()
    del du
    # 2 u of the scale, floored at the dtype's smallest spacing (dy may be subnormal), plus a du rounded the other way
    _judge(f"bn_act_bwd dy {tag}", (dy.double() - dy_ref).abs(), 2 * EPS[dtype] * scale + _MIN_ULP[dtype] + flip * a64.abs())


BN_BF16 = {(48, BATCH * 320 * 320), (96, BATCH * 160 * 160), (192, BATCH * 80 * 80), (384, BATCH * 40 * 40), (256, BATCH * 160 * 160), (8, 4096)}


@pytest.mark.parametrize("C_,rows,dtype", [(c, r, torch.float16) for c, r in bn_classes()]
                         + [(c, r, torch.bfloat16) for c, r in bn_classes() if (c, r) in BN_BF16])
def test_bn_passes_at_training_shapes(cuda, C_, rows, dtype):
    _bn_case(cuda, C_, rows, dtype, seed=C_ * 7 + rows % 9973)


BN_VIEW_SHAPES = [(48, 1000), (96, BATCH * 160 * 160)]  # small, production (yolov5m 96 x 409 600)


@pytest.mark.parametrize("variant", ["sliced", "alias", "act_none", "residual", "eval"])
@pytest.mark.parametrize("C_,rows", BN_VIEW_SHAPES)
def test_bn_views_and_contracts(cuda, C_, rows, variant):
    """Channel-slice views of y, z, dz, dy and the residual (offset 8, wider pitch, guards checked); dy aliasing dz (also
    sliced); act = Y5_ACT_NONE in the backward; the eval form of the forward (sums = NULL)."""
    kw = dict(sliced=variant in ("sliced", "residual"), alias=variant == "alias", act=0 if variant == "act_none" else 1,
              residual=variant == "residual", eval_form=variant == "eval")
    if variant == "alias":
        _bn_case(cuda, C_, rows, torch.float16, seed=11, alias=True, sliced=True)
    _bn_case(cuda, C_, rows, torch.float16, seed=11, **kw)


@pytest.mark.parametrize("rows", [1000, BATCH * 80 * 80])
@pytest.mark.parametrize("C_", [48, 80, 320])
def test_bn_partly_empty_last_block(cuda, C_, rows):
    """Channel counts whose last block of cgx groups is partly empty."""
    _bn_case(cuda, C_, rows, torch.float16, seed=13 + C_)


# ---------------------------------------------------------------------------------------------------------------------
# 2. weight gradient
# ---------------------------------------------------------------------------------------------------------------------
def _wgrad_check(tag, got, x64, dy64, k, s, p, kw=None, pw=None):
    kw = k if kw is None else kw
    pw = p if pw is None else pw
    ref = wgrad_ref(x64, dy64, k, kw, s, p, pw)
    l1 = wgrad_ref(x64.abs(), dy64.abs(), k, kw, s, p, pw)
    bound = 1e-5 * l1
    r = _judge(f"wgrad {tag}", (got.double() - ref).abs(), bound)
    M = dy64.shape[0] * dy64.shape[2] * dy64.shape[3]
    m0 = (M // 2) // 64 * 64
    lost = wgrad_ref(x64, dy64, k, kw, s, p, pw, pixels=slice(m0, min(M, m0 + 64)))
    _reject(f"wgrad lost 64-pixel K block {tag}", lost.abs(), bound)
    return r


def _conv_layers():
    return [l for l in layer_table() if l[2] != 6]  # the stem runs through the wide-pixel path (section 3)


@pytest.mark.parametrize("cin,cout,k,s,H,W", _conv_layers())
def test_conv_wgrad_every_layer(cuda, cin, cout, k, s, H, W):
    """train_ops.conv_wgrad at every distinct yolov5m layer of the 16 x 640^2 step (Detect's 255 outputs padded to 256,
    as the training step pads them); fp16, and bf16 on the 3x3 layers."""
    p = k // 2
    co = (cout + 7) // 8 * 8
    ho, wo = out_hw(H, W, k, s)
    g = _gen(cuda, cin * 31 + cout + H)
    for dtype in (torch.float16, torch.bfloat16) if k == 3 else (torch.float16,):
        x = _cl(_urand((BATCH, cin, H, W), g, cuda).to(dtype))
        dy = _cl(_urand((BATCH, co, ho, wo), g, cuda).to(dtype))
        got = train_ops.conv_wgrad(x, dy, k, s, p)
        _wgrad_check(f"{cin}->{co} k{k} s{s} {H}x{W} {str(dtype)[6:]}", got, x.double(), dy.double(), k, s, p)
        del x, dy, got


@pytest.mark.parametrize("case", [(2, 20, 20, 96, 48, 3, 1), (BATCH, 80, 80, 192, 96, 1, 1), (BATCH, 40, 40, 384, 192, 3, 2),
                                  (BATCH, 20, 20, 1536, 768, 1, 1)])
def test_conv_wgrad_slices_and_accumulate(cuda, case):
    """x and dy as channel slices of concat buffers (in_pitch != in_c, dout_pitch != out_c, what _nhwc hands over), and
    accumulate = 1 onto a non-zero dW through the C ABI."""
    B, H, W, cin, cout, k, s = case
    p = k // 2
    ho, wo = out_hw(H, W, k, s)
    dtype = torch.float16
    g = _gen(cuda, 17 + cin)
    xbuf = _cl(torch.full((B, cin + 48, H, W), float("nan"), dtype=dtype, device=cuda))
    xbuf[:, 8 : 8 + cin] = _urand((B, cin, H, W), g, cuda).to(dtype)
    dbuf = _cl(torch.full((B, cout + 56, ho, wo), float("nan"), dtype=dtype, device=cuda))
    dbuf[:, 48 : 48 + cout] = _urand((B, cout, ho, wo), g, cuda).to(dtype)
    x, dy = xbuf[:, 8 : 8 + cin], dbuf[:, 48 : 48 + cout]
    tag = f"{cin}->{cout} k{k} s{s} {B}x{H}x{W}"
    got = train_ops.conv_wgrad(x, dy, k, s, p)
    x64, dy64 = x.double(), dy.double()
    _wgrad_check(f"slices {tag}", got, x64, dy64, k, s, p)
    # accumulate = 1: dW (KRSC) += gradient
    dw0 = torch.randn(cout, k, k, cin, generator=g, device=cuda)
    dw = dw0.clone()
    d = _lib.WgradDesc()
    d.inp, d.in_pitch = x.data_ptr(), xbuf.shape[1]
    d.batch, d.in_h, d.in_w, d.in_c = B, H, W, cin
    d.dout, d.dout_pitch, d.out_c = dy.data_ptr(), dbuf.shape[1], cout
    d.dweight = dw.data_ptr()
    d.ksize, d.stride, d.pad = k, s, p
    d.dtype, d.accumulate = _lib.dtype_code(dtype), 1
    _lib.check(_lib.lib().y5_conv_wgrad(C.byref(d), _st(cuda)), "conv_wgrad accumulate")
    ref = wgrad_ref(x64, dy64, k, k, s, p, p).permute(0, 2, 3, 1) + dw0.double()
    l1 = wgrad_ref(x64.abs(), dy64.abs(), k, k, s, p, p).permute(0, 2, 3, 1)
    _judge(f"wgrad accumulate {tag}", (dw.double() - ref).abs(), 1e-5 * l1 + 2.0 ** -23 * ref.abs())
    _reject(f"wgrad accumulate ignored {tag}", dw0.double().abs(), 1e-5 * l1 + 2.0 ** -23 * ref.abs())


# ---------------------------------------------------------------------------------------------------------------------
# 3. wide-pixel stem and the generalised conv descriptor
# ---------------------------------------------------------------------------------------------------------------------
STEM_SHAPES = [(BATCH, 640, 640), (2, 64, 96), (1, 32, 608)]


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("O", [16, 32, 48, 64, 80])
@pytest.mark.parametrize("B,H,W", STEM_SHAPES)
def test_wide_pixel_stem_matches_6x6_conv(cuda, B, H, W, O, dtype):
    """y5_stem_s2d (one zero cell either side of every row) + stem_conv_wide / stem_wgrad_wide (3x1 conv over overlapping
    48-channel pixels) + the _stem_index mapping, against float64 conv2d(img, w, stride 2, padding 2) and its weight
    gradient."""
    lib, code = _lib.lib(), _lib.dtype_code(dtype)
    g = _gen(cuda, O * 13 + H + W)
    img = torch.rand(B, 3, H, W, generator=g, device=cuda).to(dtype)
    w = _urand((O, 3, 6, 6), g, cuda) * 0.2
    buf = torch.zeros(B, H // 2, W // 2 + 2, 16, dtype=dtype, device=cuda)
    _lib.check(lib.y5_stem_s2d(img.data_ptr(), code, buf.data_ptr(), code, B, H, W, W // 2 + 2, 1, _st(cuda)), "stem_s2d")
    fwd_idx, inv_idx = train_ops._stem_index(cuda)
    wf = w.flatten(1)
    w3 = torch.cat((wf, wf.new_zeros(O, 1)), 1)[:, fwd_idx].view(O, 16, 3, 3)
    y = train_ops.stem_conv_wide(buf, w3)
    img64, w64 = img.double(), w.to(dtype).double()
    tag = f"O{O} {B}x{H}x{W} {str(dtype)[6:]}"
    ref = conv_ref(img64, w64, 2, 2, 2)
    bound = ulp(ref.to(dtype).double(), dtype) + 2.0 ** -16 * conv_ref(img64.abs(), w64.abs(), 2, 2, 2)
    _judge(f"stem fwd {tag}", (y.double() - ref).abs(), bound)
    # control: one cell of the wide pixel (filter columns 0-1 of the 6x6 filter) dropped
    _reject(f"stem fwd lost wide-pixel cell {tag}", conv_ref(img64, w64, 2, 2, 2, taps={(r, c) for r in range(6) for c in (0, 1)}).abs(), bound)
    del ref, bound, y
    dy = _cl(_urand((B, O, H // 2, W // 2), g, cuda).to(dtype))
    gw = train_ops.stem_wgrad_wide(buf, dy)
    g6 = gw.reshape(O, -1)[:, inv_idx].view(O, 3, 6, 6)
    _wgrad_check(f"stem {tag}", g6, img64, dy.double(), 6, 2, 2)


def _conv_desc_run(dev, dtype, B, H, W, cin, cout, kh, kw, s, ph, pw, a_mode, gap_y=0, gap_n=0, seed=0):
    """y5_conv_bn_silu_fwd with kw / pad_w and (optionally) gapped row / image strides; gaps and padding channels hold NaN.
    Returns (return code, output, float64 reference, bound, (x, w, b) in float64)."""
    lib = _lib.lib()
    g = _gen(dev, seed)
    x = _urand((B, cin, H, W), g, dev).to(dtype)
    w = _urand((cout, cin, kh, kw), g, dev) / math.sqrt(cin * kh * kw) * 2
    b = torch.rand(cout, generator=g, device=dev) - 0.5
    pitch = cin + 8
    ys = (W + gap_y) * pitch
    ns = (H * (W + gap_y) + gap_n) * pitch
    flat = torch.full((B * ns + 64,), float("nan"), dtype=dtype, device=dev)
    flat.as_strided((B, H, W, cin), (ns, ys, pitch, 1)).copy_(x.permute(0, 2, 3, 1))
    Ho, Wo = (H + 2 * ph - kh) // s + 1, (W + 2 * pw - kw) // s + 1
    out = torch.full((B, Ho, Wo, cout), SENTINEL, dtype=dtype, device=dev)
    bk = C.c_int32()
    _lib.check(lib.y5_conv_pick(cin, cout, B * Ho * Wo, C.byref(bk), None), "conv_pick")
    wp = pack_weight(w, bk.value, dtype)
    d = _lib.ConvDesc()
    d.inp, d.in_pitch = flat.data_ptr(), pitch
    d.batch, d.in_h, d.in_w, d.in_c = B, H, W, cin
    d.weight, d.bias = wp.data_ptr(), b.data_ptr()
    d.out, d.out_pitch, d.out_c = out.data_ptr(), cout, cout
    d.ksize, d.stride, d.pad = kh, s, ph
    d.kw, d.pad_w = kw, pw
    d.in_x_stride, d.in_y_stride, d.in_n_stride = (pitch, ys, ns) if (gap_y or gap_n) else (0, 0, 0)
    d.act, d.dtype, d.block_k, d.block_n, d.a_mode = _lib.ACT_SILU, _lib.dtype_code(dtype), bk.value, 0, a_mode
    rc = lib.y5_conv_bn_silu_fwd(C.byref(d), _st(dev))
    x64, w64 = x.double(), w.to(dtype).double()
    acc = conv_ref(x64, w64, s, ph, pw) + b.double().view(1, -1, 1, 1)
    ref = acc * torch.sigmoid(acc)
    bound = ulp(ref.to(dtype).double(), dtype) + 2.0 ** -16 * (conv_ref(x64.abs(), w64.abs(), s, ph, pw) + b.double().abs().view(1, -1, 1, 1))
    return rc, out.permute(0, 3, 1, 2), ref, bound, (x64, w64, b.double().view(1, -1, 1, 1))


@pytest.mark.parametrize("a_mode", [1, 2])
@pytest.mark.parametrize("case", [
    # B, H, W, cin, cout, kh, kw, s, ph, pw, gap_y, gap_n
    (2, 20, 24, 64, 64, 3, 1, 1, 1, 0, 0, 0),       # 3x1
    (2, 20, 24, 64, 32, 1, 3, 1, 0, 1, 0, 0),       # 1x3
    (2, 24, 24, 32, 64, 5, 3, 1, 2, 1, 0, 0),       # 5x3
    (2, 13, 27, 64, 64, 3, 3, 1, 1, 1, 3, 40),      # gapped row and image strides, partial tiles
    (BATCH, 40, 40, 48, 96, 3, 3, 1, 1, 1, 2, 8),   # yolov5m widths, gapped
    (2, 16, 24, 32, 64, 3, 3, 2, 1, 1, 1, 16),      # stride 2 (TMA im2col only)
])
def test_conv_descriptor_generalisations(cuda, case, a_mode):
    """y5_conv_bn_silu_fwd with kw != ksize, pad_w != pad and gapped in_y_stride / in_n_stride (gaps hold NaN), in both
    activation fetch modes where the stride is 1, against float64 conv2d on the dense tensor."""
    B, H, W, cin, cout, kh, kw, s, ph, pw, gy, gn = case
    if s != 1 and a_mode == 2:
        pytest.skip("shifted-patch fetch is stride-1 only")
    rc, got, ref, bound, (x64, w64, b64) = _conv_desc_run(cuda, torch.float16, B, H, W, cin, cout, kh, kw, s, ph, pw, a_mode, gy, gn, seed=sum(case))
    _lib.check(rc, "conv (generalised descriptor)")
    tag = f"{kh}x{kw} s{s} pad {ph},{pw} gaps {gy},{gn} a_mode {a_mode}"
    _judge(f"conv desc {tag}", (got.double() - ref).abs(), bound)
    # control: the taps of the last filter column dropped
    acc = conv_ref(x64, w64, s, ph, pw, taps={(r, c) for r in range(kh) for c in range(kw - 1)}) + b64 if kw > 1 else b64 + conv_ref(
        x64, w64, s, ph, pw, taps={(r, 0) for r in range(kh - 1)})
    _reject(f"conv desc lost filter column {tag}", (acc * torch.sigmoid(acc) - ref).abs(), bound)


@pytest.mark.parametrize("kh,kw,ph,pw", [(3, 9, 1, 4), (8, 1, 0, 0), (1, 3, 0, 4), (3, 3, 4, 1)])
def test_conv_descriptor_rejects_unimplemented_shapes(cuda, kh, kw, ph, pw):
    """filters wider than 7 taps or padding wider than the filter: Y5_E_UNSUPPORTED, output untouched"""
    lib = _lib.lib()
    dt = torch.float16
    x = torch.zeros(1, 8, 8, 16, dtype=dt, device=cuda)
    w = torch.zeros(16, 8 * 8 * 16, dtype=dt, device=cuda)
    b = torch.zeros(16, device=cuda)
    out = torch.full((1, 16, 16, 16), SENTINEL, dtype=dt, device=cuda)
    d = _lib.ConvDesc()
    d.inp, d.in_pitch, d.batch, d.in_h, d.in_w, d.in_c = x.data_ptr(), 16, 1, 8, 8, 16
    d.weight, d.bias, d.out, d.out_pitch, d.out_c = w.data_ptr(), b.data_ptr(), out.data_ptr(), 16, 16
    d.ksize, d.stride, d.pad, d.kw, d.pad_w = kh, 1, ph, kw, pw
    d.act, d.dtype, d.block_k = _lib.ACT_SILU, _lib.Y5_F16, 16
    assert lib.y5_conv_bn_silu_fwd(C.byref(d), _st(cuda)) == -2  # Y5_E_UNSUPPORTED
    torch.cuda.synchronize()
    assert bool((out == SENTINEL).all())


# ---------------------------------------------------------------------------------------------------------------------
# 4. data gradient and glue
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,cout,k,s,H,W", _conv_layers())
def test_conv_dgrad_every_layer(cuda, cin, cout, k, s, H, W):
    """train_ops.conv_dgrad (stride 2 through y5_zero_stuff2x) at every distinct yolov5m layer of the 16 x 640^2 step; the
    first and the last image against float64."""
    p = k // 2
    co = (cout + 7) // 8 * 8
    ho, wo = out_hw(H, W, k, s)
    dtype = torch.float16
    g = _gen(cuda, cin * 17 + cout + W)
    w = torch.zeros(co, cin, k, k, device=cuda)
    w[:cout] = _urand((cout, cin, k, k), g, cuda) / math.sqrt(cout * k * k) * 2
    dy = _cl(_urand((BATCH, co, ho, wo), g, cuda).to(dtype))
    dx = train_ops.conv_dgrad(dy, w, k, s, p, (H, W))
    sel = [0, BATCH - 1]
    dy64, w64 = dy[sel].double(), w.to(dtype).double()
    ref = dgrad_ref(dy64, w64, s, p, H, W)
    bound = ulp(dgrad_ref(dy64.abs(), w64.abs(), s, p, H, W), dtype)
    tag = f"{cin}<-{co} k{k} s{s} {H}x{W}"
    _judge(f"dgrad {tag}", (dx[sel].double() - ref).abs(), bound)
    _reject(f"dgrad lost 64-channel K block {tag}", dgrad_ref(dy64, w64, s, p, H, W, taps={(0, 0)}, out_ch=slice(0, 64)).abs(), bound)


@pytest.mark.parametrize("hw", [80, 40, 20])
def test_col_sum_detect_levels(cuda, hw):
    """y5_col_sum over the gradient of a Detect level (255 outputs padded to 256 channels), 16 images."""
    rows, c = BATCH * hw * hw, 256
    dy = _urand((rows, c), _gen(cuda, hw), cuda).to(torch.float16)
    out = torch.empty(c, device=cuda)
    ws = torch.empty(2 * c, dtype=torch.float64, device=cuda)
    _lib.check(_lib.lib().y5_col_sum(dy.data_ptr(), c, rows, c, _lib.Y5_F16, out.data_ptr(), ws.data_ptr(), _st(cuda)), "col_sum")
    d64 = dy.double()
    ref = d64.sum(0)
    bound = 2e-6 * d64.abs().sum(0) + 2.0 ** -23 * ref.abs()
    _judge(f"col_sum {hw}x{hw}", (out.double() - ref).abs(), bound)
    _, rpb = row_geom(c, rows, True, STATS_RESIDENT, torch.cuda.get_device_properties(cuda).multi_processor_count)
    _reject(f"col_sum lost row block {hw}x{hw}", d64[rpb : 2 * rpb].sum(0).abs(), bound)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("c,h", [(384, 20), (192, 40)])
def test_upsample2x_bwd_from_concat_slice(cuda, c, h, dtype):
    """y5_upsample2x_bwd at the two yolov5m upsamples of the 16 x 640^2 step, reading dy as the leading channel slice of the
    following Concat's gradient (pitch 2c), as torch.cat's backward hands it over."""
    g = _gen(cuda, c + h)
    dcat = _cl(_urand((BATCH, 2 * c, 2 * h, 2 * h), g, cuda).to(dtype))
    dy = dcat[:, :c]
    dx = _cl(torch.empty(BATCH, c, h, h, dtype=dtype, device=cuda))
    _lib.check(_lib.lib().y5_upsample2x_bwd(dy.data_ptr(), 2 * c, dx.data_ptr(), c, BATCH, h, h, c, _lib.dtype_code(dtype), _st(cuda)),
               "upsample2x_bwd")
    ref = F.avg_pool2d(dy.double(), 2) * 4
    _judge(f"upsample2x_bwd {c}x{h} {str(dtype)[6:]}", (dx.double() - ref).abs(), ulp(ref.to(dtype).double(), dtype))


@pytest.mark.parametrize("dtype,levels", [(torch.float16, 4), (torch.float16, 1000), (torch.bfloat16, 4)])
def test_sppf_pool_bwd_config4(cuda, dtype, levels):
    """y5_sppf_pool_bwd at yolov5m's SPPF (16 x 20 x 20 x 384); 4 distinct input values put arg-max ties everywhere (the
    first maximum in row-major window order takes the gradient, as torch's max_pool2d backward does)."""
    B, c, h, w = BATCH, 384, 20, 20
    g = _gen(cuda, levels)
    a = (torch.randint(0, levels, (B, c, h, w), generator=g, device=cuda).double() / levels - 0.5).to(dtype)
    y1 = F.max_pool2d(a, 5, 1, 2)
    y2 = F.max_pool2d(y1, 5, 1, 2)
    cat = _cl(torch.cat((a, y1, y2, F.max_pool2d(y2, 5, 1, 2)), 1))
    dcat = _cl(_urand((B, 4 * c, h, w), g, cuda).to(dtype))
    da = _cl(torch.empty(B, c, h, w, dtype=dtype, device=cuda))
    ws = torch.empty(3 * B * h * w * c, dtype=torch.float32, device=cuda)
    _lib.check(_lib.lib().y5_sppf_pool_bwd(cat.data_ptr(), 4 * c, dcat.data_ptr(), 4 * c, da.data_ptr(), c, B, h, w, c, 5, _lib.dtype_code(dtype),
                                          ws.data_ptr(), _st(cuda)), "sppf_pool_bwd")

    def route(gcat):
        ar = a.double().requires_grad_(True)
        z1 = F.max_pool2d(ar, 5, 1, 2)
        z2 = F.max_pool2d(z1, 5, 1, 2)
        torch.cat((ar, z1, z2, F.max_pool2d(z2, 5, 1, 2)), 1).backward(gcat)
        return ar.grad

    ref = route(dcat.double())
    bound = ulp(ref.to(dtype).double(), dtype) + 2.0 ** -20 * route(dcat.double().abs())
    _judge(f"sppf_pool_bwd levels {levels} {str(dtype)[6:]}", (da.double() - ref).abs(), bound)
