"""GPU: the bfloat16 2x2x2 maximum (MaxDown2x2x2 on bfloat16 volumes) and LSSViewTransformerRaw's
`ds_dtype=torch.bfloat16`.

Contract.  MaxDown2x2x2 on a bfloat16 tensor is, bit for bit, the reference expression on that
tensor (view / permute / reshape, then torch.max(dim=-1).values) and its gradient.  The Raw neck
with ds_dtype=bfloat16 returns, when a gradient is wanted, the float32 neck's output cast to
bfloat16, and the float32 neck's depth / feature gradients for the widened output gradient; without
a gradient it returns the same values (==), and the same bits on inputs whose window sums are
never nonzero below 2^-134.  NaN positions must match; NaN payloads are not compared."""
import pytest
import torch

from tests.test_channels_last_gpu import _is_cl_view, _neck_inputs
from veon_b200 import synthetic as S

pytestmark = pytest.mark.gpu
CL = torch.channels_last_3d
BF = torch.bfloat16
FORMATS = (torch.contiguous_format, CL)


def same_bits(a, b):
    """equal dtype, shape and bits, NaN positions included (payloads not compared)"""
    assert a.dtype == b.dtype and a.shape == b.shape
    na, nb = torch.isnan(a), torch.isnan(b)
    assert torch.equal(na, nb)
    view = torch.int16 if a.dtype == BF else torch.int32
    assert torch.equal(a.masked_fill(na, 0).contiguous().view(view),
                       b.masked_fill(nb, 0).contiguous().view(view))


def reference_max(x):
    """view_transformer_raw.py:549-553 (rearrange + torch.max(dim=-1).values) on x's values"""
    b, c, z, y, w = x.shape
    v = x.view(b, c, z // 2, 2, y // 2, 2, w // 2, 2).permute(0, 1, 2, 4, 6, 3, 5, 7)
    return torch.max(v.reshape(b, c, z // 2, y // 2, w // 2, -1), dim=-1).values


def _bf16_volume(shape, g):
    """ties (few distinct values), zeros of both signs, NaN"""
    x = (torch.randint(-3, 4, shape, generator=g).float() * 0.5)
    x = torch.where(torch.rand(shape, generator=g) < 0.3, torch.randn(shape, generator=g), x)
    x[torch.rand(shape, generator=g) < 0.1] = -0.0
    x.view(-1)[3] = float("nan")
    x.view(-1)[-5] = float("nan")
    return x.to(BF).cuda()


@pytest.mark.parametrize("fmt", FORMATS)
def test_maxdown2x2x2_bf16_is_the_reference_expression(fmt):
    from veon_b200 import bev_pool as BP
    g = torch.Generator().manual_seed(21)
    shapes = [(2, 5, 6, 10, 24), (1, 7, 4, 6, 8), (3, 64, 2, 4, 4), (1, 3, 8, 8, 16)]
    if fmt is CL:
        shapes.append((2, 3, 4, 6, 6))            # X % 4 != 0: channels-last only
    for shape in shapes:
        x = _bf16_volume(shape, g)
        ours = x.contiguous(memory_format=fmt).clone().requires_grad_()
        ref = x.clone().requires_grad_()
        assert BP.MaxDown2x2x2.supports(ours), shape
        BP.enable_kernel_timing(True)
        o = BP.MaxDown2x2x2.apply(ours)
        r = reference_max(ref)
        assert o.dtype == BF and (_is_cl_view(o) if fmt is CL else o.is_contiguous())
        same_bits(o, r)
        go = torch.randn(r.shape, generator=g).to(BF).cuda()
        o.backward(go.contiguous(memory_format=fmt))
        r.backward(go)
        used = set(BP.kernel_timings_ms())
        BP.enable_kernel_timing(False)
        sfx = "_cl" if fmt is CL else ""
        assert {f"maxdown{sfx}_fwd_bf16", f"maxdown{sfx}_bwd_bf16"} <= used, used
        assert ours.grad.dtype == BF and ours.grad.is_contiguous(memory_format=fmt)
        same_bits(ours.grad, ref.grad)
    # -0 against +0 in one window, either order: the first one is the maximum and takes the
    # gradient, as in torch.max
    x = torch.zeros(1, 1, 2, 2, 4)
    x[0, 0, 0, 0, 0] = -0.0
    x[0, 0, 0, 0, 2:] = torch.tensor([0.0, -0.0])
    x = x.to(BF).cuda()
    for f in FORMATS:
        same_bits(BP.MaxDown2x2x2.apply(x.contiguous(memory_format=f)).contiguous(),
                  reference_max(x))


def test_zero_sign_caveat_of_the_bf16_maximum():
    """bfloat16 maximum of x.to(bf16) against the float32 maximum of x cast: equal values; the
    bits differ only at zero results (a nonzero sum below 2^-134 rounds to a signed zero)"""
    from veon_b200 import bev_pool as BP
    g = torch.Generator().manual_seed(5)
    shape = (2, 3, 4, 6, 8)
    tiny = float.fromhex("0x1p-140")
    x = torch.randn(shape, generator=g)
    pick = torch.rand(shape, generator=g)
    x[pick < 0.5] = tiny * torch.sign(x[pick < 0.5])
    x[pick < 0.15] = 0.0
    x[pick < 0.05] = -0.0
    x[0, 0, 0, 0, 0:2] = torch.tensor([-0.0, tiny])     # float32: +tiny -> +0; bfloat16: -0 first
    x[0, 0, 0, 1, 0:2] = -1.0
    x[0, 0, 1, 0:2, 0:2] = -1.0
    x = x.cuda()
    assert bool(((x != 0) & (x.abs() < 2.0 ** -134)).any())
    for fmt in FORMATS:
        xf = x.contiguous(memory_format=fmt)
        a = BP.MaxDown2x2x2.apply(xf.to(BF))
        b = BP.MaxDown2x2x2.apply(xf).to(BF)
        assert torch.equal(a, b)
        differ = a.contiguous().view(torch.int16) != b.contiguous().view(torch.int16)
        assert bool(differ.any()) and bool((a.contiguous()[differ] == 0).all())


# ---------------------------------------------------------------- the Raw neck
def _raw(fmt, ds_dtype, C, cfg=None, **kw):
    from veon_b200.view_transformer import LSSViewTransformerRaw
    cfg = cfg or S.CONFIGS["small"]
    return LSSViewTransformerRaw(kw.pop("grid_config", cfg.grid_config), cfg.input_size,
                                 cfg.downsample, 8, C, memory_format=fmt, ds_dtype=ds_dtype, **kw)


def _train(neck, feat5, depth5, metas, go):
    from veon_b200 import bev_pool as BP
    f = feat5.detach().clone().requires_grad_()
    d = depth5.detach().clone().requires_grad_()
    BP.enable_kernel_timing(True)
    out = neck([f] + metas, d)
    out.backward(go)
    used = set(BP.kernel_timings_ms())
    BP.enable_kernel_timing(False)
    return out.detach(), d.grad, f.grad, used


def _infer(neck, feat5, depth5, metas):
    from veon_b200 import bev_pool as BP
    BP.enable_kernel_timing(True)
    with torch.no_grad():
        out = neck([feat5] + metas, depth5)
    used = set(BP.kernel_timings_ms())
    BP.enable_kernel_timing(False)
    return out, used


def _check_training(fmt, C, feat5, depth5, metas, go_bf, cfg=None, **kw):
    """bf16 output = float32 output cast; gradients = float32 neck's for go_bf.float()"""
    a, da, fa, ua = _train(_raw(fmt, torch.float32, C, cfg, **kw), feat5, depth5, metas,
                           go_bf.float())
    b, db, fb, ub = _train(_raw(fmt, BF, C, cfg, **kw), feat5, depth5, metas, go_bf)
    assert b.dtype == BF and b.stride() == a.stride()
    same_bits(b, a.to(BF))
    same_bits(db, da)
    assert fb.dtype == feat5.dtype
    same_bits(fb, fa)
    return ub, b


def _check_inference(fmt, C, feat5, depth5, metas, cfg=None, **kw):
    """the values and (no sum below 2^-134 here) the bits of the float32 neck cast"""
    a, _ = _infer(_raw(fmt, torch.float32, C, cfg, **kw), feat5, depth5, metas)
    b, ub = _infer(_raw(fmt, BF, C, cfg, **kw), feat5, depth5, metas)
    assert b.dtype == BF and b.stride() == a.stride()
    nan = torch.isnan(a)
    assert bool(((b == a.to(BF)) | nan).all())
    same_bits(b, a.to(BF))
    return ub, b


def _small_inputs(feat_dtype, B=2, C=64):
    cfg = S.CONFIGS["small"]
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=6)
    H, W = cfg.feat_hw
    feat = feat.clamp(min=0.0)                    # many sums exactly 0: ties beside empty voxels
    feat[:, 3, 4, :] = float("nan")               # NaNs that reach the volume
    feat5 = feat.view(B, cfg.n_cams, C, H, W).to(feat_dtype)
    depth5 = depth.view(B, cfg.n_cams, cfg.D, H, W)
    go = torch.randn(B, C, 8, 100, 100, generator=torch.Generator().manual_seed(7))
    return feat5, depth5, metas, go.to(BF).cuda()


@pytest.mark.parametrize("feat_dtype", [torch.float32, BF])
def test_raw_neck_bf16_training_channels_first(feat_dtype):
    feat5, depth5, metas, go = _small_inputs(feat_dtype)
    used, out = _check_training(torch.contiguous_format, 64, feat5, depth5, metas, go)
    sfx = "_bf16feat" if feat_dtype == BF else ""
    assert out.is_contiguous()
    assert {"maxdown_fwd_mask_bf16", "pool_bwd_ds_bf16" + sfx} <= used, used
    # one node: no full-resolution gradient, no float32 reduced volume
    assert not used & {"maxdown_fwd", "maxdown_bwd", "pool_bwd", "pool_bwd_bf16",
                       "pool_bwd_ds" + sfx}, used


@pytest.mark.parametrize("feat_dtype", [torch.float32, BF])
def test_raw_neck_bf16_training_channels_last(feat_dtype):
    feat5, depth5, metas, go = _small_inputs(feat_dtype)
    used, out = _check_training(CL, 64, feat5, depth5, metas, go)
    sfx = "_bf16feat" if feat_dtype == BF else ""
    assert _is_cl_view(out)
    assert {"pool_fwd_cl" + sfx, "maxdown_cl_fwd", "maxdown_cl_bwd", "pool_bwd_cl" + sfx} <= used


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("feat_dtype", [torch.float32, BF])
def test_raw_neck_bf16_inference(fmt, feat_dtype):
    feat5, depth5, metas, _ = _small_inputs(feat_dtype)
    used, out = _check_inference(fmt, 64, feat5, depth5, metas)
    sfx = "_bf16feat" if feat_dtype == BF else ""
    cl = "_cl" if fmt is CL else ""
    assert _is_cl_view(out) if fmt is CL else out.is_contiguous()
    assert {f"pool_fwd{cl}_bf16{sfx}", f"maxdown{cl}_fwd_bf16"} <= used, used
    # no float32 full-resolution volume
    assert not used & {f"pool_fwd{cl}{sfx}", f"maxdown{cl}_fwd"}, used


def test_raw_neck_bf16_fallbacks_are_the_float32_route_cast():
    """ds=(1, 2, 2), X % 4 != 0 (channels-first) and accelerate: the float32 route and one cast,
    with and without a gradient"""
    feat5, depth5, metas, go = _small_inputs(torch.float32)
    cfg = S.CONFIGS["small"]
    wide = dict(cfg.grid_config, x=[-40.0, 40.8, 0.4])        # X = 202
    cases = [(dict(ds=(1, 2, 2)), (2, 64, 16, 100, 100), {"pool_fwd"}),
             (dict(grid_config=wide), (2, 64, 8, 100, 101), {"pool_fwd"}),
             (dict(accelerate=True), (2, 64, 8, 100, 100), {"pool_fwd"})]
    for kw, shape, names in cases:
        g = torch.randn(shape, generator=torch.Generator().manual_seed(9)).to(BF).cuda()
        used, out = _check_training(torch.contiguous_format, 64, feat5, depth5, metas, g, **kw)
        assert out.shape == shape and names <= used, (kw, used)
        assert "maxdown_fwd_mask_bf16" not in used
        used, out = _check_inference(torch.contiguous_format, 64, feat5, depth5, metas, **kw)
        assert out.shape == shape and names <= used, (kw, used)
        assert not used & {"pool_fwd_bf16", "maxdown_fwd_bf16"}, (kw, used)


def test_raw_neck_bf16_at_the_veon_real_shape():
    """VEON-real with B = 1: C = 256, 32 x 88 features, D = 88, two-hot depth, 16 x 200 x 200"""
    cfg = S.CONFIGS["C3"]
    B, C = 1, 256
    H, W = cfg.feat_hw
    g = torch.Generator(device="cuda").manual_seed(5)
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).cuda() for k in
             ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")]
    neck = _raw(torch.contiguous_format, torch.float32, C, cfg)
    metric = torch.from_numpy(S.metric_depth_np(cfg, batch=B)).cuda()
    with torch.no_grad():
        depth5 = neck.get_two_hot_depth(metric)
    feat5 = torch.randn(B, cfg.n_cams, C, H, W, device="cuda", generator=g)
    go = torch.randn(B, C, 8, 100, 100, device="cuda", generator=g).to(BF)
    used, out = _check_training(torch.contiguous_format, C, feat5, depth5, metas, go, cfg)
    assert "pool_bwd_ds_bf16" in used and out.shape == (B, C, 8, 100, 100)
    for fmt in FORMATS:
        used, out = _check_inference(fmt, C, feat5, depth5, metas, cfg)
        assert ("maxdown_cl_fwd_bf16" if fmt is CL else "maxdown_fwd_bf16") in used
