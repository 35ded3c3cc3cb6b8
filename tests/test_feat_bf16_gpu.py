"""GPU: bfloat16 image features read natively by bev_pool_v2, pool_prepared, LSSViewTransformer and
LSSViewTransformerRaw.

The contract is exact.  For a bfloat16 `feat`, every volume (float32 or bfloat16, either memory
format) and depth_grad are the bits of the same call on `feat.float()`; feat_grad is bfloat16 and
equals that call's float32 feat_grad cast to bfloat16 on the device (NaN positions must match,
payloads are not compared)."""
import pytest
import torch

from tests.test_bf16_gpu import FWD_CASES, _rejected
from tests.test_channels_last_gpu import _case, _neck_inputs
from tests.test_pool_gpu import gpu_ranks, make_case
from veon_b200 import synthetic as S

pytestmark = pytest.mark.gpu
CL = torch.channels_last_3d
BF = torch.bfloat16
FORMATS = (torch.contiguous_format, CL)
DTYPES = (torch.float32, BF)


def same_bits(a, b):
    """equal dtype, shape and bits, NaN positions included (payloads not compared)"""
    assert a.dtype == b.dtype and a.shape == b.shape
    na, nb = torch.isnan(a), torch.isnan(b)
    assert torch.equal(na, nb)
    view = torch.int16 if a.dtype == BF else torch.int32
    assert torch.equal(a.masked_fill(na, 0).contiguous().view(view),
                       b.masked_fill(nb, 0).contiguous().view(view))


def same_volume(a, b):
    assert a.stride() == b.stride()
    same_bits(a, b)


def _pool_args(case):
    rb, rd, rf, st, ln = gpu_ranks(case["ranks"])
    return rd, rf, rb, case["shape"], st, ln


def _bf16_feat(case):
    return case["feat"].to(BF).cuda()


def _check_forward(depth, feat, rd, rf, rb, shape, st, ln):
    from veon_b200.bev_pool import bev_pool_v2
    for fmt in FORMATS:
        for dt in DTYPES:
            got = bev_pool_v2(depth, feat, rd, rf, rb, shape, st, ln, memory_format=fmt, dtype=dt)
            want = bev_pool_v2(depth, feat.float(), rd, rf, rb, shape, st, ln, memory_format=fmt,
                               dtype=dt)
            same_volume(got, want)


@pytest.mark.parametrize("cfg_name,batch,C", FWD_CASES)
def test_forward_bf16_features_are_the_widened_features(cfg_name, batch, C):
    case = _case(cfg_name, batch, C)
    rd, rf, rb, shape, st, ln = _pool_args(case)
    _check_forward(case["depth"].cuda(), _bf16_feat(case), rd, rf, rb, shape, st, ln)


def test_forward_bf16_features_c2_geometry():
    """B = 8 over the C2 grid, heavy tiles: C = 64 (the float32 channels-first volume widens for
    the streaming kernel, every other route is native) and C = 20 (narrow rows)"""
    from veon_b200 import bev_pool as BP
    cfg = S.CONFIGS["C2"]
    B = 8
    lower, interval, size = S.grid_vectors(cfg.grid_config)
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B)).cuda()
    _, N, D, H, W, _ = coor.shape
    g = torch.Generator(device="cuda").manual_seed(0)
    depth = torch.softmax(torch.randn(B, N, D, H, W, device="cuda", generator=g) * 4, dim=2)
    prep = BP.prepare_ranks(coor, lower, interval, size)
    assert int(prep.plan.tile_heavy[0]) > 0
    for C in (64, 20):
        feat = torch.randn(B, N, H, W, C, device="cuda", generator=g).to(BF)
        shape = (B, 16, 200, 200, C)
        for fmt in FORMATS:
            for dt in DTYPES:
                same_volume(BP.pool_prepared(depth, feat, prep, shape, fmt, dtype=dt),
                            BP.pool_prepared(depth, feat.float(), prep, shape, fmt, dtype=dt))


def test_forward_bf16_features_voxel_with_thousands_of_points():
    B, N, D, H, W = 1, 1, 40, 8, 16
    Z, Y, X = 1, 2, 64
    g = torch.Generator().manual_seed(5)
    n_a = 3000
    rd = torch.randperm(D * H * W, generator=g)[:n_a + 333].int()
    rd[:n_a] = rd[:n_a].sort().values
    rd[n_a:] = rd[n_a:].sort().values
    rf = (rd % (H * W)).int()
    rb = torch.cat([torch.full((n_a,), 37), torch.full((333,), 41)]).int()
    st, ln = torch.tensor([0, n_a]).int(), torch.tensor([n_a, 333]).int()
    for C in (64, 20, 8, 33, 300):
        depth = torch.rand(B, N, D, H, W, generator=g).cuda()
        feat = torch.randn(B, N, H, W, C, generator=g).to(BF).cuda()
        _check_forward(depth, feat, rd.cuda(), rf.cuda(), rb.cuda(), (B, Z, Y, X, C), st.cuda(),
                       ln.cuda())


def _leaf(feat_rows, how):
    """(leaf tensor, [B,N,H,W,C] input built from it): the neck's channels-first maps seen
    channels-last, contiguous rows, or another strided view"""
    if how == "view":
        leaf = feat_rows.permute(0, 1, 4, 2, 3).contiguous().requires_grad_()
        return leaf, leaf.permute(0, 1, 3, 4, 2)
    if how == "strided":
        leaf = feat_rows.transpose(2, 3).contiguous().requires_grad_()
        return leaf, leaf.transpose(2, 3)
    leaf = feat_rows.clone().requires_grad_()
    return leaf, leaf


def _grads(case, feat_rows, how, fwd_format, vol_dtype, og, timing=False):
    from veon_b200 import bev_pool as BP
    rd, rf, rb, shape, st, ln = _pool_args(case)
    depth = case["depth"].cuda().requires_grad_()
    leaf, feat_in = _leaf(feat_rows, how)
    out = BP.bev_pool_v2(depth, feat_in, rd, rf, rb, shape, st, ln, memory_format=fwd_format,
                         dtype=vol_dtype)
    BP.enable_kernel_timing(timing)
    out.backward(og)
    used = BP.kernel_timings_ms() if timing else {}
    BP.enable_kernel_timing(False)
    return depth.grad, leaf.grad, used


def _gradient_storages(case, seed):
    B, Z, Y, X, C = case["shape"]
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(seed)).cuda()
    og_bf = og.to(BF)
    return [(og_bf.float(), torch.float32, "pool_bwd_bf16feat"),
            (og_bf, BF, "pool_bwd_bf16_bf16feat"),
            (og_bf.float().contiguous(memory_format=CL), torch.float32, "pool_bwd_cl_bf16feat"),
            (og_bf.contiguous(memory_format=CL), BF, "pool_bwd_cl_bf16_bf16feat")]


@pytest.mark.parametrize("cfg_name,batch,C", [("tiny", 2, 4), ("tiny", 2, 20), ("small", 2, 64),
                                              ("C1", 2, 100), ("small", 2, 256), ("small", 3, 512),
                                              ("ragged", 2, 36), ("ragged", 2, 64)])
@pytest.mark.parametrize("how", ["rows", "view"])
def test_backward_bf16_features_in_each_gradient_storage(cfg_name, batch, C, how):
    case = _case(cfg_name, batch, C, seed=1)
    feat = _bf16_feat(case)
    for og, vol_dtype, name in _gradient_storages(case, 2):
        for fwd_format in FORMATS:
            dg_ref, fg_ref, _ = _grads(case, feat.float(), how, fwd_format, vol_dtype,
                                       og.float() if vol_dtype is torch.float32 else og)
            dg, fg, used = _grads(case, feat, how, fwd_format, vol_dtype, og, timing=True)
            assert name in used, (name, used)
            assert not {k for k in used if k.startswith("pool_bwd") and k != name}, used
            same_bits(dg, dg_ref)
            assert fg.dtype == BF
            same_bits(fg, fg_ref.to(BF))


@pytest.mark.parametrize("C", [20, 64, 512])
def test_nan_inf_misaligned_and_strided_features(C):
    """NaN / +-inf features; a bfloat16 tensor two bytes off its 8-byte alignment (scalar or
    fallback paths: no 8-byte loads); contiguous rows, the channels-first view and another
    strided view -- all the bits of the widened call, forward and backward"""
    case = make_case("small", 2, C, seed=3)
    feat = _bf16_feat(case)
    feat[0, 1, 2, :5] = float("nan")
    feat[1, 0, 3, 4:9] = float("inf")
    feat[1, 2, 1, :3] = -float("inf")
    buf = torch.empty(feat.numel() + 1, dtype=BF, device="cuda")
    odd = buf[1:].view(feat.shape)
    odd.copy_(feat)
    assert odd.data_ptr() % 8 == 2
    rd, rf, rb, shape, st, ln = _pool_args(case)
    depth = case["depth"].cuda()
    _check_forward(depth, feat, rd, rf, rb, shape, st, ln)
    _check_forward(depth, odd, rd, rf, rb, shape, st, ln)
    for how in ("rows", "view", "strided"):
        for og, vol_dtype, name in _gradient_storages(case, 4):
            for fwd_format in FORMATS:
                dg_ref, fg_ref, _ = _grads(case, feat.float(), how, fwd_format, vol_dtype, og)
                dg, fg, _ = _grads(case, feat, how, fwd_format, vol_dtype, og)
                same_bits(dg, dg_ref)
                same_bits(fg, fg_ref.to(BF))
    # the misaligned rows themselves through the autograd node
    from veon_b200.bev_pool import bev_pool_v2
    for og, vol_dtype, _ in _gradient_storages(case, 5):
        res = []
        for f in (odd, feat.float()):
            d = depth.clone().requires_grad_()
            f = f.detach().requires_grad_()
            bev_pool_v2(d, f, rd, rf, rb, shape, st, ln, dtype=vol_dtype).backward(og)
            res.append((d.grad, f.grad))
        same_bits(res[0][0], res[1][0])
        same_bits(res[0][1], res[1][1].to(BF))


def _pool_node(out):
    todo, seen = [out.grad_fn], set()
    while todo:
        fn = todo.pop()
        if fn is None or fn in seen:
            continue
        seen.add(fn)
        if "QuickCumsum" in type(fn).__name__:
            return fn
        todo.extend(f for f, _ in fn.next_functions)
    raise AssertionError("no QuickCumsumCuda node")


@pytest.mark.parametrize("C", [20, 64, 128])
def test_native_entries_and_bf16_rows_saved(C):
    """the `_bf16feat` entries run (the float32 channels-first C = 64 volume excepted: the
    streaming kernel on widened rows), and the autograd node keeps the bfloat16 rows"""
    from veon_b200 import bev_pool as BP
    case = make_case("small", 2, C, seed=6)
    rd, rf, rb, shape, st, ln = _pool_args(case)
    depth = case["depth"].cuda().requires_grad_()
    leaf = _bf16_feat(case).permute(0, 1, 4, 2, 3).contiguous().requires_grad_()
    for fmt in FORMATS:
        for dt in DTYPES:
            BP.enable_kernel_timing(True)
            out = BP.bev_pool_v2(depth, leaf.permute(0, 1, 3, 4, 2), rd, rf, rb, shape, st, ln,
                                 memory_format=fmt, dtype=dt)
            used = set(BP.kernel_timings_ms())
            BP.enable_kernel_timing(False)
            name = "pool_fwd" + ("_cl" if fmt is CL else "") + ("_bf16" if dt is BF else "")
            assert name + "_bf16feat" in used, used
            if C == 64 and fmt is not CL and dt is torch.float32:
                assert name in used                # refused natively, widened for the stream
            else:
                assert name not in used, used
            saved = _pool_node(out).saved_tensors
            rows = [t for t in saved if t.dtype == BF]
            assert len(rows) == 1 and rows[0].is_contiguous()
            assert rows[0].shape == leaf.permute(0, 1, 3, 4, 2).shape
            assert not any(t.dtype == torch.float32 and t.shape == rows[0].shape for t in saved)


# ---------------------------------------------------------------- necks
def _lss_routes(cfg, metas, img, B, C):
    H, W = cfg.feat_hw

    def fused(neck, d, f):
        return neck.view_transform([img] + metas, d, f)[0]

    def coor_route(neck, d, f):
        coor = neck.get_lidar_coor(*metas)
        return neck.voxel_pooling_v2(coor, d.view(B, cfg.n_cams, cfg.D, H, W),
                                     f.view(B, cfg.n_cams, C, H, W))

    def accelerate(neck, d, f):
        neck.accelerate = True
        try:
            return neck.view_transform([img] + metas, d, f)[0]
        finally:
            neck.accelerate = False
    return fused, coor_route, accelerate


@pytest.mark.parametrize("sync_free", [False, True])
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("dt", DTYPES)
def test_lss_neck_bf16_tran_feat(sync_free, fmt, dt):
    """view_transform with a bfloat16 tran_feat [B*N, C, H, W] against the same call on
    tran_feat.float(): fused geometry, voxel_pooling_v2 and accelerate"""
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 64
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=3)
    feat = feat.to(BF)
    og = torch.randn(B, C, 16, 200, 200, generator=torch.Generator().manual_seed(4)).cuda().to(dt)
    og = og.contiguous(memory_format=fmt)
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                              collapse_z=False, sync_free=sync_free, memory_format=fmt, dtype=dt)
    for route in _lss_routes(cfg, metas, img, B, C):
        res = []
        for f0 in (feat, feat.float()):
            d = depth.detach().clone().requires_grad_()
            f = f0.detach().clone().requires_grad_()
            bev = route(neck, d, f)
            bev.backward(og)
            res.append((bev.detach(), d.grad, f.grad))
        (a, da, fa), (b, db, fb) = res
        same_volume(a, b)
        same_bits(da, db)
        assert fa.dtype == BF and fa.is_contiguous(), route.__name__
        same_bits(fa, fb.to(BF))


def test_lss_neck_forward_under_autocast():
    """LSSViewTransformer.forward under bfloat16 autocast: depth_net hands over bfloat16 maps,
    which reach the pooling as they are; the volume is the one of its widened maps"""
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 64
    _, metas, _, _ = _neck_inputs(cfg, B, C, seed=8)
    H, W = cfg.feat_hw
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 16, C,
                              collapse_z=False, dtype=BF).cuda()
    img = torch.randn(B, cfg.n_cams, 16, H, W, generator=torch.Generator().manual_seed(9)).cuda()
    seen = []
    hook = neck.depth_net.register_forward_hook(lambda m, i, o: seen.append(o.detach()))
    BP.enable_kernel_timing(True)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        bev, depth = neck([img] + metas)
    used = set(BP.kernel_timings_ms())
    BP.enable_kernel_timing(False)
    hook.remove()
    x, = seen
    assert x.dtype == BF and depth.dtype == torch.float32
    assert "pool_fwd_bf16_bf16feat" in used, used
    tran_feat = x[:, neck.D:neck.D + C]
    want, _ = neck.view_transform([img] + metas, depth, tran_feat.float())
    same_volume(bev, want)


def test_raw_neck_bf16_features():
    """the Raw neck pools bfloat16 features into its float32 volume: the one-node training route
    (native `_ds` backward), the channels-last plain route, and no-grad inference (widened)"""
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformerRaw
    cfg = S.CONFIGS["small"]
    B, C = 2, 64
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=6)
    H, W = cfg.feat_hw
    feat5 = feat.view(B, cfg.n_cams, C, H, W).to(BF)
    feat5[0, 1, 3, 4, :] = float("nan")
    depth5 = depth.view(B, cfg.n_cams, cfg.D, H, W)
    go = torch.randn(B, C, 8, 100, 100, generator=torch.Generator().manual_seed(7)).cuda()
    for fmt, names in ((torch.contiguous_format, {"pool_bwd_ds_bf16feat"}),
                       (CL, {"pool_fwd_cl_bf16feat", "pool_bwd_cl_bf16feat"})):
        neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                     memory_format=fmt)
        res = []
        for f0 in (feat5, feat5.float()):
            f = f0.detach().clone().requires_grad_()
            d = depth5.detach().clone().requires_grad_()
            BP.enable_kernel_timing(True)
            out = neck([f] + metas, d)
            out.backward(go.contiguous(memory_format=fmt))
            used = set(BP.kernel_timings_ms())
            BP.enable_kernel_timing(False)
            res.append((out.detach(), d.grad, f.grad, used))
        (a, da, fa, ua), (b, db, fb, _) = res
        assert names <= ua, ua
        assert a.dtype == torch.float32
        same_volume(a, b)
        same_bits(da, db)
        assert fa.dtype == BF
        same_bits(fa, fb.to(BF))
    neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C)
    with torch.no_grad():
        a = neck([feat5] + metas, depth5)
        b = neck([feat5.float()] + metas, depth5)
    same_volume(a, b)


# ---------------------------------------------------------------- graphs and plans
@pytest.mark.parametrize("fmt", FORMATS)
def test_sync_free_bf16_features_in_a_cuda_graph(fmt):
    """a sync-free bf16-feature forward and backward captured once and replayed: same bits as
    eager and as the widened call"""
    from veon_b200 import bev_pool as BP
    case = make_case("C1", 2, 64, seed=7)
    lower, interval, size = case["grid"]
    B, Z, Y, X, C = case["shape"]
    prep = BP.prepare_ranks(torch.from_numpy(case["coor"]).cuda(), lower, interval, size)
    prep.plan.sync_free = True
    depth = case["depth"].cuda().requires_grad_()
    leaf = _bf16_feat(case).permute(0, 1, 4, 2, 3).contiguous().requires_grad_()
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(3)).cuda()
    og = og.to(BF).contiguous(memory_format=fmt)

    def step(f_leaf):
        depth.grad = None
        f_leaf.grad = None
        out = BP.pool_prepared(depth, f_leaf.permute(0, 1, 3, 4, 2), prep, case["shape"], fmt,
                               dtype=BF)
        out.backward(og)
        return out

    wleaf = leaf.detach().float().requires_grad_()
    want = step(wleaf).detach()
    want_dg, want_fg = depth.grad.clone(), wleaf.grad.to(BF)
    eager = step(leaf).detach()
    same_volume(eager, want)
    same_bits(depth.grad, want_dg)
    same_bits(leaf.grad, want_fg)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step(leaf)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        vol = step(leaf)
        copy = vol.detach().clone(memory_format=fmt)
    for _ in range(3):
        copy.zero_()
        depth.grad.zero_()
        leaf.grad.zero_()
        graph.replay()
        torch.cuda.synchronize()
        same_volume(vol, want)
        same_volume(copy, want)
        same_bits(depth.grad, want_dg)
        same_bits(leaf.grad, want_fg)


@pytest.mark.parametrize("how", ["shuffled", "hand-made"])
def test_rejected_plans_bf16_features(how):
    """a rejected plan takes the generic kernels on widened rows: the volume is the widened
    call's; feat_grad comes back in bfloat16"""
    from veon_b200 import bev_pool as BP
    case = make_case("tiny", 2, 24, seed=7)
    case2 = dict(case, ranks=_rejected(case, how))
    rd, rf, rb, shape, st, ln = _pool_args(case2)
    B, Z, Y, X, C = shape
    assert not BP._plan_for(rd, rf, rb, st, ln, case["dims"], Z * Y * X).ok
    feat = _bf16_feat(case)
    _check_forward(case["depth"].cuda(), feat, rd, rf, rb, shape, st, ln)
    for og, vol_dtype, _ in _gradient_storages(case, 8):
        for fmt in FORMATS:
            dg_ref, fg_ref, _ = _grads(case2, feat.float(), "view", fmt, vol_dtype, og)
            dg, fg, _ = _grads(case2, feat, "view", fmt, vol_dtype, og)
            same_bits(dg, dg_ref)
            assert fg.dtype == BF
            # the generic backward accumulates feat_grad with float atomics (order varies run to
            # run, in the float32 route as well)
            torch.testing.assert_close(fg.float(), fg_ref.to(BF).float(), rtol=1e-2, atol=1e-5)
