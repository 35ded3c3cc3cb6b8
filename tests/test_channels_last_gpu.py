"""GPU: channels-last volumes (memory_format=torch.channels_last_3d) for bev_pool_v2, the
single-pass backward on a channels-last gradient, the channels-last 2x2x2 max-downsample and
the necks built on them.  Everything here must be the same bits as the channels-first route."""
import numpy as np
import pytest
import torch

from oracle import lift_oracle as O
from tests.test_pool_gpu import gpu_ranks, make_case, rel_max_err
from veon_b200 import synthetic as S

pytestmark = pytest.mark.gpu
CL = torch.channels_last_3d


def _is_cl_view(x):
    """channels-last-3d strides over a storage of exactly its own size (not a copy's view)"""
    return (x.is_contiguous(memory_format=CL) and x.permute(0, 2, 3, 4, 1).is_contiguous()
            and x.untyped_storage().nbytes() == x.numel() * x.element_size())


def _pool(case, memory_format, depth=None, feat=None):
    from veon_b200.bev_pool import bev_pool_v2
    rb, rd, rf, st, ln = gpu_ranks(case["ranks"])
    depth = case["depth"].cuda() if depth is None else depth
    feat = case["feat"].cuda() if feat is None else feat
    return bev_pool_v2(depth, feat, rd, rf, rb, case["shape"], st, ln, memory_format=memory_format)


def _ragged_case(C, B=2, seed=0):
    """X, Y, Z = 7, 5, 3: V = 105 (V % 32 != 0, V % 4 != 0), ~35 points per voxel (heavy tiles)"""
    g = np.random.RandomState(seed)
    N, D, H, W = 2, 30, 8, 8
    coor = (g.rand(B, N, D, H, W, 3) * np.array([7.6, 5.6, 3.6]) - 0.3).astype(np.float32)
    lower, interval, size = (np.zeros(3, np.float32), np.ones(3, np.float32),
                             np.array([7, 5, 3], np.float32))
    ranks = O.prepare_v2(coor, lower, interval, size)
    t = torch.Generator().manual_seed(seed)
    depth = torch.softmax(torch.randn(B, N, D, H, W, generator=t) * 4, dim=2)
    feat = torch.randn(B, N, H, W, C, generator=t)
    return dict(coor=coor, grid=(lower, interval, size), ranks=ranks, depth=depth, feat=feat,
                shape=(B, 3, 5, 7, C), dims=(B, N, D, H, W))


FWD_CASES = [("tiny", 2, 4), ("tiny", 2, 7), ("tiny", 2, 20), ("C1", 2, 28), ("tiny", 2, 32),
             ("small", 2, 64), ("C1", 1, 64), ("tiny", 1, 100), ("small", 2, 256),
             ("C1", 1, 512), ("tiny", 2, 768), ("ragged", 2, 7), ("ragged", 2, 20),
             ("ragged", 3, 64), ("ragged", 2, 100), ("ragged", 1, 1024)]


def _case(name, batch, C, seed=0):
    return _ragged_case(C, batch, seed) if name == "ragged" else make_case(name, batch, C, seed)


@pytest.mark.parametrize("cfg_name,batch,C", FWD_CASES)
def test_forward_channels_last_equals_channels_first(cfg_name, batch, C):
    case = _case(cfg_name, batch, C)
    cf = _pool(case, torch.contiguous_format)
    cl = _pool(case, CL)
    assert cl.shape == cf.shape and cf.is_contiguous() and _is_cl_view(cl)
    assert torch.equal(cl, cf)
    if C <= 256:   # the oracle's own channels-last output, bit for bit
        rb, rd, rf, st, ln = case["ranks"]
        want = O.bev_pool_v2_channels_last(case["depth"].numpy(), case["feat"].numpy(), rd, rf, rb,
                                           case["shape"], st, ln)
        np.testing.assert_array_equal(cl.permute(0, 2, 3, 4, 1).cpu().numpy(), want)


def test_forward_channels_last_voxel_with_thousands_of_points():
    """heavy-tile rounds carried over in one voxel, a second voxel starting mid-round"""
    from veon_b200.bev_pool import bev_pool_v2
    B, N, D, H, W = 1, 1, 40, 8, 16
    Z, Y, X = 1, 2, 64
    g = torch.Generator().manual_seed(5)
    n_a = 3000
    P = D * H * W
    rd = torch.randperm(P, generator=g)[:n_a + 333].int()
    rd[:n_a] = rd[:n_a].sort().values
    rd[n_a:] = rd[n_a:].sort().values
    rf = (rd % (H * W)).int()
    rb = torch.cat([torch.full((n_a,), 37), torch.full((333,), 41)]).int()
    st, ln = torch.tensor([0, n_a]).int(), torch.tensor([n_a, 333]).int()
    for C in (64, 20, 7, 300):
        depth = torch.rand(B, N, D, H, W, generator=g)
        feat = torch.randn(B, N, H, W, C, generator=g)
        args = (depth.cuda(), feat.cuda(), rd.cuda(), rf.cuda(), rb.cuda(), (B, Z, Y, X, C),
                st.cuda(), ln.cuda())
        cl = bev_pool_v2(*args, memory_format=CL)
        want = O.bev_pool_v2_channels_last(depth.numpy(), feat.numpy(), rd.numpy(), rf.numpy(),
                                           rb.numpy(), (B, Z, Y, X, C), st.numpy(), ln.numpy())
        np.testing.assert_array_equal(cl.permute(0, 2, 3, 4, 1).cpu().numpy(), want)
        assert torch.equal(cl, bev_pool_v2(*args))


def _grads(case, fwd_format, og, timing=False):
    from veon_b200 import bev_pool as BP
    depth = case["depth"].cuda().requires_grad_()
    feat = case["feat"].cuda().requires_grad_()
    out = _pool(case, fwd_format, depth, feat)
    BP.enable_kernel_timing(timing)
    out.backward(og)
    used = BP.kernel_timings_ms() if timing else {}
    BP.enable_kernel_timing(False)
    torch.cuda.synchronize()
    return depth.grad, feat.grad, used


@pytest.mark.parametrize("cfg_name,batch,C", [("tiny", 2, 7), ("tiny", 2, 20), ("small", 2, 64),
                                              ("C1", 2, 100), ("small", 2, 256), ("small", 3, 512),
                                              ("tiny", 2, 768), ("ragged", 2, 36),
                                              ("ragged", 2, 1024)])
def test_backward_channels_last_gradient_is_bit_identical(cfg_name, batch, C):
    case = _case(cfg_name, batch, C, seed=1)
    B, Z, Y, X, _ = case["shape"]
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(2)).cuda()
    og_cl = og.contiguous(memory_format=CL)
    dg_cf, fg_cf, used = _grads(case, torch.contiguous_format, og, True)
    assert "pool_bwd" in used and "pool_bwd_cl" not in used
    for fwd_format in (torch.contiguous_format, CL):
        dg, fg, used = _grads(case, fwd_format, og_cl, True)
        assert "pool_bwd_cl" in used and "pool_bwd" not in used      # the single pass ran
        assert torch.equal(dg, dg_cf) and torch.equal(fg, fg_cf)
    # a gradient in neither layout is copied to channels-first and takes the two passes
    odd = og.permute(0, 1, 4, 3, 2).contiguous().permute(0, 1, 4, 3, 2)
    dg, fg, _ = _grads(case, CL, odd)
    assert torch.equal(dg, dg_cf) and torch.equal(fg, fg_cf)
    # run to run
    dg2, fg2, _ = _grads(case, CL, og_cl)
    assert torch.equal(dg2, dg_cf) and torch.equal(fg2, fg_cf)
    rb, rd, rf, st, ln = case["ranks"]
    dg_want, fg_want = O.bev_pool_v2_backward(og.cpu().numpy(), case["depth"].numpy(),
                                              case["feat"].numpy(), rd, rf, rb)
    dg_np = dg_cf.cpu().numpy()
    assert rel_max_err(dg_np, dg_want) <= 2e-5
    assert rel_max_err(fg_cf.cpu().numpy(), fg_want) <= 2e-5
    kept = np.zeros(dg_np.size, bool)
    kept[rd] = True
    assert np.all(dg_np.reshape(-1)[~kept] == 0)       # dropped points: exactly zero


def test_generic_fallback_channels_last():
    """unsorted ranks (interval order shuffled): the plan is rejected and the interval-driven
    kernels run in the channels-last layout; forward and backward still match the oracle"""
    case = make_case("tiny", 2, 24, seed=7)
    rb, rd, rf, st, ln = case["ranks"]
    perm = np.random.RandomState(0).permutation(st.size)
    parts = [(rb[st[k]:st[k] + ln[k]], rd[st[k]:st[k] + ln[k]], rf[st[k]:st[k] + ln[k]])
             for k in perm]
    lens = np.array([len(p[0]) for p in parts], np.int32)
    shuf = (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
            np.concatenate([p[2] for p in parts]),
            np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int32), lens)
    case2 = dict(case, ranks=shuf)
    B, Z, Y, X, C = case["shape"]
    want = O.bev_pool_v2(case["depth"].numpy(), case["feat"].numpy(), rd, rf, rb, case["shape"],
                         st, ln)
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(8)).cuda()
    dg_want, fg_want = O.bev_pool_v2_backward(og.cpu().numpy(), case["depth"].numpy(),
                                              case["feat"].numpy(), rd, rf, rb)
    depth = case["depth"].cuda().requires_grad_()
    feat = case["feat"].cuda().requires_grad_()
    out = _pool(case2, CL, depth, feat)
    assert _is_cl_view(out)
    np.testing.assert_array_equal(out.detach().cpu().numpy(), want)
    out.backward(og.contiguous(memory_format=CL))
    assert rel_max_err(depth.grad.cpu().numpy(), dg_want) <= 2e-5
    assert rel_max_err(feat.grad.cpu().numpy(), fg_want) <= 2e-5


@pytest.mark.parametrize("C", [64, 20, 100])
def test_next_kernel_in_the_stream_sees_the_whole_channels_last_volume(C):
    """the heavy-tile grid is a programmatic dependent of the main grid (C=20: the other way
    round); the kernel launched right behind them must find every row written"""
    from veon_b200 import bev_pool as BP
    cfg = S.CONFIGS["C2"]
    B = 8
    lower, interval, size = S.grid_vectors(cfg.grid_config)
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B)).cuda()
    _, N, D, H, W, _ = coor.shape
    g = torch.Generator(device="cuda").manual_seed(0)
    depth = torch.softmax(torch.randn(B, N, D, H, W, device="cuda", generator=g) * 4, dim=2)
    feat = torch.randn(B, N, H, W, C, device="cuda", generator=g)
    prep = BP.prepare_ranks(coor, lower, interval, size)
    assert int(prep.plan.tile_heavy[0]) > 0
    shape = (B, 16, 200, 200, C)
    ref = BP.pool_prepared(depth, feat, prep, shape)
    torch.cuda.synchronize()
    scratch = torch.empty(64 << 20, device="cuda")
    for i in range(6):
        scratch.normal_()
        vol = BP.pool_prepared(depth, feat, prep, shape, memory_format=CL)
        copy = vol.clone(memory_format=CL)                 # the very next kernel reads it
        torch.cuda.synchronize()
        assert torch.equal(copy, ref), f"iteration {i}: a consumer ran before the volume was complete"


@pytest.mark.parametrize("C", [64, 20])
def test_channels_last_forward_inside_a_cuda_graph(C):
    from veon_b200 import bev_pool as BP
    case = make_case("C1", 2, C, seed=7)
    rb, rd, rf, st, ln = gpu_ranks(case["ranks"])
    B, Z, Y, X, C = case["shape"]
    V = Z * Y * X
    plan = BP._plan_for(rd, rf, rb, st, ln, case["dims"], V)
    assert plan.ok and int(plan.tile_heavy[0]) > 0
    depth, feat = case["depth"].cuda(), case["feat"].cuda()
    shape = (B, Z, Y, X, C)
    eager = BP._fwd_planar_cl(depth, feat, rd, rf, rb, plan, B, C, V, shape).clone()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        BP._fwd_planar_cl(depth, feat, rd, rf, rb, plan, B, C, V, shape)     # warm-up
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(graph):
        vol = BP._fwd_planar_cl(depth, feat, rd, rf, rb, plan, B, C, V, shape)
        copy = vol.clone()
    for _ in range(3):
        copy.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(vol, eager) and torch.equal(copy, eager)


def test_sync_free_backward_reads_no_interval_past_the_count():
    """prepare_ranks returns capacity-sized interval tables (one slot per point); only the first
    n_int are valid.  Overwrite the rest with in-range but wrong values: a single pass that read
    one of them would change the gradient."""
    from veon_b200 import bev_pool as BP
    case = make_case("small", 2, 64, seed=4)
    lower, interval, size = case["grid"]
    B, Z, Y, X, C = case["shape"]
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(5)).cuda()
    coor = case["coor"].copy()
    coor[:, :, 6:] = 1e4                  # only the first depth bins inside the grid
    grads = []
    for poison in (False, True):
        prep = BP.prepare_ranks(torch.from_numpy(coor).cuda(), lower, interval, size)
        n_int = prep.plan.n_intervals
        assert 4 * n_int < prep.interval_starts.numel()        # capacity far above the count
        if poison:
            prep.interval_starts[n_int:] = 0                   # -> ranks_bev[0]: a real voxel
            prep.plan.sync_free = True
        depth = case["depth"].cuda().requires_grad_()
        feat = case["feat"].cuda().requires_grad_()
        out = BP.pool_prepared(depth, feat, prep, case["shape"], memory_format=CL)
        out.backward(og.contiguous(memory_format=CL))
        grads.append((out.detach(), depth.grad, feat.grad))
    for a, b in zip(*grads):
        assert torch.equal(a, b)


# ---------------------------------------------------------------- necks
KEYS = ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")


def _neck_inputs(cfg, B, C, seed):
    g = torch.Generator().manual_seed(seed)
    H, W = cfg.feat_hw
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).cuda() for k in KEYS]
    depth = torch.softmax(torch.randn(B * cfg.n_cams, cfg.D, H, W, generator=g) * 4, dim=1).cuda()
    feat = torch.randn(B * cfg.n_cams, C, H, W, generator=g).cuda()
    img = torch.zeros(B, cfg.n_cams, 8, H, W, device="cuda")
    return img, metas, depth, feat


@pytest.mark.parametrize("sync_free", [False, True])
def test_neck_routes_give_channels_last_volumes(sync_free):
    """fused geometry, voxel_pooling_v2(coor, ...) and accelerate: the channels-last neck's
    volume equals the default neck's, stored channels-last; gradients are the same bits"""
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 32
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=3)
    H, W = cfg.feat_hw
    og = torch.randn(B, C, 16, 200, 200, generator=torch.Generator().manual_seed(4)).cuda()
    necks = [LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                collapse_z=False, sync_free=sync_free, memory_format=fmt)
             for fmt in (torch.contiguous_format, CL)]

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

    for route in (fused, coor_route, accelerate):
        res = []
        for neck in necks:
            d = depth.detach().clone().requires_grad_()
            f = feat.detach().clone().requires_grad_()
            bev = route(neck, d, f)
            bev.backward(og)
            res.append((bev.detach(), d.grad, f.grad))
        (a, da, fa), (b, db, fb) = res
        assert a.is_contiguous() and _is_cl_view(b), route.__name__
        assert torch.equal(a, b) and torch.equal(b, a.contiguous(memory_format=CL)), route.__name__
        assert torch.equal(da, db) and torch.equal(fa, fb), route.__name__
    # collapse_z works on a channels-last volume, whatever layout torch.cat gives
    for neck in necks:
        neck.collapse_z = True
    a, b = (fused(n, depth, feat) for n in necks)
    assert a.shape == (B, C * 16, 200, 200) and torch.equal(a, b)


def test_raw_neck_channels_last_equals_default_bit_for_bit():
    """channels-last Raw neck = pool channels-last + channels-last 2x2x2; the default neck takes
    the one-node PoolMaxDown route.  Same forward and gradients, NaN and ties at zero included."""
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformerRaw
    cfg = S.CONFIGS["small"]
    B, C = 2, 64
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=6)
    H, W = cfg.feat_hw
    feat = feat.clamp(min=0.0)                    # many sums exactly 0: ties beside empty voxels
    feat[:, 3, 4, :] = float("nan")               # NaNs that reach the volume
    feat5 = feat.view(B, cfg.n_cams, C, H, W)
    depth5 = depth.view(B, cfg.n_cams, cfg.D, H, W)
    go = torch.randn(B, C, 8, 100, 100, generator=torch.Generator().manual_seed(7)).cuda()
    res = []
    for fmt in (torch.contiguous_format, CL):
        neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                     memory_format=fmt)
        f = feat5.detach().clone().requires_grad_()
        d = depth5.detach().clone().requires_grad_()
        BP.enable_kernel_timing(True)
        out = neck([f] + metas, d)
        out.backward(go)
        used = BP.kernel_timings_ms()
        BP.enable_kernel_timing(False)
        res.append((out.detach(), d.grad, f.grad, used))
    (a, da, fa, ua), (b, db, fb, ub) = res
    assert "pool_bwd_ds" in ua                                     # the one-node route
    assert {"pool_fwd_cl", "maxdown_cl_fwd", "maxdown_cl_bwd", "pool_bwd_cl"} <= set(ub)
    assert b.shape == (B, C, 8, 100, 100) and _is_cl_view(b)
    assert bool(torch.isnan(a).any())

    def bits(t):
        return t.contiguous().view(torch.int32)
    assert torch.equal(bits(a), bits(b))
    assert torch.equal(bits(da), bits(db)) and torch.equal(bits(fa), bits(fb))
    # inference (no gradient): the plain channels-last route as well, fuse_ds skipped
    neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                 fuse_ds=True, memory_format=CL)
    with torch.no_grad():
        c = neck([feat5] + metas, depth5)
    assert _is_cl_view(c) and torch.equal(bits(c), bits(a))


def test_maxdown2x2x2_channels_last_matches_channels_first():
    """odd C, NaN, ties at zero, -0 against +0: same values and gradients as the channels-first
    kernels, in the channels-last layout"""
    from veon_b200.bev_pool import MaxDown2x2x2
    g = torch.Generator().manual_seed(11)
    for shape in [(2, 5, 6, 10, 24), (1, 7, 4, 6, 8), (3, 64, 2, 4, 4)]:
        x = torch.randn(*shape, generator=g)
        x[x.abs() < 0.6] = 0.0
        x[torch.rand(*shape, generator=g) < 0.1] = -0.0
        x.view(-1)[3] = float("nan")
        x = x.cuda()
        xc = x.contiguous(memory_format=CL)
        assert MaxDown2x2x2.supports(xc)
        a = x.clone().requires_grad_()
        b = xc.clone().requires_grad_()
        assert _is_cl_view(b)
        oa, ob = MaxDown2x2x2.apply(a), MaxDown2x2x2.apply(b)
        assert _is_cl_view(ob)
        assert torch.equal(oa.view(torch.int32), ob.contiguous().view(torch.int32))
        go = torch.randn(oa.shape, generator=g).cuda()
        oa.backward(go)
        ob.backward(go.contiguous(memory_format=CL))
        assert b.grad.is_contiguous(memory_format=CL)
        assert torch.equal(a.grad.view(torch.int32), b.grad.contiguous().view(torch.int32))
    # channels-last needs only an even X (the channels-first kernels take X % 4 == 0)
    x = torch.randn(2, 3, 4, 6, 6, generator=g).cuda().contiguous(memory_format=CL)
    assert MaxDown2x2x2.supports(x) and not MaxDown2x2x2.supports(x.contiguous())
    want = x.view(2, 3, 2, 2, 3, 2, 3, 2).amax(dim=(3, 5, 7))
    assert torch.equal(MaxDown2x2x2.apply(x), want)
