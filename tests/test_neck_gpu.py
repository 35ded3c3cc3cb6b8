"""GPU: the host-side mirror of the neck (LSSViewTransformer / LSSViewTransformerRaw) end to
end.  (The DROP-IN checks -- the reference's own, unmodified files running on top of our
operators -- are in tests/test_dropin_reference.py.)"""
import numpy as np
import pytest
import torch

from oracle import lift_oracle as O
from veon_b200 import synthetic as S

pytestmark = pytest.mark.gpu
KEYS = ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def inputs(cfg, B, C, seed=0):
    g = torch.Generator().manual_seed(seed)
    H, W = cfg.feat_hw
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).cuda() for k in KEYS]
    depth = torch.softmax(torch.randn(B * cfg.n_cams, cfg.D, H, W, generator=g) * 4, dim=1).cuda()
    feat = torch.randn(B * cfg.n_cams, C, H, W, generator=g).cuda()
    img = torch.zeros(B, cfg.n_cams, 8, H, W, device="cuda")
    return img, metas, depth, feat


def test_get_lidar_coor_kernel_matches_reference_geometry(golden_dir):
    """CUDA get_lidar_coor vs the reference's own get_lidar_coor output (golden) and vs the
    torch formulation, incl. non-trivial post_rots / bda"""
    import os
    from veon_b200.view_transformer import LSSViewTransformer
    geo = np.load(os.path.join(golden_dir, "geometry_tiny.npz"))
    for name in ("tiny", "C1"):
        cfg = S.CONFIGS[name]
        neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, cfg.channels)
        cal = S.calibration(cfg, batch=1)
        metas = [torch.from_numpy(cal[k]).cuda() for k in KEYS]
        coor = neck.get_lidar_coor(*metas).cpu().numpy()
        if name == "tiny":
            np.testing.assert_allclose(coor, geo["tiny.coor"], rtol=0, atol=3e-5)
        else:
            np.testing.assert_allclose(coor[:, :, ::11, ::5, ::7], geo["C1.coor_sample"], rtol=0, atol=3e-4)
    # random rotations in post_rots (flip / rotate augmentation) and bda
    cfg = S.CONFIGS["tiny"]
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4)
    g = torch.Generator().manual_seed(0)
    B, N = 3, cfg.n_cams
    cal = S.calibration(cfg, batch=B)
    th = torch.rand(B, N, generator=g) * 0.4 - 0.2
    pr = torch.zeros(B, N, 3, 3)
    sc = 0.4 + 0.2 * torch.rand(B, N, generator=g)
    pr[..., 0, 0] = sc * th.cos(); pr[..., 0, 1] = -sc * th.sin()
    pr[..., 1, 0] = sc * th.sin(); pr[..., 1, 1] = sc * th.cos(); pr[..., 2, 2] = 1
    bda = torch.eye(3).repeat(B, 1, 1) * torch.tensor([1.0, -1.0, 1.0]) * 1.05
    metas = [torch.from_numpy(cal[k]) for k in KEYS]
    metas[3], metas[5] = pr, bda
    metas[4] = metas[4] + torch.randn(B, N, 3, generator=g) * torch.tensor([5.0, 5.0, 0.0])
    want = O.lidar_coor_torch(neck.frustum, *metas).numpy()
    got = neck.get_lidar_coor(*[m.cuda() for m in metas]).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-4)


@pytest.mark.parametrize("sync_free", [False, True])
def test_view_transform_matches_cpu_lift(sync_free):
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 32
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                              collapse_z=False, sync_free=sync_free)
    img, metas, depth, feat = inputs(cfg, B, C)
    bev, _ = neck.view_transform([img] + metas, depth, feat)
    assert bev.shape == (B, C, 16, 200, 200)
    coor = neck.get_lidar_coor(*metas)
    H, W = cfg.feat_hw
    want, _, _ = O.torch_cpu_lift(coor.cpu(), depth.view(B, cfg.n_cams, cfg.D, H, W).cpu(),
                                  feat.view(B, cfg.n_cams, C, H, W).cpu(), neck.grid_lower_bound,
                                  neck.grid_interval, neck.grid_size)
    assert rel(bev.cpu().numpy(), want.numpy()) <= 1e-5


def test_sync_free_backward_equals_faithful_backward():
    """sync_free sizes the backward scratch by an upper bound instead of reading the
    interval count back; gradients must be the same bits as on the faithful path."""
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 32
    img, metas, depth, feat = inputs(cfg, B, C, seed=2)
    og = torch.randn(B, C, 16, 200, 200, generator=torch.Generator().manual_seed(9)).cuda()
    grads = []
    for sync_free in (False, True):
        neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                  collapse_z=False, sync_free=sync_free)
        d = depth.detach().clone().requires_grad_()
        f = feat.detach().clone().requires_grad_()
        bev, _ = neck.view_transform([img] + metas, d, f)
        bev.backward(og)
        grads.append((bev.detach(), d.grad, f.grad))
    for a, b in zip(*grads):
        assert torch.equal(a, b)


def test_accelerate_equals_non_accelerate():
    """the idea of the reference's own neck test (tests/test_models/test_necks/test_necks.py:137-195)"""
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 1, 64
    # collapse_z=False: the reference's accelerate branch squeezes Z (view_transformer.py:284)
    # instead of collapsing it, so the two paths only agree in shape for un-collapsed volumes
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C, collapse_z=False)
    img, metas, depth, feat = inputs(cfg, B, C, seed=1)
    a, _ = neck.view_transform([img] + metas, depth, feat)
    neck.accelerate = True
    b, _ = neck.view_transform([img] + metas, depth, feat)
    c, _ = neck.view_transform([img] + metas, depth, feat)       # cached ranks + cached plan
    assert a.shape == (B, C, 16, 200, 200)
    assert torch.equal(a, b) and torch.equal(b, c)


def test_raw_neck_forward_downsamples():
    from veon_b200.view_transformer import LSSViewTransformerRaw
    cfg = S.CONFIGS["small"]
    B, C = 1, 16
    neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C)
    img, metas, depth, feat = inputs(cfg, B, C, seed=2)
    H, W = cfg.feat_hw
    out = neck([feat.view(B, cfg.n_cams, C, H, W)] + metas, depth.view(B, cfg.n_cams, cfg.D, H, W))
    assert out.shape == (B, C, 8, 100, 100)
    neck.use_ds = False
    full = neck([feat.view(B, cfg.n_cams, C, H, W)] + metas, depth.view(B, cfg.n_cams, cfg.D, H, W))
    want = full.view(B, C, 8, 2, 100, 2, 100, 2).amax(dim=(3, 5, 7))
    assert torch.equal(out, want)


def test_no_point_in_grid_matches_reference_dummy():
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["tiny"]
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4, collapse_z=True)
    B, N, D = 1, cfg.n_cams, cfg.D
    H, W = cfg.feat_hw
    coor = torch.full((B, N, D, H, W, 3), 1000.0, device="cuda")
    out = neck.voxel_pooling_v2(coor, torch.rand(B, N, D, H, W, device="cuda"),
                                torch.rand(B, N, 4, H, W, device="cuda"))
    assert out.shape == (1, 4 * 16, 200, 200) and float(out.abs().sum()) == 0.0


@pytest.mark.parametrize("C", [64, 128])
def test_raw_neck_inference_equals_gradient_route(C):
    """The no-grad Raw neck pools, then max-reduces 2x2x2 with its own kernel; the result must
    equal the gradient route's (the one-node pool + maximum) bit for bit, and that route must still
    give a gradient."""
    from veon_b200.view_transformer import LSSViewTransformerRaw
    cfg = S.CONFIGS["small"]
    B = 2
    neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C)
    img, metas, depth, feat = inputs(cfg, B, C, seed=4)
    H, W = cfg.feat_hw
    feat5 = feat.view(B, cfg.n_cams, C, H, W)
    depth5 = depth.view(B, cfg.n_cams, cfg.D, H, W)
    from veon_b200 import bev_pool as BP
    BP.enable_kernel_timing(True)
    with torch.no_grad():
        fused = neck([feat5] + metas, depth5)
    used = BP.kernel_timings_ms()
    BP.enable_kernel_timing(False)
    assert {"pool_fwd", "maxdown_fwd"} <= set(used), used
    assert fused.shape == (B, C, 8, 100, 100)
    f = feat5.detach().clone().requires_grad_()                   # gradient wanted -> plain route
    plain = neck([f] + metas, depth5)
    assert torch.equal(fused, plain.detach())
    plain.sum().backward()
    assert f.grad is not None and torch.isfinite(f.grad).all()


def ref_maxdown(x):
    """the reference's expression, view_transformer_raw.py:549-553"""
    from einops import rearrange
    x = rearrange(x, 'b c (z dz) (h dh) (w dw) -> b c z h w (dz dh dw)', dz=2, dh=2, dw=2)
    return torch.max(x, dim=-1).values


def test_maxdown2x2x2_matches_the_reference_expression_forward_and_backward():
    """own 2x2x2 max-downsample kernels vs the reference's expression
    (view_transformer_raw.py:549-553: rearrange + torch.max(dim=-1).values), whose backward
    routes the whole gradient to the FIRST arg-max of a block -- ties are structural in a
    pooled volume (empty voxels are exactly 0.0)"""
    from veon_b200.bev_pool import MaxDown2x2x2
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 5, 6, 10, 24, generator=g).cuda()
    x[x.abs() < 0.6] = 0.0                      # plenty of ties at zero, like an occupancy volume
    x[0, 0, 0, 0, 0] = float("nan")
    assert MaxDown2x2x2.supports(x)
    a = x.clone().requires_grad_()
    b = x.clone().requires_grad_()
    out = MaxDown2x2x2.apply(a)
    B, C, Z, Y, X = x.shape
    want = ref_maxdown(b)
    assert torch.equal(torch.nan_to_num(out, nan=-7.0), torch.nan_to_num(want, nan=-7.0))
    go = torch.randn(out.shape, generator=g).cuda()
    out.backward(go)
    want.backward(go)
    assert torch.equal(a.grad, b.grad)                      # incl. the block that holds the NaN
    # every block hands its gradient to exactly one input
    nz = (a.grad != 0).view(B, C, Z // 2, 2, Y // 2, 2, X // 2, 2).sum(dim=(3, 5, 7))
    assert int(nz.max()) == 1


def test_raw_neck_training_route_uses_own_downsample_and_matches_amax():
    from veon_b200.view_transformer import LSSViewTransformerRaw
    from veon_b200 import bev_pool as BP
    cfg = S.CONFIGS["small"]
    B, C = 1, 64
    img, metas, depth, feat = inputs(cfg, B, C, seed=6)
    H, W = cfg.feat_hw
    feat5 = feat.view(B, cfg.n_cams, C, H, W)
    depth5 = depth.view(B, cfg.n_cams, cfg.D, H, W)
    neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C)
    f1 = feat5.detach().clone().requires_grad_()
    BP.enable_kernel_timing(True)
    out = neck([f1] + metas, depth5)
    go = torch.randn(out.shape, generator=torch.Generator().manual_seed(3)).cuda()
    out.backward(go)
    used = BP.kernel_timings_ms()
    BP.enable_kernel_timing(False)
    # one autograd node: the backward goes from grad_ds + mask straight to the gradient rows
    assert "maxdown_fwd" in used and "pool_bwd_ds" in used
    assert "maxdown_bwd" not in used and "pool_bwd" not in used
    # the reference's expression on the same pooled volume
    f2 = feat5.detach().clone().requires_grad_()
    bev, _ = neck.view_transform([f2] + metas, depth5.reshape(B * cfg.n_cams, cfg.D, H, W),
                                 f2.reshape(B * cfg.n_cams, C, H, W))
    b, c, z, y, x = bev.shape
    want = ref_maxdown(bev)
    d2 = depth5.detach().clone().requires_grad_()
    bev2, _ = neck.view_transform([f2] + metas, d2.reshape(B * cfg.n_cams, cfg.D, H, W),
                                  f2.reshape(B * cfg.n_cams, C, H, W))
    want2 = ref_maxdown(bev2)
    f2.grad = None
    want2.backward(go)
    assert torch.equal(out, want) and torch.equal(out, want2)
    assert torch.equal(f1.grad, f2.grad)
    # depth gradient through the fused node as well
    d1 = depth5.detach().clone().requires_grad_()
    f3 = feat5.detach().clone().requires_grad_()
    neck([f3] + metas, d1).backward(go)
    assert torch.equal(d1.grad, d2.grad) and torch.equal(f3.grad, f2.grad)


def test_fused_geometry_gives_the_same_ranks_and_volume():
    """SURVEY 8f-3: get_lidar_coor folded into the preparation kernel = the two-step route"""
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 64
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C, collapse_z=False)
    img, metas, depth, feat = inputs(cfg, B, C, seed=8)
    # non-trivial augmentation so that every matrix matters
    metas[3] = metas[3] + 0.01 * torch.randn(metas[3].shape, generator=torch.Generator().manual_seed(1)).cuda()
    metas[4] = metas[4] + torch.tensor([3.0, -2.0, 0.0]).cuda()
    coor = neck.get_lidar_coor(*metas)
    a = BP.prepare_ranks(coor, neck.grid_lower_bound, neck.grid_interval, neck.grid_size)
    b = BP.prepare_ranks_calib(neck._frustum_on(coor.device), metas[0], metas[2], metas[3], metas[4],
                               metas[5], neck.grid_lower_bound, neck.grid_interval, neck.grid_size)
    n, m = a.plan.n_points, a.plan.n_intervals
    assert (n, m) == (b.plan.n_points, b.plan.n_intervals) and n > 0
    for x, y in ((a.ranks_bev, b.ranks_bev), (a.ranks_depth, b.ranks_depth),
                 (a.ranks_feat, b.ranks_feat)):
        assert torch.equal(x[:n], y[:n])
    assert torch.equal(a.interval_starts[:m], b.interval_starts[:m])
    assert torch.equal(a.plan.tile_start, b.plan.tile_start)
    fused, _ = neck.view_transform([img] + metas, depth, feat)
    neck.fuse_geometry = False
    plain, _ = neck.view_transform([img] + metas, depth, feat)
    assert torch.equal(fused, plain)


# ---- round 2: calibration-keyed rank cache (8f-3), negligible-depth skip (8f-2), range check ------
def test_rank_cache_keyed_on_the_calibration():
    """`rank_cache=N` keeps the prepared ranks of the last N calibrations (64-bit hash of the
    calibration tensors' bits): same volume bit for bit, the preparation runs once per rig, a
    changed calibration is a miss, and the least recently used rig is the one that is dropped."""
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 32
    plain = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C, collapse_z=False)
    cached = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                collapse_z=False, rank_cache=2)
    img, metas, depth, feat = inputs(cfg, B, C, seed=21)
    rigs = [metas]
    for k in (1, 2):                       # two more rigs: a shifted and a rotated one
        m = [t.clone() for t in metas]
        m[0][..., :3, 3] += 0.05 * k
        m[4][..., 0] += 2.0 * k
        rigs.append(m)
    want = [plain.view_transform([img] + m, depth, feat)[0] for m in rigs]
    order = [0, 0, 1, 0, 1, 2, 0, 1]
    BP.enable_kernel_timing(True)
    for i in order:
        # fresh tensor objects every call: the key is the VALUES, not the objects
        got, _ = cached.view_transform([img] + [t.clone() for t in rigs[i]], depth, feat)
        assert torch.equal(got, want[i])
    n_prepare = len(BP.kernel_timings_ms().get("prepare_v2", []))
    BP.enable_kernel_timing(False)
    # two slots, least recently used out: misses at calls 1 (rig 0), 3 (rig 1), 6 (rig 2, drops
    # rig 0), 7 (rig 0, drops rig 1), 8 (rig 1, drops rig 2) => 5 preparations for 8 calls
    assert cached.rank_cache_misses == n_prepare == 5 and cached.rank_cache_hits == 3
    # a single changed bit is a different rig
    assert BP.calib_hash(*[rigs[0][k] for k in (0, 2, 3, 4, 5)]) != \
        BP.calib_hash(*[rigs[1][k] for k in (0, 2, 3, 4, 5)])
    assert BP.calib_hash(*[rigs[0][k] for k in (0, 2, 3, 4, 5)]) == \
        BP.calib_hash(*[rigs[0][k].clone() for k in (0, 2, 3, 4, 5)])


def test_negligible_depth_bins_can_be_skipped_at_inference():
    """SURVEY 8f-2: with VEON's two-hot depth (view_transformer_raw.py:406-429, clamp at -16) most
    bins weigh ~e^-16 of their pixel.  depth_eps drops them before they are ranked: far fewer
    points, the pooled volume within the north_star tolerance (max-abs <= 1e-3 relative; in fact
    ~1e-6), and the exact path whenever a gradient is wanted."""
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformerRaw
    cfg = S.CONFIGS["C1"]
    B, C = 2, 64
    H, W = cfg.feat_hw
    img, metas, _, feat = inputs(cfg, B, C, seed=22)
    exact = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C, use_ds=False)
    sparse = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C, use_ds=False,
                                   depth_eps=1e-6)
    metric = torch.from_numpy(S.metric_depth_np(cfg, batch=B)).cuda()
    depth5 = exact.get_two_hot_depth(metric)                       # [B,N,D,H,W], peaky
    assert float((depth5 > 1e-6).float().mean()) < 0.15
    feat5 = feat.view(B, cfg.n_cams, C, H, W)
    with torch.no_grad():
        a = exact([feat5] + metas, depth5)
        b = sparse([feat5] + metas, depth5)
    assert a.shape == b.shape == (B, C, 16, 200, 200)
    err = float((a - b).abs().max() / a.abs().max())
    assert err <= 1e-3, err
    assert err <= 1e-5, err
    # the point list really shrank
    fr = exact._frustum_on(metas[0].device)
    grid = (exact.grid_lower_bound, exact.grid_interval, exact.grid_size)
    full = BP.prepare_ranks_calib(fr, metas[0], metas[2], metas[3], metas[4], metas[5], *grid)
    thin = BP.prepare_ranks_calib(fr, metas[0], metas[2], metas[3], metas[4], metas[5], *grid,
                                  depth=depth5, depth_eps=1e-6)
    assert thin.plan.n_points < 0.2 * full.plan.n_points
    kept = thin.ranks_depth[:thin.plan.n_points].long()
    assert bool((depth5.reshape(-1)[kept] > 1e-6).all())
    # training: depth_eps is ignored, gradients are the exact ones
    f1 = feat5.detach().clone().requires_grad_()
    f2 = feat5.detach().clone().requires_grad_()
    go = torch.randn(a.shape, generator=torch.Generator().manual_seed(1)).cuda()
    exact([f1] + metas, depth5).backward(go)
    sparse([f2] + metas, depth5).backward(go)
    assert torch.equal(f1.grad, f2.grad)


def test_out_of_range_ranks_are_refused():
    """The reference checks nothing (bev_pool.cpp has no CHECK_* macros: a bad rank is a silent
    out-of-bounds access); here a plan flagged VEON_PLAN_OUT_OF_RANGE raises."""
    from veon_b200.bev_pool import bev_pool_v2
    B, N, D, H, W, C = 1, 1, 2, 2, 2, 4
    depth = torch.rand(B, N, D, H, W, device="cuda")
    feat = torch.rand(B, N, H, W, C, device="cuda")
    rd = torch.tensor([0, 4, 1, 6], dtype=torch.int32, device="cuda")
    rf = torch.tensor([0, 0, 1, 2], dtype=torch.int32, device="cuda")
    st = torch.tensor([0, 2], dtype=torch.int32, device="cuda")
    ln = torch.tensor([2, 2], dtype=torch.int32, device="cuda")
    for bad in (dict(rb=[0, 0, 1, 99]), dict(rd=[0, 4, 1, 8]), dict(rf=[0, 0, 1, 4])):
        r = dict(rb=[0, 0, 1, 1], rd=rd.tolist(), rf=rf.tolist())
        r.update(bad)
        t = {k: torch.tensor(v, dtype=torch.int32, device="cuda") for k, v in r.items()}
        with pytest.raises(ValueError):
            bev_pool_v2(depth, feat, t["rd"], t["rf"], t["rb"], (1, 1, 2, 2, C), st, ln)


def test_inference_ranks_without_backward_tables():
    """prepare_ranks_calib(backward_tables=False): same ranks, plan and pooled volume, no
    point -> interval table; a backward through them is refused, not wrong."""
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 16
    H, W = cfg.feat_hw
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C, collapse_z=False)
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).cuda() for k in KEYS]
    g = torch.Generator().manual_seed(5)
    depth = torch.softmax(torch.randn(B, cfg.n_cams, cfg.D, H, W, generator=g) * 4, dim=2).cuda()
    feat = torch.randn(B, cfg.n_cams, C, H, W, generator=g).cuda()
    full = neck._prepare_calib(metas, depth)
    lean = neck._prepare_calib(metas, depth, backward_tables=False)
    torch.cuda.synchronize()
    assert lean.plan.point_interval is None and full.plan.point_interval is not None
    for a, b in ((full.ranks_bev, lean.ranks_bev), (full.ranks_depth, lean.ranks_depth),
                 (full.ranks_feat, lean.ranks_feat), (full.plan.tile_start, lean.plan.tile_start),
                 (full.plan.tile_occ, lean.plan.tile_occ)):
        n = full.plan.n_points if a.numel() >= full.plan.n_points and a is not full.plan.tile_start \
            and a is not full.plan.tile_occ else a.numel()
        assert torch.equal(a[:n], b[:n])
    with torch.no_grad():
        assert torch.equal(neck._pool_prepared(full, depth, feat), neck._pool_prepared(lean, depth, feat))
    d = depth.clone().requires_grad_()
    out = neck._pool_prepared(lean, d, feat)
    with pytest.raises(RuntimeError, match="backward_tables=False"):
        out.sum().backward()


def test_prefetched_ranks_are_picked_up_and_give_the_same_volume():
    """prefetch_ranks(coor) on the side stream + voxel_pooling_v2(coor, ...): same volume and
    gradients as the plain call; another tensor (or a modified one) is prepared afresh."""
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 16
    H, W = cfg.feat_hw
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C, collapse_z=False)
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B)).cuda()
    other = torch.from_numpy(S.lidar_coor_np(cfg, batch=B, sample_offset=7)).cuda()
    g = torch.Generator().manual_seed(9)
    depth = torch.softmax(torch.randn(B, cfg.n_cams, cfg.D, H, W, generator=g) * 4, dim=2).cuda()
    feat = torch.randn(B, cfg.n_cams, C, H, W, generator=g).cuda()
    og = torch.randn(B, C, 16, 200, 200, generator=g).cuda()

    def run(c, prefetch):
        d, f = depth.clone().requires_grad_(), feat.clone().requires_grad_()
        if prefetch is not None:
            neck.prefetch_ranks(prefetch)
        out = neck.voxel_pooling_v2(c, d, f)
        out.backward(og)
        torch.cuda.synchronize()
        return out.detach(), d.grad, f.grad

    plain = run(coor, None)
    for a, b in zip(plain, run(coor, coor)):            # prefetched and used
        assert torch.equal(a, b)
    assert neck.__dict__["_prefetched"] is None
    for a, b in zip(plain, run(coor, other)):           # prefetched for another tensor: ignored
        assert torch.equal(a, b)
    for a, b in zip(run(other, None), run(other, other)):
        assert torch.equal(a, b)
