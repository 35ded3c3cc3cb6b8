"""GPU: bfloat16 volumes (dtype=torch.bfloat16) for bev_pool_v2, pool_prepared and
LSSViewTransformer, in both memory formats, and the backward that reads their bfloat16 gradient.

The contract is exact: the bfloat16 volume is the float32 volume cast to bfloat16 ON THE DEVICE,
bit for bit (NaN positions must match, payloads are not compared), and the float32 depth / feat
gradients of a bfloat16 gradient are the float32 route's given that gradient widened."""
import numpy as np
import pytest
import torch

from tests.test_channels_last_gpu import _case, _is_cl_view, _neck_inputs, _pool
from tests.test_pool_gpu import gpu_ranks, make_case
from veon_b200 import synthetic as S

pytestmark = pytest.mark.gpu
CL = torch.channels_last_3d
BF = torch.bfloat16


def assert_bits(bf, want):
    """bf (bfloat16) equals want (float32, cast here on the device) bit for bit, NaN positions
    included; both are compared in their logical [B,C,Z,Y,X] order"""
    assert bf.dtype == BF and bf.shape == want.shape
    want = want.to(BF)
    na, nb = torch.isnan(bf), torch.isnan(want)
    assert torch.equal(na, nb)
    a = bf.masked_fill(na, 0).contiguous().view(torch.int16)
    b = want.masked_fill(nb, 0).contiguous().view(torch.int16)
    assert torch.equal(a, b)


FWD_CASES = [("tiny", 2, 4), ("tiny", 2, 20), ("C1", 2, 28), ("tiny", 2, 32), ("tiny", 2, 33),
             ("small", 2, 64), ("C1", 1, 64), ("small", 2, 96), ("small", 2, 128),
             ("C1", 1, 512), ("ragged", 2, 4), ("ragged", 2, 20), ("ragged", 3, 33),
             ("ragged", 2, 64), ("ragged", 2, 96), ("ragged", 1, 512), ("tiny", 8, 64),
             ("tiny", 8, 28)]


@pytest.mark.parametrize("cfg_name,batch,C", FWD_CASES)
def test_forward_bf16_is_the_float32_volume_cast(cfg_name, batch, C):
    case = _case(cfg_name, batch, C)
    from veon_b200.bev_pool import bev_pool_v2
    rb, rd, rf, st, ln = gpu_ranks(case["ranks"])
    args = (case["depth"].cuda(), case["feat"].cuda(), rd, rf, rb, case["shape"], st, ln)
    for fmt in (torch.contiguous_format, CL):
        f32 = bev_pool_v2(*args, memory_format=fmt)
        bf = bev_pool_v2(*args, memory_format=fmt, dtype=BF)
        assert bf.is_contiguous() if fmt is torch.contiguous_format else _is_cl_view(bf)
        assert_bits(bf, f32)


def test_forward_bf16_c2_geometry():
    """B = 8, C = 64 and C = 20 over the C2 grid: the general kernel (no streaming kernel for
    bfloat16) and the narrow-row kernel, heavy tiles in both"""
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
        feat = torch.randn(B, N, H, W, C, device="cuda", generator=g)
        shape = (B, 16, 200, 200, C)
        for fmt in (torch.contiguous_format, CL):
            f32 = BP.pool_prepared(depth, feat, prep, shape, fmt)
            bf = BP.pool_prepared(depth, feat, prep, shape, fmt, dtype=BF)
            assert_bits(bf, f32)
            del f32, bf


def test_forward_bf16_voxel_with_thousands_of_points():
    """heavy-tile rounds carried over in one voxel, a second voxel starting mid-round"""
    from veon_b200.bev_pool import bev_pool_v2
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
        depth = torch.rand(B, N, D, H, W, generator=g)
        feat = torch.randn(B, N, H, W, C, generator=g)
        args = (depth.cuda(), feat.cuda(), rd.cuda(), rf.cuda(), rb.cuda(), (B, Z, Y, X, C),
                st.cuda(), ln.cuda())
        for fmt in (torch.contiguous_format, CL):
            assert_bits(bev_pool_v2(*args, memory_format=fmt, dtype=BF),
                        bev_pool_v2(*args, memory_format=fmt))


def _edge_values():
    """float32 values whose bfloat16 rounding is an edge case"""
    def f(bits):
        return np.array(bits, np.uint32).view(np.float32)
    return np.concatenate([
        f([0x3F808000, 0x3F818000, 0xBF808000, 0xBF818000,     # exact half-way: to even, down / up
           0x3F808001, 0x3F807FFF, 0x4049FFFF, 0x7F7F8000]),   # just off half-way; 0x7F7F8000 -> inf
        f([0x7F7FFFFF, 0xFF7FFFFF, 0x7F7F7FFF]),                # the largest floats: +-inf; below: finite
        f([0x00010000, 0x00008000, 0x80018000, 0x00000001,     # bfloat16 subnormals and below them
           0x007FFFFF, 0x00800000]),
        np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, 1.0, -3.5], np.float32)])


@pytest.mark.parametrize("C", [8, 64, 36])
def test_store_rounding_edges(C):
    """single-point voxels with depth 1.0: the stored value is fma(feat, 1, 0), so the volume holds
    the hand-set features and pins the store rule: round to nearest even like the device cast"""
    from veon_b200.bev_pool import bev_pool_v2
    vals = _edge_values()
    P = 64
    feat = np.resize(vals, P * C).reshape(1, 1, 1, P, C)
    feat = np.ascontiguousarray(np.roll(feat, 3, axis=4))
    idx = np.arange(P, dtype=np.int32)
    rb = idx * 2                                          # every other voxel, X = 128
    depth = torch.ones(1, 1, 1, 1, P).cuda()
    args = (depth, torch.from_numpy(feat).cuda(), torch.from_numpy(idx).cuda(),
            torch.from_numpy(idx).cuda(), torch.from_numpy(rb).cuda(), (1, 1, 1, 2 * P, C),
            torch.from_numpy(idx).cuda(), torch.ones(P, dtype=torch.int32).cuda())
    for fmt in (torch.contiguous_format, CL):
        f32 = bev_pool_v2(*args, memory_format=fmt)
        bf = bev_pool_v2(*args, memory_format=fmt, dtype=BF)
        assert_bits(bf, f32)
        got = bf[0, :, 0, 0, ::2].t().float().cpu().numpy()          # [P, C]
        # the sum is fma(f, 1, +0) = f + 0 (so -0 is stored as +0); the host cast rounds the
        # same way as the device
        want = torch.from_numpy(feat[0, 0, 0] + np.float32(0)).to(BF).float().numpy()
        fin = ~np.isnan(want)
        assert np.array_equal(np.isnan(got), ~fin)
        assert np.array_equal(got[fin].view(np.uint32), want[fin].view(np.uint32))
        assert np.isinf(got).sum() >= 3                               # the overflows happened


def _grads(case, fwd_format, og, dtype, feat_view=False, timing=True, spy=None):
    from veon_b200 import bev_pool as BP
    depth = case["depth"].cuda().requires_grad_()
    if feat_view:   # the neck's channels-last view of channels-first maps
        f = case["feat"].permute(0, 1, 4, 2, 3).contiguous().cuda().requires_grad_()
        feat_in, leaf = f.permute(0, 1, 3, 4, 2), f
    else:
        leaf = feat_in = case["feat"].cuda().requires_grad_()
    out = _pool(case, fwd_format, depth, feat_in) if dtype is torch.float32 else \
        _pool_dtype(case, fwd_format, depth, feat_in, dtype)
    BP.enable_kernel_timing(timing)
    out.backward(og)
    used = BP.kernel_timings_ms() if timing else {}
    BP.enable_kernel_timing(False)
    torch.cuda.synchronize()
    fg = leaf.grad.permute(0, 1, 3, 4, 2) if feat_view else leaf.grad
    return depth.grad, fg, used


def _pool_dtype(case, memory_format, depth, feat, dtype):
    from veon_b200.bev_pool import bev_pool_v2
    rb, rd, rf, st, ln = gpu_ranks(case["ranks"])
    return bev_pool_v2(depth, feat, rd, rf, rb, case["shape"], st, ln,
                       memory_format=memory_format, dtype=dtype)


@pytest.mark.parametrize("cfg_name,batch,C", [("tiny", 2, 4), ("tiny", 2, 20), ("small", 2, 64),
                                              ("C1", 2, 100), ("small", 2, 256), ("small", 3, 512),
                                              ("ragged", 2, 36), ("ragged", 2, 64)])
@pytest.mark.parametrize("feat_view", [False, True])
def test_backward_bf16_gradient_in_each_storage(cfg_name, batch, C, feat_view, monkeypatch):
    from veon_b200 import bev_pool as BP
    case = _case(cfg_name, batch, C, seed=1)
    B, Z, Y, X, _ = case["shape"]
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(2)).cuda().to(BF)
    dg_ref, fg_ref, used = _grads(case, torch.contiguous_format, og.float(), torch.float32,
                                  feat_view)
    assert "pool_bwd" in used
    scratch = []
    real = BP._bwd_rows
    monkeypatch.setattr(BP, "_bwd_rows", lambda *a: scratch.append(1) or real(*a))
    odd = og.permute(0, 1, 4, 3, 2).contiguous().permute(0, 1, 4, 3, 2)
    for fwd_format in (torch.contiguous_format, CL):
        for g, name in ((og, "pool_bwd_bf16"), (og.contiguous(memory_format=CL), "pool_bwd_cl_bf16"),
                        (odd, "pool_bwd_bf16")):
            del scratch[:]
            dg, fg, used = _grads(case, fwd_format, g, BF, feat_view)
            assert name in used and not ({"pool_bwd", "pool_bwd_cl", "pool_bwd_bf16",
                                          "pool_bwd_cl_bf16"} - {name}) & set(used), used
            assert bool(scratch) == (name == "pool_bwd_bf16")   # the single pass: no rows scratch
            assert torch.equal(dg, dg_ref) and torch.equal(fg, fg_ref), (fwd_format, name)


def _rejected(case, how):
    rb, rd, rf, st, ln = case["ranks"]
    if how == "shuffled":   # interval order shuffled: unsorted ranks_bev
        perm = np.random.RandomState(0).permutation(st.size)
        parts = [(rb[st[k]:st[k] + ln[k]], rd[st[k]:st[k] + ln[k]], rf[st[k]:st[k] + ln[k]])
                 for k in perm]
        lens = np.array([len(p[0]) for p in parts], np.int32)
        return (np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
                np.concatenate([p[2] for p in parts]),
                np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int32), lens)
    # hand-made: the right runs, but every point reads another pixel's feature row
    B, N, D, H, W = case["dims"]
    rf2 = ((rf + 7) % (B * N * H * W)).astype(np.int32)
    return rb, rd, rf2, st, ln


@pytest.mark.parametrize("how", ["shuffled", "hand-made"])
def test_rejected_plans_bf16(how):
    """the plan is rejected: the generic kernel pools into a float32 volume that is then cast, and
    the backward widens the bfloat16 gradient for it"""
    from veon_b200 import bev_pool as BP
    case = make_case("tiny", 2, 24, seed=7)
    case2 = dict(case, ranks=_rejected(case, how))
    rb, rd, rf, st, ln = gpu_ranks(case2["ranks"])
    B, Z, Y, X, C = case["shape"]
    plan = BP._plan_for(rd, rf, rb, st, ln, case["dims"], Z * Y * X)
    assert not plan.ok
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(8)).cuda().to(BF)
    for fmt in (torch.contiguous_format, CL):
        dg_ref, fg_ref, _ = _grads(case2, fmt, og.float(), torch.float32, timing=False)
        f32 = _pool(case2, fmt)
        bf = _pool_dtype(case2, fmt, case["depth"].cuda(), case["feat"].cuda(), BF)
        assert_bits(bf, f32)
        for g in (og, og.contiguous(memory_format=CL)):
            dg, fg, _ = _grads(case2, fmt, g, BF, timing=False)
            assert torch.equal(dg, dg_ref)
            # the generic backward accumulates feat_grad with float atomics (order varies run
            # to run, in the float32 route as well)
            torch.testing.assert_close(fg, fg_ref, rtol=1e-5, atol=1e-6)


def test_sync_free_bf16_single_pass_reads_no_interval_past_the_count():
    from veon_b200 import bev_pool as BP
    case = make_case("small", 2, 64, seed=4)
    lower, interval, size = case["grid"]
    B, Z, Y, X, C = case["shape"]
    og = torch.randn(B, C, Z, Y, X, generator=torch.Generator().manual_seed(5)).cuda().to(BF)
    coor = case["coor"].copy()
    coor[:, :, 6:] = 1e4
    grads = []
    for poison in (False, True):
        prep = BP.prepare_ranks(torch.from_numpy(coor).cuda(), lower, interval, size)
        n_int = prep.plan.n_intervals
        assert 4 * n_int < prep.interval_starts.numel()
        if poison:
            prep.interval_starts[n_int:] = 0
            prep.plan.sync_free = True
        depth = case["depth"].cuda().requires_grad_()
        feat = case["feat"].cuda().requires_grad_()
        out = BP.pool_prepared(depth, feat, prep, case["shape"], CL, dtype=BF)
        out.backward(og.contiguous(memory_format=CL))
        grads.append((out.detach(), depth.grad, feat.grad))
    for a, b in zip(*grads):
        assert torch.equal(a, b)


@pytest.mark.parametrize("C", [64, 20, 100])
@pytest.mark.parametrize("fmt", [torch.contiguous_format, CL])
def test_next_kernel_in_the_stream_sees_the_whole_bf16_volume(C, fmt):
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
    ref = BP.pool_prepared(depth, feat, prep, shape).to(BF)
    torch.cuda.synchronize()
    scratch = torch.empty(64 << 20, device="cuda")
    for i in range(4):
        scratch.normal_()
        vol = BP.pool_prepared(depth, feat, prep, shape, fmt, dtype=BF)
        copy = vol.clone(memory_format=fmt)                # the very next kernel reads it
        torch.cuda.synchronize()
        assert torch.equal(copy, ref), f"iteration {i}: a consumer ran before the volume was complete"


@pytest.mark.parametrize("C", [64, 20])
@pytest.mark.parametrize("channels_last", [False, True])
def test_bf16_forward_inside_a_cuda_graph(C, channels_last):
    from veon_b200 import bev_pool as BP
    case = make_case("C1", 2, C, seed=7)
    rb, rd, rf, st, ln = gpu_ranks(case["ranks"])
    B, Z, Y, X, C = case["shape"]
    V = Z * Y * X
    plan = BP._plan_for(rd, rf, rb, st, ln, case["dims"], V)
    assert plan.ok and int(plan.tile_heavy[0]) > 0
    depth, feat = case["depth"].cuda(), case["feat"].cuda()
    shape = (B, Z, Y, X, C) if channels_last else (B, C, Z, Y, X)

    def run():
        return BP._fwd_planar(depth, feat, rd, rf, rb, plan, B, C, V, shape, channels_last, BF)
    want = BP._fwd_planar(depth, feat, rd, rf, rb, plan, B, C, V, shape, channels_last)
    eager = run().clone()
    assert_bits(eager, want)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    with torch.cuda.graph(graph):
        vol = run()
        copy = vol.clone()
    for _ in range(3):
        copy.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(vol.view(torch.int16), eager.view(torch.int16))
        assert torch.equal(copy.view(torch.int16), eager.view(torch.int16))


# ---------------------------------------------------------------- necks
@pytest.mark.parametrize("sync_free", [False, True])
@pytest.mark.parametrize("fmt", [torch.contiguous_format, CL])
def test_neck_bf16_routes(sync_free, fmt):
    """fused geometry, voxel_pooling_v2(coor, ...), accelerate, collapse_z: the bfloat16 neck's
    volume is the float32 neck's cast; its input gradients are the float32 neck's for the same
    gradient widened"""
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["small"]
    B, C = 2, 32
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=3)
    H, W = cfg.feat_hw
    og = torch.randn(B, C, 16, 200, 200, generator=torch.Generator().manual_seed(4)).cuda().to(BF)
    necks = [LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                collapse_z=False, sync_free=sync_free, memory_format=fmt,
                                dtype=dt)
             for dt in (torch.float32, BF)]

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
        for neck, g in zip(necks, (og.float(), og)):
            d = depth.detach().clone().requires_grad_()
            f = feat.detach().clone().requires_grad_()
            bev = route(neck, d, f)
            bev.backward(g)
            res.append((bev.detach(), d.grad, f.grad))
        (a, da, fa), (b, db, fb) = res
        assert b.dtype == BF and (b.is_contiguous() if fmt is torch.contiguous_format
                                  else _is_cl_view(b)), route.__name__
        assert_bits(b, a)
        assert torch.equal(da, db) and torch.equal(fa, fb), route.__name__
    for neck in necks:
        neck.collapse_z = True
    a, b = (fused(n, depth, feat) for n in necks)
    assert a.shape == (B, C * 16, 200, 200)
    assert_bits(b, a)


@pytest.mark.parametrize("sync_free", [False, True])
def test_neck_bf16_with_no_points_in_the_grid(sync_free):
    """the reference's dummy (or, sync-free, the all-zero volume) in the requested dtype"""
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["tiny"]
    B, C = 1, 8
    img, metas, depth, feat = _neck_inputs(cfg, B, C, seed=9)
    metas[0] = metas[0].clone()
    metas[0][..., :3, 3] += 1e5          # every camera far outside the grid
    outs = []
    for dt in (torch.float32, BF):
        neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                  sync_free=sync_free, dtype=dt)
        outs.append(neck.view_transform([img] + metas, depth, feat)[0])
        coor = neck.get_lidar_coor(*metas)[:0]
        H, W = cfg.feat_hw
        empty = neck.voxel_pooling_v2(coor, depth.view(B, cfg.n_cams, cfg.D, H, W),
                                      feat.view(B, cfg.n_cams, C, H, W))
        assert empty.dtype == dt and not bool(empty.any())
    a, b = outs
    assert not bool(a.any()) and b.dtype == BF
    assert_bits(b, a)
