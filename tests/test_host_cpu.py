"""CPU: C-ABI surface, host-side mirror logic, multi-process sharding (gloo)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "veon_lift.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(veon_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from veon_b200 import _lib
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), f"libveonlift.so does not export {n}"
    assert set(names) == set(_lib.EXPORTED_SYMBOLS), "ctypes table and header disagree"
    header = open(os.path.join(ROOT, "include", "veon_lift.h")).read()
    declared = int(re.search(r"#define\s+VEON_ABI_VERSION\s+(\d+)", header).group(1))
    assert lib.veon_abi_version() == declared >= 3
    assert b"bad argument" in lib.veon_error_string(-1)


def test_argument_errors_do_not_need_a_gpu():
    from veon_b200 import _lib
    lib = _lib.load()
    null = ctypes.c_void_p(0)
    assert lib.veon_bev_pool_v2(64, 10, null, null, null, null, null, null, null, null, null) == -1
    assert lib.veon_bev_pool_v2_fwd_planar(null, null, null, null, null, null, null, null, null, 0,
                                           1, 64, 640000, 4224, null, null, 0, null) == -1
    assert lib.veon_bev_pool_v2_fwd_workspace_bytes(8, 64, 640000) > (32 << 20)
    assert lib.veon_bev_pool_v2_fwd_workspace_bytes(0, 64, 640000) == 0
    gs = _lib.float3([200, 200, 16])
    assert lib.veon_prepare_v2_workspace_bytes(8, 6, 88, 16, 44, gs) > 0
    assert lib.veon_prepare_v2_workspace_bytes(0, 6, 88, 16, 44, gs) == 0
    assert lib.veon_pool_num_tiles(8, 640000) == 8 * 20000
    assert lib.veon_pool_num_tiles(2, 33) == 4
    # the entry points added for the neck's other steps validate before touching CUDA as well
    f1 = ctypes.c_float(1.0)
    assert lib.veon_two_hot_depth(null, 1, 4, 4, 8, 88, f1, ctypes.c_float(0.5), f1, null, null) == -1
    assert lib.veon_maxdown2_fwd(null, 1, 16, 200, 200, null, null) == -1
    assert lib.veon_maxdown2_fwd_mask(null, 1, 16, 200, 200, null, null, null) == -1
    assert lib.veon_maxdown2_bwd(null, null, null, 1, 16, 200, 200, null, null) == -1
    assert lib.veon_transpose_batched(null, 1, 4, 4, null, null) == -1
    assert lib.veon_bev_pool_v2_bwd_planar_ds(null, null, null, null, null, null, null, 0, 1, 1, 2, 2,
                                              2, 64, 16, 200, 200, null, null, null, null) == -1
    assert lib.veon_pool_heavy_list_ints(1000, 10) == 12 and lib.veon_pool_heavy_list_ints(64, 10) == 4
    # fused lift + classify: argument and shape errors are decided before any launch
    assert lib.veon_lift_classify_fwd(null, null, null, null, null, null, null, 0, 1, 20, 18, 16, 200,
                                      200, 10, null, 17, null, null) == -1
    buf4 = ctypes.cast((ctypes.c_float * 64)(), ctypes.c_void_p)
    args = lambda Cp, Q, Z: (buf4, buf4, buf4, buf4, buf4, buf4, buf4, 8, 1, Cp, Q, Z, 200, 200, 10, buf4,
                             17, buf4, null)
    assert lib.veon_lift_classify_fwd(*args(22, 18, 16)) == -4      # Cp % 4
    assert lib.veon_lift_classify_fwd(*args(20, 19, 16)) == -4      # Q + 2 > Cp
    assert lib.veon_lift_classify_fwd(*args(100, 94, 16)) == -4     # Cp > 96
    assert lib.veon_lift_classify_fwd(buf4, buf4, buf4, buf4, buf4, buf4, buf4, 8, 1, 20, 18, 3, 5, 7,
                                      10, buf4, 17, buf4, null) == -4   # V = 105: not whole tiles
    # the SM reservation is a plain process-wide setting (no device needed)
    assert lib.veon_reserve_sms(5) == 0 and lib.veon_reserve_sms(-3) == 5 and lib.veon_reserve_sms(0) == 0
    # the tail's entry points
    assert lib.veon_semantic_inference_3d(null, null, 1, 64, 18, 8, 100, 100, null, null, null) == -1
    # the classifier's tensor-core operand image: [W_hi ; W_lo] of every 32-channel chunk
    assert lib.veon_text_classifier_image_bytes(18, 512) == 16 * 2 * 32 * 32 * 4
    assert lib.veon_text_classifier_image_bytes(67, 512) == 16 * 2 * 80 * 32 * 4
    assert lib.veon_text_classifier_image_bytes(18, 100) == 0       # C % 32: the FFMA kernel's shapes
    assert lib.veon_text_classifier_image_bytes(200, 512) == 0
    assert lib.veon_text_classifier_image(null, 18, 512, null, 0, null) == -1
    assert lib.veon_upsample_classify(null, null, null, 1, 18, 8, 100, 100, 16, 200, 200, 17,
                                      null, null) == -1
    assert lib.veon_classify_logits(null, 0, null, 0, null, 1, 18, 16, 200, 200, 17, null, null) == -1
    assert lib.veon_voxel_text_argmax_lowres_workspace_bytes(2, 18, 8, 100, 100) == 2 * 18 * 80000 * 4
    assert lib.veon_voxel_text_argmax_lowres_workspace_bytes(0, 18, 8, 100, 100) == 0
    some = ctypes.cast((ctypes.c_float * 4)(), ctypes.c_void_p)
    assert lib.veon_voxel_text_argmax_lowres(some, some, some, some, 1, 64, 18, 8, 100, 100, 16, 200,
                                             200, 17, some, null, 0, null, null) == -1  # no workspace
    assert lib.veon_voxel_text_argmax_lowres(some, some, some, some, 1, 64, 18, 8, 100, 100, 16, 200,
                                             200, 17, some, some, 16, null, null) == -2  # too small
    # a pooled volume that the fused / down-sample kernels do not take is refused, not mangled
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert lib.veon_maxdown2_fwd(p, 1, 3, 4, 8, p, null) == -4          # odd Z
    assert lib.veon_maxdown2_fwd(p, 1, 2, 4, 6, p, null) == -4          # X % 4 != 0


def test_cpu_tensors_are_refused_loudly():
    from veon_b200.bev_pool import bev_pool_v2, voxel_pooling_prepare_v2
    from veon_b200 import synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer
    cfg = S.CONFIGS["tiny"]
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4)
    cal = S.calibration(cfg, batch=1)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        neck.get_lidar_coor(*[torch.from_numpy(cal[k]) for k in
                              ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        voxel_pooling_prepare_v2(torch.zeros(1, 1, 2, 2, 2, 3), [0, 0, 0], [1, 1, 1], [4, 4, 2])
    z = torch.zeros(1, 1, 2, 2, 2)
    i = torch.zeros(2, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        bev_pool_v2(z, z, i, i, i, (1, 1, 2, 2, 2), i, i)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from veon_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.VeonLibraryError):
        _lib.load()


def test_view_transformer_mirror_geometry(golden_dir):
    """frustum and get_lidar_coor against the reference's outputs"""
    from oracle import lift_oracle as O
    from veon_b200 import synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer
    geo = np.load(os.path.join(golden_dir, "geometry_tiny.npz"))
    for name in ("tiny", "C1"):
        cfg = S.CONFIGS[name]
        neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, cfg.channels)
        assert neck.D == int(geo[f"{name}.D"]) == cfg.D
        np.testing.assert_array_equal(neck.frustum.numpy(), geo[f"{name}.frustum"])
        lower, interval, size = S.grid_vectors(cfg.grid_config)
        np.testing.assert_array_equal(neck.grid_size.numpy(), size)
        np.testing.assert_array_equal(neck.grid_lower_bound.numpy(), lower)
        np.testing.assert_array_equal(neck.grid_interval.numpy(), interval)
        cal = S.calibration(cfg, batch=1)
        coor = O.lidar_coor_torch(neck.frustum, *[torch.from_numpy(cal[k]) for k in
                                     ("sensor2ego", "ego2global", "intrins", "post_rots",
                                      "post_trans", "bda")]).numpy()
        if name == "tiny":
            np.testing.assert_allclose(coor, geo["tiny.coor"], rtol=0, atol=2e-5)
        else:
            np.testing.assert_allclose(coor[:, :, ::11, ::5, ::7], geo["C1.coor_sample"],
                                       rtol=0, atol=2e-4)
        # and the bit-reproducible rig generator describes the same geometry
        np.testing.assert_allclose(S.lidar_coor_np(cfg, batch=1), coor, rtol=0, atol=2e-4)


def test_tail_class_of_prompt_matches_oracle():
    from oracle.lift_oracle import class_groups
    from veon_b200.tail import class_of_prompt
    sizes = [16, 1, 1, 1, 8, 1, 1, 3, 1, 1, 1, 1, 5, 3, 5, 13, 4]
    refl = [k for k, n in enumerate(sizes) for _ in range(n)]
    assert class_of_prompt(refl).tolist() == class_groups(refl).tolist()
    assert class_of_prompt(list(range(17))).tolist() == list(range(18))


def test_pipeline_heads_and_cpu_refusal():
    """lift_classify stacks [W ; gate] and pads the row count for the 16-byte row copies of the
    pooling kernels; like every operator it refuses CPU tensors."""
    from veon_b200 import pipeline, tail
    w, g = torch.randn(18, 64), torch.randn(2, 64)
    rows = pipeline._heads(w, g)
    assert rows.shape == (20, 64) and torch.equal(rows[:18], w) and torch.equal(rows[18:], g)
    rows = pipeline._heads(torch.randn(67, 64), g)
    assert rows.shape == (72, 64) and torch.all(rows[69:] == 0)
    assert pipeline._heads(w, g, 32).shape == (32, 64)
    with pytest.raises(ValueError):
        pipeline._heads(w, torch.randn(3, 64))
    for fn, args in ((tail.semantic_inference_3d, (w, torch.randn(1, 64, 2, 2, 4))),
                     (tail.classify_logits, (torch.randn(1, 18, 2, 2, 4), torch.randn(1, 2, 2, 2, 4),
                                             torch.arange(18, dtype=torch.int32))),
                     (tail.voxel_text_argmax_lowres, (torch.randn(1, 64, 2, 2, 4), w,
                                                      torch.arange(18, dtype=torch.int32),
                                                      torch.randn(1, 2, 2, 2, 4)))):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(*args)
    # channel slices of one volume are passed through without a copy, anything else is copied
    vol = torch.randn(3, 12, 4, 5, 6)
    assert tail._sample_contiguous(vol[:, :8]).data_ptr() == vol.data_ptr()
    assert tail._sample_contiguous(vol[:, 8:10]).stride(0) == vol.stride(0)
    assert tail._sample_contiguous(vol[:, :, ::2]).is_contiguous()
    assert tail._sample_contiguous(vol[:1].expand(3, 12, 4, 5, 6)).data_ptr() != vol.data_ptr()


def test_shard_samples():
    from veon_b200.dist import shard_samples
    for n, g in ((8, 1), (8, 2), (9, 4), (3, 8), (64, 8)):
        seen = sorted(i for r in range(g) for i in shard_samples(n, g, r))
        assert seen == list(range(n))


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
from veon_b200.dist import shard_samples, all_gather_occupancy, gathered_row
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
r = dist.get_rank()
for n in (5, 4, 1):
    mine = shard_samples(n, 2, r)
    local = torch.stack([torch.full((3, 4, 2), 10 * i + 1, dtype=torch.uint8) for i in mine]) if mine \
        else torch.zeros((0, 3, 4, 2), dtype=torch.uint8)
    full = all_gather_occupancy(local, n)
    assert full.shape == (n, 3, 4, 2), full.shape
    for i in range(n):
        assert int(full[i, 0, 0, 0]) == 10 * i + 1 and bool((full[i] == 10 * i + 1).all())
    raw = all_gather_occupancy(local, n, sample_order=False)      # rank-major, no reordering pass
    assert raw.shape[0] == 2 * ((n + 1) // 2)
    for i in range(n):
        assert bool((raw[gathered_row(i, n, 2)] == 10 * i + 1).all())
dist.destroy_process_group()
print("rank", r, "ok")
"""


def test_all_gather_occupancy_world_size_2_gloo(tmp_path):
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "w.py"
    script.write_text(_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


def test_shard_cameras():
    from veon_b200.dist import shard_cameras
    for n, g in ((6, 1), (6, 2), (6, 4), (6, 8), (5, 3)):
        seen = sorted(c for r in range(g) for c in shard_cameras(n, g, r))
        assert seen == list(range(n))
    with pytest.raises(ValueError):
        shard_cameras(6, 2, 2)


_CAM_WORKER = r"""
import os, sys, types, torch, torch.distributed as dist
sys.path.insert(0, {root!r})
import veon_b200.dist as VD, veon_b200.pipeline as VP, veon_b200.tail as VT
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
r = dist.get_rank()
# stand-ins for the two CUDA stages (this test is about the sharding logic, on the CPU): the
# "lift" of a camera group is the sum of its cameras' per-camera volumes, the classifier an argmax
B, N, Q, Z, Y, X = 2, 6, 5, 2, 3, 4
g = torch.Generator().manual_seed(0)
per_cam = torch.randn(N, B, 8, Z, Y, X, generator=g)            # same on both ranks
seen = []
def fake_lift_logits(neck, input, depth, feat, w, gate, channel_pad=4, cameras=None):
    seen.append(list(cameras))
    return per_cam[list(cameras)].sum(0).clone()
def fake_classify(sem, gate, cls, free_label=17):
    return sem.argmax(1).to(torch.uint8)
VP.lift_logits = fake_lift_logits
VT.classify_logits = fake_classify
neck = types.SimpleNamespace()
inp = [torch.zeros(B, N, 1, 2, 2)] + [None] * 6
w = torch.zeros(Q, 4)
lab = VD.lift_classify_camera_sharded(neck, inp, None, torch.zeros(B * N, 4, 2, 2), w, None, None)
assert seen == [VD.shard_cameras(N, 2, r)], seen
want = per_cam.sum(0)[:, :Q].argmax(1).to(torch.uint8)
assert torch.equal(lab, want), (lab.shape, want.shape)
dist.destroy_process_group()
print("rank", r, "ok")
"""


def test_camera_group_sharding_world_size_2_gloo(tmp_path):
    """every rank lifts ITS cameras, one all-reduce sums the logit volumes, all ranks classify the
    same sum (the CUDA stages are replaced by stand-ins: the host logic is what runs here)"""
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    script = tmp_path / "c.py"
    script.write_text(_CAM_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


@pytest.mark.needs_reference
def test_operator_surface_matches_reference_call_sites():
    """CPU-side drop-in check (the GPU-side one needs both a GPU and
    /root/reference): run the UNMODIFIED reference neck with a recording stub
    bound as `bev_pool_v2` and verify that exactly that call is accepted by our
    operator's signature, and that our prepare wrapper has the reference
    method's shape of result."""
    import inspect
    from _ref_loader import load_reference_view_transformer
    from veon_b200 import bev_pool as BP, synthetic as S
    calls = []

    def recorder(*args, **kwargs):
        calls.append((args, kwargs))
        depth, feat = args[0], args[1]
        B, Z, Y, X, C = args[5]
        return torch.zeros(B, C, Z, Y, X)

    mod = load_reference_view_transformer(recorder)
    cfg = S.CONFIGS["tiny"]
    neck = mod.LSSViewTransformer(grid_config=cfg.grid_config, input_size=cfg.input_size,
                                  downsample=cfg.downsample, in_channels=8, out_channels=4,
                                  collapse_z=False)
    B, N, D = 1, cfg.n_cams, cfg.D
    H, W = cfg.feat_hw
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B))
    neck.voxel_pooling_v2(coor, torch.rand(B, N, D, H, W), torch.rand(B, N, 4, H, W))
    (args, kwargs), = calls
    sig = inspect.signature(BP.bev_pool_v2)
    bound = sig.bind(*args, **kwargs)               # raises TypeError if the surface differs
    assert list(bound.arguments) == ["depth", "feat", "ranks_depth", "ranks_feat", "ranks_bev",
                                     "bev_feat_shape", "interval_starts", "interval_lengths"]
    assert bound.arguments["feat"].shape == (B, N, H, W, 4)          # permuted view, :190
    assert not bound.arguments["feat"].is_contiguous()
    assert all(bound.arguments[k].dtype == torch.int32 for k in
               ("ranks_depth", "ranks_feat", "ranks_bev", "interval_starts", "interval_lengths"))
    # same names on the module as the reference's bev_pool.py
    for name in ("bev_pool_v2", "QuickCumsumCuda", "TRTBEVPoolv2"):
        assert hasattr(BP, name)
    ref_fwd = inspect.signature(BP.QuickCumsumCuda.forward)
    assert list(ref_fwd.parameters)[:9] == ["ctx", "depth", "feat", "ranks_depth", "ranks_feat",
                                            "ranks_bev", "bev_feat_shape", "interval_starts",
                                            "interval_lengths"]
    # the neck mirror exposes the reference neck's methods / attributes
    from veon_b200.view_transformer import LSSViewTransformer
    ours = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4, collapse_z=False)
    for name in ("create_grid_infos", "create_frustum", "get_lidar_coor", "init_acceleration_v2",
                 "voxel_pooling_v2", "voxel_pooling_prepare_v2", "pre_compute", "view_transform_core",
                 "view_transform", "forward"):
        assert callable(getattr(ours, name)) and hasattr(neck, name)
        ref_params = list(inspect.signature(getattr(neck, name)).parameters)
        our_params = list(inspect.signature(getattr(ours, name)).parameters)
        assert ref_params == our_params, (name, ref_params, our_params)
    for attr in ("grid_lower_bound", "grid_interval", "grid_size", "frustum", "D", "accelerate",
                 "initial_flag", "collapse_z", "out_channels", "in_channels", "downsample", "sid"):
        assert hasattr(ours, attr) and hasattr(neck, attr)


# ---- INTEGRATION route B plumbing (no GPU needed) -----------------------------------------------
@pytest.mark.needs_reference
def test_reference_operator_file_runs_on_a_substituted_ext(golden_dir):
    """mmdet3d/ops/bev_pool_v2/bev_pool.py, unmodified, imports whatever module is registered
    as `bev_pool_v2_ext` (bev_pool.py:6).  With an ext made of the C oracle it reproduces the
    reference's known-answer test (bev_pool.py:145-176) on the CPU -- the same substitution
    tests/test_dropin_reference.py makes with veon_b200.bev_pool_v2_ext on the GPU."""
    import json
    import types
    import torch
    from _ref_loader import load_reference_bev_pool
    from oracle import lift_oracle as O

    def fwd(depth, feat, out, rd, rf, rb, ln, st):
        out.copy_(torch.from_numpy(O.bev_pool_v2_channels_last(
            depth.numpy(), feat.numpy(), rd.numpy(), rf.numpy(), rb.numpy(), tuple(out.shape),
            st.numpy(), ln.numpy())))

    mod = load_reference_bev_pool(types.SimpleNamespace(bev_pool_v2_forward=fwd,
                                                        bev_pool_v2_backward=None))
    with open(os.path.join(golden_dir, "kat_bev_pool_v2.json")) as f:
        k = json.load(f)
    depth = torch.tensor(k["depth"]).float().view(*k["depth_shape"])
    feat = torch.ones(size=k["feat_shape"])
    rd, rf, rb = (torch.tensor(k[n]).int() for n in ("ranks_depth", "ranks_feat", "ranks_bev"))
    bev = mod.bev_pool_v2(depth, feat, rd, rf, rb, tuple(k["bev_feat_shape"]),
                          torch.tensor([0, 2]).int(), torch.tensor([2, 2]).int())
    assert abs(float(bev.sum()) - k["loss"]) < 1e-6


def test_ext_stand_in_has_the_pybind_surface_and_refuses_cpu_tensors():
    """veon_b200.bev_pool_v2_ext mirrors bev_pool.cpp:106-111 (two functions, lengths before
    starts) and has no CPU path."""
    import inspect
    import torch
    from veon_b200 import bev_pool_v2_ext as ext
    assert list(inspect.signature(ext.bev_pool_v2_forward).parameters) == [
        "depth", "feat", "out", "ranks_depth", "ranks_feat", "ranks_bev", "interval_lengths",
        "interval_starts"]
    assert list(inspect.signature(ext.bev_pool_v2_backward).parameters) == [
        "out_grad", "depth_grad", "feat_grad", "depth", "feat", "ranks_depth", "ranks_feat",
        "ranks_bev", "interval_lengths", "interval_starts"]
    t = torch.zeros(1, 1, 1, 1, 1)
    i = torch.zeros(1, dtype=torch.int32)
    with pytest.raises(RuntimeError):
        ext.bev_pool_v2_forward(t, t, t, i, i, i, i, i)


def test_prepare_vocabulary_matches_the_reference_expression():
    """san_in_veon_temporal.py:261-266 over clip_utils/classifier.py:107-112: exp(logit_scale) x
    L2-normalised [text rows ; background row], detached; and the semkitti re-ordering is refused"""
    import torch
    import torch.nn.functional as F
    from veon_b200.tail import class_of_prompt, prepare_vocabulary
    g = torch.Generator().manual_seed(0)
    emb = torch.randn(66, 512, generator=g)
    bg = torch.randn(1, 512, generator=g) * 512 ** -0.5
    logit_scale = torch.tensor(4.6052, requires_grad=True)
    want = logit_scale.exp() * F.normalize(torch.cat([emb, bg], dim=0), p=2, dim=-1)
    got = prepare_vocabulary(emb, bg, logit_scale)
    assert got.shape == (67, 512) and not got.requires_grad
    assert torch.allclose(got, want.detach(), rtol=0, atol=1e-5)
    with pytest.raises(NotImplementedError):
        class_of_prompt([0, 0, 1], mode="semkitti")
    # loss-side grouping (no background row): occ3d_nuscenes.py:249-265
    assert class_of_prompt([0, 0, 1, 2, 2], background=False).tolist() == [0, 0, 1, 2, 2]
    assert class_of_prompt([0, 0, 1, 2, 2]).tolist() == [0, 0, 1, 2, 2, 3]


# ---- bench.py --dump-outputs ----------------------------------------------------------------------
def test_bench_dump_outputs_stores_a_fixed_sample_of_large_arrays(tmp_path):
    """Arrays up to DUMP_MAX_ELEMENTS are stored whole with their shape, larger ones at flat indices
    that depend on their size alone (seed 0), so two runs store the same positions; the three
    outputs of a step stay under 64 MB."""
    import bench
    cap = bench.DUMP_MAX_ELEMENTS
    assert 3 * cap * 4 <= 64 << 20
    n = cap + 1000                                  # < 2^24: float32 holds every index exactly
    big = torch.arange(n, dtype=torch.float32)      # element value == its flat index
    small = torch.randn(5, 4, dtype=torch.float64).t()          # non-contiguous, float64
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"bev": big.view(2, -1), "feat_grad": small})
    assert sorted(os.listdir(tmp_path / "a")) == ["bev_sample.npy", "feat_grad.npy"]
    a = np.load(tmp_path / "a" / "bev_sample.npy")
    want = np.unique(np.random.default_rng(0).integers(0, n, cap)).astype(np.float32)
    assert a.dtype == np.float32 and np.array_equal(a, want)
    assert np.array_equal(a, np.load(tmp_path / "b" / "bev_sample.npy"))
    f = np.load(tmp_path / "a" / "feat_grad.npy")
    assert f.dtype == np.float32 and f.shape == (4, 5)
    np.testing.assert_array_equal(f, small.float().numpy())


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_bench_refuses_arguments_it_cannot_honour(monkeypatch, argv):
    import bench
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.parse()
