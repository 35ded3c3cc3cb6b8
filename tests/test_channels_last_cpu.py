"""CPU: the channels-last entry points and options -- argument errors decided before any device
work, `memory_format` validation, and the reference's call sites still binding."""
import ctypes
import inspect

import pytest
import torch

NULL = ctypes.c_void_p(0)


def _buf():
    return ctypes.cast((ctypes.c_float * 64)(), ctypes.c_void_p)


def test_channels_last_entry_points_reject_bad_arguments():
    from veon_b200 import _lib
    lib = _lib.load()
    b = _buf()
    # forward: NULL pointers, non-positive sizes, a heavy list too short to hold its header
    assert lib.veon_bev_pool_v2_fwd_planar_cl(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 0,
                                              1, 64, 640000, 4224, NULL, NULL) == -1
    fwd = lambda B, C, V, rows, heavy_ints=8: lib.veon_bev_pool_v2_fwd_planar_cl(
        b, b, b, b, b, b, b, heavy_ints, B, C, V, rows, b, NULL)
    assert fwd(0, 64, 640000, 4224) == -1
    assert fwd(1, 0, 640000, 4224) == -1
    assert fwd(1, 64, 0, 4224) == -1
    assert fwd(1, 64, 640000, 0) == -1
    assert fwd(1, 64, 640000, 4224, heavy_ints=1) == -1
    # single-pass backward: NULL pointers (no workspace argument at all), sizes, B*V >= 2^31
    assert lib.veon_bev_pool_v2_bwd_planar_cl(NULL, NULL, NULL, NULL, NULL, NULL, 1, 6, 88, 16, 44,
                                              64, 640000, NULL, NULL, NULL) == -1
    bwd = lambda B, N, D, H, W, C, V: lib.veon_bev_pool_v2_bwd_planar_cl(
        b, b, b, b, b, b, B, N, D, H, W, C, V, b, b, NULL)
    for args in [(0, 6, 88, 16, 44, 64, 640000), (1, 0, 88, 16, 44, 64, 640000),
                 (1, 6, 0, 16, 44, 64, 640000), (1, 6, 88, 0, 44, 64, 640000),
                 (1, 6, 88, 16, 0, 64, 640000), (1, 6, 88, 16, 44, 0, 640000),
                 (1, 6, 88, 16, 44, 64, 0)]:
        assert bwd(*args) == -1, args
    assert bwd(4096, 6, 88, 16, 44, 64, 640000) == -3
    # channels-last 2x2x2 max: NULL, non-positive sizes, odd grids, too many output voxels
    assert lib.veon_maxdown2_cl_fwd(NULL, 1, 64, 16, 200, 200, NULL, NULL) == -1
    assert lib.veon_maxdown2_cl_bwd(NULL, NULL, NULL, 1, 64, 16, 200, 200, NULL, NULL) == -1
    assert lib.veon_maxdown2_cl_bwd(b, b, NULL, 1, 64, 16, 200, 200, b, NULL) == -1
    assert lib.veon_maxdown2_cl_bwd(b, b, b, 1, 64, 16, 200, 200, NULL, NULL) == -1
    for B, C, Z, Y, X in [(0, 64, 16, 200, 200), (1, 0, 16, 200, 200), (1, 64, 0, 200, 200),
                          (1, 64, 16, -2, 200), (1, 64, 16, 200, 0)]:
        assert lib.veon_maxdown2_cl_fwd(b, B, C, Z, Y, X, b, NULL) == -1
        assert lib.veon_maxdown2_cl_bwd(b, b, b, B, C, Z, Y, X, b, NULL) == -1
    for Z, Y, X in [(15, 200, 200), (16, 199, 200), (16, 200, 201)]:
        assert lib.veon_maxdown2_cl_fwd(b, 1, 64, Z, Y, X, b, NULL) == -4
        assert lib.veon_maxdown2_cl_bwd(b, b, b, 1, 64, Z, Y, X, b, NULL) == -4
    assert lib.veon_maxdown2_cl_fwd(b, 1 << 20, 1, 64, 128, 128, b, NULL) == -3   # 2^32 outputs


@pytest.mark.parametrize("fmt", [torch.channels_last, torch.preserve_format, "channels_last_3d",
                                 None])
def test_memory_format_is_validated_before_any_device_work(fmt):
    """Only torch.contiguous_format and torch.channels_last_3d are accepted; the check comes
    first, so CPU tensors (which the operators refuse) are never even looked at."""
    from veon_b200 import bev_pool as BP
    from veon_b200 import synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer, LSSViewTransformerRaw
    t = torch.zeros(1)
    with pytest.raises(ValueError, match="memory_format"):
        BP.bev_pool_v2(t, t, t, t, t, (1, 1, 1, 1, 1), t, t, memory_format=fmt)
    with pytest.raises(ValueError, match="memory_format"):
        BP.pool_prepared(t, t, None, (1, 1, 1, 1, 1), memory_format=fmt)
    cfg = S.CONFIGS["tiny"]
    for cls in (LSSViewTransformer, LSSViewTransformerRaw):
        with pytest.raises(ValueError, match="memory_format"):
            cls(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4, memory_format=fmt)


def test_necks_accept_both_memory_formats():
    from veon_b200 import synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer, LSSViewTransformerRaw
    cfg = S.CONFIGS["tiny"]
    for cls in (LSSViewTransformer, LSSViewTransformerRaw):
        assert cls(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4).memory_format \
            is torch.contiguous_format
        neck = cls(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4,
                   memory_format=torch.channels_last_3d)
        assert neck.memory_format is torch.channels_last_3d


def test_reference_call_sites_still_bind():
    """bev_pool.py:86-92 is called with eight positional arguments, and QuickCumsumCuda.apply
    likewise; memory_format is keyword-only and defaults to the reference's layout."""
    from veon_b200.bev_pool import QuickCumsumCuda, bev_pool_v2, pool_prepared
    args = ("depth", "feat", "ranks_depth", "ranks_feat", "ranks_bev", "bev_feat_shape",
            "interval_starts", "interval_lengths")
    sig = inspect.signature(bev_pool_v2)
    bound = sig.bind(*args)
    bound.apply_defaults()
    assert bound.arguments["memory_format"] is torch.contiguous_format
    assert sig.parameters["memory_format"].kind is inspect.Parameter.KEYWORD_ONLY
    with pytest.raises(TypeError):
        sig.bind(*args, torch.channels_last_3d)           # not a ninth positional argument
    inspect.signature(QuickCumsumCuda.forward).bind("ctx", *args)
    assert inspect.signature(pool_prepared).parameters["memory_format"].default \
        is torch.contiguous_format
