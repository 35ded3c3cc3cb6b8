"""CPU: the bfloat16 entry points and options -- argument errors decided before any device work
(the same codes as their float32 twins), `dtype` validation, and the ABI version."""
import ctypes

import pytest
import torch

NULL = ctypes.c_void_p(0)


def _buf():
    return ctypes.cast((ctypes.c_float * 64)(), ctypes.c_void_p)


def test_abi_version_is_10():
    from veon_b200 import _lib
    assert _lib.load().veon_abi_version() == 10


@pytest.mark.parametrize("suffix", ["", "_bf16"])
def test_bf16_forward_entry_points_reject_bad_arguments(suffix):
    """the float32 twins ("") and the bfloat16 entry points give the same codes"""
    from veon_b200 import _lib
    lib = _lib.load()
    b = _buf()
    fwd = getattr(lib, "veon_bev_pool_v2_fwd_planar" + suffix)
    fwd_cl = getattr(lib, "veon_bev_pool_v2_fwd_planar_cl" + suffix)
    assert fwd(NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, 0, 1, 64, 640000, 4224, NULL,
               NULL, 0, NULL) == -1
    assert fwd_cl(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 0, 1, 64, 640000, 4224, NULL,
                  NULL) == -1
    for i in range(6):   # one NULL input at a time (tile_istart / tile_occ / heavy may be NULL)
        p = [b] * 6
        p[i] = NULL
        assert fwd(*p, NULL, NULL, b, 8, 1, 64, 640000, 4224, b, NULL, 0, NULL) == -1, i
        assert fwd_cl(*p, b, 8, 1, 64, 640000, 4224, b, NULL) == -1, i
    assert fwd(b, b, b, b, b, b, NULL, NULL, b, 8, 1, 64, 640000, 4224, NULL, NULL, 0, NULL) == -1
    assert fwd_cl(b, b, b, b, b, b, b, 8, 1, 64, 640000, 4224, NULL, NULL) == -1

    def both(B, C, V, rows, heavy_ints=8):
        a = fwd(b, b, b, b, b, b, NULL, NULL, b, heavy_ints, B, C, V, rows, b, NULL, 0, NULL)
        c = fwd_cl(b, b, b, b, b, b, b, heavy_ints, B, C, V, rows, b, NULL)
        assert a == c
        return a
    assert both(0, 64, 640000, 4224) == -1
    assert both(-1, 64, 640000, 4224) == -1
    assert both(1, 0, 640000, 4224) == -1
    assert both(1, 64, 0, 4224) == -1
    assert both(1, 64, 640000, 0) == -1
    assert both(1, 64, 640000, 4224, heavy_ints=1) == -1
    # size limits (32-bit feature row offsets, B < 65536, B*V < 2^31): checked before any launch
    # but after the one-time launch-configuration query, so without a device that query's CUDA
    # error comes back instead of VEON_E_RANGE -- the same one from both twins
    for args in [(1, 64, 640000, 1 << 24), (65536, 4, 32, 4224), (8, 64, 1 << 28, 4224)]:
        rc = both(*args)
        assert rc == -3 or rc > 0, (args, rc)


@pytest.mark.parametrize("suffix", ["", "_bf16"])
def test_bf16_backward_entry_points_reject_bad_arguments(suffix):
    from veon_b200 import _lib
    lib = _lib.load()
    b = _buf()
    bwd = getattr(lib, "veon_bev_pool_v2_bwd_planar" + suffix)
    bwd_cl = getattr(lib, "veon_bev_pool_v2_bwd_planar_cl" + suffix)
    # two passes: NULL pointers, sizes, a negative interval count, too small a rows scratch
    assert bwd(NULL, NULL, NULL, NULL, NULL, NULL, 10, 1, 6, 88, 16, 44, 64, 640000, NULL, 640,
               NULL, NULL, NULL) == -1
    for i in range(6):
        p = [b] * 6
        p[i] = NULL
        assert bwd(*p, 10, 1, 6, 88, 16, 44, 64, 640000, b, 640, b, b, NULL) == -1, i
    assert bwd(b, b, b, b, b, b, 10, 1, 6, 88, 16, 44, 64, 640000, NULL, 640, b, b, NULL) == -1
    assert bwd(b, b, b, b, b, b, 10, 1, 6, 88, 16, 44, 64, 640000, b, 640, NULL, b, NULL) == -1
    assert bwd(b, b, b, b, b, b, 10, 1, 6, 88, 16, 44, 64, 640000, b, 640, b, NULL, NULL) == -1
    for dims in [(0, 6, 88, 16, 44, 64, 640000), (1, 0, 88, 16, 44, 64, 640000),
                 (1, 6, 0, 16, 44, 64, 640000), (1, 6, 88, 0, 44, 64, 640000),
                 (1, 6, 88, 16, 0, 64, 640000), (1, 6, 88, 16, 44, 0, 640000),
                 (1, 6, 88, 16, 44, 64, 0)]:
        assert bwd(b, b, b, b, b, b, 10, *dims, b, 640, b, b, NULL) == -1, dims
    assert bwd(b, b, b, b, b, b, -1, 1, 6, 88, 16, 44, 64, 640000, b, 640, b, b, NULL) == -1
    assert bwd(b, b, b, b, b, b, 10, 1, 6, 88, 16, 44, 64, 640000, b, 639, b, b, NULL) == -2
    # single pass: NULL pointers, sizes, B*V >= 2^31
    assert bwd_cl(NULL, NULL, NULL, NULL, NULL, NULL, 1, 6, 88, 16, 44, 64, 640000, NULL, NULL,
                  NULL) == -1
    for i in range(6):
        p = [b] * 6
        p[i] = NULL
        assert bwd_cl(*p, 1, 6, 88, 16, 44, 64, 640000, b, b, NULL) == -1, i
    for dims in [(0, 6, 88, 16, 44, 64, 640000), (1, 0, 88, 16, 44, 64, 640000),
                 (1, 6, 0, 16, 44, 64, 640000), (1, 6, 88, 0, 44, 64, 640000),
                 (1, 6, 88, 16, 0, 64, 640000), (1, 6, 88, 16, 44, 0, 640000),
                 (1, 6, 88, 16, 44, 64, 0)]:
        assert bwd_cl(b, b, b, b, b, b, *dims, b, b, NULL) == -1, dims
    assert bwd_cl(b, b, b, b, b, b, 4096, 6, 88, 16, 44, 64, 640000, b, b, NULL) == -3


@pytest.mark.parametrize("dtype", [torch.float16, torch.float64, "bfloat16", None, torch.int32])
def test_dtype_is_validated_before_any_device_work(dtype):
    """Only torch.float32 and torch.bfloat16 are accepted; the check comes first, so CPU tensors
    (which the operators refuse) are never even looked at."""
    from veon_b200 import bev_pool as BP
    from veon_b200 import synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer
    t = torch.zeros(1)
    for fmt in (torch.contiguous_format, torch.channels_last_3d):
        with pytest.raises(ValueError, match="dtype"):
            BP.bev_pool_v2(t, t, t, t, t, (1, 1, 1, 1, 1), t, t, memory_format=fmt, dtype=dtype)
        with pytest.raises(ValueError, match="dtype"):
            BP.pool_prepared(t, t, None, (1, 1, 1, 1, 1), fmt, dtype=dtype)
    cfg = S.CONFIGS["tiny"]
    with pytest.raises(ValueError, match="dtype"):
        LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4, dtype=dtype)


def test_necks_take_the_dtype_option():
    import inspect
    from veon_b200 import synthetic as S
    from veon_b200.bev_pool import bev_pool_v2, pool_prepared
    from veon_b200.view_transformer import LSSViewTransformer, LSSViewTransformerRaw
    cfg = S.CONFIGS["tiny"]
    args = (cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4)
    assert LSSViewTransformer(*args).dtype is torch.float32
    for fmt in (torch.contiguous_format, torch.channels_last_3d):
        assert LSSViewTransformer(*args, memory_format=fmt, dtype=torch.bfloat16).dtype \
            is torch.bfloat16
    assert LSSViewTransformerRaw(*args, dtype=torch.float32).dtype is torch.float32
    with pytest.raises(ValueError, match="float32 only"):
        LSSViewTransformerRaw(*args, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="dtype"):
        LSSViewTransformerRaw(*args, dtype=torch.float16)
    for fn in (bev_pool_v2, pool_prepared):
        p = inspect.signature(fn).parameters["dtype"]
        assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is torch.float32
