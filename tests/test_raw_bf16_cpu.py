"""CPU: the bfloat16 2x2x2 maximum and the bfloat16 `_ds` backward in the C ABI (declared, bound,
the argument errors of their float32 twins, decided before any device work), and the `ds_dtype`
option of LSSViewTransformerRaw."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NULL = ctypes.c_void_p(0)
# bfloat16 entry -> its float32 twin
TWINS = {
    "veon_maxdown2_fwd_bf16": "veon_maxdown2_fwd",
    "veon_maxdown2_fwd_mask_bf16": "veon_maxdown2_fwd_mask",
    "veon_maxdown2_bwd_bf16": "veon_maxdown2_bwd",
    "veon_maxdown2_cl_fwd_bf16": "veon_maxdown2_cl_fwd",
    "veon_maxdown2_cl_bwd_bf16": "veon_maxdown2_cl_bwd",
    "veon_bev_pool_v2_bwd_planar_ds_bf16": "veon_bev_pool_v2_bwd_planar_ds",
    "veon_bev_pool_v2_bwd_planar_ds_bf16_bf16feat": "veon_bev_pool_v2_bwd_planar_ds_bf16feat",
}


def _buf(offset=0):
    """a 256-byte aligned host buffer (never dereferenced: every call here fails its checks)"""
    return ctypes.c_void_p(0x10000 + offset)


def test_new_entries_are_declared_bound_and_take_the_twins_arguments():
    from veon_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "veon_lift.h")).read()
    declared = set(re.findall(r"\b(veon_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", header,
                                                                   flags=re.S)))
    for name, twin in TWINS.items():
        assert name in declared and name in _lib.EXPORTED_SYMBOLS and hasattr(lib, name), name
        assert _lib._SIGNATURES[name] == _lib._SIGNATURES[twin], name
    assert re.search(r"#define\s+VEON_ABI_VERSION\s+11\b", header)
    assert lib.veon_abi_version() == 11


@pytest.mark.parametrize("suffix", ["", "_bf16"])
def test_channels_first_maximum_rejects_bad_arguments(suffix):
    """NULL pointers, non-positive sizes, odd Z / Y, X % 4 != 0: the twins' codes"""
    from veon_b200 import _lib
    lib = _lib.load()
    p = _buf()
    fwd = getattr(lib, "veon_maxdown2_fwd" + suffix)
    mask = getattr(lib, "veon_maxdown2_fwd_mask" + suffix)
    bwd = getattr(lib, "veon_maxdown2_bwd" + suffix)
    for dims, rc in [((4, 16, 200, 200), None), ((0, 16, 200, 200), -1), ((4, -2, 200, 200), -1),
                     ((4, 15, 200, 200), -4), ((4, 16, 199, 200), -4), ((4, 16, 200, 202), -4),
                     ((4, 16, 200, 6), -4)]:
        if rc is None:          # valid sizes: the NULL pointers decide
            rc = -1
            assert fwd(NULL, *dims, p, NULL) == rc and fwd(p, *dims, NULL, NULL) == rc
            assert mask(p, *dims, p, NULL, NULL) == rc and mask(NULL, *dims, p, p, NULL) == rc
            assert bwd(p, p, NULL, *dims, p, NULL) == rc and bwd(p, p, p, *dims, NULL, NULL) == rc
            assert bwd(NULL, p, p, *dims, p, NULL) == rc
            continue
        assert fwd(p, *dims, p, NULL) == rc, dims
        assert mask(p, *dims, p, p, NULL) == rc, dims
        assert bwd(p, p, p, *dims, p, NULL) == rc, dims


def test_channels_first_bf16_alignment():
    """bfloat16: the volume 8-byte aligned, the reduced volume 4-byte aligned, else UNSUPPORTED
    (the float32 volume of the mask entry 16-byte aligned, as its twin; its mask 2-byte)"""
    from veon_b200 import _lib
    lib = _lib.load()
    p, dims = _buf(), (4, 16, 200, 200)
    for off in (2, 4, 6):
        assert lib.veon_maxdown2_fwd_bf16(_buf(off), *dims, p, NULL) == -4, off
        assert lib.veon_maxdown2_bwd_bf16(_buf(off), p, p, *dims, p, NULL) == -4, off
        assert lib.veon_maxdown2_bwd_bf16(p, p, p, *dims, _buf(off), NULL) == -4, off
        assert lib.veon_maxdown2_fwd_mask_bf16(_buf(off), *dims, p, p, NULL) == -4, off
    for off in (2, 6):
        assert lib.veon_maxdown2_fwd_bf16(p, *dims, _buf(off), NULL) == -4, off
        assert lib.veon_maxdown2_bwd_bf16(p, _buf(off), p, *dims, p, NULL) == -4, off
        assert lib.veon_maxdown2_bwd_bf16(p, p, _buf(off), *dims, p, NULL) == -4, off
        assert lib.veon_maxdown2_fwd_mask_bf16(p, *dims, _buf(off), p, NULL) == -4, off
    assert lib.veon_maxdown2_fwd_mask_bf16(_buf(8), *dims, p, p, NULL) == -4
    assert lib.veon_maxdown2_fwd_mask_bf16(p, *dims, p, _buf(1), NULL) == -4


@pytest.mark.parametrize("suffix", ["", "_bf16"])
def test_channels_last_maximum_rejects_bad_arguments(suffix):
    """NULL pointers, non-positive sizes, odd Z / Y / X, and 2^32 output voxels or more"""
    from veon_b200 import _lib
    lib = _lib.load()
    p = _buf()
    fwd = getattr(lib, "veon_maxdown2_cl_fwd" + suffix)
    bwd = getattr(lib, "veon_maxdown2_cl_bwd" + suffix)
    dims = (4, 256, 16, 200, 200)
    assert fwd(NULL, *dims, p, NULL) == -1 and fwd(p, *dims, NULL, NULL) == -1
    for i in range(4):
        ptrs = [p] * 4
        ptrs[i] = NULL
        assert bwd(*ptrs[:3], *dims, ptrs[3], NULL) == -1, i
    for bad, rc in [((0, 256, 16, 200, 200), -1), ((4, 0, 16, 200, 200), -1),
                    ((4, 256, 15, 200, 200), -4), ((4, 256, 16, 201, 200), -4),
                    ((4, 256, 16, 200, 199), -4),
                    ((1 << 16, 1, 256, 256, 256), -3),      # 2^32 output voxels
                    ((4096, 1, 2048, 2048, 4), -3)]:
        assert fwd(p, *bad, p, NULL) == rc, bad
        assert bwd(p, p, p, *bad, p, NULL) == rc, bad


@pytest.mark.parametrize("name", ["veon_bev_pool_v2_bwd_planar_ds",
                                  "veon_bev_pool_v2_bwd_planar_ds_bf16feat",
                                  "veon_bev_pool_v2_bwd_planar_ds_bf16",
                                  "veon_bev_pool_v2_bwd_planar_ds_bf16_bf16feat"])
def test_ds_backward_rejects_bad_arguments(name):
    from veon_b200 import _lib
    f = getattr(_lib.load(), name)
    p = _buf()
    grid = (16, 200, 200)
    assert f(NULL, p, p, p, p, p, p, 10, 1, 6, 8, 16, 44, 64, *grid, p, p, p, NULL) == -1
    for i in range(7):
        ptrs = [p] * 7
        ptrs[i] = NULL
        assert f(*ptrs, 10, 1, 6, 8, 16, 44, 64, *grid, p, p, p, NULL) == -1, i
    assert f(p, p, p, p, p, p, p, -1, 1, 6, 8, 16, 44, 64, *grid, p, p, p, NULL) == -1
    assert f(p, p, p, p, p, p, p, 10, 1, 6, 8, 16, 44, 0, *grid, p, p, p, NULL) == -1
    for bad in [(15, 200, 200), (16, 199, 200), (16, 200, 201)]:
        assert f(p, p, p, p, p, p, p, 10, 1, 6, 8, 16, 44, 64, *bad, p, p, p, NULL) == -4, bad
    # B * Z * Y * X >= 2^31
    assert f(p, p, p, p, p, p, p, 10, 64, 6, 8, 16, 44, 64, 64, 1024, 1024, p, p, p, NULL) == -3


def _raw_args():
    from veon_b200 import synthetic as S
    cfg = S.CONFIGS["tiny"]
    return (cfg.grid_config, cfg.input_size, cfg.downsample, 8, 4)


@pytest.mark.parametrize("ds_dtype", [torch.float16, torch.float64, "bfloat16", None, torch.int32])
def test_ds_dtype_is_validated_before_any_device_work(ds_dtype):
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformerRaw
    with pytest.raises(ValueError, match="ds_dtype"):
        LSSViewTransformerRaw(*_raw_args(), ds_dtype=ds_dtype)
    with pytest.raises(ValueError, match="dtype"):
        BP.pool_prepared_maxdown(torch.zeros(1), torch.zeros(1), None, (1, 2, 2, 4, 4),
                                 dtype=ds_dtype)


def test_ds_dtype_default_and_use_ds():
    import inspect
    from veon_b200 import bev_pool as BP
    from veon_b200.view_transformer import LSSViewTransformerRaw
    assert LSSViewTransformerRaw(*_raw_args()).ds_dtype is torch.float32
    assert LSSViewTransformerRaw(*_raw_args(), use_ds=False).ds_dtype is torch.float32
    neck = LSSViewTransformerRaw(*_raw_args(), ds_dtype=torch.bfloat16,
                                 memory_format=torch.channels_last_3d)
    assert neck.ds_dtype is torch.bfloat16 and neck.dtype is torch.float32
    with pytest.raises(ValueError, match="use_ds"):
        LSSViewTransformerRaw(*_raw_args(), use_ds=False, ds_dtype=torch.bfloat16)
    # the pooled volume's dtype stays float32 only, whatever ds_dtype says
    with pytest.raises(ValueError, match="float32 only"):
        LSSViewTransformerRaw(*_raw_args(), dtype=torch.bfloat16, ds_dtype=torch.bfloat16)
    p = inspect.signature(BP.pool_prepared_maxdown).parameters["dtype"]
    assert p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is torch.float32
