"""CPU: the C ABI of the bfloat16-feature pooling entry points (declared, bound, argument checks
decided before any device work) and the refusal of CPU tensors with bfloat16 features."""
import ctypes
import re
import os

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FWD = ("veon_bev_pool_v2_fwd_planar_bf16feat", "veon_bev_pool_v2_fwd_planar_bf16_bf16feat")
FWD_CL = ("veon_bev_pool_v2_fwd_planar_cl_bf16feat", "veon_bev_pool_v2_fwd_planar_cl_bf16_bf16feat")
BWD = ("veon_bev_pool_v2_bwd_planar_bf16feat", "veon_bev_pool_v2_bwd_planar_bf16_bf16feat")
BWD_CL = ("veon_bev_pool_v2_bwd_planar_cl_bf16feat", "veon_bev_pool_v2_bwd_planar_cl_bf16_bf16feat")
BWD_DS = "veon_bev_pool_v2_bwd_planar_ds_bf16feat"
NEW = FWD + FWD_CL + BWD + BWD_CL + (BWD_DS, "veon_transpose_batched_u16")


def test_every_new_entry_is_declared_and_bound():
    from veon_b200 import _lib
    lib = _lib.load()
    text = open(os.path.join(ROOT, "include", "veon_lift.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    declared = set(re.findall(r"\b(veon_[a-z0-9_]+)\s*\(", text))
    for name in NEW:
        assert name in declared and name in _lib.EXPORTED_SYMBOLS and hasattr(lib, name), name
        # the same arguments as the twin without `_bf16feat`
        twin = name.replace("_bf16feat", "").replace("_u16", "")
        assert _lib._SIGNATURES[name] == _lib._SIGNATURES[twin], name
    assert re.search(r"#define\s+VEON_ABI_VERSION\s+11\b", open(os.path.join(
        ROOT, "include", "veon_lift.h")).read())


def _buf():
    return ctypes.cast((ctypes.c_float * 64)(), ctypes.c_void_p)


def test_null_and_non_positive_arguments_are_refused():
    from veon_b200 import _lib
    lib = _lib.load()
    null, p = ctypes.c_void_p(0), _buf()
    for name in FWD:
        f = getattr(lib, name)
        assert f(null, null, null, null, null, null, null, null, null, 0, 1, 64, 640000, 4224,
                 null, null, 0, null) == -1
        assert f(p, p, p, p, p, p, p, p, p, 8, 0, 64, 640000, 4224, p, null, 0, null) == -1   # B
        assert f(p, p, p, p, p, p, p, p, p, 8, 1, 0, 640000, 4224, p, null, 0, null) == -1    # C
        assert f(p, p, p, p, p, p, p, p, p, 8, 1, 64, 0, 4224, p, null, 0, null) == -1        # V
        assert f(p, p, p, p, p, p, p, p, p, 8, 1, 64, 640000, 0, p, null, 0, null) == -1      # rows
        assert f(p, p, p, p, p, p, p, p, p, 1, 1, 64, 640000, 4224, p, null, 0, null) == -1   # heavy
    for name in FWD_CL:
        f = getattr(lib, name)
        assert f(null, null, null, null, null, null, null, 0, 1, 64, 640000, 4224, null, null) == -1
        assert f(p, p, p, p, p, p, p, 8, 1, -4, 640000, 4224, p, null) == -1
        assert f(p, p, p, p, p, p, p, 8, 1, 64, 640000, -1, p, null) == -1
    for name in BWD:
        f = getattr(lib, name)
        assert f(null, null, null, null, null, null, 0, 1, 1, 2, 2, 2, 64, 640000, null, 0, null,
                 null, null) == -1
        assert f(p, p, p, p, p, p, 0, 1, 0, 2, 2, 2, 64, 640000, p, 0, p, p, null) == -1       # N
        assert f(p, p, p, p, p, p, -1, 1, 1, 2, 2, 2, 64, 640000, p, 0, p, p, null) == -1      # n_int
        assert f(p, p, p, p, p, p, 10, 1, 1, 2, 2, 2, 64, 640000, p, 639, p, p, null) == -2    # rows_ws
    for name in BWD_CL:
        f = getattr(lib, name)
        assert f(null, null, null, null, null, null, 1, 1, 2, 2, 2, 64, 640000, null, null,
                 null) == -1
        assert f(p, p, p, p, p, p, 1, 1, 2, 2, 2, 64, 0, p, p, null) == -1
    f = getattr(lib, BWD_DS)
    assert f(null, null, null, null, null, null, null, 0, 1, 1, 2, 2, 2, 64, 16, 200, 200, null,
             null, null, null) == -1
    assert f(p, p, p, p, p, p, p, 0, 1, 1, 2, 2, 2, 64, 15, 200, 200, p, p, p, null) == -4    # odd Z


def test_u16_transpose_checks_match_the_float_one():
    from veon_b200 import _lib
    lib = _lib.load()
    null, p = ctypes.c_void_p(0), _buf()
    for args in ((null, 1, 4, 4, null), (p, 0, 4, 4, p), (p, 1, 0, 4, p), (p, 1, 4, -1, p),
                 (p, 1, 4, 4, null), (p, 65536, 4, 4, p)):
        want = lib.veon_transpose_batched(*args, null)
        assert want in (-1, -3)
        assert lib.veon_transpose_batched_u16(*args, null) == want


def test_cpu_tensors_with_bf16_features_are_refused():
    from veon_b200.bev_pool import bev_pool_v2
    d = torch.zeros(1, 1, 2, 2, 2)
    f = torch.zeros(1, 1, 2, 2, 8, dtype=torch.bfloat16)
    i = torch.zeros(2, dtype=torch.int32)
    for kw in ({}, {"dtype": torch.bfloat16}, {"memory_format": torch.channels_last_3d}):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            bev_pool_v2(d, f, i, i, i, (1, 1, 2, 2, 8), i, i, **kw)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            bev_pool_v2(d, f.permute(0, 1, 4, 2, 3).contiguous().permute(0, 1, 3, 4, 2), i, i, i,
                        (1, 1, 2, 2, 8), i, i, **kw)
