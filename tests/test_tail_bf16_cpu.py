"""CPU: the bfloat16 tail entry points decide argument errors before any device work, with the
same codes as their float32 twins, and the Python layer refuses CPU bfloat16 tensors."""
import ctypes

import pytest
import torch

NULL = ctypes.c_void_p(0)


def _buf():
    return ctypes.cast((ctypes.c_float * 64)(), ctypes.c_void_p)


def _entries(suffix):
    from veon_b200 import _lib
    lib = _lib.load()
    return (getattr(lib, "veon_voxel_text_argmax" + suffix),
            getattr(lib, "veon_semantic_inference_3d" + suffix),
            getattr(lib, "veon_voxel_text_argmax_lowres" + suffix))


def _codes(suffix):
    """every argument error of the three entries, in a fixed order"""
    argmax, sem3d, lowres = _entries(suffix)
    b = _buf()
    dims = (1, 64, 18, 16, 200, 200)
    bad_dims = [(0, 64, 18, 16, 200, 200), (1, 0, 18, 16, 200, 200), (1, 64, 0, 16, 200, 200),
                (1, 64, 18, 0, 200, 200), (1, 64, 18, 16, 0, 200), (1, 64, 18, 16, 200, 0),
                (-1, 64, 18, 16, 200, 200), (65536, 64, 18, 16, 200, 200)]
    codes = []
    for i in range(5):                     # feat, text_w, class_of_prompt, bin_occ, labels
        p = [b] * 5
        p[i] = NULL
        codes.append(argmax(p[0], p[1], p[2], p[3], *dims, 17, p[4], NULL, NULL))
    for d in bad_dims:
        codes.append(argmax(b, b, b, b, *d, 17, b, NULL, NULL))
    for i in range(3):                     # text_w, feat, sem_occ
        p = [b] * 3
        p[i] = NULL
        codes.append(sem3d(p[0], p[1], *dims, p[2], NULL, NULL))
    for d in bad_dims:
        codes.append(sem3d(b, b, *d, b, NULL, NULL))
    lr = (8, 100, 100, 16, 200, 200)
    need = 4 * 1 * 18 * 8 * 100 * 100
    codes.append(lowres(b, b, b, b, 1, 64, 18, *lr, 17, b, NULL, need, NULL, NULL))   # no workspace
    codes.append(lowres(b, b, b, b, 1, 64, 18, *lr, 17, b, b, need - 4, NULL, NULL))  # short one
    codes.append(lowres(b, b, b, b, 1, 64, 18, *lr, 17, b, b, 0, NULL, NULL))
    codes.append(lowres(NULL, b, b, b, 1, 64, 18, *lr, 17, b, b, need, NULL, NULL))
    codes.append(lowres(b, NULL, b, b, 1, 64, 18, *lr, 17, b, b, need, NULL, NULL))
    codes.append(lowres(b, b, b, b, 65536, 64, 18, *lr, 17, b, b, 1 << 62, NULL, NULL))
    codes.append(lowres(b, b, b, b, 1, 64, 0, *lr, 17, b, b, need, NULL, NULL))
    return codes


def test_bf16_tail_entries_return_the_float32_codes():
    f32, bf16 = _codes(""), _codes("_bf16")
    assert bf16 == f32
    assert all(c == -1 for c in f32[:24]), f32
    assert f32[24:27] == [-1, -2, -2] and all(c == -1 for c in f32[27:]), f32


def test_bf16_tail_entries_are_declared():
    import os
    from veon_b200 import _lib
    with open(os.path.join(os.path.dirname(_lib.__file__), "..", "include", "veon_lift.h")) as f:
        header = f.read()
    for name in ("veon_voxel_text_argmax_bf16", "veon_semantic_inference_3d_bf16",
                 "veon_voxel_text_argmax_lowres_bf16"):
        assert name + "(" in header and name in _lib.EXPORTED_SYMBOLS


def test_cpu_bfloat16_tensors_are_refused():
    from veon_b200.tail import semantic_inference_3d, voxel_text_argmax, voxel_text_argmax_lowres
    feat = torch.zeros(1, 32, 2, 2, 8, dtype=torch.bfloat16)
    w = torch.zeros(4, 32)
    cls = torch.arange(4, dtype=torch.int32)
    gate = torch.zeros(1, 2, 2, 2, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        voxel_text_argmax(feat, w, cls, gate)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        semantic_inference_3d(w, feat)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        voxel_text_argmax_lowres(feat, w, cls, gate, occ_size=(4, 4, 16))
