"""CPU: the channels-last tail entry points are declared and exported, decide argument errors
before any device work with the codes of their channels-first twins, and the Python layer refuses
CPU channels-last tensors."""
import os

import pytest
import torch

from tests.test_tail_bf16_cpu import _codes

NAMES = ("veon_voxel_text_argmax", "veon_semantic_inference_3d", "veon_voxel_text_argmax_lowres")


def test_channels_last_tail_entries_are_declared_and_exported():
    from veon_b200 import _lib
    with open(os.path.join(os.path.dirname(_lib.__file__), "..", "include", "veon_lift.h")) as f:
        header = f.read()
    lib = _lib.load()
    for name in NAMES:
        for suffix in ("_cl", "_cl_bf16"):
            assert name + suffix + "(" in header and name + suffix in _lib.EXPORTED_SYMBOLS
            assert getattr(lib, name + suffix) is not None


@pytest.mark.parametrize("suffix,twin", [("_cl", ""), ("_cl_bf16", "_bf16")])
def test_channels_last_tail_entries_return_the_channels_first_codes(suffix, twin):
    assert _codes(suffix) == _codes(twin)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_cpu_channels_last_tensors_are_refused(dtype):
    from veon_b200.tail import semantic_inference_3d, voxel_text_argmax, voxel_text_argmax_lowres
    feat = torch.zeros(1, 32, 2, 2, 8, dtype=dtype).contiguous(memory_format=torch.channels_last_3d)
    assert not feat.is_contiguous()
    w = torch.zeros(4, 32)
    cls = torch.arange(4, dtype=torch.int32)
    gate = torch.zeros(1, 2, 2, 2, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        voxel_text_argmax(feat, w, cls, gate)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        semantic_inference_3d(w, feat)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        voxel_text_argmax_lowres(feat, w, cls, gate, occ_size=(4, 4, 16))
