"""ctypes binding of libveonlift.so (the C ABI declared in include/veon_lift.h).

There is no CPU or PyTorch fallback: if the shared library is missing the
import of any operator fails loudly (`VeonLibraryError`).
"""
import ctypes
import os
from ctypes import c_char_p, c_int, c_int32, c_int64, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libveonlift.so")


class VeonLibraryError(RuntimeError):
    pass


class VeonError(RuntimeError):
    def __init__(self, code, what):
        self.code = code
        super().__init__(f"{what} failed: [{code}] {error_string(code)}")


_P = c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "veon_abi_version": (c_int, []),
    "veon_reserve_sms": (c_int, [c_int]),
    "veon_error_string": (c_char_p, [c_int]),
    "veon_kernel_launch_count": (ctypes.c_uint64, []),
    "veon_bev_pool_v2": (c_int, [c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "veon_bev_pool_v2_grad": (c_int, [c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "veon_bev_pool_v2_generic": (c_int, [c_int, c_int, c_int, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "veon_bev_pool_v2_grad_generic": (c_int, [c_int, c_int64, c_int, c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "veon_lidar_coor_workspace_bytes": (c_size_t, [c_int, c_int]),
    "veon_lidar_coor": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P,
                                c_size_t, _P]),
    "veon_transpose_batched": (c_int, [_P, c_int64, c_int, c_int, _P, _P]),
    "veon_prepare_v2_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, _P]),
    "veon_pool_num_tiles": (c_int64, [c_int, c_int64]),
    "veon_two_hot_depth": (c_int, [_P, c_int64, c_int, c_int, c_int, c_int, ctypes.c_float,
                                   ctypes.c_float, ctypes.c_float, _P, _P]),
    "veon_maxdown2_fwd": (c_int, [_P, c_int64, c_int, c_int, c_int, _P, _P]),
    "veon_maxdown2_fwd_mask": (c_int, [_P, c_int64, c_int, c_int, c_int, _P, _P, _P]),
    "veon_bev_pool_v2_bwd_planar_ds": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64,
                                               c_int, c_int, c_int, c_int, c_int, c_int,
                                               c_int, c_int, c_int, _P, _P, _P, _P]),
    "veon_maxdown2_bwd": (c_int, [_P, _P, _P, c_int64, c_int, c_int, c_int, _P, _P]),
    "veon_maxdown2_cl_fwd": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "veon_maxdown2_cl_bwd": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "veon_prepare_v2_voxel_start_offset": (c_size_t, [c_int, c_int, c_int, c_int, c_int, _P]),
    "veon_bev_pool_v2_ds_fwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                        c_int64, _P, _P]),
    "veon_pool_heavy_list_ints": (c_int64, [c_int64, c_int64]),
    "veon_prepare_v2": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P,
                                _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "veon_prepare_v2_calib": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                      _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                      _P, c_size_t, _P, c_size_t, _P]),
    "veon_prepare_v2_calib_sparse": (c_int, [_P, _P, _P, _P, _P, _P, _P, ctypes.c_float,
                                             c_int, c_int, c_int, c_int, c_int,
                                             _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                             _P, c_size_t, _P, c_size_t, _P]),
    "veon_calib_hash": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P, _P]),
    "veon_pool_plan_build": (c_int, [_P, _P, _P, _P, _P, c_int64, c_int64,
                                     c_int, c_int, c_int, c_int, c_int, c_int64,
                                     _P, _P, _P, _P, _P, _P, _P]),
    "veon_bev_pool_v2_fwd_workspace_bytes": (c_size_t, [c_int, c_int, c_int64]),
    "veon_bev_pool_v2_fwd_planar": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64,
                                            c_int, c_int, c_int64, c_int64, _P, _P, c_size_t, _P]),
    "veon_bev_pool_v2_fwd_planar_cl": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64,
                                               c_int, c_int, c_int64, c_int64, _P, _P]),
    "veon_bev_pool_v2_bwd_planar_cl": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int,
                                               c_int, c_int, c_int64, _P, _P, _P]),
    "veon_bev_pool_v2_fwd_planar_bf16": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64,
                                                 c_int, c_int, c_int64, c_int64, _P, _P, c_size_t,
                                                 _P]),
    "veon_bev_pool_v2_fwd_planar_cl_bf16": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64,
                                                    c_int, c_int, c_int64, c_int64, _P, _P]),
    "veon_bev_pool_v2_bwd_planar_bf16": (c_int, [_P, _P, _P, _P, _P, _P, c_int64,
                                                 c_int, c_int, c_int, c_int, c_int, c_int, c_int64,
                                                 _P, c_int64, _P, _P, _P]),
    "veon_bev_pool_v2_bwd_planar_cl_bf16": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int,
                                                    c_int, c_int, c_int, c_int64, _P, _P, _P]),
    "veon_bev_pool_v2_fwd_planar_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64,
                                                     c_int, c_int, c_int64, c_int64, _P, _P,
                                                     c_size_t, _P]),
    "veon_bev_pool_v2_fwd_planar_bf16_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P,
                                                          c_int64, c_int, c_int, c_int64, c_int64,
                                                          _P, _P, c_size_t, _P]),
    "veon_bev_pool_v2_fwd_planar_cl_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64,
                                                        c_int, c_int, c_int64, c_int64, _P, _P]),
    "veon_bev_pool_v2_fwd_planar_cl_bf16_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64,
                                                             c_int, c_int, c_int64, c_int64, _P,
                                                             _P]),
    "veon_bev_pool_v2_bwd_planar_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, c_int64,
                                                     c_int, c_int, c_int, c_int, c_int, c_int,
                                                     c_int64, _P, c_int64, _P, _P, _P]),
    "veon_bev_pool_v2_bwd_planar_bf16_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, c_int64,
                                                          c_int, c_int, c_int, c_int, c_int, c_int,
                                                          c_int64, _P, c_int64, _P, _P, _P]),
    "veon_bev_pool_v2_bwd_planar_cl_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int,
                                                        c_int, c_int, c_int, c_int, c_int64, _P,
                                                        _P, _P]),
    "veon_bev_pool_v2_bwd_planar_cl_bf16_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int,
                                                             c_int, c_int, c_int, c_int, c_int64,
                                                             _P, _P, _P]),
    "veon_bev_pool_v2_bwd_planar_ds_bf16feat": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64,
                                                        c_int, c_int, c_int, c_int, c_int, c_int,
                                                        c_int, c_int, c_int, _P, _P, _P, _P]),
    "veon_transpose_batched_u16": (c_int, [_P, c_int64, c_int, c_int, _P, _P]),
    "veon_bev_pool_v2_bwd_workspace_floats": (c_size_t, [c_int64, c_int, c_int, c_int, c_int, c_int,
                                                         c_int, c_int64]),
    "veon_bev_pool_v2_bwd_planar": (c_int, [_P, _P, _P, _P, _P, _P, c_int64,
                                            c_int, c_int, c_int, c_int, c_int, c_int, c_int64,
                                            _P, c_int64, _P, _P, _P]),
    "veon_voxel_text_argmax": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_int, _P, _P, _P]),
    "veon_text_classifier_image_bytes": (c_size_t, [c_int, c_int]),
    "veon_text_classifier_image": (c_int, [_P, c_int, c_int, _P, c_size_t, _P]),
    "veon_semantic_inference_3d": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P,
                                           _P]),
    "veon_point_text_argmax": (c_int, [_P, _P, c_int, c_int64, c_int64, _P, _P, _P]),
    "veon_upsample_classify": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_int, c_int, _P, _P]),
    "veon_classify_logits": (c_int, [_P, c_int64, _P, c_int64, _P, c_int, c_int, c_int, c_int, c_int,
                                     c_int, _P, _P]),
    "veon_lift_classify_fwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, c_int, c_int, c_int, c_int,
                                       c_int, c_int, c_int64, _P, c_int, _P, _P]),
    "veon_voxel_text_argmax_lowres_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "veon_voxel_text_argmax_lowres": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                              c_int, c_int, c_int, c_int, c_int, _P, _P, c_size_t,
                                              _P, _P]),
    "veon_voxel_text_argmax_bf16": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                            c_int, _P, _P, _P]),
    "veon_semantic_inference_3d_bf16": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P,
                                                _P, _P]),
    "veon_voxel_text_argmax_lowres_bf16": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                                   c_int, c_int, c_int, c_int, c_int, _P, _P, c_size_t,
                                                   _P, _P]),
    "veon_voxel_text_argmax_cl": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                          c_int, _P, _P, _P]),
    "veon_voxel_text_argmax_cl_bf16": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                               c_int, c_int, _P, _P, _P]),
    "veon_semantic_inference_3d_cl": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P,
                                              _P, _P]),
    "veon_semantic_inference_3d_cl_bf16": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                                                   _P, _P, _P]),
    "veon_voxel_text_argmax_lowres_cl": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                                 c_int, c_int, c_int, c_int, c_int, _P, _P, c_size_t,
                                                 _P, _P]),
    "veon_voxel_text_argmax_lowres_cl_bf16": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int,
                                                      c_int, c_int, c_int, c_int, c_int, c_int, _P, _P,
                                                      c_size_t, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)
E_UNSUPPORTED = -4   # VEON_E_UNSUPPORTED: the shape does not fit this entry point
_lib = None


def load():
    """Load libveonlift.so once and bind every exported symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise VeonLibraryError(
            f"{LIB_PATH} not found: build it with `make -C veon_b200/csrc` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
            "veon_b200 has no CPU / PyTorch fallback.")
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise VeonLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise VeonLibraryError(f"{LIB_PATH} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def error_string(code):
    return load().veon_error_string(int(code)).decode()


def check(code, what):
    if code != 0:
        raise VeonError(code, what)


def float3(values):
    """[host] float32[3] argument."""
    return (ctypes.c_float * 3)(*[float(v) for v in values])


def ptr(t):
    """A tensor's data as a pointer argument."""
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr(device):
    """torch's current stream on `device` as a cudaStream_t argument."""
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(*tensors):
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError(
                "veon_b200 runs on CUDA tensors only (there is no CPU fallback); "
                f"got a tensor on {t.device}")
