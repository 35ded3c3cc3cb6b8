"""Stand-in for the reference's pybind extension `mmdet3d.ops.bev_pool_v2.bev_pool_v2_ext`
(bev_pool.cpp:106-111): the same two functions with the same argument order, over the two
literal C-ABI drop-ins of libveonlift (INTEGRATION.md route B).

    bev_pool_v2_forward(depth, feat, out, ranks_depth, ranks_feat, ranks_bev,
                        interval_lengths, interval_starts)            bev_pool.cpp:30-57
    bev_pool_v2_backward(out_grad, depth_grad, feat_grad, depth, feat, ranks_depth,
                         ranks_feat, ranks_bev, interval_lengths, interval_starts)   :74-104

Note the lengths-before-starts order (bev_pool.py:36-37).  Semantics are the reference's:
channels-last `out` / `out_grad`, caller-zeroed outputs, intervals taken as given, nothing
returned.  Unlike the reference (legacy default stream, bev_pool_cuda.cu:127,136) the
kernels go to torch's current stream.  A reference checkout uses it with

    sys.modules["mmdet3d.ops.bev_pool_v2.bev_pool_v2_ext"] = veon_b200.bev_pool_v2_ext

before `mmdet3d.ops.bev_pool_v2.bev_pool` is imported; its own QuickCumsumCuda (memset,
permute, argsort and all) then runs unchanged on our kernels.
"""
import torch

from . import _lib
from ._lib import ptr, require_cuda, stream_ptr

__all__ = ["bev_pool_v2_forward", "bev_pool_v2_backward"]


def _check(*tensors):
    require_cuda(*tensors)
    if not all(t.is_contiguous() for t in tensors):
        raise RuntimeError("bev_pool_v2_ext: tensors must be contiguous")


def bev_pool_v2_forward(depth, feat, out, ranks_depth, ranks_feat, ranks_bev,
                        interval_lengths, interval_starts):
    _check(depth, feat, out, ranks_depth, ranks_feat, ranks_bev, interval_lengths, interval_starts)
    lib = _lib.load()
    with torch.cuda.device(depth.device):                    # OptionalCUDAGuard, bev_pool.cpp:42
        rc = lib.veon_bev_pool_v2(int(feat.size(4)), int(interval_lengths.size(0)), ptr(depth),
                                  ptr(feat), ptr(ranks_depth), ptr(ranks_feat), ptr(ranks_bev),
                                  ptr(interval_starts), ptr(interval_lengths), ptr(out),
                                  stream_ptr(depth.device))
    _lib.check(rc, "veon_bev_pool_v2")


def bev_pool_v2_backward(out_grad, depth_grad, feat_grad, depth, feat, ranks_depth, ranks_feat,
                         ranks_bev, interval_lengths, interval_starts):
    _check(out_grad, depth_grad, feat_grad, depth, feat, ranks_depth, ranks_feat, ranks_bev,
           interval_lengths, interval_starts)
    lib = _lib.load()
    with torch.cuda.device(out_grad.device):                 # bev_pool.cpp:88
        rc = lib.veon_bev_pool_v2_grad(int(out_grad.size(4)), int(interval_lengths.size(0)),
                                       ptr(out_grad), ptr(depth), ptr(feat), ptr(ranks_depth),
                                       ptr(ranks_feat), ptr(ranks_bev), ptr(interval_starts),
                                       ptr(interval_lengths), ptr(depth_grad), ptr(feat_grad),
                                       stream_ptr(out_grad.device))
    _lib.check(rc, "veon_bev_pool_v2_grad")
