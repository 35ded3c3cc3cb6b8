"""BEVPoolv2 operator surface on libveonlift (B200 / sm_100a).

Mirrors `mmdet3d/ops/bev_pool_v2/bev_pool.py` of the reference:

    bev_pool_v2(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                bev_feat_shape, interval_starts, interval_lengths)   :86-92
    QuickCumsumCuda (torch.autograd.Function)                         :11-83
    TRTBEVPoolv2                                                      :95-142

plus the index preparation the necks call before it,

    voxel_pooling_prepare_v2(coor, grid_lower_bound, grid_interval, grid_size)
        = LSSViewTransformer.voxel_pooling_prepare_v2, view_transformer.py:202-260

What differs underneath (DESIGN.md): the volume is produced channels-first
in one pass (no memset, no permute copy), the backward needs no argsort, and a
"plan" (tile tables + point->interval table) rides along with the rank
tensors.  Everything runs in CUDA through the C ABI; there is no CPU path.

`memory_format=torch.channels_last_3d` (bev_pool_v2 / pool_prepared) returns the
same [B,C,Z,Y,X] values stored channels-last ([B,Z,Y,X,C] underneath), written
that way by the kernels; a channels-last gradient is consumed in place by a
single-pass backward, whichever layout the forward produced.

`dtype=torch.bfloat16` (bev_pool_v2 / pool_prepared, either memory format) returns
the volume in bfloat16, written so by the kernels: float32 sums rounded once, at
the store, so the result is bit for bit the float32 volume cast to bfloat16.  Its
bfloat16 gradient is read in place and widened exactly (depth / feat gradients
stay float32).

A bfloat16 `feat` (what a network under bfloat16 autocast hands the lift) is read as it is: the
kernels widen each value exactly where they load it, so every volume is bit for bit the one the
same call makes from `feat.float()`, depth_grad is that call's, and feat_grad comes back in
bfloat16, that call's feat_grad rounded once.  Only the bfloat16 rows are kept for the backward.
"""
import collections
import functools
import weakref
import ctypes

import torch

from . import _lib
from ._lib import ptr as _ptr, require_cuda as _require_cuda, stream_ptr as _stream_ptr

__all__ = ["bev_pool_v2", "QuickCumsumCuda", "TRTBEVPoolv2",
           "voxel_pooling_prepare_v2", "prepare_ranks", "PreparedRanks",
           "pool_prepared", "lidar_coor"]

LAYOUT_BZYXC, LAYOUT_BCZYX = 0, 1
PLAN_OUT_OF_RANGE = 8       # VEON_PLAN_OUT_OF_RANGE
TILE_VOXELS = 32


_MEMORY_FORMATS = (torch.contiguous_format, torch.channels_last_3d)


def _channels_last(memory_format):
    """True for torch.channels_last_3d, False for torch.contiguous_format; ValueError otherwise."""
    if memory_format not in _MEMORY_FORMATS:
        raise ValueError("memory_format must be torch.contiguous_format or torch.channels_last_3d, "
                         f"got {memory_format!r}")
    return memory_format is torch.channels_last_3d


_DTYPES = (torch.float32, torch.bfloat16)


def _bf16(dtype):
    """True for torch.bfloat16, False for torch.float32; ValueError otherwise (float16 overflows
    where the float32 sums do not: another contract)."""
    if not isinstance(dtype, torch.dtype) or dtype not in _DTYPES:
        raise ValueError(f"dtype must be torch.float32 or torch.bfloat16, got {dtype!r}")
    return dtype is torch.bfloat16


# Opt-in device timing of the library calls (bench.py / profiling only): CUDA
# events recorded on the stream the kernels are launched on.
_TIMERS = None


def enable_kernel_timing(on=True):
    global _TIMERS
    _TIMERS = {} if on else None


def kernel_timings_ms():
    """{call name: [ms, ...]} of everything recorded since enable_kernel_timing()."""
    torch.cuda.synchronize()
    return {k: [s.elapsed_time(e) for s, e in v] for k, v in (_TIMERS or {}).items()}


class _timed:
    def __init__(self, name, dev):
        self.name, self.dev = name, dev

    def __enter__(self):
        if _TIMERS is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.e = torch.cuda.Event(enable_timing=True)
            self.s.record(torch.cuda.current_stream(self.dev))

    def __exit__(self, *exc):
        if _TIMERS is not None:
            self.e.record(torch.cuda.current_stream(self.dev))
            _TIMERS.setdefault(self.name, []).append((self.s, self.e))
        return False


def lidar_coor(frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda):
    """get_lidar_coor (view_transformer.py:114-152) as one fused CUDA pass.
    frustum [D,H,W,3]; returns coor [B,N,D,H,W,3] float32."""
    _require_cuda(frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda)
    lib = _lib.load()
    dev = sensor2ego.device
    B, N = sensor2ego.shape[:2]
    D, H, W, _ = frustum.shape
    args = [t.detach().contiguous().float() for t in
            (frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda)]
    with torch.cuda.device(dev):
        coor = torch.empty((B, N, D, H, W, 3), dtype=torch.float32, device=dev)
        ws_bytes = lib.veon_lidar_coor_workspace_bytes(B, N)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with _timed("lidar_coor", dev):
            rc = lib.veon_lidar_coor(*[_ptr(a) for a in args], B, N, D, H, W, _ptr(coor), _ptr(ws),
                                     ws_bytes, _stream_ptr(dev))
    _lib.check(rc, "veon_lidar_coor")
    return coor


class PoolPlan:
    """By-products of the index preparation used by the planar kernels."""
    __slots__ = ("__weakref__", "tile_start", "tile_istart", "tile_occ", "tile_heavy", "voxel_start",
                 "point_interval", "dims", "V",
                 "flags", "_n_intervals", "_n_points", "counts_dev", "counts_host",
                 "counts_event", "keepalive", "sync_free")

    def __init__(self, tiles, heavy, point_interval, dims, V, flags=0, voxel_start=None,
                 counts=(None, None, None), n_points=None, n_intervals=None):
        """tiles: the [3, n_tiles + 1] start / interval-start / occupancy table; counts: the
        (device, pinned host, event) of counts still in flight, else n_points / n_intervals."""
        self.tile_start, self.tile_istart, self.tile_occ = tiles[0], tiles[1], tiles[2]
        self.tile_heavy = heavy
        self.point_interval = point_interval
        self.voxel_start = voxel_start
        self.dims, self.V, self.flags = dims, V, flags
        self.counts_dev, self.counts_host, self.counts_event = counts
        self._n_points, self._n_intervals = n_points, n_intervals
        self.keepalive = None
        self.sync_free = False

    def _resolve(self):
        if self._n_intervals is None:
            self.counts_event.synchronize()
            self._n_points = int(self.counts_host[0])
            self._n_intervals = int(self.counts_host[1])

    @property
    def n_intervals(self):
        self._resolve()
        return self._n_intervals

    @property
    def n_points(self):
        self._resolve()
        return self._n_points

    @property
    def ok(self):
        return self.flags == 0

    def interval_capacity(self):
        """Rows the backward scratch needs.  Exact when the counts are known (or have
        already arrived); a `sync_free` plan whose counts are still in flight answers
        with the upper bound (every point its own interval) instead of blocking."""
        if (self._n_intervals is None and self.sync_free and self.counts_event is not None
                and not self.counts_event.query()):
            B, N, D, H, W = self.dims
            return B * N * D * H * W
        return self.n_intervals


class PreparedRanks:
    """Device-side result of the index preparation (capacity-sized buffers;
    the valid prefix lengths live in `plan.counts_dev` / `plan.n_points`)."""
    __slots__ = ("ranks_bev", "ranks_depth", "ranks_feat", "interval_starts",
                 "interval_lengths", "plan", "shape")


# Pinned host slots the scan kernel writes {n_kept, n_int} into.  A ring owned by this
# module (never returned to torch's host allocator while a kernel may still write to it);
# a slot is reused only after the event of its previous prepare call has completed.
_COUNTS_RING = {}
_GEOMETRY_CACHE = {}   # per (shape, grid objects): float3 arrays, sizes (host-side only)
_COUNTS_SLOTS = 64


def _counts_slot(dev):
    ring = _COUNTS_RING.get(dev.index)
    if ring is None:
        ring = [torch.zeros((_COUNTS_SLOTS, 2), dtype=torch.int64).pin_memory(),
                [None] * _COUNTS_SLOTS, 0]
        _COUNTS_RING[dev.index] = ring
    buf, owners, nxt = ring
    ring[2] = (nxt + 1) % _COUNTS_SLOTS
    if owners[nxt] is not None:
        ev, plan_ref = owners[nxt]
        old = plan_ref()
        if old is not None:
            old._resolve()          # a plan that is still alive keeps its numbers
        else:
            ev.synchronize()        # the kernel that wrote the slot has finished
    return buf[nxt], nxt


def prepare_ranks_calib(frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda,
                        grid_lower_bound, grid_interval, grid_size, depth=None, depth_eps=None,
                        backward_tables=True):
    """`prepare_ranks(lidar_coor(...))` in one call with the geometry fused into the
    classification kernel (SURVEY 8f-3): the [B,N,D,H,W,3] coordinate tensor is never written.
    Same ranks, bit for bit.

    depth [B,N,D,H,W] + depth_eps (inference only, SURVEY 8f-2): points whose depth weight is
    <= depth_eps are dropped as well (`veon_prepare_v2_calib_sparse`).
    backward_tables=False (inference): the point -> interval table of the backward is not built;
    a backward through such ranks raises."""
    _require_cuda(frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda)
    calib = [t.detach().contiguous().float() for t in
             (frustum, sensor2ego, cam2imgs, post_rots, post_trans, bda)]
    B, N = sensor2ego.shape[:2]
    D, H, W, _ = frustum.shape
    sparse = None
    if depth_eps is not None:
        if depth is None or tuple(depth.shape) != (B, N, D, H, W):
            raise ValueError("depth_eps needs depth [B,N,D,H,W]")
        _require_cuda(depth)
        sparse = (depth.detach().contiguous().float(), float(depth_eps))
    return _prepare(None, calib, (B, N, D, H, W), sensor2ego.device, grid_lower_bound,
                    grid_interval, grid_size, sparse, backward_tables)


# Pinned host slots for calibration hashes (same life-cycle rules as the counts ring)
_HASH_RING = {}


def calib_hash(sensor2ego, cam2imgs, post_rots, post_trans, bda):
    """64-bit hash of the calibration tensors' bits (`veon_calib_hash`): one tiny kernel that
    writes into pinned host memory + an event wait (no copy queued on the stream).  Returns a
    python int."""
    _require_cuda(sensor2ego, cam2imgs, post_rots, post_trans, bda)
    lib = _lib.load()
    dev = sensor2ego.device
    B, N = sensor2ego.shape[:2]
    args = [t.detach().contiguous().float() for t in (sensor2ego, cam2imgs, post_rots, post_trans, bda)]
    ring = _HASH_RING.get(dev.index)
    if ring is None:
        ring = _HASH_RING[dev.index] = [torch.zeros(16, dtype=torch.int64).pin_memory(), 0]
    slot = ring[1] = (ring[1] + 1) % 16
    out = ring[0][slot:slot + 1]
    with torch.cuda.device(dev):
        rc = lib.veon_calib_hash(*[_ptr(a) for a in args], B, N, _ptr(out), _stream_ptr(dev))
        _lib.check(rc, "veon_calib_hash")
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
    ev.synchronize()
    return int(out[0])


def prepare_ranks(coor, grid_lower_bound, grid_interval, grid_size, stream=None):
    """Launch the GPU index preparation; returns without a host sync.

    coor: [B,N,D,H,W,3] float tensor on CUDA.  The three grid vectors are the
    reference's float32 tensors (view_transformer.py:79-82) or any 3-sequence.
    stream: a torch.cuda.Stream to launch on instead of the current one; the outputs are still
    allocated in the CURRENT stream's pool (the caller consumes them there, after waiting for
    `plan.counts_event`).
    """
    _require_cuda(coor)
    if coor.dim() != 6 or coor.shape[-1] != 3:
        raise ValueError(f"coor must be [B,N,D,H,W,3], got {tuple(coor.shape)}")
    coor = coor.detach().contiguous().float()
    return _prepare(coor, None, tuple(coor.shape[:5]), coor.device, grid_lower_bound,
                    grid_interval, grid_size, stream=stream)


_TENSOR_VALUES = {}


def _values(x):
    """The floats of a 3-vector as a tuple.  Reading a tensor element by element costs a few
    microseconds per call, so tensors are remembered by (object, in-place version); plain
    sequences / ndarrays (which have no version counter) are simply re-read every time."""
    if isinstance(x, torch.Tensor):
        hit = _TENSOR_VALUES.get(id(x))
        if hit is not None and hit[0]() is x and hit[1] == x._version:
            return hit[2]
        vals = tuple(float(v) for v in x.tolist())
        if len(_TENSOR_VALUES) > 256:
            _TENSOR_VALUES.clear()
        _TENSOR_VALUES[id(x)] = (weakref.ref(x), x._version, vals)
        return vals
    return tuple(float(v) for v in x)


def _prepare(coor, calib, dims, dev, grid_lower_bound, grid_interval, grid_size, sparse=None,
             backward_tables=True, stream=None):
    lib = _lib.load()
    launch_on = stream if stream is not None else torch.cuda.current_stream(dev)
    sp = ctypes.c_void_p(launch_on.cuda_stream)
    B, N, D, H, W = (int(v) for v in dims)
    P = B * N * D * H * W
    # keyed on the VALUES (three small tuples): a list / ndarray mutated in place, or a
    # recycled id(), can never hand back stale geometry
    lower, interval, size = _values(grid_lower_bound), _values(grid_interval), _values(grid_size)
    key = (B, N, D, H, W, lower, interval, size)
    geo = _GEOMETRY_CACHE.get(key)
    if geo is None:
        V = int(size[0]) * int(size[1]) * int(size[2])
        c_size = _lib.float3(size)
        ws_bytes = lib.veon_prepare_v2_workspace_bytes(B, N, D, H, W, c_size)
        if ws_bytes == 0:
            raise _lib.VeonError(-3, "veon_prepare_v2_workspace_bytes")
        n_tiles = lib.veon_pool_num_tiles(B, V)
        if len(_GEOMETRY_CACHE) > 64:
            _GEOMETRY_CACHE.clear()
        geo = (_lib.float3(lower), _lib.float3(interval), c_size, V, ws_bytes, n_tiles,
               lib.veon_pool_heavy_list_ints(P, n_tiles),
               lib.veon_prepare_v2_voxel_start_offset(B, N, D, H, W, c_size))
        _GEOMETRY_CACHE[key] = geo
    c_lower, c_interval, c_size, V, ws_bytes, n_tiles, nh, vs_off = geo
    with torch.cuda.device(dev):
        # one allocation for every int32 output + the kernel workspace (fewer allocator
        # round-trips per call); the pieces below are views of it
        nt1 = (n_tiles + 1 + 3) // 4 * 4
        ws_ints = (ws_bytes + 3) // 4
        nh4 = (nh + 3) // 4 * 4
        pool = torch.empty(6 * P + 3 * nt1 + nh4 + 4 + ws_ints + 64, dtype=torch.int32,
                           device=dev)
        ranks = pool[:5 * P].view(5, P)
        point_interval = pool[5 * P:6 * P]
        o = 6 * P
        tiles = pool[o:o + 3 * nt1].view(3, nt1)[:, :n_tiles + 1]
        o += 3 * nt1
        heavy = pool[o:o + nh]
        o += nh4
        counts = pool[o:o + 4].view(torch.int64)
        o = (o + 4 + 63) // 64 * 64           # 256-byte aligned workspace
        ws = pool[o:o + ws_ints]
        # The two counts come back through pinned host memory the scan kernel writes
        # directly (no D2H copy that could queue behind the caller's bulk transfers on
        # the copy engine); they are valid once `ev` has completed.
        counts_host, slot = _counts_slot(dev)
        # the pixel-major point -> interval table only serves the backward: an inference caller
        # saves its 4-byte-per-point fill and the scattered writes of the ranking kernel
        outs = (_ptr(ranks[0]), _ptr(ranks[1]), _ptr(ranks[2]), _ptr(ranks[3]), _ptr(ranks[4]),
                _ptr(counts), _ptr(counts_host), _ptr(tiles[0]), _ptr(tiles[1]), _ptr(tiles[2]),
                _ptr(heavy), _ptr(point_interval) if backward_tables else None)
        with _timed("prepare_v2", dev):
            if calib is None:
                rc = lib.veon_prepare_v2(_ptr(coor), B, N, D, H, W, c_lower, c_interval, c_size,
                                         *outs, _ptr(ws), ws_bytes, sp)
            else:
                xbytes = lib.veon_lidar_coor_workspace_bytes(B, N)
                xws = torch.empty(xbytes, dtype=torch.uint8, device=dev)
                if sparse is None:
                    rc = lib.veon_prepare_v2_calib(*[_ptr(a) for a in calib], B, N, D, H, W,
                                                   c_lower, c_interval, c_size, *outs, _ptr(xws),
                                                   xbytes, _ptr(ws), ws_bytes, sp)
                else:
                    rc = lib.veon_prepare_v2_calib_sparse(
                        *[_ptr(a) for a in calib], _ptr(sparse[0]), sparse[1], B, N, D, H, W,
                        c_lower, c_interval, c_size, *outs, _ptr(xws), xbytes, _ptr(ws), ws_bytes,
                        sp)
        _lib.check(rc, "veon_prepare_v2")
        ev = torch.cuda.Event()
        ev.record(launch_on)
    # first point of every voxel: lives in the preparation workspace (kept alive by this view)
    voxel_start = (ws[vs_off // 4: vs_off // 4 + B * V + 1]
                   if B * V < (1 << 24) and vs_off % 4 == 0 else None)
    plan = PoolPlan(tiles, heavy, point_interval if backward_tables else None, (B, N, D, H, W), V,
                    voxel_start=voxel_start, counts=(counts, counts_host, ev))
    _COUNTS_RING[dev.index][1][slot] = (ev, weakref.ref(plan))
    out = PreparedRanks()
    out.ranks_bev, out.ranks_depth, out.ranks_feat = ranks[0], ranks[1], ranks[2]
    out.interval_starts, out.interval_lengths = ranks[3], ranks[4]
    out.plan = plan
    out.shape = (B, N, D, H, W)
    return out


# ---------------------------------------------------------------- plan cache
_PLAN_CACHE = collections.OrderedDict()
_PLAN_CACHE_SIZE = 8


def _plan_key(rd, rf, rb, ist, iln, dims, V):
    return (rd.data_ptr(), rf.data_ptr(), rb.data_ptr(), ist.data_ptr(), iln.data_ptr(),
            rd.numel(), ist.numel(), rd._version, rf._version, rb._version,
            ist._version, iln._version, dims, V, rd.device.index)


def _remember_plan(key, plan, tensors):
    plan.keepalive = tensors  # pins the addresses the key is made of
    _PLAN_CACHE[key] = plan
    _PLAN_CACHE.move_to_end(key)
    while len(_PLAN_CACHE) > _PLAN_CACHE_SIZE:
        _PLAN_CACHE.popitem(last=False)


def _plan_for(rd, rf, rb, ist, iln, dims, V):
    """Plan for caller-held rank tensors: cached, else built + validated."""
    key = _plan_key(rd, rf, rb, ist, iln, dims, V)
    plan = _PLAN_CACHE.get(key)
    if plan is not None:
        _PLAN_CACHE.move_to_end(key)
        return plan
    lib = _lib.load()
    B, N, D, H, W = dims
    dev = rb.device
    P = B * N * D * H * W
    n_tiles = lib.veon_pool_num_tiles(B, V)
    with torch.cuda.device(dev):
        tiles = torch.empty((3, n_tiles + 1), dtype=torch.int32, device=dev)
        heavy = torch.empty(lib.veon_pool_heavy_list_ints(rd.numel(), n_tiles),
                            dtype=torch.int32, device=dev)
        point_interval = torch.empty(P, dtype=torch.int32, device=dev)
        flags = torch.zeros(1, dtype=torch.int32, device=dev)
        rc = lib.veon_pool_plan_build(
            _ptr(rd), _ptr(rf), _ptr(rb), _ptr(ist), _ptr(iln), rd.numel(), ist.numel(),
            B, N, D, H, W, V, _ptr(tiles[0]), _ptr(tiles[1]), _ptr(tiles[2]), _ptr(heavy),
            _ptr(point_interval), _ptr(flags), _stream_ptr(dev))
        _lib.check(rc, "veon_pool_plan_build")
        plan = PoolPlan(tiles, heavy, point_interval, dims, V,
                        flags=int(flags.item()),  # one sync per distinct rank set
                        n_points=rd.numel(), n_intervals=ist.numel())
    _remember_plan(key, plan, (rd, rf, rb, ist, iln))
    return plan


def pool_prepared_downsampled(depth, feat, prep, bev_feat_shape):
    """bev_pool_v2 fused with the neck's 2x2x2 max-downsample (view_transformer_raw.py:549-553),
    forward only: returns [B, C, Z/2, Y/2, X/2] without materialising the full volume, or None
    when the shape is outside what the fused kernel takes (the caller then pools and reduces).

    depth [B,N,D,H,W]; feat [B,N,H,W,C] (a permuted view of channels-first maps is fine);
    prep from `prepare_ranks` (its workspace holds the per-voxel point prefix)."""
    B, Z, Y, X, C = (int(v) for v in bev_feat_shape)
    vs = prep.plan.voxel_start
    if vs is None or (Z | Y | X) & 1 or C % 64 != 0:
        return None
    _require_cuda(depth, feat)
    lib = _lib.load()
    dev = feat.device
    depth = depth.detach().contiguous().float()
    feat = _feat_rows(feat.detach())[0].float()     # the fused kernel reads float32 rows
    with torch.cuda.device(dev):
        out = torch.empty((B, C, Z // 2, Y // 2, X // 2), dtype=torch.float32, device=dev)
        with _timed("pool_ds_fwd", dev):
            rc = lib.veon_bev_pool_v2_ds_fwd(
                _ptr(depth), _ptr(feat), _ptr(prep.ranks_depth), _ptr(prep.ranks_feat),
                _ptr(prep.ranks_bev), _ptr(vs), B, C, Z, Y, X, feat.numel() // C, _ptr(out),
                _stream_ptr(dev))
    if rc == -4:        # VEON_E_UNSUPPORTED: shape outside the fused kernel
        return None
    _lib.check(rc, "veon_bev_pool_v2_ds_fwd")
    return out


def two_hot_depth(depths, depth_cfg, D, gamma=4.0, downsample=0):
    """LSSViewTransformerRaw.get_two_hot_depth (+ downsample_depth), forward only
    (view_transformer_raw.py:393-429): depths [B,N,H,W] metric depth on CUDA ->
    [B,N,D,H/s,W/s] float32 (contiguous; the reference returns a permuted view of the same
    values)."""
    _require_cuda(depths)
    lib = _lib.load()
    d = depths.detach().contiguous().float()
    B, N, H, W = d.shape
    s = int(downsample) if downsample else 1
    if H % s or W % s:
        raise ValueError("depth map size must be a multiple of the downsample factor")
    with torch.cuda.device(d.device):
        out = torch.empty((B, N, D, H // s, W // s), dtype=torch.float32, device=d.device)
        with _timed("two_hot_depth", d.device):
            rc = lib.veon_two_hot_depth(_ptr(d), B * N, H // s, W // s, s, int(D),
                                        float(depth_cfg[0]), float(depth_cfg[2]), float(gamma),
                                        _ptr(out), _stream_ptr(d.device))
    _lib.check(rc, "veon_two_hot_depth")
    return out


class MaxDown2x2x2(torch.autograd.Function):
    """The neck's 2x2x2 reduction, `rearrange(... '(dz dh dw)') -> torch.max(dim=-1).values`
    (view_transformer_raw.py:549-553), and its gradient (all of it to the first arg-max of a
    block, as max(dim) does) as two streaming kernels.  A channels-last-3d input (even Z, Y, X)
    goes through the channels-last kernels and gives a channels-last-3d result."""

    @staticmethod
    def supports(x):
        if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 5
                and x.shape[2] % 2 == 0 and x.shape[3] % 2 == 0):
            return False
        if x.is_contiguous():
            return x.shape[4] % 4 == 0
        return x.shape[4] % 2 == 0 and x.is_contiguous(memory_format=torch.channels_last_3d)

    @staticmethod
    def forward(ctx, x):
        lib = _lib.load()
        B, C, Z, Y, X = x.shape
        ctx.channels_last = not x.is_contiguous()
        if ctx.channels_last:
            with torch.cuda.device(x.device):
                out = torch.empty((B, Z // 2, Y // 2, X // 2, C), dtype=torch.float32,
                                  device=x.device).permute(0, 4, 1, 2, 3)
                with _timed("maxdown_cl_fwd", x.device):
                    rc = lib.veon_maxdown2_cl_fwd(_ptr(x), B, C, Z, Y, X, _ptr(out),
                                                  _stream_ptr(x.device))
            _lib.check(rc, "veon_maxdown2_cl_fwd")
            ctx.save_for_backward(x, out)
            return out
        with torch.cuda.device(x.device):
            out = torch.empty((B, C, Z // 2, Y // 2, X // 2), dtype=torch.float32, device=x.device)
            with _timed("maxdown_fwd", x.device):
                rc = lib.veon_maxdown2_fwd(_ptr(x), B * C, Z, Y, X, _ptr(out), _stream_ptr(x.device))
        _lib.check(rc, "veon_maxdown2_fwd")
        ctx.save_for_backward(x, out)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, out = ctx.saved_tensors
        lib = _lib.load()
        B, C, Z, Y, X = x.shape
        if ctx.channels_last:
            g = grad_out.float().contiguous(memory_format=torch.channels_last_3d)
            with torch.cuda.device(x.device):
                grad_in = torch.empty_like(x)          # channels-last, like x
                with _timed("maxdown_cl_bwd", x.device):
                    rc = lib.veon_maxdown2_cl_bwd(_ptr(x), _ptr(out), _ptr(g), B, C, Z, Y, X,
                                                  _ptr(grad_in), _stream_ptr(x.device))
            _lib.check(rc, "veon_maxdown2_cl_bwd")
            return grad_in
        g = grad_out.contiguous().float()
        with torch.cuda.device(x.device):
            grad_in = torch.empty_like(x)
            with _timed("maxdown_bwd", x.device):
                rc = lib.veon_maxdown2_bwd(_ptr(x), _ptr(out), _ptr(g), B * C, Z, Y, X,
                                           _ptr(grad_in), _stream_ptr(x.device))
        _lib.check(rc, "veon_maxdown2_bwd")
        return grad_in


class PoolMaxDown(torch.autograd.Function):
    """bev_pool_v2 followed by the neck's 2x2x2 max-downsample as ONE autograd node
    (view_transformer.py:175-200 + view_transformer_raw.py:549-553).  Forward: the two kernels
    of the plain route, plus an 8-bit mask per output (one bit: which input is the arg-max,
    the first one on ties).  Backward: the gradient rows of the occupied voxels come straight
    from grad_ds and the mask (the gradient of torch.max(dim): everything to the arg-max), so
    neither the 1.31 GB full-resolution gradient nor the volume is kept or touched."""

    @staticmethod
    def forward(ctx, depth, feat, prep, bev_feat_shape):
        lib = _lib.load()
        B, Z, Y, X, C = (int(v) for v in bev_feat_shape)
        plan = prep.plan
        depth = depth.contiguous().float()
        feat, ctx.feat_transposed = _feat_rows(feat)
        vol = _fwd_planar(depth, feat, prep.ranks_depth, prep.ranks_feat, prep.ranks_bev, plan,
                          B, C, Z * Y * X, (B, C, Z, Y, X))
        dev = vol.device
        with torch.cuda.device(dev):
            out = torch.empty((B, C, Z // 2, Y // 2, X // 2), dtype=torch.float32, device=dev)
            mask = torch.empty(out.shape, dtype=torch.uint8, device=dev)
            with _timed("maxdown_fwd", dev):
                rc = lib.veon_maxdown2_fwd_mask(_ptr(vol), B * C, Z, Y, X, _ptr(out), _ptr(mask),
                                                _stream_ptr(dev))
        _lib.check(rc, "veon_maxdown2_fwd_mask")
        ctx.save_for_backward(depth, feat, mask)
        ctx.plan, ctx.grid = plan, (Z, Y, X)
        return out

    @staticmethod
    def backward(ctx, grad_ds):
        depth, feat, mask = ctx.saved_tensors
        lib = _lib.load()
        plan = ctx.plan
        Z, Y, X = ctx.grid
        B, N, D, H, W = plan.dims
        C = feat.shape[-1]
        dev = feat.device
        g = grad_ds.contiguous().float()
        _need_backward_tables(plan)
        suffix = "_bf16feat" if feat.dtype == torch.bfloat16 else ""
        with torch.cuda.device(dev):
            depth_grad = torch.empty_like(depth)
            feat_grad = torch.empty_like(feat)          # in the rows' dtype
            n_int, rows = _bwd_rows(lib, plan, C, dev)
            with _timed("pool_bwd_ds" + suffix, dev):
                rc = getattr(lib, "veon_bev_pool_v2_bwd_planar_ds" + suffix)(
                    _ptr(g), _ptr(mask), _ptr(depth), _ptr(feat), _ptr(plan.tile_istart),
                    _ptr(plan.tile_occ), _ptr(plan.point_interval), n_int, B, N, D, H, W, C,
                    Z, Y, X, _ptr(rows), _ptr(depth_grad), _ptr(feat_grad), _stream_ptr(dev))
        _lib.check(rc, "veon_bev_pool_v2_bwd_planar_ds" + suffix)
        return depth_grad, _feat_grad_back(feat_grad, ctx.feat_transposed), None, None


def pool_prepared_maxdown(depth, feat, prep, bev_feat_shape):
    """Pool + 2x2x2 max as one differentiable node (see PoolMaxDown); None when the grid is not
    even / X % 4 != 0 or the plan is not a prepared one (the caller then takes the plain route)."""
    B, Z, Y, X, C = (int(v) for v in bev_feat_shape)
    if (Z | Y) & 1 or X & 3 or not prep.plan.ok:
        return None
    _require_cuda(depth, feat)
    return PoolMaxDown.apply(depth, feat, prep, bev_feat_shape)


def voxel_pooling_prepare_v2(coor, grid_lower_bound, grid_interval, grid_size):
    """Same contract as the reference method (view_transformer.py:202-260):
    returns (ranks_bev, ranks_depth, ranks_feat, interval_starts,
    interval_lengths), int32 contiguous on coor.device, or five `None`s when
    nothing can be pooled (:236-237, :253-254)."""
    if coor.numel() == 0:
        return None, None, None, None, None
    prep = prepare_ranks(coor, grid_lower_bound, grid_interval, grid_size)
    n_kept, n_int = prep.plan.n_points, prep.plan.n_intervals  # host sync
    if n_int == 0:
        return None, None, None, None, None
    rb, rd, rf = prep.ranks_bev[:n_kept], prep.ranks_depth[:n_kept], prep.ranks_feat[:n_kept]
    ist, iln = prep.interval_starts[:n_int], prep.interval_lengths[:n_int]
    key = _plan_key(rd, rf, rb, ist, iln, prep.shape, prep.plan.V)
    _remember_plan(key, prep.plan, (rd, rf, rb, ist, iln))
    return rb, rd, rf, ist, iln


# ------------------------------------------------------------------ pooling
def _transpose_batched(src, batch, R, S, out_shape):
    """[batch][R][S] -> [batch][S][R] of a contiguous float32 or bfloat16 tensor (bfloat16 bits
    are moved, not rounded), returned as `out_shape` in the same dtype."""
    lib = _lib.load()
    dev = src.device
    what = "veon_transpose_batched_u16" if src.dtype == torch.bfloat16 else "veon_transpose_batched"
    with torch.cuda.device(dev):
        dst = torch.empty(out_shape, dtype=src.dtype, device=dev)
        rc = getattr(lib, what)(_ptr(src), batch, R, S, _ptr(dst), _stream_ptr(dev))
    _lib.check(rc, what)
    return dst


def _feat_rows(feat):
    """feat [B,N,H,W,C] as contiguous rows, and whether they were transposed: float32 and bfloat16
    rows keep their dtype, any other dtype is widened to float32.  The necks hand over a
    channels-last VIEW of channels-first maps, which our own transpose kernel turns into rows
    instead of a strided copy."""
    if (feat.dtype in _DTYPES and not feat.is_contiguous()
            and feat.permute(0, 1, 4, 2, 3).is_contiguous()):
        B, N, H, W, C = feat.shape
        return _transpose_batched(feat.permute(0, 1, 4, 2, 3), B * N, C, H * W,
                                  (B, N, H, W, C)), True
    if feat.dtype == torch.bfloat16:
        return feat.contiguous(), False
    return feat.contiguous().float(), False


def _feat_grad_back(feat_grad, transposed):
    """The gradient of `_feat_rows`' rows, transposed back to channels-first storage (as a
    [B,N,H,W,C] view) when the rows were transposed."""
    if not transposed:
        return feat_grad
    B, N, H, W, C = feat_grad.shape
    return _transpose_batched(feat_grad, B * N, H * W, C, (B, N, C, H, W)).permute(0, 1, 3, 4, 2)


# Scratch of the streaming forward (control block + the L2-resident ring of compact rows):
# one buffer per (device, stream) -- calls on one stream are ordered, calls on different
# streams may overlap and must not share it.  FWD_RING_BYTES: None = the library's default size
# (tools/fwd_check.py sweeps it: the buffer size decides how many ring slots an SM gets).
_FWD_WS = {}
FWD_RING_BYTES = None


def _fwd_workspace(lib, dev, B, C, V):
    need = lib.veon_bev_pool_v2_fwd_workspace_bytes(B, C, V)
    if FWD_RING_BYTES is not None:
        need = int(FWD_RING_BYTES)
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream)
    ws = _FWD_WS.get(key)
    if ws is None or ws.numel() != need:
        ws = _FWD_WS[key] = torch.empty(need, dtype=torch.uint8, device=dev)
    return ws


def _fwd_planar(depth, feat, rd, rf, rb, plan, B, C, V, shape5, channels_last=False,
                dtype=torch.float32):
    """Planar forward of a valid plan from float32 or bfloat16 rows `feat` into a new volume
    `shape5` of `dtype` (float32 or bfloat16): [B,C,Z,Y,X], or [B,Z,Y,X,C] with channels_last
    (the streaming kernel and its workspace are float32 channels-first only, from float32 rows:
    where it would run, bfloat16 rows are widened first)."""
    lib = _lib.load()
    dev = feat.device
    bf16 = dtype is torch.bfloat16
    bf16feat = feat.dtype == torch.bfloat16
    suffix = ("_bf16" if bf16 else "") + ("_bf16feat" if bf16feat else "")
    with torch.cuda.device(dev):
        out = torch.empty(shape5, dtype=dtype, device=dev)
        if channels_last:
            what = "veon_bev_pool_v2_fwd_planar_cl" + suffix
            with _timed("pool_fwd_cl" + suffix, dev):
                rc = getattr(lib, what)(
                    _ptr(depth), _ptr(feat), _ptr(rd), _ptr(rf), _ptr(rb), _ptr(plan.tile_start),
                    _ptr(plan.tile_heavy), plan.tile_heavy.numel(), B, C, V, feat.numel() // C,
                    _ptr(out), _stream_ptr(dev))
        else:
            what = "veon_bev_pool_v2_fwd_planar" + suffix
            ws = None if bf16 else _fwd_workspace(lib, dev, B, C, V)
            with _timed("pool_fwd" + suffix, dev):
                rc = getattr(lib, what)(
                    _ptr(depth), _ptr(feat), _ptr(rd), _ptr(rf), _ptr(rb), _ptr(plan.tile_start),
                    _ptr(plan.tile_istart), _ptr(plan.tile_occ),
                    _ptr(plan.tile_heavy), plan.tile_heavy.numel(),
                    B, C, V, feat.numel() // C, _ptr(out), None if bf16 else _ptr(ws),
                    0 if bf16 else ws.numel(), _stream_ptr(dev))
    if bf16feat and rc == _lib.E_UNSUPPORTED:
        # a 64-channel float32 channels-first volume: the streaming kernel, on widened rows
        return _fwd_planar(depth, feat.float(), rd, rf, rb, plan, B, C, V, shape5, channels_last,
                           dtype)
    _lib.check(rc, what)
    return out


_fwd_planar_cl = functools.partial(_fwd_planar, channels_last=True)


def _need_backward_tables(plan):
    if plan.point_interval is None:
        raise RuntimeError("these ranks were prepared with backward_tables=False (inference): "
                           "no gradient can flow through the pooling")


def _bwd_rows(lib, plan, C, dev):
    """The intervals a row pass covers (a bound while a sync-free plan's count is still in
    flight) and its scratch: one C-float row per interval."""
    B, N, D, H, W = plan.dims
    n_int = plan.interval_capacity()
    n_rows = lib.veon_bev_pool_v2_bwd_workspace_floats(n_int, B, N, D, H, W, C, plan.V)
    return n_int, torch.empty(max(n_rows, 1), dtype=torch.float32, device=dev)


def _pool_bwd(out_grad, depth, feat, rd, rf, rb, ist, plan):
    """(depth_grad, feat_grad) for the gradient of a [B,Z,Y,X,C] volume, routed by its storage:
    float32 or bfloat16 channels-last (out_grad contiguous, its [B,C,Z,Y,X] view not) with a
    valid plan -> the single pass, which reads the gradient rows in place; otherwise a valid plan
    -> the two passes on a channels-first copy (bfloat16 stays bfloat16, anything else becomes
    float32); a rejected plan -> the generic kernel on a float32 copy.  feat_grad has the dtype of
    the rows `feat` (float32 or bfloat16)."""
    lib = _lib.load()
    dev = feat.device
    _, Z, Y, X, C = out_grad.shape
    g = out_grad.permute(0, 4, 1, 2, 3)  # back to the channels-first storage order
    bf16 = out_grad.dtype == torch.bfloat16 and plan.ok
    suffix = ("_bf16" if bf16 else "") + ("_bf16feat" if feat.dtype == torch.bfloat16 else "")
    single = ((out_grad.dtype == torch.float32 or bf16) and not g.is_contiguous()
              and out_grad.is_contiguous() and plan.ok)
    if not single:
        g = g.contiguous() if bf16 else g.float().contiguous()
    with torch.cuda.device(dev):
        if not plan.ok:
            what = "veon_bev_pool_v2_grad_generic"
            featf = feat.float()                 # the generic kernels read float32 rows
            depth_grad, feat_grad = torch.zeros_like(depth), torch.zeros_like(featf)
            rc = lib.veon_bev_pool_v2_grad_generic(
                C, rb.numel(), LAYOUT_BCZYX, Z * Y * X, _ptr(g), _ptr(depth), _ptr(featf),
                _ptr(rd), _ptr(rf), _ptr(rb), _ptr(depth_grad), _ptr(feat_grad), _stream_ptr(dev))
            _lib.check(rc, what)
            return depth_grad, feat_grad.to(feat.dtype)
        else:
            _need_backward_tables(plan)
            B, N, D, H, W = plan.dims
            depth_grad, feat_grad = torch.empty_like(depth), torch.empty_like(feat)
            if single:
                what = "veon_bev_pool_v2_bwd_planar_cl" + suffix
                with _timed("pool_bwd_cl" + suffix, dev):
                    rc = getattr(lib, what)(
                        _ptr(out_grad), _ptr(depth), _ptr(feat), _ptr(rb), _ptr(ist),
                        _ptr(plan.point_interval), B, N, D, H, W, C, plan.V, _ptr(depth_grad),
                        _ptr(feat_grad), _stream_ptr(dev))
            else:
                what = "veon_bev_pool_v2_bwd_planar" + suffix
                n_int, rows = _bwd_rows(lib, plan, C, dev)
                with _timed("pool_bwd" + suffix, dev):
                    rc = getattr(lib, what)(
                        _ptr(g), _ptr(depth), _ptr(feat), _ptr(plan.tile_istart),
                        _ptr(plan.tile_occ), _ptr(plan.point_interval), n_int, B, N, D, H, W, C,
                        plan.V, _ptr(rows), rows.numel(), _ptr(depth_grad), _ptr(feat_grad),
                        _stream_ptr(dev))
    _lib.check(rc, what)
    return depth_grad, feat_grad


class QuickCumsumCuda(torch.autograd.Function):
    """Same signature and result as the reference Function (bev_pool.py:11-83):
    returns the pooled volume shaped [B,Z,Y,X,C].  It is a permuted VIEW of a
    channels-first buffer, so the `.permute(0,4,1,2,3).contiguous()` that
    `bev_pool_v2` applies next (bev_pool.py:91) is free.  With the extra
    `channels_last` argument it is a contiguous [B,Z,Y,X,C] tensor instead.

    The backward takes the gradient in the layout it arrives in: channels-first
    storage -> the two-pass kernels; channels-last storage (a contiguous
    [B,Z,Y,X,C] gradient) with a valid plan -> the single-pass kernel, which reads
    the gradient rows in place; anything else is copied to channels-first first.
    All routes give the same bits.  With the extra `dtype` torch.bfloat16 the volume is
    bfloat16 (the float32 one rounded once), and so is the gradient the backward reads.  A
    bfloat16 `feat` is pooled and saved as bfloat16 rows; its gradient is bfloat16."""

    @staticmethod
    def forward(ctx, depth, feat, ranks_depth, ranks_feat, ranks_bev,
                bev_feat_shape, interval_starts, interval_lengths, *extra):
        # `extra` = (PoolPlan or None[, channels_last[, dtype]]) when called from this package;
        # the reference's 8-argument call is accepted unchanged
        plan = extra[0] if extra else None
        channels_last = bool(extra[1]) if len(extra) > 1 else False
        dtype = extra[2] if len(extra) > 2 else torch.float32
        ctx.n_extra = len(extra)
        _require_cuda(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                     interval_starts, interval_lengths)
        if depth.dim() != 5 or feat.dim() != 5:
            raise ValueError("depth must be [B,N,D,H,W] and feat [B,N,H,W,C]")
        ranks_bev = ranks_bev.int().contiguous()
        depth = depth.contiguous().float()
        feat, ctx.feat_transposed = _feat_rows(feat)
        ranks_depth = ranks_depth.contiguous().int()
        ranks_feat = ranks_feat.contiguous().int()
        interval_lengths = interval_lengths.contiguous().int()
        interval_starts = interval_starts.contiguous().int()
        B, Z, Y, X, C = (int(v) for v in bev_feat_shape)
        if feat.shape[-1] != C:
            raise ValueError("bev_feat_shape[-1] must equal feat.shape[-1]")
        V = Z * Y * X
        dims = tuple(int(v) for v in depth.shape)
        if plan is None:
            plan = _plan_for(ranks_depth, ranks_feat, ranks_bev, interval_starts,
                             interval_lengths, dims, V)
        if plan.flags & PLAN_OUT_OF_RANGE:
            # the reference would read / write out of bounds here (it checks nothing,
            # bev_pool.cpp has no CHECK_* macros); so would the unchecked generic kernels
            raise ValueError("bev_pool_v2: a rank lies outside its tensor (ranks_depth >= "
                             "depth.numel(), ranks_feat >= feat rows or ranks_bev >= B*Z*Y*X)")
        shape5 = (B, Z, Y, X, C) if channels_last else (B, C, Z, Y, X)
        if plan.ok:
            out = _fwd_planar(depth, feat, ranks_depth, ranks_feat, ranks_bev, plan, B, C, V,
                              shape5, channels_last, dtype)
        else:
            # the interval-driven generic kernel adds float32 rows into a zeroed volume
            lib = _lib.load()
            featf = feat.float()
            out = featf.new_zeros(shape5)
            with torch.cuda.device(feat.device):
                rc = lib.veon_bev_pool_v2_generic(
                    C, interval_starts.numel(), LAYOUT_BZYXC if channels_last else LAYOUT_BCZYX, V,
                    _ptr(depth), _ptr(featf), _ptr(ranks_depth), _ptr(ranks_feat), _ptr(ranks_bev),
                    _ptr(interval_starts), _ptr(interval_lengths), _ptr(out),
                    _stream_ptr(feat.device))
            _lib.check(rc, "veon_bev_pool_v2_generic")
            out = out.to(dtype)     # bfloat16: the same single rounding of the float32 sums
        ctx.save_for_backward(ranks_bev, depth, feat, ranks_feat, ranks_depth, interval_starts)
        ctx.plan = plan
        return out if channels_last else out.permute(0, 2, 3, 4, 1)

    @staticmethod
    def backward(ctx, out_grad):
        ranks_bev, depth, feat, ranks_feat, ranks_depth, interval_starts = ctx.saved_tensors
        depth_grad, feat_grad = _pool_bwd(out_grad, depth, feat, ranks_depth, ranks_feat,
                                          ranks_bev, interval_starts, ctx.plan)
        feat_grad = _feat_grad_back(feat_grad, ctx.feat_transposed)
        return (depth_grad, feat_grad, None, None, None, None, None, None) + (None,) * ctx.n_extra


def bev_pool_v2(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                bev_feat_shape, interval_starts, interval_lengths, *,
                memory_format=torch.contiguous_format, dtype=torch.float32):
    """Drop-in for the reference `bev_pool_v2` (bev_pool.py:86-92).

    depth [B,N,D,H,W]; feat [B,N,H,W,C] (any strides); int32 rank / interval
    tensors; bev_feat_shape = (B,Z,Y,X,C).  Returns [B,C,Z,Y,X] float32,
    differentiable w.r.t. depth and feat: contiguous, or with
    memory_format=torch.channels_last_3d the same values stored channels-last
    (written so by the kernels, not copied).  dtype=torch.bfloat16 returns the
    volume in bfloat16: the float32 result rounded to nearest even, bit for bit,
    with no float32 volume in between."""
    cl = _channels_last(memory_format)
    bf16 = _bf16(dtype)
    extra = (None, cl, dtype) if bf16 else ((None, True) if cl else ())
    x = QuickCumsumCuda.apply(depth, feat, ranks_depth, ranks_feat, ranks_bev,
                              bev_feat_shape, interval_starts, interval_lengths, *extra)
    x = x.permute(0, 4, 1, 2, 3)
    # no copy either way: the storage already has the requested order
    return x if cl else x.contiguous()


def pool_prepared(depth, feat, prep, bev_feat_shape, memory_format=torch.contiguous_format, *,
                  dtype=torch.float32):
    """bev_pool_v2 on a `PreparedRanks` without any host synchronisation in the
    forward (the counts are only needed, and by then long available, when the
    backward sizes its scratch).  memory_format and dtype as in bev_pool_v2."""
    cl = _channels_last(memory_format)
    bf16 = _bf16(dtype)
    extra = (prep.plan, cl, dtype) if bf16 else ((prep.plan, True) if cl else (prep.plan,))
    x = QuickCumsumCuda.apply(depth, feat, prep.ranks_depth, prep.ranks_feat, prep.ranks_bev,
                              bev_feat_shape, prep.interval_starts, prep.interval_lengths, *extra)
    x = x.permute(0, 4, 1, 2, 3)
    return x if cl else x.contiguous()


def lift_classify_prepared(depth, pix, prep, Q, prompt_class, grid_zyx, free_label=17):
    """Fused lift + classify (`veon_lift_classify_fwd`): depth [B,N,D,H,W]; pix [B,N,Cp,H,W]
    channels-first per-pixel rows ordered [gate 0, gate 1, logit 0..Q-1, zero padding]; prep from
    `prepare_ranks*`; -> uint8 labels [B,X,Y,Z], or None when the kernel does not take the shape
    (the caller then pools the volume and classifies it).  No gradient."""
    _require_cuda(depth, pix, prompt_class)
    lib = _lib.load()
    Z, Y, X = (int(v) for v in grid_zyx)
    B, N, Cp, H, W = (int(v) for v in pix.shape)
    if not prep.plan.ok or prep.plan.tile_heavy is None:
        return None
    dev = pix.device
    depth = depth.detach().contiguous().float()
    rows = _transpose_batched(pix.detach().contiguous().float(), B * N, Cp, H * W, (B, N, H, W, Cp))
    cls = prompt_class.contiguous().int()
    with torch.cuda.device(dev):
        labels = torch.empty((B, X, Y, Z), dtype=torch.uint8, device=dev)
        with _timed("lift_classify_fwd", dev):
            rc = lib.veon_lift_classify_fwd(
                _ptr(depth), _ptr(rows), _ptr(prep.ranks_depth), _ptr(prep.ranks_feat),
                _ptr(prep.ranks_bev), _ptr(prep.plan.tile_start), _ptr(prep.plan.tile_heavy),
                prep.plan.tile_heavy.numel(), B, Cp, int(Q), Z, Y, X, rows.numel() // Cp, _ptr(cls),
                int(free_label), _ptr(labels), _stream_ptr(dev))
    if rc in (-4, -5):      # VEON_E_UNSUPPORTED / VEON_E_RANGE: shape outside the fused kernel
        return None
    _lib.check(rc, "veon_lift_classify_fwd")
    return labels


class TRTBEVPoolv2(torch.autograd.Function):
    """ONNX/TensorRT export shim with the reference's symbolic
    (bev_pool.py:95-142): emits `mmdeploy::bev_pool_v2`; eager `forward`
    evaluates through `bev_pool_v2` for a single un-batched sample."""

    @staticmethod
    def symbolic(g, depth, feat, ranks_depth, ranks_feat, ranks_bev, interval_starts,
                 interval_lengths, out_height=128, out_width=128):
        return g.op("mmdeploy::bev_pool_v2", depth, feat, ranks_depth, ranks_feat, ranks_bev,
                    interval_starts, interval_lengths, out_height_i=out_height,
                    out_width_i=out_width)

    @staticmethod
    def forward(g, depth, feat, ranks_depth, ranks_feat, ranks_bev, interval_starts,
                interval_lengths, out_height=128, out_width=128):
        depth5, feat5 = depth[None], feat[None]          # N,D,H,W -> 1,N,D,H,W
        shape = (1, 1, out_height, out_width, feat5.shape[-1])
        bev = bev_pool_v2(depth5, feat5, ranks_depth, ranks_feat, ranks_bev, shape,
                          interval_starts, interval_lengths)
        return bev[:, :, 0].permute(0, 2, 3, 1)         # [1, Y, X, C]
