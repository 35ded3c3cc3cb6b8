"""Host-side mirror of the reference's Lift-Splat view transformer, restricted
to the lifting path (SURVEY.md 8a rows a1-a4, a10, a11).

Same class name, constructor arguments, attribute names and method names as
`mmdet3d/models/necks/view_transformer.py::LSSViewTransformer` (and the
`forward` convention of `view_transformer_raw.py::LSSViewTransformerRaw`,
:537-555), so reference-side code and tests that drive the neck read the same.
The tensor work underneath goes to libveonlift through `veon_b200.bev_pool`.

Out of scope here (SURVEY.md 2, rows 10-14): DepthNet / ASPP / stereo cost
volumes and every other conv stack of the reference file.
"""
import torch
import torch.nn as nn

from . import bev_pool as _bp

__all__ = ["LSSViewTransformer", "LSSViewTransformerRaw"]


class LSSViewTransformer(nn.Module):
    """Lift-Splat view transformer (reference: view_transformer.py:15-319).

    Args mirror the reference (:40-50): grid_config {x,y,z,depth: (lo,hi,step)},
    input_size (H_in, W_in), downsample, in_channels, out_channels,
    accelerate, sid, collapse_z.

    Extra (not in the reference): `sync_free` -- when True the non-accelerated
    path never reads the point / interval counts back to the host (the default
    reads them AFTER the pooling has been queued, where the reference's
    boolean-mask indexing syncs before it); the only behavioural difference is
    that an input with no point inside the grid yields an all-zero volume of
    the regular shape instead of the reference's warning + dummy tensor
    (:179-189).

    Extra: `memory_format` -- torch.channels_last_3d makes every pooling route
    (fused geometry, voxel_pooling_v2, accelerate) return the same values stored
    channels-last, written that way by the pooling kernels (the layout a
    channels-last 3D encoder wants; its channels-last gradient is consumed
    without a copy).  The default, torch.contiguous_format, is the reference's.

    Extra: `dtype` -- torch.bfloat16 makes every pooling route return the
    volume in bfloat16 (the float32 volume rounded once, bit for bit, written
    so by the kernels; the layout a bfloat16 3D encoder under autocast wants),
    combined with either memory format.  Its bfloat16 gradient is read as it
    arrives; the depth / feature gradients stay float32.
    """

    def __init__(self, grid_config, input_size, downsample=16, in_channels=512,
                 out_channels=64, accelerate=False, sid=False, collapse_z=True,
                 sync_free=False, rank_cache=0, depth_eps=None,
                 memory_format=torch.contiguous_format, dtype=torch.float32):
        super().__init__()
        _bp._channels_last(memory_format)     # ValueError for anything but the two formats
        _bp._bf16(dtype)                      # ValueError for anything but float32 / bfloat16
        self.memory_format = memory_format
        self.dtype = dtype
        self.grid_config = grid_config
        self.downsample = downsample
        self.create_grid_infos(**grid_config)
        self.sid = sid
        self.frustum = self.create_frustum(grid_config["depth"], input_size, downsample)
        self.out_channels = out_channels
        self.in_channels = in_channels
        # the reference's 1x1 depth/context head (:59-60); a library conv, kept
        # so that `forward` is a complete drop-in
        self.depth_net = nn.Conv2d(in_channels, self.D + self.out_channels, kernel_size=1)
        self.accelerate = accelerate
        self.initial_flag = True
        self.collapse_z = collapse_z
        self.sync_free = sync_free
        # Optional callable (not in the reference), invoked on the host right after the
        # index-preparation kernels of a call have been queued and before the pooling
        # kernels.  A pipelined caller uses it to release its bulk host<->device copies
        # there: the dozen short launches before this point are latency-bound and measurably
        # slower while PCIe is saturated (command fetch shares the link), the long pooling
        # kernels after it are not (bench.py, tools/e2e_timeline.py).
        self.prepared_hook = None
        # Extra (not in the reference): fold get_lidar_coor into the index preparation inside
        # view_transform (SURVEY 8f-3).  Same float operations in the same order, so the pooled
        # volume is the same bits; set False to run the two steps separately.
        self.fuse_geometry = True
        # Extra (not in the reference), SURVEY 8f-3: keep the prepared ranks of the last
        # `rank_cache` distinct calibrations, keyed by a 64-bit hash of the calibration tensors'
        # bits (one tiny kernel + an 8-byte read instead of the whole index preparation).  It
        # generalises `accelerate` (:154-173), which caches ONE rig for ever.  0 = off.
        self.rank_cache = int(rank_cache)
        self._rank_cache = {}
        self.rank_cache_hits = self.rank_cache_misses = 0
        # Extra (not in the reference), SURVEY 8f-2, INFERENCE only: drop the points whose depth
        # weight is <= depth_eps before they are ranked (VEON's two-hot depth leaves ~90 % of
        # the bins at the e^-16 clamp).  Ignored whenever a gradient is wanted; None = exact.
        self.depth_eps = depth_eps

    # -- a1 ------------------------------------------------------------------
    def create_grid_infos(self, x, y, z, **kwargs):
        """float32 grid vectors exactly as the reference builds them (:66-82):
        python-float arithmetic, then a float32 tensor."""
        axes = (x, y, z)
        self.grid_lower_bound = torch.tensor([a[0] for a in axes], dtype=torch.float32)
        self.grid_interval = torch.tensor([a[2] for a in axes], dtype=torch.float32)
        self.grid_size = torch.tensor([(a[1] - a[0]) / a[2] for a in axes],
                                      dtype=torch.float32)

    def create_frustum(self, depth_cfg, input_size, downsample):
        """[D,H,W,3] frustum of (x_img, y_img, depth) (reference :84-112)."""
        h_in, w_in = input_size
        h, w = h_in // downsample, w_in // downsample
        depth = torch.arange(*depth_cfg, dtype=torch.float)
        self.D = depth.numel()
        if self.sid:
            lo = torch.tensor(float(depth_cfg[0]))
            hi = torch.tensor(float(depth_cfg[1]))
            idx = torch.arange(self.D).float()
            depth = torch.exp(torch.log(lo) + idx / (self.D - 1) * torch.log((hi - 1) / lo))
        xs = torch.linspace(0, w_in - 1, w, dtype=torch.float)
        ys = torch.linspace(0, h_in - 1, h, dtype=torch.float)
        fr = torch.empty(self.D, h, w, 3, dtype=torch.float)
        fr[..., 0] = xs.view(1, 1, w)
        fr[..., 1] = ys.view(1, h, 1)
        fr[..., 2] = depth.view(self.D, 1, 1)
        return fr

    # -- a2 ------------------------------------------------------------------
    def get_lidar_coor(self, sensor2ego, ego2global, cam2imgs, post_rots, post_trans, bda):
        """Frustum points in the ego/lidar frame, [B,N,D,H,W,3]
        (reference :114-152; same operation order so that float32 results
        agree to rounding): undo image augmentation, un-project with depth,
        camera->ego, BEV augmentation."""
        return _bp.lidar_coor(self._frustum_on(sensor2ego.device), sensor2ego, cam2imgs,
                              post_rots, post_trans, bda)

    def _frustum_on(self, device):
        cache = self.__dict__.setdefault("_frustum_cache", {})
        if device not in cache:
            cache[device] = self.frustum.to(device).contiguous()
        return cache[device]

    # -- a3 ------------------------------------------------------------------
    def voxel_pooling_prepare_v2(self, coor):
        """(ranks_bev, ranks_depth, ranks_feat, interval_starts,
        interval_lengths) or five Nones -- reference :202-260."""
        return _bp.voxel_pooling_prepare_v2(coor, self.grid_lower_bound, self.grid_interval,
                                            self.grid_size)

    def init_acceleration_v2(self, coor):
        """Cache the ranks for constant calibration (reference :154-173)."""
        ranks_bev, ranks_depth, ranks_feat, interval_starts, interval_lengths = \
            self.voxel_pooling_prepare_v2(coor)
        self.ranks_bev = ranks_bev.int().contiguous()
        self.ranks_feat = ranks_feat.int().contiguous()
        self.ranks_depth = ranks_depth.int().contiguous()
        self.interval_starts = interval_starts.int().contiguous()
        self.interval_lengths = interval_lengths.int().contiguous()

    def _bev_shape(self, depth, channels):
        zyx = self.__dict__.get("_zyx")
        if zyx is None or zyx[0] is not self.grid_size:   # cached: three .item() calls
            gs = self.grid_size
            zyx = self.__dict__["_zyx"] = (gs, int(gs[2]), int(gs[1]), int(gs[0]))
        return (depth.shape[0], zyx[1], zyx[2], zyx[3], channels)  # B,Z,Y,X,C

    # -- a4 ------------------------------------------------------------------
    def voxel_pooling_v2(self, coor, depth, feat):
        """coor [B,N,D,H,W,3], depth [B,N,D,H,W], feat [B,N,C,H,W] ->
        [B,C,Z,Y,X] (or [B,C*Z,Y,X] with collapse_z) -- reference :175-200."""
        if coor.numel() == 0:
            return self._no_points_dummy(feat)
        prep = self._take_prefetched(coor)
        if prep is None:
            prep = _bp.prepare_ranks(coor, self.grid_lower_bound, self.grid_interval,
                                     self.grid_size)
        return self._pool_prepared(prep, depth, feat)

    # -- pipelined index preparation ----------------------------------------------------------
    def prefetch_ranks(self, coor):
        """Queue `voxel_pooling_prepare_v2(coor)` on a side stream, behind everything the caller
        has launched so far on the current stream; the next `voxel_pooling_v2(coor, ...)` with
        this very tensor picks the ranks up instead of preparing them.  The preparation depends
        on the geometry only, so a loop can prepare step i+1 while the backward of step i runs
        (call this between the forward and the backward): its dozen short, latency-bound
        launches then cost nothing on the critical path."""
        if not coor.is_cuda or coor.numel() == 0:
            return
        dev = coor.device
        streams = self.__dict__.setdefault("_prep_streams", {})
        side = streams.get(dev)
        if side is None:
            side = streams[dev] = torch.cuda.Stream(dev)
        here = torch.cuda.Event()
        here.record(torch.cuda.current_stream(dev))
        side.wait_event(here)
        # launched on the side stream, allocated in the current stream's pool (where the ranks
        # are consumed): no allocator traffic between the two streams
        prep = _bp.prepare_ranks(coor, self.grid_lower_bound, self.grid_interval, self.grid_size,
                                 stream=side)
        self.__dict__["_prefetched"] = (coor, coor._version, prep, prep.plan.counts_event)

    def _take_prefetched(self, coor):
        pf = self.__dict__.get("_prefetched")
        if pf is None:
            return None
        self.__dict__["_prefetched"] = None
        if pf[0] is not coor or pf[1] != coor._version:
            return None                      # another tensor (or modified since): prepare afresh
        torch.cuda.current_stream(coor.device).wait_event(pf[3])   # the side stream's kernels are done
        return pf[2]

    def _voxel_pooling_calib(self, calib, depth, feat):
        """voxel_pooling_v2 with get_lidar_coor folded into the index preparation (SURVEY 8f-3):
        `calib` = the six tensors get_lidar_coor takes; no coordinate tensor is written."""
        wants_grad = torch.is_grad_enabled() and (depth.requires_grad or feat.requires_grad)
        return self._pool_prepared(self._prepare_calib(calib, depth, wants_grad), depth, feat)

    def _prepare_calib(self, calib, depth, wants_grad=False, backward_tables=True):
        """The prepared ranks + plan for a calibration (fused geometry; rank cache / negligible
        depth bins when configured).  backward_tables=False: inference, the backward's point ->
        interval table is not built (never combined with the rank cache, whose entries may
        serve a training step later)."""
        sensor2ego, _ego2global, cam2imgs, post_rots, post_trans, bda = calib
        frustum = self._frustum_on(sensor2ego.device)
        grid = (self.grid_lower_bound, self.grid_interval, self.grid_size)
        if self.depth_eps is not None and not wants_grad:
            # depth-dependent ranks: nothing to cache
            prep = _bp.prepare_ranks_calib(frustum, sensor2ego, cam2imgs, post_rots, post_trans,
                                           bda, *grid, depth=depth, depth_eps=self.depth_eps)
        elif self.rank_cache > 0:
            key = (_bp.calib_hash(sensor2ego, cam2imgs, post_rots, post_trans, bda),
                   tuple(depth.shape), sensor2ego.device.index)
            prep = self._rank_cache.pop(key, None)
            if prep is None:
                self.rank_cache_misses += 1
                prep = _bp.prepare_ranks_calib(frustum, sensor2ego, cam2imgs, post_rots,
                                               post_trans, bda, *grid)
            else:
                self.rank_cache_hits += 1
            self._rank_cache[key] = prep                      # most recently used last
            while len(self._rank_cache) > self.rank_cache:
                self._rank_cache.pop(next(iter(self._rank_cache)))
        else:
            prep = _bp.prepare_ranks_calib(frustum, sensor2ego, cam2imgs, post_rots, post_trans,
                                           bda, *grid, backward_tables=backward_tables)
        return prep

    def lift_labels_calib(self, calib, depth, pix, Q, prompt_class, free_label=17):
        """Fused lift + classify of per-pixel rows `pix` [B,N,Cp,H,W] = [gate 0, gate 1,
        logit 0..Q-1, padding] (veon_b200.pipeline.lift_classify): uint8 labels [B,X,Y,Z], or None
        when the fused kernel does not take the shape.  Inference only."""
        with torch.no_grad():
            prep = self._prepared(self._prepare_calib(calib, depth, backward_tables=False))
            gs = self.grid_size
            return _bp.lift_classify_prepared(depth, pix, prep, Q, prompt_class,
                                              (int(gs[2]), int(gs[1]), int(gs[0])), free_label)

    def _prepared(self, prep):
        """A freshly prepared rank set on its way to the pooling kernels: a sync-free plan's
        backward sizes its scratch by a bound; `prepared_hook` (see __init__) runs here."""
        prep.plan.sync_free = self.sync_free
        if self.prepared_hook is not None:
            self.prepared_hook()
        return prep

    def _no_points(self, prep):
        """The reference's empty-input case: no interval at all.  Read back after the pooling
        has been queued, so the host read-back (the reference syncs at the same place in its
        boolean-mask indexing) overlaps the forward kernel; never asked when sync_free."""
        return not self.sync_free and prep.plan.n_intervals == 0

    def _pool_prepared(self, prep, depth, feat):
        feat_last = feat.permute(0, 1, 3, 4, 2)
        shape = self._bev_shape(depth, feat_last.shape[-1])
        bev_feat = _bp.pool_prepared(depth, feat_last, self._prepared(prep), shape,
                                     self.memory_format, dtype=self.dtype)
        if self._no_points(prep):
            return self._no_points_dummy(feat)
        if self.collapse_z:
            bev_feat = torch.cat(bev_feat.unbind(dim=2), 1)
        return bev_feat

    def _no_points_dummy(self, feat):
        """reference :179-189 (note its X/Y order and that Z is always collapsed)"""
        print("warning ---> no points within the predefined bev receptive field")
        gs = self.grid_size
        dummy = torch.zeros(size=[feat.shape[0], feat.shape[2], int(gs[2]), int(gs[0]),
                                  int(gs[1])]).to(feat)
        if self.dtype is torch.bfloat16:
            dummy = dummy.to(torch.bfloat16)
        return torch.cat(dummy.unbind(dim=2), 1)

    # -- a10 -----------------------------------------------------------------
    def pre_compute(self, input):
        if self.initial_flag:
            coor = self.get_lidar_coor(*input[1:7])
            self.init_acceleration_v2(coor)
            self.initial_flag = False

    def view_transform_core(self, input, depth, tran_feat):
        """reference :268-290"""
        B, N, C, H, W = input[0].shape
        if self.accelerate:
            feat = tran_feat.view(B, N, self.out_channels, H, W).permute(0, 1, 3, 4, 2)
            depth = depth.view(B, N, self.D, H, W)
            bev_feat = _bp.bev_pool_v2(depth, feat, self.ranks_depth, self.ranks_feat,
                                       self.ranks_bev, self._bev_shape(depth, feat.shape[-1]),
                                       self.interval_starts, self.interval_lengths,
                                       memory_format=self.memory_format, dtype=self.dtype)
            bev_feat = bev_feat.squeeze(2)
        elif self.fuse_geometry and input[1].is_cuda:
            # get_lidar_coor folded into the index preparation: same ranks, no coor tensor
            bev_feat = self._voxel_pooling_calib(input[1:7], depth.view(B, N, self.D, H, W),
                                                 tran_feat.view(B, N, self.out_channels, H, W))
        else:
            coor = self.get_lidar_coor(*input[1:7])
            bev_feat = self.voxel_pooling_v2(coor, depth.view(B, N, self.D, H, W),
                                             tran_feat.view(B, N, self.out_channels, H, W))
        return bev_feat, depth

    def view_transform(self, input, depth, tran_feat):
        if self.accelerate:
            self.pre_compute(input)
        return self.view_transform_core(input, depth, tran_feat)

    def forward(self, input):
        """input = (img_feat [B,N,C_in,H,W], sensor2ego, ego2global, cam2imgs,
        post_rots, post_trans, bda) -> (bev_feat, depth) -- reference :297-319."""
        x = input[0]
        B, N, C, H, W = x.shape
        x = self.depth_net(x.view(B * N, C, H, W))
        depth = x[:, :self.D].softmax(dim=1)
        tran_feat = x[:, self.D:self.D + self.out_channels]
        return self.view_transform(input, depth, tran_feat)


class LSSViewTransformerRaw(LSSViewTransformer):
    """VEON's neck entry (reference view_transformer_raw.py:537-555): takes
    ready-made features and a depth distribution, lifts, then (use_ds)
    max-pools the volume 2x2x2.  With memory_format=torch.channels_last_3d it
    pools channels-last and reduces with the channels-last 2x2x2 kernels (the
    one-node PoolMaxDown training route is channels-first only and is not
    taken); the result is channels-last-3d.

    `dtype` (the pooled full-resolution volume) is float32 only: any other raises ValueError.

    Extra: `ds_dtype` -- the dtype of the 2x2x2-reduced output, torch.float32 (the default) or
    torch.bfloat16 (what a 3D decoder under bfloat16 autocast reads; needs use_ds).  With bfloat16:
    - a gradient wanted: the output is, bit for bit, the float32 neck's output cast to bfloat16,
      and the depth / feature gradients are the float32 neck's for the widened output gradient.
      The maximum and its first arg-max are taken over the float32 sums, as the reference's are
      under autocast.  Channels-first 2x2x2 takes the one-node PoolMaxDown route, which stores a
      bfloat16 result and reads its bfloat16 gradient in place; channels-last takes the float32
      route followed by a cast (which keeps the layout).
    - no gradient (2x2x2, even grid, fused geometry): the neck pools straight into a bfloat16
      volume (either layout) and takes the maximum in bfloat16, so no float32 full-resolution
      volume is written.  Rounding to nearest even is monotone, so every value equals the float32
      route cast (==), and so do the bits, except that a zero result may carry the other sign: a
      window whose float32 sums include a nonzero one of magnitude below 2^-134, which bfloat16
      rounds to a signed zero, may then return the zero of another element.  Which element is the arg-max is not observable without a gradient.
    - any other case (other `ds`, odd grids, `accelerate`, `collapse_z`, the empty-input dummy):
      the float32 route, then one cast."""

    def __init__(self, *args, use_ds=True, ds=(2, 2, 2), ds_dtype=torch.float32, **kwargs):
        if not isinstance(ds_dtype, torch.dtype) or ds_dtype not in _bp._DTYPES:
            raise ValueError(f"ds_dtype must be torch.float32 or torch.bfloat16, got {ds_dtype!r}")
        if ds_dtype is torch.bfloat16 and not use_ds:
            raise ValueError("ds_dtype=torch.bfloat16 is the dtype of the 2x2x2-reduced volume "
                             "and needs use_ds=True")
        kwargs.setdefault("collapse_z", False)
        super().__init__(*args, **kwargs)
        if self.dtype is not torch.float32:
            raise ValueError(f"LSSViewTransformerRaw is float32 only, got dtype={self.dtype!r}")
        self.ds_dtype = ds_dtype
        self.use_ds = use_ds
        self.ds = tuple(ds)

    # -- depth-distribution producer (SURVEY 8f-2) ------------------------------
    def downsample_depth(self, depths, downsample):
        """reference view_transformer_raw.py:393-404 (plain torch: it is only a helper of the
        autograd route below; the CUDA route fuses it)"""
        B, N, H, W = depths.shape
        d = depths.view(B * N, H // downsample, downsample, W // downsample, downsample)
        d = torch.where(d == 0.0, torch.full_like(d, 1e5), d)
        return d.amin(dim=(2, 4)).view(B, N, H // downsample, W // downsample)

    def get_two_hot_depth(self, depths, gamma=4, downsample=False):
        """reference view_transformer_raw.py:406-429: [B,N,H,W] metric depth -> [B,N,D,h,w]
        distribution.  One CUDA kernel when no gradient is wanted (`veon_two_hot_depth`);
        otherwise the reference's own expression, so that autograd sees the same graph."""
        if depths.is_cuda and not (torch.is_grad_enabled() and depths.requires_grad):
            return _bp.two_hot_depth(depths, self.grid_config["depth"], self.D, gamma,
                                     self.downsample if downsample else 0)
        if downsample:
            depths = self.downsample_depth(depths, self.downsample)
        B, N, H, W = depths.shape
        cfg = self.grid_config["depth"]
        centers = torch.arange(self.D + 1, device=depths.device) * cfg[2] + (cfg[0] + cfg[2] / 2)
        gap = -torch.abs(depths.reshape(B * N, H, W, 1) - centers) * gamma
        gap = torch.where(gap >= -16, gap, gap + (-16 - gap.detach()))
        dist = torch.softmax(gap, dim=-1)[..., :-1]
        return dist.view(B, N, H, W, self.D).permute(0, 1, 4, 2, 3)

    def forward(self, input, depth, stereo_metas=None):
        tran_feat = input[0]
        B, N, C, H, W = tran_feat.shape
        fused = None
        if self.ds_dtype is torch.bfloat16:
            fused = self._forward_bf16_inference(input, depth)
        if fused is None:
            fused = self._forward_pool_maxdown(input, depth)
        if fused is not None:
            return fused
        tran_feat = tran_feat.reshape(B * N, C, H, W)
        Bd, Nd, Dd, Hd, Wd = depth.shape
        depth = depth.reshape(Bd * Nd, Dd, Hd, Wd)
        bev_feat, _ = self.view_transform(input, depth, tran_feat)
        if self.use_ds:
            dz, dy, dx = self.ds
            b, c, z, y, x = bev_feat.shape
            if self.ds == (2, 2, 2) and _bp.MaxDown2x2x2.supports(bev_feat):
                bev_feat = _bp.MaxDown2x2x2.apply(bev_feat)      # same values, own kernels
            else:   # other factors / odd grids: the reference's expression (:549-553)
                bev_feat = bev_feat.view(b, c, z // dz, dz, y // dy, dy, x // dx, dx) \
                    .permute(0, 1, 2, 4, 6, 3, 5, 7).reshape(b, c, z // dz, y // dy, x // dx, -1)
                bev_feat = torch.max(bev_feat, dim=-1).values
        return bev_feat.to(self.ds_dtype)      # (float32: the tensor itself)

    def _forward_pool_maxdown(self, input, depth):
        """Training path: pooling and the 2x2x2 maximum as ONE autograd node whose backward never
        forms the full-resolution gradient (bev_pool.PoolMaxDown).  None -> plain route."""
        tran_feat = input[0]
        if (not self.use_ds or self.ds != (2, 2, 2) or self.accelerate or self.collapse_z
                or self.memory_format is not torch.contiguous_format
                or not tran_feat.is_cuda or not torch.is_grad_enabled()
                or not (tran_feat.requires_grad or depth.requires_grad)):
            return None
        B, N, C, H, W = tran_feat.shape
        sensor2ego, _e2g, cam2imgs, post_rots, post_trans, bda = input[1:7]
        prep = self._prepared(_bp.prepare_ranks_calib(
            self._frustum_on(sensor2ego.device), sensor2ego, cam2imgs, post_rots, post_trans, bda,
            self.grid_lower_bound, self.grid_interval, self.grid_size))
        feat_last = tran_feat.reshape(B, N, C, H, W).permute(0, 1, 3, 4, 2)
        d5 = depth.reshape(B, N, self.D, H, W)
        out = _bp.pool_prepared_maxdown(d5, feat_last, prep, self._bev_shape(d5, C),
                                        dtype=self.ds_dtype)
        # None also lets the plain route reproduce the reference's empty-input behaviour
        return None if out is None or self._no_points(prep) else out

    def _forward_bf16_inference(self, input, depth):
        """ds_dtype=bfloat16 without a gradient: pool into a bfloat16 volume in the neck's memory
        format and take the 2x2x2 maximum of it in bfloat16 (see the class docstring for what
        that returns).  Same ranks as the plain route (fused geometry, rank cache, depth_eps).
        None -> another route."""
        tran_feat = input[0]
        if (self.ds != (2, 2, 2) or self.accelerate or self.collapse_z or not self.fuse_geometry
                or not tran_feat.is_cuda or not input[1].is_cuda
                or (torch.is_grad_enabled() and (tran_feat.requires_grad or depth.requires_grad))):
            return None
        B, N, C, H, W = tran_feat.shape
        d5 = depth.reshape(B, N, self.D, H, W)
        shape = self._bev_shape(d5, C)
        _, Z, Y, X, _ = shape
        cl = self.memory_format is torch.channels_last_3d
        if (Z | Y) & 1 or X % (2 if cl else 4):     # what MaxDown2x2x2 takes
            return None
        feat_last = tran_feat.reshape(B, N, C, H, W).permute(0, 1, 3, 4, 2)
        prep = self._prepare_calib(input[1:7], d5)
        vol = _bp.pool_prepared(d5, feat_last, self._prepared(prep), shape, self.memory_format,
                                dtype=torch.bfloat16)
        # None also lets the plain route reproduce the reference's empty-input behaviour
        return None if self._no_points(prep) else _bp.MaxDown2x2x2.apply(vol)
