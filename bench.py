#!/usr/bin/env python
"""bench.py -- 6-camera samples/s of the lift (voxel_pooling_prepare_v2 +
bev_pool_v2 forward + backward) on N B200s, with the roofline of the dominant
kernel, the other BASELINE workloads, the reference's own CUDA kernels on the
same GPU and the CPU baseline beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of synthetic
nuScenes-shaped input: BASELINE.json configs[1] (6 cams 16x44 feats, D=88,
C=64, batch 8 per GPU; weak scaling: every rank lifts its own 8 samples, no
data-path collective).  Exactly K steps are timed after W warm-up steps
(--min-seconds S repeats the K-step region until S seconds of GPU time have
been measured and reports the median repeat).  Prints ONE JSON line on rank 0.

--dump-outputs DIR writes what the last timed step returned to its caller --
the pooled volume and the gradients of depth and features -- as float32 .npy
files (see dump_outputs); the inputs depend on the arguments only, so two
builds can be compared output for output.

Secondary objects of the line (all device-timed with CUDA events):
  workloads        C3 (C=512), C4 (C=768, D=118, B=16) lift fwd+bwd and the real VEON neck
                   (C=256, 32x88, two-hot depth, 2x2x2 max) -- N=1 only
  reference_cuda   the reference's own kernels (oracle/_ref, compiled unmodified) in the
                   reference's own flow (memset, permute, argsort) on the same inputs -- N=1 only
  pipeline         lift + classify (C3 geometry, Q=18 / Q=67) INCLUDING the NCCL all-gather of
                   the uint8 occupancy volumes on a side stream, per-GPU batch 8..64 -- every N
  tail, tail_lowres, downsample   as in round 1
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "6-cam samples/sec for lift (bev_pool_v2 fwd+bwd)"
UNIT = "samples/s"
KEYS = ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")
VOX = 640000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # 1300 C2 steps of 0.76 ms (one B200): the default timed region lasts about a second
    ap.add_argument("--steps", type=int, default=1300, help="timed steps K")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", help="veon_b200.synthetic.CONFIGS key")
    ap.add_argument("--batch", type=int, default=0, help="override samples per GPU per step")
    ap.add_argument("--cpu-seconds", type=float, default=15.0,
                    help="budget of the cpu_baseline leg (rank 0, N=1 only)")
    ap.add_argument("--min-seconds", type=float, default=0.0,
                    help="repeat the K-step region until this much GPU time is measured and "
                         "report the median (default 0: one region, exactly K timed steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="headline + e2e only (no workloads / comparator / pipeline / tail legs)")
    ap.add_argument("--host-sync", type=int, default=0,
                    help="1: read the point / interval counts back every step (the reference's "
                         "empty-input check); default 0 = LSSViewTransformer(sync_free=True)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy "
                         "(rank 0's outputs when several GPUs run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computes: it needs --impl ours")
    return args


DUMP_MAX_ELEMENTS = 4 << 20      # 16 MB of float32 per array, three arrays: under 64 MB in all


def dump_outputs(directory, arrays):
    """Writes each tensor of `arrays` as float32 `directory/<name>.npy`.  A tensor of more than
    DUMP_MAX_ELEMENTS elements is stored as `<name>_sample.npy`: its elements at a fixed set of
    flat indices (drawn with seed 0 from its size alone, sorted), so two runs of the same
    arguments store the same positions."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), DUMP_MAX_ELEMENTS))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
            name += "_sample"
        np.save(os.path.join(directory, name + ".npy"), t.float().cpu().numpy())


def workload_dict(cfg, batch, extra=None):
    H, W = cfg.feat_hw
    d = {"workload": f"{cfg.name}: {cfg.n_cams} cams {cfg.input_size[0]}x{cfg.input_size[1]} -> "
                     f"{H}x{W} feats, D={cfg.D}, C={cfg.channels} -> 200x200x16, "
                     f"prepare_v2 + bev_pool_v2 fwd + bwd",
         "samples_per_gpu_per_step": batch, "parallelism": "sample-sharded, no collective"}
    if extra:
        d.update(extra)
    return d


# ---------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi-equivalent (NVML) clock / throttle sampling during the timed region."""

    def __init__(self, index):
        self.samples, self.reasons = [], set()
        self._stop = threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) \
                    if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join(timeout=1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------ CPU baseline
def cpu_lift_once(cfg, batch, seed=0):
    """inputs for the CPU port (oracle.lift_oracle.torch_cpu_lift)"""
    import torch
    from veon_b200 import synthetic as S
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=batch, sample_offset=seed))
    B, N, D, H, W, _ = coor.shape
    g = torch.Generator().manual_seed(seed)
    depth = torch.softmax(torch.randn(B, N, D, H, W, generator=g) * 4, dim=2)
    feat = torch.randn(B, N, cfg.channels, H, W, generator=g)
    og = torch.randn(B, cfg.channels, 16, 200, 200, generator=g)
    return coor, depth, feat, og


def time_cpu_port(cfg, budget_s, steps=None, warmup=1, batch=1):
    """Times the reference's pure-PyTorch CPU lift (BASELINE.json configs[0]) as restated in
    oracle/ (kind "port").  Returns (samples/s, cores, description, ms per step)."""
    import torch
    from oracle import lift_oracle as O
    from veon_b200 import synthetic as S
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    lower, interval, size = S.grid_vectors(cfg.grid_config)
    coor, depth, feat, og = cpu_lift_once(cfg, batch)
    for _ in range(warmup):
        O.torch_cpu_lift(coor, depth, feat, lower, interval, size, og)
    times = []
    t_end = time.perf_counter() + budget_s
    while True:
        t0 = time.perf_counter()
        O.torch_cpu_lift(coor, depth, feat, lower, interval, size, og)
        times.append(time.perf_counter() - t0)
        if steps is not None and len(times) >= steps:
            break
        if steps is None and (time.perf_counter() > t_end and len(times) >= 3):
            break
    times.sort()
    med = times[len(times) // 2]
    desc = (f"{len(times)} timed passes (median) of prepare_v2 + scatter-add pool fwd + autograd bwd "
            f"on {batch} sample(s) of {cfg.name} (6 cams, D={cfg.D}, C={cfg.channels}), torch CPU fp32, "
            f"{cores} threads")
    return batch / med, cores, desc, med * 1e3, len(times)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; the
    reference is Python + CUDA, its CPU path is the pure-PyTorch lift of BASELINE configs[0])."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from veon_b200 import synthetic as S
    cfg = S.CONFIGS[args.workload]
    # each step = ONE sample of the workload (bounded so K steps end in minutes)
    val, cores, desc, ms, n = time_cpu_port(cfg, 0.0, steps=max(args.steps, 1),
                                            warmup=max(args.warmup, 1), batch=1)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": workload_dict(cfg, 1, {"note": "CPU port; one sample per step"}),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": desc},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------- ours
def algorithmic_bytes(cfg, B, n_kept, n_int, C=None):
    """SURVEY.md 8(d): compulsory traffic per step (every input element read once, every
    output element written once)."""
    C = cfg.channels if C is None else C
    H, W = cfg.feat_hw
    NHW = cfg.n_cams * H * W
    P = NHW * cfg.D * B
    fwd = 4 * VOX * C * B + 4 * NHW * C * B + 4 * n_kept + 8 * n_kept + 12 * n_int
    n_bp = NHW * B
    bwd = 4 * n_int * C + 4 * NHW * C * B + 4 * n_kept + 4 * P + 4 * NHW * C * B + 12 * n_kept + 8 * n_bp
    prep = 12 * P + 12 * n_kept + 8 * n_int
    return {"prepare": prep, "pool_fwd": fwd, "pool_bwd": bwd}


def numa_info(local):
    """NUMA placement of this rank's GPU.  Binding the rank's threads (and so, by first touch, its
    pinned buffers) to the GPU's node is attempted; on a single-node guest there is nothing to
    bind to and the reason is reported instead of a silent null."""
    info = {"node": None}
    try:
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")]
        info["host_nodes"] = len(nodes)
    except Exception:
        info["host_nodes"] = None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:          # nvml pads the PCI domain to 8 hex digits
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            info["why"] = "sysfs reports numa_node=-1 for the GPU (single-node guest): nothing to bind"
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        info["node"] = node
        info["cpus_bound"] = len(cpus)
    except Exception as e:   # noqa: BLE001
        info["why"] = f"{type(e).__name__}: {e}"
    return info


def reference_cuda_leg(cfg, B, dev, peak_gbs):
    """The GPU comparator SURVEY 8(d) asks for: the reference's OWN kernels (bev_pool_cuda.cu,
    compiled unmodified into oracle/_ref) driven by the reference's OWN operator file (memset
    :27, permute :91, argsort :47-57, contiguous :69) and the reference's own
    voxel_pooling_prepare_v2 (view_transformer.py:202-260), on the same C2 inputs, same GPU,
    CUDA events.  Comparator only: nothing of it is on the product path."""
    import torch
    so = os.path.join(ROOT, "oracle", "_ref", "libbev_pool_v2_ref.so")
    if not os.path.isfile(so):
        return {"unavailable": "oracle/_ref not built (make -C oracle ref)"}
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    try:
        from _ref_loader import (load_reference_bev_pool, load_reference_view_transformer,
                                 reference_available)
        if not reference_available():
            return {"unavailable": "reference python files not staged"}
        lib = ctypes.CDLL(so)
        fwd = getattr(lib, "_Z11bev_pool_v2iiPKfS0_PKiS2_S2_S2_S2_Pf")
        bwd = getattr(lib, "_Z16bev_pool_v2_gradiiPKfS0_S0_PKiS2_S2_S2_S2_PfS3_")
    except Exception as e:   # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}
    vp = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731

    # torch's default stream IS the legacy default stream the reference launches on
    def f_fwd(depth, feat, out, rd, rf, rb, ln, st):
        fwd(ctypes.c_int(feat.size(4)), ctypes.c_int(ln.size(0)), vp(depth), vp(feat), vp(rd),
            vp(rf), vp(rb), vp(st), vp(ln), vp(out))

    def f_bwd(og, dg, fg, depth, feat, rd, rf, rb, ln, st):
        bwd(ctypes.c_int(og.size(4)), ctypes.c_int(ln.size(0)), vp(og), vp(depth), vp(feat),
            vp(rd), vp(rf), vp(rb), vp(st), vp(ln), vp(dg), vp(fg))

    ext = types.SimpleNamespace(bev_pool_v2_forward=f_fwd, bev_pool_v2_backward=f_bwd)
    ref_op = load_reference_bev_pool(ext)
    ref_vt = load_reference_view_transformer(ref_op.bev_pool_v2)
    from veon_b200 import synthetic as S
    C = cfg.channels
    assert B * VOX * C < 2 ** 31, "the reference kernels index with 32-bit ints"
    neck = ref_vt.LSSViewTransformer(grid_config=cfg.grid_config, input_size=cfg.input_size,
                                     downsample=cfg.downsample, in_channels=8, out_channels=C,
                                     collapse_z=False)
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B)).to(dev)
    _, N, D, H, W, _ = coor.shape
    g = torch.Generator(device=dev).manual_seed(99)
    depth = torch.softmax(torch.randn(B, N, D, H, W, device=dev, generator=g) * 4, dim=2)
    feat = torch.randn(B, N, H, W, C, device=dev, generator=g)
    og = torch.randn(B, C, 16, 200, 200, device=dev, generator=g)
    shape = (B, 16, 200, 200, C)

    def ev():
        return torch.cuda.Event(enable_timing=True)
    n, warm = 10, 3
    tp, tf, tb = [], [], []
    for i in range(n + warm):
        e = [ev() for _ in range(4)]
        e[0].record()
        rb, rd, rf, st, ln = neck.voxel_pooling_prepare_v2(coor)
        e[1].record()
        d = depth.detach().requires_grad_()
        f = feat.detach().requires_grad_()
        out = ref_op.bev_pool_v2(d, f, rd, rf, rb, shape, st, ln)
        e[2].record()
        out.backward(og)
        e[3].record()
        torch.cuda.synchronize()
        if i >= warm:
            tp.append(e[0].elapsed_time(e[1]))
            tf.append(e[1].elapsed_time(e[2]))
            tb.append(e[2].elapsed_time(e[3]))
        del out, d, f
    med = lambda v: sorted(v)[len(v) // 2]   # noqa: E731
    alg = algorithmic_bytes(cfg, B, int(rb.numel()), int(st.numel()))
    res = {"what": "reference voxel_pooling_prepare_v2 (ATen ops) + reference QuickCumsumCuda / "
                   "bev_pool_v2 (its memset, permute, argsort, contiguous) on the reference's own "
                   "kernels compiled unmodified for sm_100a; same inputs, same GPU, CUDA events, "
                   f"median of {n}",
           "samples_per_call": B,
           "prepare_ms": med(tp), "pool_fwd_ms": med(tf), "pool_bwd_ms": med(tb),
           "step_ms": med(tp) + med(tf) + med(tb),
           "samples_per_s": B / ((med(tp) + med(tf) + med(tb)) * 1e-3),
           "fwd_gbs_algorithmic": alg["pool_fwd"] / (med(tf) * 1e-3) / 1e9,
           "bwd_gbs_algorithmic": alg["pool_bwd"] / (med(tb) * 1e-3) / 1e9,
           "fwd_bwd_frac_of_hbm_peak": (alg["pool_fwd"] + alg["pool_bwd"]) /
                                       ((med(tf) + med(tb)) * 1e-3) / 1e9 / peak_gbs}
    del coor, depth, feat, og
    torch.cuda.empty_cache()
    return res


def lift_workload(name, cfg_name, B, C, dev, peak_gbs, raw_neck=False, n_min=6, seconds=0.4):
    """One of the other BASELINE workloads through the public neck API on device-resident
    inputs: whole-step samples/s + the per-call device times of prepare / forward / backward
    with their algorithmic GB/s and fraction of the measured HBM peak."""
    import torch
    from veon_b200 import bev_pool as BP, synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer, LSSViewTransformerRaw
    cfg = S.CONFIGS[cfg_name]
    H, W = cfg.feat_hw
    N, D = cfg.n_cams, cfg.D
    g = torch.Generator(device=dev).manual_seed(5)
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).to(dev) for k in KEYS]
    feat = torch.randn(B, N, C, H, W, device=dev, generator=g)
    if raw_neck:
        neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                     sync_free=True)
        metric = torch.from_numpy(S.metric_depth_np(cfg, batch=B)).to(dev)
        og = torch.randn(B, C, 8, 100, 100, device=dev, generator=g)
    else:
        neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                  collapse_z=False, sync_free=True)
        depth0 = torch.softmax(torch.randn(B, N, D, H, W, device=dev, generator=g) * 4, dim=2)
        og = torch.randn(B, C, 16, 200, 200, device=dev, generator=g)
    img = torch.zeros(B, N, 1, H, W, device=dev)

    def step():
        f = feat.detach().requires_grad_()
        if raw_neck:
            with torch.no_grad():   # the depth estimator is frozen in VEON: two-hot forward only
                d = neck.get_two_hot_depth(metric)
            d = d.requires_grad_()
            out = neck([f] + metas, d)
        else:
            d = depth0.detach().requires_grad_()
            out, _ = neck.view_transform([img] + metas, d.view(B * N, D, H, W),
                                         f.view(B * N, C, H, W))
        out.backward(og)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    step()
    e1.record()
    torch.cuda.synchronize()
    n = max(n_min, int(seconds * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(n):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / n
    BP.enable_kernel_timing(True)
    for _ in range(min(n, 10)):
        step()
    t = BP.kernel_timings_ms()
    BP.enable_kernel_timing(False)
    avg = {k: sum(v) / len(v) for k, v in t.items()}
    coor = neck.get_lidar_coor(*metas)
    prep = BP.prepare_ranks(coor, neck.grid_lower_bound, neck.grid_interval, neck.grid_size)
    n_kept, n_int = prep.plan.n_points, prep.plan.n_intervals
    del coor, prep
    alg = algorithmic_bytes(cfg, B, n_kept, n_int, C)
    fwd_ms = avg.get("pool_fwd")
    bwd_ms = avg.get("pool_bwd", avg.get("pool_bwd_ds"))
    out = {"workload": name, "samples_per_call": B, "channels": C, "D": D, "feat_hw": [H, W],
           "ms_per_step": ms_step, "samples_per_s": B / (ms_step * 1e-3), "timed_steps": n,
           "n_kept": n_kept, "n_intervals": n_int,
           "phases_ms": {k: round(v, 4) for k, v in avg.items()}}
    if fwd_ms:
        out["fwd_gbs_algorithmic"] = alg["pool_fwd"] / (fwd_ms * 1e-3) / 1e9
        out["fwd_frac_of_hbm_peak"] = out["fwd_gbs_algorithmic"] / peak_gbs
    if bwd_ms and not raw_neck:
        out["bwd_gbs_algorithmic"] = alg["pool_bwd"] / (bwd_ms * 1e-3) / 1e9
        out["bwd_frac_of_hbm_peak"] = out["bwd_gbs_algorithmic"] / peak_gbs
    if fwd_ms and bwd_ms and not raw_neck:
        out["fwd_bwd_frac_of_hbm_peak"] = (alg["pool_fwd"] + alg["pool_bwd"]) / \
            ((fwd_ms + bwd_ms) * 1e-3) / 1e9 / peak_gbs
    if raw_neck:
        out["note"] = ("LSSViewTransformerRaw training step: two-hot depth producer (no grad) + "
                       "geometry + prepare + pool + 2x2x2 max as one autograd node + backward from "
                       "the [B,C,8,100,100] gradient; the forward fraction counts the full-"
                       "resolution volume the pooling kernel writes")
    del feat, og, neck
    torch.cuda.empty_cache()
    return out


def pipeline_leg(dev, world, rank, peak_gbs, batches=(8, 16, 32, 64), Qs=(18, 67)):
    """BASELINE configs[2] + [4]: lift + classify on C3 geometry (C=512 image features, Q prompt
    rows) with the NCCL all-gather of the finished uint8 occupancy volumes on a side stream
    (it overlaps the next step's compute), per-GPU batch swept.  Gathered volumes are verified
    once against the local ones outside the timed region."""
    import torch
    import torch.distributed as dist
    from veon_b200 import synthetic as S
    from veon_b200.dist import all_gather_occupancy, reserve_sms
    from veon_b200.pipeline import lift_classify
    from veon_b200.tail import class_of_prompt
    from veon_b200.view_transformer import LSSViewTransformer
    SIZES = [16, 1, 1, 1, 8, 1, 1, 3, 1, 1, 1, 1, 5, 3, 5, 13, 4]   # nuscenes_brief prompts per class
    c3 = S.CONFIGS["C3"]
    Ct, N, D = 512, c3.n_cams, c3.D
    H, W = c3.feat_hw
    neck = LSSViewTransformer(c3.grid_config, c3.input_size, c3.downsample, 8, Ct, collapse_z=False,
                              sync_free=True)
    side = torch.cuda.Stream(dev)
    rows = []
    g = torch.Generator(device=dev).manual_seed(11 + rank)
    # with a collective running beside the path, leave it a few SMs: the persistent grids would
    # otherwise make its CTAs wait for a kernel boundary (veon_reserve_sms; 8 GPUs, 8 samples per
    # step: 0.773 -> 0.751 ms)
    reserved = 16 if world > 1 else 0
    reserve_sms(reserved)
    for Q in Qs:
        refl = list(range(Q - 1)) if Q == 18 else [k for k, n in enumerate(SIZES) for _ in range(n)]
        cls_t = class_of_prompt(refl).to(dev)
        wt = torch.randn(Q, Ct, device=dev, generator=g)
        wt = 100.0 * wt / wt.norm(dim=1, keepdim=True)
        gate_w = torch.randn(2, Ct, device=dev, generator=g)
        for Bp in (batches if Q == 18 else batches[:1]):
            cal = S.calibration(c3, batch=min(Bp, 8), sample_offset=rank * 1000)
            metas = [torch.from_numpy(cal[k]).to(dev) for k in KEYS]
            if Bp > 8:   # repeat the 8 calibrated rigs (the index preparation still runs per sample)
                metas = [m.repeat((Bp // 8,) + (1,) * (m.dim() - 1)) for m in metas]
            depth = torch.softmax(torch.randn(Bp * N, D, H, W, device=dev, generator=g) * 4, 1)
            feat = torch.randn(Bp * N, Ct, H, W, device=dev, generator=g) * 0.05
            img = torch.zeros(Bp, N, 1, H, W, device=dev)
            n_total = Bp * world
            # one call lifts at most 16 samples: the reference's float32 voxel rank is exact only
            # while B * 640 000 < 2^24 (B <= 26, SURVEY 7), so larger batches go in chunks
            CH = 16

            def one():
                if Bp <= CH:
                    return lift_classify(neck, [img] + metas, depth, feat, wt, cls_t, gate_w)
                labs = []
                for b0 in range(0, Bp, CH):
                    sl = slice(b0, b0 + CH)
                    labs.append(lift_classify(neck, [img[sl]] + [m[sl] for m in metas],
                                              depth[b0 * N:(b0 + CH) * N], feat[b0 * N:(b0 + CH) * N],
                                              wt, cls_t, gate_w))
                return torch.cat(labs, 0)

            def gather(lab):
                # sample i -> rank i mod world (veon_b200.dist.shard_samples); the gathered buffer
                # stays rank-major (the reference's collector orders its results on the host too)
                return all_gather_occupancy(lab, n_total, sample_order=False) if world > 1 else lab
            # correctness of the collective, outside the timed region: this rank's block of the
            # rank-major buffer, and the sample-ordered form against it
            lab = one()
            allv = gather(lab)
            torch.cuda.synchronize()
            ok = True
            if world > 1:
                ok = bool(torch.equal(allv[rank * Bp:(rank + 1) * Bp], lab)) and \
                    bool(torch.equal(all_gather_occupancy(lab, n_total)[rank::world], lab))
            # the all-gather alone
            ag_us = None
            if world > 1:
                dist.barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(10):
                    gather(lab)
                b.record()
                torch.cuda.synchronize()
                ag_us = a.elapsed_time(b) * 100.0
            main = torch.cuda.current_stream(dev)
            for _ in range(3):                 # warm-up of the whole loop, side stream included
                lab = one()
                done = torch.cuda.Event()
                done.record(main)
                with torch.cuda.stream(side):
                    side.wait_event(done)
                    lab.record_stream(side)
                    allv = gather(lab)
            main.wait_stream(side)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            def timed(steps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    lab = one()
                    done = torch.cuda.Event()
                    done.record(main)
                    with torch.cuda.stream(side):
                        side.wait_event(done)
                        lab.record_stream(side)
                        gather(lab)
                main.wait_stream(side)
                e1.record()
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                return float(t.item())
            ms = timed(10)
            steps = max(10, min(400, int(300.0 / max(ms, 1e-3))))     # ~0.3 s per row
            ms = timed(steps)
            rows.append({"Q": Q, "samples_per_gpu_per_step": Bp, "ms_per_step": ms, "timed_steps": steps,
                         "samples_per_s": n_total / (ms * 1e-3),
                         "all_gather_us": ag_us, "gathered_bytes": n_total * VOX,
                         "gather_verified": ok})
            del depth, feat, img, metas
            torch.cuda.empty_cache()
    reserve_sms(0)
    # ---- a static rig: the calibration-keyed rank cache (SURVEY 8f-3) skips the index preparation
    static_row = None
    if rank == 0 or world > 1:
        Q, Bp = 18, 8
        neck_c = LSSViewTransformer(c3.grid_config, c3.input_size, c3.downsample, 8, Ct,
                                    collapse_z=False, sync_free=True, rank_cache=2)
        cls_t = class_of_prompt(list(range(Q - 1))).to(dev)
        wt = torch.randn(Q, Ct, device=dev, generator=g)
        wt = 100.0 * wt / wt.norm(dim=1, keepdim=True)
        gate_w = torch.randn(2, Ct, device=dev, generator=g)
        cal = S.calibration(c3, batch=Bp, sample_offset=rank * 1000)
        metas = [torch.from_numpy(cal[k]).to(dev) for k in KEYS]
        depth = torch.softmax(torch.randn(Bp * N, D, H, W, device=dev, generator=g) * 4, 1)
        feat = torch.randn(Bp * N, Ct, H, W, device=dev, generator=g) * 0.05
        img = torch.zeros(Bp, N, 1, H, W, device=dev)
        want = lift_classify(neck, [img] + metas, depth, feat, wt, cls_t, gate_w)
        for _ in range(3):
            got = lift_classify(neck_c, [img] + metas, depth, feat, wt, cls_t, gate_w)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(200):
            lift_classify(neck_c, [img] + metas, depth, feat, wt, cls_t, gate_w)
        e1.record()
        torch.cuda.synchronize()
        ms_c = e0.elapsed_time(e1) / 200
        static_row = {"what": "the same step on a static rig: LSSViewTransformer(rank_cache=2) finds the "
                              "calibration's ranks by its device-side hash and skips the preparation",
                      "Q": Q, "samples_per_gpu_per_step": Bp, "ms_per_step": ms_c,
                      "samples_per_s_per_gpu": Bp / (ms_c * 1e-3),
                      "cache_hits": neck_c.rank_cache_hits, "cache_misses": neck_c.rank_cache_misses,
                      "labels_equal_uncached": bool(torch.equal(got, want))}
        del depth, feat, img, metas
    sharded = None
    if world > 1:
        # ---- fewer samples than GPUs (SURVEY 8e): the CAMERAS of every sample are dealt over the
        # ranks, one NCCL all-reduce sums the [B,Q+2,Z,Y,X] logit volumes, everyone classifies
        from veon_b200.dist import lift_classify_camera_sharded
        Bc, Q = 2, 18
        gs = torch.Generator(device=dev).manual_seed(77)            # the SAME inputs on every rank
        cls_t = class_of_prompt(list(range(Q - 1))).to(dev)
        wt = torch.randn(Q, Ct, device=dev, generator=gs)
        wt = 100.0 * wt / wt.norm(dim=1, keepdim=True)
        gate_w = torch.randn(2, Ct, device=dev, generator=gs)
        cal = S.calibration(c3, batch=Bc, sample_offset=5000)
        metas = [torch.from_numpy(cal[k]).to(dev) for k in KEYS]
        depth = torch.softmax(torch.randn(Bc * N, D, H, W, device=dev, generator=gs) * 4, 1)
        feat = torch.randn(Bc * N, Ct, H, W, device=dev, generator=gs) * 0.05
        img = torch.zeros(Bc, N, 1, H, W, device=dev)

        def one_sharded():
            return lift_classify_camera_sharded(neck, [img] + metas, depth, feat, wt, cls_t, gate_w)
        lab = one_sharded()
        ref = lift_classify(neck, [img] + metas, depth, feat, wt, cls_t, gate_w)
        agree = float((lab == ref).float().mean())
        for _ in range(2):
            one_sharded()
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            one_sharded()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / 10], device=dev, dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        e0.record()
        for _ in range(10):
            lift_classify(neck, [img] + metas, depth, feat, wt, cls_t, gate_w)
        e1.record()
        torch.cuda.synchronize()
        sharded = {"what": f"camera-group sharding: {Bc} samples on {world} GPUs, each rank lifts the "
                           f"logits of its cameras (6 cameras dealt round-robin), one all-reduce of the "
                           f"[{Bc},20,16,200,200] volume ({Bc * 20 * VOX * 4 / 1e6:.0f} MB), classify",
                   "samples": Bc, "ms_per_step": float(ms.item()),
                   "samples_per_s": Bc / (float(ms.item()) * 1e-3),
                   "one_gpu_unsharded_ms": e0.elapsed_time(e1) / 10,
                   "labels_agree_with_unsharded": agree}
    return {"camera_sharded": sharded, "static_rig": static_row,
            "what": "lift_classify (C3 geometry: 6 cams 32x88, D=88, C=512 image features -> per-pixel "
                    "gate + logit rows on tcgen05 -> get_lidar_coor + prepare_v2 -> veon_lift_classify_fwd: "
                    "bev_pool_v2 of the Q+2 channels with merge/argmax/gate in the pooling kernel's "
                    "registers, the logit volume is never written -> uint8 [B,200,200,16]) + "
                    "all_gather_occupancy over NCCL on a side stream; weak scaling, samples dealt "
                    "round-robin (the gathered buffer stays rank-major, as the reference's collector "
                    "orders results on the host); max over ranks",
            "reserved_sms": reserved,
            "n_gpus": world, "rows": rows}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from veon_b200 import _lib, bev_pool as BP, synthetic as S
    from veon_b200.view_transformer import LSSViewTransformer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    numa = numa_info(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner to STDOUT when the first communicator comes up; the
        # contract is ONE JSON line there, so stdout points at stderr until that has happened
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.load()

    cfg = S.CONFIGS[args.workload]
    B = args.batch or cfg.batch
    C = cfg.channels
    sync_free = not bool(args.host_sync)
    neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, in_channels=8,
                              out_channels=C, collapse_z=False, sync_free=sync_free)
    lower, interval, size = S.grid_vectors(cfg.grid_config)

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback)"

    # rotating input sets so that a step's inputs are not L2-hot from the previous step
    n_sets = 4
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    host_sets, dev_sets = [], []
    for i in range(n_sets):
        coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B, sample_offset=rank * 1000 + i * B))
        Bc, N, D, H, W, _ = coor.shape
        depth = torch.softmax(torch.randn(B, N, D, H, W, device=dev, generator=g) * 4, dim=2)
        feat = torch.randn(B, N, C, H, W, device=dev, generator=g)
        host_sets.append((depth.cpu(), feat.cpu()))
        dev_sets.append((coor.to(dev), depth, feat))
    out_grad = torch.randn(B, C, 16, 200, 200, device=dev, generator=g)

    def step_device(i):
        coor, depth, feat = dev_sets[i % n_sets]
        depth = depth.detach().requires_grad_()
        feat = feat.detach().requires_grad_()
        bev = neck.voxel_pooling_v2(coor, depth, feat)
        bev.backward(out_grad)
        return bev, depth.grad, feat.grad

    # --dump-outputs: the outputs of the last step of the final timed region only, so that no
    # earlier region runs with a step's outputs held alive
    last, capture = {}, {"on": False}

    def step_headline(i):
        out = step_device(i)
        if capture["on"] and i == K - 1:
            last.update(zip(("bev", "depth_grad", "feat_grad"), out))

    def final_region_of_headline():
        capture["on"] = bool(args.dump_outputs) and rank == 0

    def step_device_lookahead(i):
        """The same step with the index preparation of step i+1 queued on the neck's side stream
        behind the forward of step i (LSSViewTransformer.prefetch_ranks): it depends on the
        geometry only, and its dozen short launches then overlap the backward."""
        coor, depth, feat = dev_sets[i % n_sets]
        depth = depth.detach().requires_grad_()
        feat = feat.detach().requires_grad_()
        bev = neck.voxel_pooling_v2(coor, depth, feat)
        neck.prefetch_ranks(dev_sets[(i + 1) % n_sets][0])
        bev.backward(out_grad)
        return depth.grad, feat.grad

    # ---- end to end: the user's call, view_transform(input, depth, tran_feat), on HOST data.
    # Per step ONE pinned buffer travels each way: [calibration | depth | feat] host -> device on a
    # copy stream (overlapped with the previous step's compute), get_lidar_coor + prepare + pool
    # forward + backward on device, [depth_grad | feat_grad] device -> host on a D2H stream.
    n_d, n_f = B * N * D * H * W, B * N * C * H * W
    e2e_host, meta_shapes, n_meta = [], None, 0
    for i in range(n_sets):
        cal = S.calibration(cfg, batch=B, sample_offset=rank * 1000 + i * B)
        parts = [torch.from_numpy(cal[k]).reshape(-1) for k in KEYS]
        meta_shapes = [tuple(cal[k].shape) for k in KEYS]
        hd, hf = host_sets[i]
        n_meta = (sum(p.numel() for p in parts) + 63) // 64 * 64      # keeps the pieces 256-B aligned
        packed = torch.zeros(n_meta + n_d + n_f, dtype=torch.float32)
        packed[:sum(p.numel() for p in parts)] = torch.cat(parts)
        packed[n_meta:n_meta + n_d] = hd.reshape(-1)
        packed[n_meta + n_d:] = hf.reshape(-1)
        e2e_host.append(packed.pin_memory())
    del host_sets

    def unpack(packed_dev):
        out, o = [], 0
        for shp in meta_shapes:
            n = 1
            for v in shp:
                n *= v
            out.append(packed_dev[o:o + n].view(shp))
            o += n
        depth = packed_dev[n_meta:n_meta + n_d].view(B * N, D, H, W)
        feat = packed_dev[n_meta + n_d:].view(B * N, C, H, W)
        return out, depth, feat

    img_shape = torch.zeros(B, N, 1, H, W, device=dev)      # only its shape is read
    copy_stream, d2h_stream = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    grad_host = [torch.empty(n_d + n_f, dtype=torch.float32).pin_memory() for _ in range(2)]
    grad_dev = [torch.empty(n_d + n_f, dtype=torch.float32, device=dev) for _ in range(2)]
    dev_in = [torch.empty_like(e2e_host[0], device=dev) for _ in range(2)]   # static staging

    def e2e_h2d(i, gate=None):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])          # the slot's previous user is done
            if gate is not None:
                copy_stream.wait_event(gate)
            dev_in[slot].copy_(e2e_host[i % n_sets], non_blocking=True)
            ready[slot].record(copy_stream)

    def e2e_d2h(slot, gate):
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(gate)
            grad_host[slot].copy_(grad_dev[slot], non_blocking=True)
            d2h_done[slot].record(d2h_stream)

    d2h_done = [torch.cuda.Event(), torch.cuda.Event()]

    def run_e2e(steps, compute=True):
        """Every step copies its inputs in and its gradients out.  The copies are queued from
        the neck's `prepared_hook`: H2D of step i+1 and D2H of step i-1 are released when the
        index preparation of step i is done, so they overlap the two long pooling kernels
        instead of the dozen short launches before them (those are measurably slower while
        PCIe is saturated; tools/e2e_timeline.py).  compute=False: the same copies with no
        kernels in between -- the ceiling the host side sets."""
        main = torch.cuda.current_stream(dev)
        for ev in consumed + d2h_done:
            ev.record(main)
        gate = torch.cuda.Event()
        state = {"i": 0, "pending": None}
        done = [torch.cuda.Event() for _ in range(4)]   # bounds the host's run-ahead to 2 steps

        def hook():
            gate.record(main)
            if state["i"] + 1 < steps:
                e2e_h2d(state["i"] + 1, gate)
            if state["pending"] is not None:
                e2e_d2h(state["pending"], gate)
                state["pending"] = None

        neck.prepared_hook = hook if compute else None
        try:
            e2e_h2d(0)
            for i in range(steps):
                slot = i % 2
                state["i"] = i
                if i >= 2:
                    done[(i - 2) % 4].synchronize()
                main.wait_event(ready[slot])
                main.wait_event(d2h_done[slot])        # grad_dev[slot] has left for the host
                if compute:
                    metas, depth, feat = unpack(dev_in[slot])
                    depth = depth.detach().requires_grad_()
                    feat = feat.detach().requires_grad_()
                    bev, _ = neck.view_transform([img_shape] + metas, depth, feat)
                    bev.backward(out_grad)
                    # one packed result buffer per step (two small device copies, one D2H)
                    grad_dev[slot][:n_d].copy_(depth.grad.reshape(-1))
                    grad_dev[slot][n_d:].copy_(feat.grad.reshape(-1))
                else:
                    hook()
                consumed[slot].record(main)
                done[i % 4].record(main)
                state["pending"] = slot
        finally:
            neck.prepared_hook = None
        gate.record(main)
        e2e_d2h(state["pending"], gate)
        main.wait_stream(d2h_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, whole_loop=False, min_seconds=0.0, max_repeats=400,
              before_final=None):
        """W warm-up steps, then the K-step region (barrier + synchronize on both sides, CUDA
        events, max over ranks), once or, with `min_seconds` > 0, repeated until that much GPU
        time: returns the MEDIAN region in ms, the launches of one region, the number of repeats
        and the total time.  `before_final` is called before the last region starts."""
        if whole_loop:
            fn(warmup)
        else:
            for i in range(warmup):
                fn(i)

        def region(final):
            barrier()
            if final and before_final is not None:
                before_final()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            l0 = lib.veon_kernel_launch_count()
            e0.record()
            if whole_loop:
                fn(steps)
            else:
                for i in range(steps):
                    fn(i)
            e1.record()
            barrier()
            launches = lib.veon_kernel_launch_count() - l0
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms.item()), launches
        ms0, launches = region(final=min_seconds <= 0)
        repeats = 1 if min_seconds <= 0 else \
            max(3, min(max_repeats, int(min_seconds * 1e3 / max(ms0, 1e-3)) + 1))
        if world > 1:      # every rank must run the same number of regions (collectives inside)
            r = torch.tensor([repeats], device=dev)
            dist.broadcast(r, 0)
            repeats = int(r.item())
        all_ms = [ms0] + [region(final=k == repeats - 2)[0] for k in range(repeats - 1)]
        s = sorted(all_ms)
        return s[len(s) // 2], launches, len(all_ms), sum(all_ms) * 1e-3, s[0], s[-1]

    K, Wm = args.steps, max(args.warmup, 3)
    with ClockSampler(local) as clocks:
        ms_total, launches, reps, total_s, ms_min, ms_max = timed(
            step_headline, K, Wm, min_seconds=args.min_seconds,
            before_final=final_region_of_headline)
        if last:
            dump_outputs(args.dump_outputs, last)
            last.clear()
        ms_look, _, reps_look, _, _, _ = timed(step_device_lookahead, K, Wm,
                                               min_seconds=args.min_seconds / 2)
    ms_e2e, _, reps_e2e, total_e2e, _, _ = timed(run_e2e, K, max(3, Wm // 2), whole_loop=True,
                                                 min_seconds=args.min_seconds / 2)
    ms_copy, _, _, _, _, _ = timed(lambda n: run_e2e(n, compute=False), K, 3, whole_loop=True,
                                   min_seconds=args.min_seconds)

    # live per-call device times (CUDA events on the launching stream) over K more steps
    BP.enable_kernel_timing(True)
    for i in range(K):
        step_device(i)
    t = BP.kernel_timings_ms()
    BP.enable_kernel_timing(False)
    avg = {k: sum(v) / len(v) for k, v in t.items()}

    # counts for the algorithmic-byte denominators
    prep = BP.prepare_ranks(dev_sets[0][0], lower, interval, size)
    n_kept, n_int = prep.plan.n_points, prep.plan.n_intervals
    del prep
    alg = algorithmic_bytes(cfg, B, n_kept, n_int)

    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            tj = json.load(f).get(args.workload, {})
            traffic = tj.get("pool_fwd_dram_bytes_per_launch")
            traffic_src = "static, from profiles/roofline_traffic.json (" + tj.get("source", "ncu --set full") + ")"
    except Exception:
        pass
    fwd_ms, bwd_ms = avg.get("pool_fwd"), avg.get("pool_bwd")
    achieved = alg["pool_fwd"] / (fwd_ms * 1e-3) / 1e9 if fwd_ms else None
    fb = (alg["pool_fwd"] + alg["pool_bwd"]) / ((fwd_ms + bwd_ms) * 1e-3) / 1e9 \
        if fwd_ms and bwd_ms else None

    value = world * B * K / (ms_total * 1e-3)
    e2e_value = world * B * K / (ms_e2e * 1e-3)
    h2d = e2e_host[0].numel() * 4
    d2h = grad_host[0].numel() * 4

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_dict(cfg, B, {
            "l2": f"inputs rotate over {n_sets} sets; each step streams a "
                  f"{4 * VOX * C * B / 1e9:.2f} GB volume (>> 126 MB L2)",
            "host_sync_per_step": 0 if sync_free else 1,
            "numa": numa,
            "n_kept": n_kept, "n_intervals": n_int}),
        "timing": {"what": (f"one {K}-step region " if reps == 1 else
                            f"median of {reps} repeats of the {K}-step region ") +
                           "(barrier + synchronize on both sides, CUDA events, max over ranks)",
                   "repeats": reps, "timed_region_s_total": round(total_s, 3),
                   "ms_per_step_min": ms_min / K, "ms_per_step_max": ms_max / K},
        "gpu_launches": int(launches),
        "lookahead": {"what": "the same K steps with the index preparation of step i+1 queued on a "
                              "side stream behind the forward of step i (prefetch_ranks): it depends "
                              "on the geometry only and overlaps the backward",
                      "value": world * B * K / (ms_look * 1e-3), "unit": UNIT,
                      "ms_per_step": ms_look / K, "repeats": reps_look},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / K,
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "repeats": reps_e2e, "timed_region_s_total": round(total_e2e, 3),
                "copies_only_samples_per_s": world * B * K / (ms_copy * 1e-3),
                "what": "ONE pinned buffer [calibration|depth|feat] host -> device, "
                        "LSSViewTransformer.view_transform (get_lidar_coor fused into prepare_v2, "
                        "bev_pool_v2) -> backward -> ONE pinned buffer [depth_grad|feat_grad] device -> "
                        "host; copies on side streams, double-buffered, released from the neck's "
                        "prepared_hook.  copies_only = the same transfers with no kernels between "
                        "them: the ceiling the host side (PCIe + pinned-memory bandwidth shared by "
                        "all ranks) sets"},
        "roofline": {"bound": "hbm",
                     "kernel": "veon_bev_pool_v2_fwd_planar: k_fwd_stream (role A rows -> L2 ring -> "
                               "role E dense volume) + k_pool_fwd_heavy queued behind it",
                     "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                     "frac": (achieved / peak_gbs) if achieved else None, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg["pool_fwd"],
                     "ms_per_launch": fwd_ms, "traffic": traffic, "traffic_source": traffic_src},
        "roofline_fwd_bwd": {
            "what": "north_star target quantity: bev_pool_v2 forward + backward, algorithmic bytes of "
                    "both over the sum of their device times, against the measured HBM copy peak",
            "achieved": fb, "peak": peak_gbs, "unit": "GB/s", "frac": (fb / peak_gbs) if fb else None,
            "algorithmic_bytes": alg["pool_fwd"] + alg["pool_bwd"],
            "ms": (fwd_ms + bwd_ms) if fwd_ms and bwd_ms else None},
        "phases_ms": {k: round(v, 4) for k, v in avg.items()},
        "phases_gbs_algorithmic": {
            k: round(alg[a] / (avg[k] * 1e-3) / 1e9, 1)
            for k, a in (("prepare_v2", "prepare"), ("pool_fwd", "pool_fwd"), ("pool_bwd", "pool_bwd"))
            if k in avg},
        "phases_frac_of_hbm_peak": {
            k: round(alg[a] / (avg[k] * 1e-3) / 1e9 / peak_gbs, 4)
            for k, a in (("prepare_v2", "prepare"), ("pool_fwd", "pool_fwd"), ("pool_bwd", "pool_bwd"))
            if k in avg},
        "clocks": clocks.summary(),
    }
    # free the headline buffers before the big secondary workloads
    del dev_sets, e2e_host, grad_host, grad_dev, dev_in
    torch.cuda.empty_cache()

    if not args.no_extras:
        # ---- the north-star pipeline with its one collective, at EVERY N
        line["pipeline"] = pipeline_leg(dev, world, rank, peak_gbs)
    if not args.no_extras and world == 1:
        # ---- the other BASELINE workloads (device-resident inputs, public neck API)
        line["workloads"] = [
            lift_workload("C3: VEON ViT-B CLIP-dim lift, C=512, batch 8", "C3", 8, 512, dev, peak_gbs),
            lift_workload("C4: VEON* ViT-L, 32x88 feats, D=118, C=768, batch 16", "C4", 16, 768,
                          dev, peak_gbs, n_min=3, seconds=0.3),
            lift_workload("VEON-real: LSSViewTransformerRaw, C=256, 32x88 feats, D=88, two-hot depth, "
                          "2x2x2 max, batch 4", "C3", 4, 256, dev, peak_gbs, raw_neck=True),
        ]
        # ---- the reference's own CUDA kernels and flow on this GPU
        rc = reference_cuda_leg(cfg, B, dev, peak_gbs)
        if "unavailable" not in rc:
            ours = {"prepare": avg.get("prepare_v2"), "pool_fwd": fwd_ms, "pool_bwd": bwd_ms}
            rc["speedup_vs_reference_cuda"] = {
                "prepare": rc["prepare_ms"] / ours["prepare"] if ours["prepare"] else None,
                "pool_fwd": rc["pool_fwd_ms"] / ours["pool_fwd"] if ours["pool_fwd"] else None,
                "pool_bwd": rc["pool_bwd_ms"] / ours["pool_bwd"] if ours["pool_bwd"] else None,
                "step": rc["step_ms"] / (ms_total / K)}
        line["reference_cuda"] = rc

        # ---- the open-vocabulary tail (tcgen05 3xTF32 logits + fused argmax): HBM-bound, 9 flop/B
        from veon_b200.tail import class_of_prompt, voxel_text_argmax, voxel_text_argmax_lowres
        Bt, Ct = 2, 512
        gt = torch.Generator(device=dev).manual_seed(7)
        feat_occ = torch.sigmoid(torch.randn(Bt, Ct, 16, 200, 200, device=dev, generator=gt)) - 0.5
        bin_occ = torch.randn(Bt, 2, 16, 200, 200, device=dev, generator=gt)

        def ev_ms(fn, seconds=0.3, n_min=10):
            for _ in range(3):
                fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            n = max(n_min, int(seconds * 1e3 / max(a.elapsed_time(b), 1e-3)))
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        def burst_ms(fn, n=20, idle_s=0.5):
            """n calls after an idle pause: the tail draws the board's whole power budget (~995 W),
            so a long back-to-back run is timed at the ~1.5 GHz the power cap leaves it"""
            fn()
            torch.cuda.synchronize()
            time.sleep(idle_s)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        SIZES = [16, 1, 1, 1, 8, 1, 1, 3, 1, 1, 1, 1, 5, 3, 5, 13, 4]
        line["tail"] = []
        for Qt in (18, 67):
            refl = list(range(Qt - 1)) if Qt == 18 else [k for k, n in enumerate(SIZES) for _ in range(n)]
            cls_t = class_of_prompt(refl).to(dev)
            wt = torch.randn(Qt, Ct, device=dev, generator=gt)
            wt = 100.0 * wt / wt.norm(dim=1, keepdim=True)
            ms_t = ev_ms(lambda: voxel_text_argmax(feat_occ, wt, cls_t, bin_occ))
            ms_tb = burst_ms(lambda: voxel_text_argmax(feat_occ, wt, cls_t, bin_occ))
            bytes_t = Bt * (4 * VOX * Ct + 8 * VOX + VOX) + 4 * Qt * Ct
            line["tail"].append({
                "what": f"veon_voxel_text_argmax, C={Ct}, Q={Qt} prompt rows, {Bt} samples/call, "
                        "3xTF32 tcgen05 + fused class-max/argmax/gate -> uint8 [B,200,200,16]",
                "samples_per_s_per_gpu": Bt / (ms_t * 1e-3), "ms_per_call": ms_t,
                "achieved_gbs_algorithmic": bytes_t / (ms_t * 1e-3) / 1e9,
                "frac_of_hbm_peak": bytes_t / (ms_t * 1e-3) / 1e9 / peak_gbs,
                "burst_ms_per_call": ms_tb,
                "burst_frac_of_hbm_peak": bytes_t / (ms_tb * 1e-3) / 1e9 / peak_gbs,
                "timing": "ms_per_call: 0.3 s back to back (sw_power_cap: ~995 W, SM clock ~1.5 GHz); "
                          "burst: 20 calls after 0.5 s idle (1.965 GHz)"})
        del feat_occ, bin_occ
        # the same tail from the decoder's resolution (SURVEY 8f-4)
        Bl, Qt = 8, 18
        cls_t = class_of_prompt(list(range(Qt - 1))).to(dev)
        wt = torch.randn(Qt, Ct, device=dev, generator=gt)
        wt = 100.0 * wt / wt.norm(dim=1, keepdim=True)
        feat_lr = torch.sigmoid(torch.randn(Bl, Ct, 8, 100, 100, device=dev, generator=gt)) - 0.5
        bin_lr = torch.randn(Bl, 2, 8, 100, 100, device=dev, generator=gt)
        ws_lr = torch.empty(Bl * Qt * 80000, dtype=torch.float32, device=dev)
        ms_l = ev_ms(lambda: voxel_text_argmax_lowres(feat_lr, wt, cls_t, bin_lr, workspace=ws_lr))
        bytes_l = Bl * (4 * 80000 * Ct + 8 * 80000 + VOX) + 4 * Qt * Ct
        line["tail_lowres"] = {
            "what": f"veon_voxel_text_argmax_lowres, C={Ct}, Q={Qt}, {Bl} samples/call, feat_occ "
                    "[B,C,8,100,100] -> logits (tcgen05 3xTF32) -> trilinear up-sampling of the Q "
                    "logits + class-max/argmax/gate -> uint8 [B,200,200,16]",
            "samples_per_s_per_gpu": Bl / (ms_l * 1e-3), "ms_per_call": ms_l,
            "achieved_gbs_algorithmic": bytes_l / (ms_l * 1e-3) / 1e9,
            "frac_of_hbm_peak": bytes_l / (ms_l * 1e-3) / 1e9 / peak_gbs}
        del feat_lr, bin_lr, ws_lr
        # the neck's 2x2x2 max-downsample of the pooled volume (SURVEY 8f-1)
        vol = out_grad.detach().clone().requires_grad_()
        go_ds = torch.randn(B, C, 8, 100, 100, device=dev, generator=gt)
        with torch.no_grad():
            ms_df = ev_ms(lambda: BP.MaxDown2x2x2.apply(vol))
        ms_dfb = ev_ms(lambda: torch.autograd.grad(BP.MaxDown2x2x2.apply(vol), vol, go_ds))
        vb = 4.0 * vol.numel()
        line["downsample"] = {
            "what": "2x2x2 max-downsample of the [B,C,16,200,200] volume "
                    "(view_transformer_raw.py:549-553) and its gradient (to the first arg-max), own kernels",
            "fwd_ms": ms_df, "fwd_gbs": 1.125 * vb / (ms_df * 1e-3) / 1e9,
            "bwd_ms": ms_dfb - ms_df, "bwd_gbs": 2.25 * vb / ((ms_dfb - ms_df) * 1e-3) / 1e9,
            "frac_of_hbm_peak_fwd": 1.125 * vb / (ms_df * 1e-3) / 1e9 / peak_gbs}
        del vol, go_ds
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        c1 = S.CONFIGS["C1"] if args.workload == "C2" else cfg
        v, cores, desc, _, _ = time_cpu_port(c1, args.cpu_seconds)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": desc}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
