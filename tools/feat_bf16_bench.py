"""bfloat16 image features vs float32 ones: the pooling forward and backward and two neck training
steps, timed with CUDA events, the variants of one group alternating in one process, every timed
region >= --region seconds after warm-up (the timing loop of tools/channels_last_bench.py).
Before any timing, every bfloat16-feature result is checked bit for bit against the same call on
the widened features: volumes and depth_grad equal, feat_grad equal to the float32 one cast.

    python tools/feat_bf16_bench.py [--region 1.0] [--rounds 3]

Shapes: C2 (B = 8, C = 64) and C3 (B = 1, C = 512), float32 channels-first volume, softmax depth;
VEON-real: the Raw neck at C = 256, B = 4, two-hot depth (C2 geometry).

Variants (the features enter as the necks hand them over: a channels-last view of channels-first
[B*N, C, H, W] maps):
  f32       float32 maps
  today     bfloat16 maps, emulated as the parent release handled them: `.float()` of the view,
            the float32 route, and feat_grad cast to bfloat16
  native    bfloat16 maps read as they are (the `_bf16feat` entries)
Timed per shape: `fwd` (feature rows + pooling), `bwd` (both gradients from a float32
channels-first volume gradient, feat_grad back to maps), and a training step of the neck
(LSSViewTransformer.view_transform for C2 / C3, LSSViewTransformerRaw for VEON-real: fused
geometry, prepare, forward, backward).  Also printed: the bytes of feature rows the forward
gathers, n_kept * C * element size, from the plan's n_kept.

Prints the device and its power limit, one line per variant (median us per call), and one JSON
line at the end."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from channels_last_bench import bench, power_limit  # noqa: E402
from veon_b200 import bev_pool as BP, synthetic as S  # noqa: E402
from veon_b200.view_transformer import LSSViewTransformer, LSSViewTransformerRaw  # noqa: E402

BF = torch.bfloat16
KEYS = ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")


def same_bits(a, b):
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    view = torch.int16 if a.dtype == BF else torch.int32
    return bool(torch.equal(na, nb)) and torch.equal(
        a.masked_fill(na, 0).contiguous().view(view), b.masked_fill(nb, 0).contiguous().view(view))


def group(name, cfg, B, C, region_s, rounds, dev, raw=False):
    lower, interval, size = S.grid_vectors(cfg.grid_config)
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).to(dev) for k in KEYS]
    N, D = cfg.n_cams, cfg.D
    H, W = cfg.feat_hw
    g = torch.Generator(device=dev).manual_seed(0)
    if raw:   # two-hot depth from metric depth maps (LSSViewTransformerRaw.get_two_hot_depth)
        metric = torch.rand(B, N, H, W, device=dev, generator=g) * 40 + 2
        depth = BP.two_hot_depth(metric, cfg.grid_config["depth"], D)
    else:
        depth = torch.softmax(torch.randn(B, N, D, H, W, device=dev, generator=g) * 4, dim=2)
    maps = torch.randn(B, N, C, H, W, device=dev, generator=g)
    maps_bf = maps.to(BF)
    if raw:
        neck = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C)
    else:
        neck = LSSViewTransformer(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                  collapse_z=False)
    coor = neck.get_lidar_coor(*metas)
    prep = BP.prepare_ranks(coor, lower, interval, size)
    plan = prep.plan
    plan._resolve()
    Z, Y, X = int(size[2]), int(size[1]), int(size[0])
    V = Z * Y * X
    rd, rf, rb, ist = prep.ranks_depth, prep.ranks_feat, prep.ranks_bev, prep.interval_starts
    shape5 = (B, C, Z, Y, X)
    og = torch.randn(shape5, device=dev, generator=g)
    og_zyxc = og.permute(0, 2, 3, 4, 1)

    def view(m):
        return m.permute(0, 1, 3, 4, 2)

    def rows(kind):
        if kind == "f32":
            return BP._feat_rows(view(maps))[0]
        if kind == "today":
            return BP._feat_rows(view(maps_bf).float())[0]
        return BP._feat_rows(view(maps_bf))[0]

    def fwd(kind):
        return lambda: BP._fwd_planar(depth, rows(kind), rd, rf, rb, plan, B, C, V, shape5)

    saved = {k: rows(k) for k in ("f32", "today", "native")}

    def bwd(kind):
        def run():
            dg, fg = BP._pool_bwd(og_zyxc, depth, saved[kind], rd, rf, rb, ist, plan)
            if kind == "today":
                return dg, BP._feat_grad_back(fg, True).to(BF)
            return dg, BP._feat_grad_back(fg, True)
        return run

    go = torch.randn(B, C, Z // 2, Y // 2, X // 2, device=dev, generator=g) if raw else og
    img = torch.zeros(B, N, 8, H, W, device=dev)

    def train(kind):
        src = {"f32": maps, "today": maps_bf, "native": maps_bf}[kind]

        def run():
            f = src.detach().requires_grad_()
            d = depth.detach().requires_grad_()
            f_in = f.float() if kind == "today" else f
            if raw:
                out = neck([f_in] + metas, d)
            else:
                out = neck.view_transform([img] + metas, d.view(B * N, D, H, W),
                                          f_in.view(B * N, C, H, W))[0]
            out.backward(go)
            return out, d.grad, f.grad
        return run

    # bit-for-bit checks at the timed sizes, outside the timed regions
    eq = dict(fwd=same_bits(fwd("native")(), fwd("today")()))
    (dn, fn), (dt, ft) = bwd("native")(), bwd("today")()
    eq["bwd"] = same_bits(dn, dt) and same_bits(fn, ft)
    (on, dn, fn), (ot, dt, ft) = train("native")(), train("today")()
    eq["train"] = same_bits(on, ot) and same_bits(dn, dt) and same_bits(fn, ft)
    del dn, fn, dt, ft, on, ot
    torch.cuda.synchronize()
    gathered = {k: plan.n_points * C * s for k, s in (("f32", 4), ("native", 2))}
    print(f"{name}: B={B} C={C} kept={plan.n_points} intervals={plan.n_intervals}; feature rows "
          f"gathered per forward: {gathered['f32'] / 1e6:.0f} MB float32, "
          f"{gathered['native'] / 1e6:.0f} MB bfloat16; native == widened: {eq}", flush=True)
    variants = {}
    for kind in ("f32", "today", "native"):
        variants[f"fwd_{kind}"] = fwd(kind)
    for kind in ("f32", "today", "native"):
        variants[f"bwd_{kind}"] = bwd(kind)
    for kind in ("f32", "today", "native"):
        variants[f"train_{kind}"] = train(kind)
    t = bench(name, variants, region_s, rounds)
    return dict(B=B, C=C, n_kept=plan.n_points, gathered_bytes=gathered, bitwise_equal=eq,
                us={k: round(v, 1) for k, v in t.items()})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--region", type=float, default=1.0, help="seconds per timed region")
    ap.add_argument("--rounds", type=int, default=3, help="timed regions per variant")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("feat_bf16_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plim = torch.cuda.get_device_name(dev), power_limit()
    print(f"device: {name}, power limit {plim}", flush=True)
    res = dict(device=name, power_limit=plim, region_s=args.region, rounds=args.rounds)
    res["C2"] = group("C2", S.CONFIGS["C2"], 8, 64, args.region, args.rounds, dev)
    torch.cuda.empty_cache()
    res["C3"] = group("C3", S.CONFIGS["C3"], 1, 512, args.region, args.rounds, dev)
    torch.cuda.empty_cache()
    res["VEON-real"] = group("VEON-real", S.CONFIGS["C2"], 4, 256, args.region, args.rounds, dev,
                             raw=True)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
