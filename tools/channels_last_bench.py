"""Channels-last volumes vs channels-first: pooling forward, backward and the Raw-neck training
step, timed with CUDA events, the variants of one group alternating in one process, every timed
region >= --region seconds after warm-up.  Volumes (1.3 GB) are far larger than L2; the inputs
(ranks, depth, features) stay L2-resident, as in a real step.  Before any timing, the
channels-last results are checked bit for bit against the channels-first ones at the same sizes.

    python tools/channels_last_bench.py [--region 1.0] [--rounds 3]

Prints the device and its power limit, one line per variant (median us per call), and one JSON
line at the end."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from veon_b200 import bev_pool as BP, synthetic as S  # noqa: E402
from veon_b200.view_transformer import LSSViewTransformerRaw  # noqa: E402

CL = torch.channels_last_3d
KEYS = ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def region_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def bench(group, variants, region_s, rounds):
    """{name: median us per call}: warm-up, calibrate the calls per region, then `rounds`
    rounds in which every variant runs one timed region, alternating"""
    calls = {}
    for name, fn in variants.items():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        n = 1
        while True:
            ms = region_ms(fn, n)
            if ms >= 0.25 * region_s * 1e3:
                break
            n *= 2
        calls[name] = max(1, int(n * region_s * 1e3 / ms) + 1)
    per_call = {k: [] for k in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            ms = region_ms(fn, calls[name])
            assert ms >= region_s * 1e3 * 0.9, (name, ms)
            per_call[name].append(ms * 1e3 / calls[name])
    res = {}
    for name, v in per_call.items():
        v = sorted(v)
        res[name] = v[len(v) // 2]
        print(f"{group:>4} {name:<28} {res[name]:9.1f} us  (rounds {', '.join(f'{x:.1f}' for x in v)};"
              f" {calls[name]} calls per region)", flush=True)
    return res


def pool_group(name, cfg, B, C, region_s, rounds, dev):
    lower, interval, size = S.grid_vectors(cfg.grid_config)
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B)).to(dev)
    _, N, D, H, W, _ = coor.shape
    g = torch.Generator(device=dev).manual_seed(0)
    depth = torch.softmax(torch.randn(B, N, D, H, W, device=dev, generator=g) * 4, dim=2)
    feat = torch.randn(B, N, H, W, C, device=dev, generator=g)
    prep = BP.prepare_ranks(coor, lower, interval, size)
    plan = prep.plan
    plan._resolve()
    Z, Y, X = int(size[2]), int(size[1]), int(size[0])
    V = Z * Y * X
    rd, rf, rb, ist = prep.ranks_depth, prep.ranks_feat, prep.ranks_bev, prep.interval_starts
    g_cf = torch.randn(B, C, Z, Y, X, device=dev, generator=g)
    g_cl = g_cf.permute(0, 2, 3, 4, 1).contiguous()          # the same values, [B,Z,Y,X,C]
    g_cl_view = g_cl.permute(0, 4, 1, 2, 3)                   # how a channels-last user holds it

    def fwd_cf():
        return BP._fwd_planar(depth, feat, rd, rf, rb, plan, B, C, V, (B, C, Z, Y, X))

    def fwd_cl():
        return BP._fwd_planar_cl(depth, feat, rd, rf, rb, plan, B, C, V, (B, Z, Y, X, C))

    def fwd_cf_convert():
        return fwd_cf().contiguous(memory_format=CL)

    # _pool_bwd takes the gradient of the [B,Z,Y,X,C] volume QuickCumsumCuda returns
    def bwd_cf():
        return BP._pool_bwd(g_cf.permute(0, 2, 3, 4, 1), depth, feat, rd, rf, rb, ist, plan)

    def bwd_cl():
        return BP._pool_bwd(g_cl, depth, feat, rd, rf, rb, ist, plan)

    def bwd_copy():
        return BP._pool_bwd(g_cl_view.contiguous().permute(0, 2, 3, 4, 1), depth, feat, rd, rf,
                            rb, ist, plan)

    # bit-for-bit checks at the timed sizes, outside the timed regions
    a, b = fwd_cf(), fwd_cl()
    eq_fwd = torch.equal(a.permute(0, 2, 3, 4, 1), b)
    del a, b
    (d1, f1), (d2, f2) = bwd_cf(), bwd_cl()
    eq_bwd = torch.equal(d1, d2) and torch.equal(f1, f2)
    del d1, f1, d2, f2
    torch.cuda.synchronize()
    print(f"{name}: B={B} C={C} intervals={plan.n_intervals} kept={plan.n_points}; "
          f"channels-last == channels-first: forward {eq_fwd}, backward {eq_bwd}", flush=True)
    t = bench(name, {"fwd_channels_first": fwd_cf, "fwd_channels_last": fwd_cl,
                     "fwd_channels_first+convert": fwd_cf_convert,
                     "bwd_cf_grad_two_pass": bwd_cf, "bwd_cl_grad_single_pass": bwd_cl,
                     "bwd_cl_grad_copy+two_pass": bwd_copy}, region_s, rounds)
    return dict(B=B, C=C, bitwise_equal_fwd=eq_fwd, bitwise_equal_bwd=eq_bwd,
                us={k: round(v, 1) for k, v in t.items()})


def raw_train_group(region_s, rounds, dev):
    """Raw-neck training step at C2 (geometry + prepare + forward + backward), as
    tools/raw_train_bench.py measures it"""
    cfg = S.CONFIGS["C2"]
    B, C = cfg.batch, cfg.channels
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).to(dev) for k in KEYS]
    N, D = cfg.n_cams, cfg.D
    H, W = cfg.feat_hw
    g = torch.Generator(device=dev).manual_seed(0)
    depth = torch.softmax(torch.randn(B, N, D, H, W, device=dev, generator=g) * 4, dim=2)
    feat = torch.randn(B, N, C, H, W, device=dev, generator=g)
    go = torch.randn(B, C, 8, 100, 100, device=dev, generator=g)
    go_cl = go.contiguous(memory_format=CL)
    neck_cf = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C)
    neck_cl = LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                    memory_format=CL)

    def step(neck, convert, grad):
        f = feat.detach().requires_grad_()
        d = depth.detach().requires_grad_()
        out = neck([f] + metas, d)
        if convert:
            out = out.contiguous(memory_format=CL)
        out.backward(grad)
        return out, d.grad, f.grad

    runs = [step(neck_cf, False, go), step(neck_cl, False, go_cl), step(neck_cf, True, go_cl)]
    same = all(torch.equal(x, y) for r in runs[1:] for x, y in zip(runs[0], r))
    del runs
    print(f"raw: channels-last step == channels-first step (output, depth.grad, feat.grad): {same}",
          flush=True)
    t = bench("raw", {"channels_first_one_node": lambda: step(neck_cf, False, go),
                      "channels_last": lambda: step(neck_cl, False, go_cl),
                      "channels_first+2_conversions": lambda: step(neck_cf, True, go_cl)},
              region_s, rounds)
    return dict(B=B, C=C, bitwise_equal=same, us={k: round(v, 1) for k, v in t.items()})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--region", type=float, default=1.0, help="seconds per timed region")
    ap.add_argument("--rounds", type=int, default=3, help="timed regions per variant")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("channels_last_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plim = torch.cuda.get_device_name(dev), power_limit()
    print(f"device: {name}, power limit {plim}", flush=True)
    res = dict(device=name, power_limit=plim, region_s=args.region, rounds=args.rounds)
    res["C2"] = pool_group("C2", S.CONFIGS["C2"], 8, 64, args.region, args.rounds, dev)
    torch.cuda.empty_cache()
    res["C3"] = pool_group("C3", S.CONFIGS["C3"], 1, 512, args.region, args.rounds, dev)
    torch.cuda.empty_cache()
    res["raw_train_C2"] = raw_train_group(args.region, args.rounds, dev)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
