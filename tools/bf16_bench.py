"""bfloat16 volumes vs float32: pooling forward in both layouts and the backward on bfloat16
gradients, timed with CUDA events, the variants of one group alternating in one process, every
timed region >= --region seconds after warm-up (the timing loop of tools/channels_last_bench.py).
Volumes (0.66 / 1.31 GB) are far larger than L2; the inputs (ranks, depth, features) stay
L2-resident, as in a real step.  Before any timing, every bfloat16 result is checked bit for bit
against its float32 counterpart at the same sizes: the forward against the float32 volume cast
on the device, the backward against the float32 route given the widened gradient.

    python tools/bf16_bench.py [--region 1.0] [--rounds 3]

Variants per configuration (C2: B = 8, C = 64; C3: B = 1, C = 512):
  fwd_{cf,cl}_f32         float32 volume, channels-first / channels-last
  fwd_{cf,cl}_f32+cast    float32 volume, then .to(torch.bfloat16) (today's autocast user)
  fwd_{cf,cl}_bf16        bfloat16 volume written by the kernels
  bwd_f32_cf_two_pass     float32 channels-first gradient: row pass + pixel pass
  bwd_bf16_cf_two_pass    bfloat16 channels-first gradient: bf16 row pass + pixel pass
  bwd_f32_cl_single_pass  float32 channels-last gradient, read in place
  bwd_bf16_cl_single_pass bfloat16 channels-last gradient, read in place
  bwd_cast_volume         a bfloat16 gradient widened by ToCopyBackward, then the float32
                          two passes (today's route for a cast volume)

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

BF = torch.bfloat16


def bits_equal(bf, f32):
    """bf == f32 cast to bfloat16 on the device, bit for bit (NaN positions only)"""
    want = f32.to(BF)
    na, nb = torch.isnan(bf), torch.isnan(want)
    return bool(torch.equal(na, nb)) and torch.equal(
        bf.masked_fill(na, 0).contiguous().view(torch.int16),
        want.masked_fill(nb, 0).contiguous().view(torch.int16))


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
    g_cf_bf, g_cl_bf = g_cf.to(BF), g_cl.to(BF)
    shape = {False: (B, C, Z, Y, X), True: (B, Z, Y, X, C)}

    def fwd(cl, dtype=torch.float32):
        return lambda: BP._fwd_planar(depth, feat, rd, rf, rb, plan, B, C, V, shape[cl], cl, dtype)

    def fwd_cast(cl):
        f = fwd(cl)
        return lambda: f().to(BF)

    # _pool_bwd takes the gradient of the [B,Z,Y,X,C] volume QuickCumsumCuda returns
    def bwd(grad_zyxc):
        return lambda: BP._pool_bwd(grad_zyxc, depth, feat, rd, rf, rb, ist, plan)

    def bwd_cast_volume():   # ToCopyBackward: the bfloat16 gradient widened to a new float32 one
        return BP._pool_bwd(g_cf_bf.float().permute(0, 2, 3, 4, 1), depth, feat, rd, rf, rb, ist,
                            plan)

    # bit-for-bit checks at the timed sizes, outside the timed regions
    eq = {}
    for cl in (False, True):
        a, b = fwd(cl)(), fwd(cl, BF)()
        eq["fwd_cl" if cl else "fwd_cf"] = bits_equal(b, a)
        del a, b
    want = bwd(g_cf_bf.float().permute(0, 2, 3, 4, 1))()
    for k, grad in (("bwd_bf16_cf", g_cf_bf.permute(0, 2, 3, 4, 1)), ("bwd_bf16_cl", g_cl_bf)):
        got = bwd(grad)()
        eq[k] = all(torch.equal(x, y) for x, y in zip(got, want))
    del want, got
    torch.cuda.synchronize()
    print(f"{name}: B={B} C={C} intervals={plan.n_intervals} kept={plan.n_points}; "
          f"bfloat16 == float32 (cast / widened): {eq}", flush=True)
    t = bench(name, {"fwd_cf_f32": fwd(False), "fwd_cf_f32+cast": fwd_cast(False),
                     "fwd_cf_bf16": fwd(False, BF),
                     "fwd_cl_f32": fwd(True), "fwd_cl_f32+cast": fwd_cast(True),
                     "fwd_cl_bf16": fwd(True, BF),
                     "bwd_f32_cf_two_pass": bwd(g_cf.permute(0, 2, 3, 4, 1)),
                     "bwd_bf16_cf_two_pass": bwd(g_cf_bf.permute(0, 2, 3, 4, 1)),
                     "bwd_f32_cl_single_pass": bwd(g_cl), "bwd_bf16_cl_single_pass": bwd(g_cl_bf),
                     "bwd_cast_volume": bwd_cast_volume}, region_s, rounds)
    return dict(B=B, C=C, bitwise_equal=eq, us={k: round(v, 1) for k, v in t.items()})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--region", type=float, default=1.0, help="seconds per timed region")
    ap.add_argument("--rounds", type=int, default=3, help="timed regions per variant")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bf16_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plim = torch.cuda.get_device_name(dev), power_limit()
    print(f"device: {name}, power limit {plim}", flush=True)
    res = dict(device=name, power_limit=plim, region_s=args.region, rounds=args.rounds)
    res["C2"] = pool_group("C2", S.CONFIGS["C2"], 8, 64, args.region, args.rounds, dev)
    torch.cuda.empty_cache()
    res["C3"] = pool_group("C3", S.CONFIGS["C3"], 1, 512, args.region, args.rounds, dev)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
