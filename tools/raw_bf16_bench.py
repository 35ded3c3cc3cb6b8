"""LSSViewTransformerRaw with a bfloat16 2x2x2-reduced output (`ds_dtype=torch.bfloat16`) against
the float32 neck, and against the float32 neck followed by a cast, timed with CUDA events, the
variants of one workload alternating in one process, every timed region >= --region seconds after
warm-up (the timing loop of tools/channels_last_bench.py).  Before any timing, every bfloat16
result is checked against the contract: with a gradient, the output is the float32 output cast and
the depth / feature gradients are the float32 neck's for the widened output gradient (bit for
bit); without one, the output equals the float32 output cast (values, and here bits).

    python tools/raw_bf16_bench.py [--region 1.0] [--rounds 3]

Workloads (geometry and calibration from veon_b200.synthetic, as bench.py):
  VEON-real  C3 geometry (32 x 88 features, D = 88), B = 4, C = 256, two-hot depth
  C2         C2 geometry (16 x 44 features, D = 88), B = 8, C = 64, softmax depth
both on the 16 x 200 x 200 grid, reduced to 8 x 100 x 100; sync_free necks, fused geometry.

Variants:
  train_f32       float32 neck, forward + backward from a float32 gradient
  train_f32_cast  float32 neck, output cast to bfloat16 in the graph, backward from a bfloat16
                  gradient (autograd widens it)
  train_bf16      ds_dtype=bfloat16, backward from the same bfloat16 gradient
  infer_f32_cast_{cf,cl}  no gradient, float32 neck then `.to(torch.bfloat16)`, either layout
  infer_bf16_{cf,cl}      no gradient, ds_dtype=bfloat16, either layout
Also printed: the algorithmic bytes of the volumes each variant writes and reads after the
pooling's sums, from the shapes.

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
from veon_b200 import synthetic as S  # noqa: E402
from veon_b200.view_transformer import LSSViewTransformerRaw  # noqa: E402

BF = torch.bfloat16
CL = torch.channels_last_3d
KEYS = ("sensor2ego", "ego2global", "intrins", "post_rots", "post_trans", "bda")


def same_bits(a, b):
    if a.dtype != b.dtype or a.shape != b.shape or a.stride() != b.stride():
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    view = torch.int16 if a.dtype == BF else torch.int32
    return bool(torch.equal(na, nb)) and torch.equal(
        a.masked_fill(na, 0).contiguous().view(view), b.masked_fill(nb, 0).contiguous().view(view))


def algorithmic_bytes(B, C, Z, Y, X):
    """GB moved after the pooling's sums: the full-resolution volume, the reduced one, the mask
    and their gradients (the pooling's own gathers and the pixel pass are the same in every
    variant and left out)"""
    full, red = B * C * Z * Y * X, B * C * (Z // 2) * (Y // 2) * (X // 2)
    gb = 1e-9
    return {
        # pool write + max read (float32), reduced write, cast read + write
        "infer_f32_cast": (4 * full + 4 * full + 4 * red + 4 * red + 2 * red) * gb,
        # pool write + max read (bfloat16), reduced write
        "infer_bf16": (2 * full + 2 * full + 2 * red) * gb,
        # forward: pool write + masked max read, reduced write + mask; backward: grad_ds + mask
        "train_f32": (4 * full + 4 * full + 4 * red + red + 4 * red + red) * gb,
        # ... + the cast (read 4, write 2) + the widening of its gradient (read 2, write 4)
        "train_f32_cast": (4 * full + 4 * full + 4 * red + red + 6 * red + 6 * red + 4 * red
                           + red) * gb,
        "train_bf16": (4 * full + 4 * full + 2 * red + red + 2 * red + red) * gb,
        "volume_f32_GB": 4 * full * gb, "volume_bf16_GB": 2 * full * gb,
        "reduced_f32_GB": 4 * red * gb, "reduced_bf16_GB": 2 * red * gb, "mask_GB": red * gb,
    }


def workload(name, cfg, B, C, region_s, rounds, dev, two_hot):
    N, D = cfg.n_cams, cfg.D
    H, W = cfg.feat_hw
    g = torch.Generator(device=dev).manual_seed(5)
    cal = S.calibration(cfg, batch=B)
    metas = [torch.from_numpy(cal[k]).to(dev) for k in KEYS]

    def neck(fmt, ds_dtype):
        return LSSViewTransformerRaw(cfg.grid_config, cfg.input_size, cfg.downsample, 8, C,
                                     sync_free=True, memory_format=fmt, ds_dtype=ds_dtype)

    n32 = {fmt: neck(fmt, torch.float32) for fmt in (torch.contiguous_format, CL)}
    n16 = {fmt: neck(fmt, BF) for fmt in (torch.contiguous_format, CL)}
    if two_hot:
        metric = torch.from_numpy(S.metric_depth_np(cfg, batch=B)).to(dev)
        with torch.no_grad():
            depth = n32[torch.contiguous_format].get_two_hot_depth(metric)
    else:
        depth = torch.softmax(torch.randn(B, N, D, H, W, device=dev, generator=g) * 4, dim=2)
    feat = torch.randn(B, N, C, H, W, device=dev, generator=g)
    Z, Y, X = (int(v) for v in reversed(n32[CL].grid_size.tolist()))
    go_bf = torch.randn(B, C, Z // 2, Y // 2, X // 2, device=dev, generator=g).to(BF)
    go_f32 = go_bf.float()

    def train(kind):
        nk = n16[torch.contiguous_format] if kind == "bf16" else n32[torch.contiguous_format]
        go = go_f32 if kind == "f32" else go_bf

        def run():
            f = feat.detach().requires_grad_()
            d = depth.detach().requires_grad_()
            out = nk([f] + metas, d)
            if kind == "f32_cast":
                out = out.to(BF)
            out.backward(go)
            return out.detach(), d.grad, f.grad
        return run

    def infer(kind, fmt):
        def run():
            with torch.no_grad():
                if kind == "bf16":
                    return n16[fmt]([feat] + metas, depth)
                return n32[fmt]([feat] + metas, depth).to(BF)
        return run

    # the contract at the timed sizes, outside the timed regions
    (o32, d32, f32), (o16, d16, f16) = train("f32")(), train("bf16")()
    ok = {"train": same_bits(o16, o32.to(BF)) and same_bits(d16, d32) and same_bits(f16, f32)}
    del o32, d32, f32, o16, d16, f16
    for fmt, tag in ((torch.contiguous_format, "cf"), (CL, "cl")):
        a, b = infer("f32_cast", fmt)(), infer("bf16", fmt)()
        ok[f"infer_{tag}"] = bool(((a == b) | torch.isnan(a)).all()) and same_bits(a, b)
        del a, b
    torch.cuda.synchronize()
    alg = algorithmic_bytes(B, C, Z, Y, X)
    print(f"{name}: B={B} C={C} grid {Z}x{Y}x{X}; contract holds: {ok}; GB after the sums: "
          + ", ".join(f"{k} {v:.3f}" for k, v in alg.items()), flush=True)
    if not all(ok.values()):
        sys.exit(f"{name}: a bfloat16 result breaks the contract, not timing it")
    variants = {f"train_{k}": train(k) for k in ("f32", "f32_cast", "bf16")}
    for fmt, tag in ((torch.contiguous_format, "cf"), (CL, "cl")):
        variants[f"infer_f32_cast_{tag}"] = infer("f32_cast", fmt)
        variants[f"infer_bf16_{tag}"] = infer("bf16", fmt)
    t = bench(name, variants, region_s, rounds)
    return dict(B=B, C=C, grid=[Z, Y, X], contract=ok, algorithmic_GB=alg,
                us={k: round(v, 1) for k, v in t.items()})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--region", type=float, default=1.0, help="seconds per timed region")
    ap.add_argument("--rounds", type=int, default=3, help="timed regions per variant")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("raw_bf16_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plim = torch.cuda.get_device_name(dev), power_limit()
    print(f"device: {name}, power limit {plim}", flush=True)
    res = dict(device=name, power_limit=plim, region_s=args.region, rounds=args.rounds)
    res["VEON-real"] = workload("VEON-real", S.CONFIGS["C3"], 4, 256, args.region, args.rounds,
                                dev, two_hot=True)
    torch.cuda.empty_cache()
    res["C2"] = workload("C2", S.CONFIGS["C2"], 8, 64, args.region, args.rounds, dev,
                         two_hot=False)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
