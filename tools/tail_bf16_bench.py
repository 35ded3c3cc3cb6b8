"""The open-vocabulary tail on bfloat16 feature volumes against float32: voxel_text_argmax at full
resolution and voxel_text_argmax_lowres at the decoder's resolution, timed with CUDA events, the
variants of one group alternating in one process, every timed region >= --region seconds after
warm-up (the timing loop of tools/channels_last_bench.py).  Volumes (0.66 to 2.6 GB) are far
larger than L2.  Before any timing, every bfloat16 result is checked byte for byte against the
float32 route on the widened volume at the same sizes.  Then one sustained region of --sustain
seconds per variant, because a long run of the tail reaches the power limit.

    python tools/tail_bf16_bench.py [--region 1.0] [--rounds 3] [--sustain 5.0]

Variants per configuration (C = 512, Q in {18, 67}):
  f32         float32 volume
  bf16+float  bfloat16 volume widened by .float(), then the float32 kernel (the route a
              bfloat16 volume took before the tail read bfloat16)
  bf16        bfloat16 volume read by the kernels as it is
Configurations: full resolution (B = 2, 16x200x200) and decoder resolution (B = 8, 8x100x100
-> 16x200x200).  TB/s is on the algorithmic bytes: the feature volume once (2 or 4 bytes a value),
the float32 gate (8 bytes a voxel) and the uint8 labels; at decoder resolution the features and
the gate are counted at the low resolution and the labels at the full one (the logits round trip
through the workspace is not counted).  bf16+float is counted with the bfloat16 bytes.

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

from channels_last_bench import bench, power_limit, region_ms  # noqa: E402
from veon_b200.tail import class_of_prompt, voxel_text_argmax, voxel_text_argmax_lowres  # noqa: E402

BF = torch.bfloat16
SIZES = [16, 1, 1, 1, 8, 1, 1, 3, 1, 1, 1, 1, 5, 3, 5, 13, 4]   # nuscenes_brief prompts per class
VOCAB = {18: list(range(17)), 67: [k for k, n in enumerate(SIZES) for _ in range(n)]}
OCC = (16, 200, 200)


def group(name, B, C, Q, vol, lowres, region_s, rounds, sustain_s, dev):
    g = torch.Generator(device=dev).manual_seed(Q)
    feat_bf = (torch.rand(B, C, *vol, device=dev, generator=g) - 0.5).to(BF)
    feat32 = feat_bf.float()
    w = torch.randn(Q, C, device=dev, generator=g)
    w = 100.0 * w / w.norm(dim=1, keepdim=True)
    gate = torch.randn(B, 2, *vol, device=dev, generator=g)
    cls = class_of_prompt(VOCAB[Q]).to(dev)
    if lowres:
        ws = torch.empty(B * Q * vol[0] * vol[1] * vol[2], dtype=torch.float32, device=dev)

        def call(f):
            return lambda: voxel_text_argmax_lowres(f, w, cls, gate, occ_size=OCC, workspace=ws)

        def call_widened():
            return voxel_text_argmax_lowres(feat_bf.float(), w, cls, gate, occ_size=OCC,
                                            workspace=ws)
    else:
        def call(f):
            return lambda: voxel_text_argmax(f, w, cls, gate)

        def call_widened():
            return voxel_text_argmax(feat_bf.float(), w, cls, gate)
    variants = {"f32": call(feat32), "bf16+float": call_widened, "bf16": call(feat_bf)}
    got, want = variants["bf16"](), variants["f32"]()
    torch.cuda.synchronize()
    equal = bool(torch.equal(got, want))
    del got, want
    print(f"{name}: B={B} C={C} Q={Q} {vol}{' -> ' + str(OCC) if lowres else ''}; "
          f"bfloat16 labels == float32 labels of the widened volume: {equal}", flush=True)
    t = bench(name, variants, region_s, rounds)
    V = vol[0] * vol[1] * vol[2]
    labels = B * OCC[0] * OCC[1] * OCC[2]
    nbytes = {k: (4 if k == "f32" else 2) * C * V * B + 8 * V * B + labels for k in variants}
    tbs = {k: nbytes[k] / (t[k] * 1e-6) / 1e12 for k in variants}
    for k in variants:
        print(f"{name:>10} {k:<12} {t[k]:8.1f} us  {tbs[k]:5.2f} TB/s", flush=True)
    sustained = {}
    for k, fn in variants.items():   # one long region each: the rate under the power limit
        n = max(1, int(sustain_s * 1e6 / t[k]))
        sustained[k] = region_ms(fn, n) * 1e3 / n
        print(f"{name:>10} {k:<12} sustained {sustain_s:.0f} s: {sustained[k]:8.1f} us", flush=True)
    return dict(B=B, C=C, Q=Q, vol=vol, lowres=lowres, bitwise_equal=equal,
                us={k: round(v, 1) for k, v in t.items()},
                tb_per_s={k: round(v, 2) for k, v in tbs.items()},
                sustained_us={k: round(v, 1) for k, v in sustained.items()})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--region", type=float, default=1.0, help="seconds per timed region")
    ap.add_argument("--rounds", type=int, default=3, help="timed regions per variant")
    ap.add_argument("--sustain", type=float, default=5.0, help="seconds of the sustained region")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tail_bf16_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plim = torch.cuda.get_device_name(dev), power_limit()
    print(f"device: {name}, power limit {plim}", flush=True)
    res = dict(device=name, power_limit=plim, region_s=args.region, rounds=args.rounds,
               sustain_s=args.sustain)
    for Q in (18, 67):
        res[f"full_q{Q}"] = group(f"full_q{Q}", 2, 512, Q, OCC, False, args.region, args.rounds,
                                  args.sustain, dev)
        torch.cuda.empty_cache()
        res[f"lowres_q{Q}"] = group(f"lowres_q{Q}", 8, 512, Q, (8, 100, 100), True, args.region,
                                    args.rounds, args.sustain, dev)
        torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
