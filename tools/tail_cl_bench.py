"""The open-vocabulary tail on channels-last feature volumes: voxel_text_argmax at full resolution
and voxel_text_argmax_lowres at the decoder's resolution, timed with CUDA events, the variants of
one group alternating in one process, every timed region >= --region seconds after warm-up (the
timing loop of tools/channels_last_bench.py).  Volumes (0.66 to 2.6 GB) are far larger than L2.
Before any timing, every `cl` result is checked byte for byte against `cf` at the same sizes.

    python tools/tail_cl_bench.py [--region 1.0] [--rounds 3]

Variants per configuration (C = 512, Q in {18, 67}), in float32 and in bfloat16:
  cf       channels-first volume
  cl+copy  channels-last volume, .contiguous() and then the call (the route a channels-last
           volume took before the tail read it as it is)
  cl       channels-last volume read by the kernel as it is
Configurations: full resolution (B = 2, 16x200x200) and decoder resolution (B = 8, 8x100x100
-> 16x200x200).  TB/s is on the algorithmic bytes of `cf`: the feature volume once (4 or 2 bytes
a value), the float32 gate (8 bytes a voxel) and the uint8 labels; at decoder resolution the
features and the gate are counted at the low resolution and the labels at the full one.

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
from veon_b200.tail import (class_of_prompt, semantic_inference_3d, voxel_text_argmax,  # noqa: E402
                            voxel_text_argmax_lowres)

SIZES = [16, 1, 1, 1, 8, 1, 1, 3, 1, 1, 1, 1, 5, 3, 5, 13, 4]   # nuscenes_brief prompts per class
VOCAB = {18: list(range(17)), 67: [k for k, n in enumerate(SIZES) for _ in range(n)]}
OCC = (16, 200, 200)
CL3 = torch.channels_last_3d


def group(name, B, C, Q, vol, lowres, dtype, region_s, rounds, dev):
    g = torch.Generator(device=dev).manual_seed(Q)
    feat_cf = (torch.rand(B, C, *vol, device=dev, generator=g) - 0.5).to(dtype)
    feat_cl = feat_cf.contiguous(memory_format=CL3)
    w = torch.randn(Q, C, device=dev, generator=g)
    w = 100.0 * w / w.norm(dim=1, keepdim=True)
    gate = torch.randn(B, 2, *vol, device=dev, generator=g)
    cls = class_of_prompt(VOCAB[Q]).to(dev)
    if lowres:
        ws = torch.empty(B * Q * vol[0] * vol[1] * vol[2], dtype=torch.float32, device=dev)

        def run(f):
            return voxel_text_argmax_lowres(f, w, cls, gate, occ_size=OCC, workspace=ws)
    else:
        def run(f):
            return voxel_text_argmax(f, w, cls, gate)
    variants = {"cf": lambda: run(feat_cf), "cl+copy": lambda: run(feat_cl.contiguous()),
                "cl": lambda: run(feat_cl)}
    got, want = variants["cl"](), variants["cf"]()
    torch.cuda.synchronize()
    equal = bool(torch.equal(got, want))
    del got, want
    if not lowres:   # the logits too, bit for bit (semantic_inference_3d, B = 1 to bound memory)
        a = semantic_inference_3d(w, feat_cl[:1])
        b = semantic_inference_3d(w, feat_cf[:1])
        torch.cuda.synchronize()
        equal = equal and bool(torch.equal(a.view(torch.int32), b.view(torch.int32)))
        del a, b
    print(f"{name}: B={B} C={C} Q={Q} {vol}{' -> ' + str(OCC) if lowres else ''} {dtype}; "
          f"cl == cf bit for bit: {equal}", flush=True)
    if not equal:
        sys.exit(f"{name}: the channels-last result differs from the channels-first one")
    t = bench(name, variants, region_s, rounds)
    V = vol[0] * vol[1] * vol[2]
    nbytes = feat_cf.element_size() * C * V * B + 8 * V * B + B * OCC[0] * OCC[1] * OCC[2]
    tbs = {k: nbytes / (t[k] * 1e-6) / 1e12 for k in variants}
    for k in variants:
        print(f"{name:>14} {k:<8} {t[k]:8.1f} us  {tbs[k]:5.2f} TB/s", flush=True)
    return dict(B=B, C=C, Q=Q, vol=vol, lowres=lowres, dtype=str(dtype), bitwise_equal=equal,
                bytes=nbytes, us={k: round(v, 1) for k, v in t.items()},
                tb_per_s={k: round(v, 2) for k, v in tbs.items()})


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--region", type=float, default=1.0, help="seconds per timed region")
    ap.add_argument("--rounds", type=int, default=3, help="timed regions per variant")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tail_cl_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, plim = torch.cuda.get_device_name(dev), power_limit()
    print(f"device: {name}, power limit {plim}", flush=True)
    res = dict(device=name, power_limit=plim, region_s=args.region, rounds=args.rounds)
    for dtype, tag in ((torch.float32, "f32"), (torch.bfloat16, "bf16")):
        for Q in (18, 67):
            key = f"full_q{Q}_{tag}"
            res[key] = group(key, 2, 512, Q, OCC, False, dtype, args.region, args.rounds, dev)
            torch.cuda.empty_cache()
            key = f"lowres_q{Q}_{tag}"
            res[key] = group(key, 8, 512, Q, (8, 100, 100), True, dtype, args.region, args.rounds,
                             dev)
            torch.cuda.empty_cache()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
