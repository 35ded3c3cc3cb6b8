"""Where the roles of k_tail_tc (CTA 0) spend their cycles on one call; needs a build with
-DVEON_TAIL_TRACE (tools/build_variant.sh) loaded through VEON_LIB.

    python tools/tail_trace.py [q67] [bf16] [cl]     (bf16: a bfloat16 feature volume;
                                                      cl: a channels_last_3d one)"""
import ctypes
import os
import sys

import torch

sys.path.insert(0, ".")
from veon_b200 import _lib  # noqa: E402
_lib.LIB_PATH = os.environ["VEON_LIB"]
from veon_b200.tail import class_of_prompt, voxel_text_argmax  # noqa: E402

SIZES = [16, 1, 1, 1, 8, 1, 1, 3, 1, 1, 1, 1, 5, 3, 5, 13, 4]
q67 = "q67" in sys.argv[1:]
dev = torch.device("cuda", 0)
C, B = 512, 2
refl = [k for k, n in enumerate(SIZES) for _ in range(n)] if q67 else list(range(17))
g = torch.Generator(device=dev).manual_seed(0)
feat = torch.sigmoid(torch.randn(B, C, 16, 200, 200, device=dev, generator=g)) - 0.5
w = torch.randn(len(refl) + 1, C, device=dev, generator=g)
bo = torch.randn(B, 2, 16, 200, 200, device=dev, generator=g)
if "bf16" in sys.argv[1:]:
    feat = feat.to(torch.bfloat16)
if "cl" in sys.argv[1:]:
    feat = feat.contiguous(memory_format=torch.channels_last_3d)
cls = class_of_prompt(refl).to(dev)
lib = ctypes.CDLL(_lib.LIB_PATH)
for _ in range(3):
    voxel_text_argmax(feat, w, cls, bo)
torch.cuda.synchronize()
buf = (ctypes.c_ulonglong * 256)()
assert lib.veon_internal_tail_trace(buf, 1) == 0
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(); voxel_text_argmax(feat, w, cls, bo); b.record()
torch.cuda.synchronize()
assert lib.veon_internal_tail_trace(buf, 0) == 0
print(f"call {a.elapsed_time(b) * 1e3:.1f} us (traced build), Q={len(refl) + 1}")
mhz = 1965.0
roles = (("converters", 0, 16, ["raw data wait", "empty wait", "read + split", "W copy + st + wait::st + arrive"]),
         ("mma", 16, 17, ["acc_empty wait", "full wait", "issue + commit"]),
         ("epilogue", 17, 21, ["acc_full wait", "work"]))
for role, lo, hi, names in roles:
    tot = [sum(buf[x * 8 + k] for x in range(lo, hi)) / (hi - lo) / mhz for k in range(len(names))]
    print(f"{role:10s} (mean over warps, us): " + ", ".join(f"{n} {t:.1f}" for n, t in zip(names, tot)))
