"""A few C2 backward calls (for ncu): python tools/bwd_profile.py [cfg B C iters]"""
import sys
import torch
sys.path.insert(0, ".")
sys.path.insert(0, "tools")
from fwd_check import setup  # noqa: E402
from veon_b200 import bev_pool as BP  # noqa: E402

cfg = sys.argv[1] if len(sys.argv) > 1 else "C2"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 8
C = int(sys.argv[3]) if len(sys.argv) > 3 else 64
iters = int(sys.argv[4]) if len(sys.argv) > 4 else 3
prep, depth, feat, shape = setup(cfg, B, C)
og = torch.randn(shape, device="cuda")
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for i in range(iters):
    a.record()
    dg, fg = BP._pool_bwd(og.permute(0, 2, 3, 4, 1), depth, feat, prep.ranks_depth,
                          prep.ranks_feat, prep.ranks_bev, prep.interval_starts, prep.plan)
    b.record()
torch.cuda.synchronize()
print("ok", float(dg.abs().sum()), float(fg.abs().sum()), f"last call {a.elapsed_time(b) * 1e3:.1f} us")
