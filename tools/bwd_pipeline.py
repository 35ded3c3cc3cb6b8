"""Experiment: the backward as per-sample row / pixel launches on two streams (rows of sample s+1
overlap the pixels of sample s), optionally with the row scratch pinned in L2 by an access-policy
window.  Compared with the library's two launches over all samples.  Needs a tools build of the
library (the per-pass entry points are not in the shipped one):
    VEON_LIB=$(tools/build_variant.sh tools "-DVEON_TOOLS" | tail -1) python tools/bwd_pipeline.py"""
import ctypes
import sys

import torch

sys.path.insert(0, ".")
sys.path.insert(0, "tools")
from fwd_check import setup, ev_ms  # noqa: E402
from veon_b200 import _lib, bev_pool as BP  # noqa: E402

B, C = 8, 64
prep, depth, feat, shape = setup("C2", B, C)
plan = prep.plan
_, N, D, H, W = plan.dims
HW, V = H * W, plan.V
tps = V // 32
og = torch.randn(shape, device="cuda")
lib = ctypes.CDLL(_lib.LIB_PATH)
n_int = plan.n_intervals
rows = torch.empty(n_int * C, dtype=torch.float32, device="cuda")
dg, fg = torch.empty_like(depth), torch.empty_like(feat)
P = ctypes.c_void_p
i64 = ctypes.c_int64


def ptr(t, off=0):
    return P(t.data_ptr() + off * t.element_size())


def reference():
    return BP._pool_bwd(og.permute(0, 2, 3, 4, 1), depth, feat, prep.ranks_depth,
                        prep.ranks_feat, prep.ranks_bev, prep.interval_starts, plan)


want_dg, want_fg = reference()
s_rows, s_pix = torch.cuda.Stream(), torch.cuda.Stream()
ev_rows = [torch.cuda.Event() for _ in range(B)]
ev_pix = [torch.cuda.Event() for _ in range(B)]


def pipelined(group=1):
    main = torch.cuda.current_stream()
    start = torch.cuda.Event()
    start.record(main)
    s_rows.wait_event(start)
    s_pix.wait_event(start)
    for s in range(0, B, group):
        g = min(group, B - s)
        rc = lib.veon_internal_bwd_rows(ptr(og, s * C * V), ptr(plan.tile_istart, s * tps),
                                        ptr(plan.tile_occ, s * tps), i64(g * tps), i64(tps), i64(V), C,
                                        ptr(rows), P(s_rows.cuda_stream))
        assert rc == 0, rc
        ev_rows[s].record(s_rows)
        s_pix.wait_event(ev_rows[s])
        rc = lib.veon_internal_bwd_pixels(ptr(rows), ptr(depth, s * N * D * HW), ptr(feat, s * N * HW * C),
                                          ptr(plan.point_interval, s * N * HW * D), i64(g * N * HW), D, HW, C,
                                          ptr(dg, s * N * D * HW), ptr(fg, s * N * HW * C),
                                          P(s_pix.cuda_stream))
        assert rc == 0, rc
    done = torch.cuda.Event()
    done.record(s_pix)
    main.wait_event(done)
    done2 = torch.cuda.Event()
    done2.record(s_rows)
    main.wait_event(done2)


pipelined()
torch.cuda.synchronize()
print("pipelined == two launches:", torch.equal(dg, want_dg), torch.equal(fg, want_fg))
print(f"two launches (library): {ev_ms(reference, n=20) * 1e3:.1f} us")
for group in (1, 2, 4):
    print(f"per-{group}-sample launches on two streams: {ev_ms(lambda: pipelined(group), n=20) * 1e3:.1f} us")
cudart = ctypes.CDLL("libcudart.so.12")
attr = ctypes.c_int()
cudart.cudaDeviceGetAttribute(ctypes.byref(attr), 108, 0)   # MaxPersistingL2CacheSize
print("max persisting L2 bytes:", attr.value)
cudart.cudaDeviceGetAttribute(ctypes.byref(attr), 109, 0)   # MaxAccessPolicyWindowSize
print("max access-policy window bytes:", attr.value)

# ring of two samples' rows, pinned
first = plan.tile_istart[::tps].cpu().tolist() + [n_int]
per_sample = max(first[i + 1] - first[i] for i in range(B))
ring = torch.empty(2 * per_sample * C, dtype=torch.float32, device="cuda")
print(f"ring: {ring.numel() * 4 / 2**20:.1f} MB")


def ringed():
    main = torch.cuda.current_stream()
    start = torch.cuda.Event()
    start.record(main)
    s_rows.wait_event(start)
    s_pix.wait_event(start)
    for s in range(B):
        base = P(ring.data_ptr() + 4 * ((s % 2) * per_sample * C - first[s] * C))
        if s >= 2:
            s_rows.wait_event(ev_pix[s - 2])
        rc = lib.veon_internal_bwd_rows(ptr(og, s * C * V), ptr(plan.tile_istart, s * tps),
                                        ptr(plan.tile_occ, s * tps), i64(tps), i64(tps), i64(V), C,
                                        base, P(s_rows.cuda_stream))
        assert rc == 0, rc
        ev_rows[s].record(s_rows)
        s_pix.wait_event(ev_rows[s])
        rc = lib.veon_internal_bwd_pixels(base, ptr(depth, s * N * D * HW), ptr(feat, s * N * HW * C),
                                          ptr(plan.point_interval, s * N * HW * D), i64(N * HW), D, HW, C,
                                          ptr(dg, s * N * D * HW), ptr(fg, s * N * HW * C),
                                          P(s_pix.cuda_stream))
        assert rc == 0, rc
        ev_pix[s].record(s_pix)
    main.wait_event(ev_pix[B - 1])
    done2 = torch.cuda.Event()
    done2.record(s_rows)
    main.wait_event(done2)


dg.zero_(); fg.zero_()
ringed()
torch.cuda.synchronize()
print("ringed == two launches:", torch.equal(dg, want_dg), torch.equal(fg, want_fg))
print(f"ring of two samples, no window: {ev_ms(ringed, n=20) * 1e3:.1f} us")
for mb in (40, 72):
    for st in (s_rows, s_pix):
        rc = lib.veon_internal_l2_window(P(st.cuda_stream), ptr(ring), ctypes.c_size_t(ring.numel() * 4),
                                         ctypes.c_float(min(1.0, mb * 2 ** 20 / (ring.numel() * 4))),
                                         ctypes.c_size_t(mb << 20))
        assert rc == 0, rc
    print(f"  + ring window, {mb} MB set aside: {ev_ms(ringed, n=20) * 1e3:.1f} us")
