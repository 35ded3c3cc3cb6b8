"""Forward pooling: streaming two-role kernel vs the general kernel (bit-exact) + timings, at
C = 64 (the only width the streaming kernel takes) and over ring sizes of 2 ... 16 slots per SM.
    python tools/fwd_check.py [check] [time]
Run under `timeout`: the streaming kernel spins on flags, a bug there hangs instead of failing."""
import sys
import time

import torch

import os
sys.path.insert(0, ".")
from veon_b200 import _lib, bev_pool as BP, synthetic as S  # noqa: E402
if os.environ.get("VEON_LIB"):          # an experimental build of tools/build_variant.sh
    _lib.LIB_PATH = os.environ["VEON_LIB"]

RING_SLOTS = (2, 4, 8, 16)              # ring slots per SM (the library's default is 8)


def setup(cfg_name, B, C, seed=0):
    cfg = S.CONFIGS[cfg_name]
    lower, interval, size = S.grid_vectors(cfg.grid_config)
    coor = torch.from_numpy(S.lidar_coor_np(cfg, batch=B)).cuda()
    _, N, D, H, W, _ = coor.shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    depth = torch.softmax(torch.randn(B, N, D, H, W, device="cuda", generator=g) * 4, dim=2)
    feat = torch.randn(B, N, H, W, C, device="cuda", generator=g)
    prep = BP.prepare_ranks(coor, lower, interval, size)
    return prep, depth, feat, (B, C, 16, 200, 200)


def ring(ns):
    """A streaming-forward workspace of `ns` slots (512 rows x 64 channels) per SM."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    return torch.empty(sms * ns * 512 * 64 * 4, dtype=torch.uint8, device="cuda")


def planar(prep, depth, feat, shape, ws=None, out=None):
    """veon_bev_pool_v2_fwd_planar: without a workspace the general kernel; with the whole plan and
    a workspace (C = 64) the streaming kernel, its ring sized by the workspace."""
    lib = _lib.load()
    B, C = shape[0], shape[1]
    V = 640000
    if out is None:
        out = torch.full(shape, float("nan"), device="cuda")
    p = prep.plan
    stream = ws is not None
    rc = lib.veon_bev_pool_v2_fwd_planar(
        BP._ptr(depth), BP._ptr(feat), BP._ptr(prep.ranks_depth), BP._ptr(prep.ranks_feat),
        BP._ptr(prep.ranks_bev), BP._ptr(p.tile_start), BP._ptr(p.tile_istart) if stream else None,
        BP._ptr(p.tile_occ) if stream else None, BP._ptr(p.tile_heavy), p.tile_heavy.numel(), B, C,
        V, feat.numel() // C, BP._ptr(out), BP._ptr(ws) if stream else None,
        ws.numel() if stream else 0, BP._stream_ptr(depth.device))
    assert rc == 0, rc
    return out


def general(prep, depth, feat, shape, out=None):
    return planar(prep, depth, feat, shape, out=out)


def ev_ms(fn, n=20, warm=3):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    what = sys.argv[1:] or ["check", "time"]
    if "check" in what:
        for cfg, B in (("C1", 1), ("C1", 2), ("C1", 4), ("small", 3), ("C3", 1), ("C3", 2),
                       ("C2", 8)):
            prep, depth, feat, shape = setup(cfg, B, 64)
            b = general(prep, depth, feat, shape)
            for ns in RING_SLOTS:
                t0 = time.time()
                ws = ring(ns)
                a = planar(prep, depth, feat, shape, ws)
                torch.cuda.synchronize()
                same = torch.equal(a, b)
                print(f"check {cfg} B={B} C=64 ring={ns} slots/SM: equal={same} "
                      f"({time.time() - t0:.2f}s)", flush=True)
                if not same:
                    d = (a != b) | (a.isnan() != b.isnan())
                    idx = d.nonzero()
                    print("  mismatches:", int(d.sum()), "first:", idx[:5].tolist())
                # twice more: the ring and its barriers are reused
                for _ in range(2):
                    assert torch.equal(planar(prep, depth, feat, shape, ws), b) == same
                del a, ws
            del b, prep, depth, feat
    if "time" in what:
        for cfg, B in (("C2", 8), ("C3", 4)):
            prep, depth, feat, shape = setup(cfg, B, 64)
            scratch = torch.empty(shape, device="cuda")
            tg = ev_ms(lambda: general(prep, depth, feat, shape, scratch), n=10)
            line = f"time {cfg} B={B} C=64: general {tg * 1e3:.1f} us"
            for ns in RING_SLOTS:
                ws = ring(ns)
                ts = ev_ms(lambda: planar(prep, depth, feat, shape, ws, scratch), n=10)
                line += f" | {ns} slots/SM: {ts * 1e3:.1f} us"
                del ws
            gb = 4.0 * 640000 * 64 * B / 1e9
            line += f"   (volume {gb:.2f} GB)"
            print(line, flush=True)
            del scratch, prep, depth, feat


if __name__ == "__main__":
    main()
