"""Compute share of one rank in the banded Poisson solve, on one GPU.

Times wr_poisson_blend on the whole atlas against the work ONE rank of the banded solve (wr_poisson_band_step) does
for N ranks: its setup, sweep launches, halo kernels and finish, with its neighbours emulated by local buffers on the
same GPU (so the halo loads and the finish's stores to the other ranks' atlases go to local HBM, not over NVLink, and
no barrier runs).  The rank timed is the busiest band: rank 1 (two neighbours, a tall band) from 3 ranks up, rank 0
for 2.  These are compute shares per rank, not a multi-GPU time.  Also times one seam padding (wr_uv_padding), which
every rank still runs on the whole atlas.  CUDA events, after warm-up; median [min-max] over the repetitions.

usage: python tools/poisson_band_probe.py [--size 4096] [--iters 1000] [--reps 7]"""
import argparse
import ctypes
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from worldrenderer_b200 import _native, parallel  # noqa: E402
from worldrenderer_b200.uv import uv_padding  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--size", type=int, default=4096)
ap.add_argument("--iters", type=int, default=1000)
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--worlds", default="2,4,8")
a = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("poisson_band_probe: no CUDA device")
dev = torch.device("cuda", 0)
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"device: {torch.cuda.get_device_name(dev)} | nvidia-smi name, power limit, max SM clock: {smi}")

H = W = a.size
C = 3
g = torch.Generator().manual_seed(0)
src = torch.rand((H, W, C), generator=g).to(dev)
tgt = torch.rand((H, W, C), generator=g).to(dev)
yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
# atlas-like: large charts separated by 12-texel gutters
mask = (((yy % 256) >= 12) & ((xx % 340) >= 12)).to(torch.uint8).to(dev).contiguous()
c = _native.NativeContext(dev)


def timed(fn):
    fn()
    fn()  # warm-up
    torch.cuda.synchronize()
    ts = []
    for _ in range(a.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def fmt(t):
    return f"{t[0]:8.3f} ms [{t[1]:.3f}-{t[2]:.3f}]"


out1 = torch.empty_like(tgt)


def full():
    c.check(_native.lib().wr_poisson_blend(c.handle, _native.ptr(src), _native.ptr(mask), _native.ptr(tgt), H, W, C,
                                           a.iters, 0, _native.ptr(out1), c.stream()), "wr_poisson_blend")


t_full = timed(full)
print(f"wr_poisson_blend {H}x{W}x{C}, {a.iters} sweeps: {fmt(t_full)}")
t_pad = timed(lambda: uv_padding(tgt, mask, 3, c))
print(f"wr_uv_padding {H}x{W}x{C} (radius 3, run by every rank): {fmt(t_pad)}")

for world in [int(w) for w in a.worlds.split(",")]:
    rank = 1 if world >= 3 else 0
    lay = [parallel.poisson_band_layout(H, W, C, world, r, a.iters) for r in range(world)]
    need = [r for r in (rank - 1, rank, rank + 1) if 0 <= r < world and lay[r].plane_bytes]
    xa = [torch.zeros(max(l.plane_bytes // 4, 4), device=dev) for l in lay]
    xb = [torch.zeros(max(l.plane_bytes // 4, 4), device=dev) for l in lay]
    bs = [torch.empty(l.plane_bytes, dtype=torch.uint8, device=dev) for l in lay]
    ms = [torch.empty(l.mask_bytes, dtype=torch.uint8, device=dev) for l in lay]
    outs = [torch.empty_like(tgt) for _ in range(world)]
    ptrs = lambda ts: [t.data_ptr() for t in ts]
    args = {r: parallel._poisson_band_args(src, mask, tgt, a.iters, 0, world, r, ptrs(xa), ptrs(xb), ptrs(outs), bs[r],
                                           ms[r]) for r in need}
    for r in need:   # the neighbours' planes hold a set-up iterate, as they would
        args[r].step = 0
        c.check(_native.lib().wr_poisson_band_step(c.handle, ctypes.byref(args[r]), c.stream()), "wr_poisson_band_step")

    def band():
        for _ in parallel._poisson_band_stages(c, args[rank]):
            pass

    t_band = timed(band)
    rows = lay[rank].row_hi - lay[rank].row_lo
    print(f"N={world}: rank {rank} ({rows} rows, {lay[rank].steps} sweep launches + halo kernels + finish into {world} "
          f"atlases): {fmt(t_band)}  = {t_band[0] / t_full[0]:.3f} of the whole solve (1/N = {1 / world:.3f})")
    del xa, xb, bs, ms, outs, args
    torch.cuda.empty_cache()
