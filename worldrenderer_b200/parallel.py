"""Multi-GPU partitioning of the geometry path (one process per GPU, torch.distributed).

The reference is single-GPU (SURVEY.md section 2b); this module is the new functionality
BASELINE.json asks for:

* Rendering shards with NO data-path collective: units (mesh, view) are independent.  `shard_bounds`
  gives rank r a contiguous, balanced slice of the meshes (config D) or of the views (config E).
* The bake has ONE exchange step.  Because
      sum_v attr_v * (w_v / max(sum_v w_v, 1e-5))  ==  (sum_v attr_v * w_v) / max(sum_v w_v, 1e-5)
  (uv.py:342-344, 421-423; the outer clamp(0, 1) is a no-op for w >= 0), each rank accumulates
  [Huv, Wuv, 5] = (sum w r, sum w g, sum w b, sum w, sum valid) over its local views with
  wr_uv_unproject, the ranks all-reduce that tensor (NCCL over NVLink / NVSwitch; gloo in the CPU
  tests) and every rank finalises with wr_uv_finalize.  The valid count travels as a float sum of small
  integers, which is exact, so `uv_valid_mask_blend` is identical on every rank and to the 1-GPU result;
  the colour sums differ from the 1-GPU result only by fp32 summation order (1e-5 relative).
"""
from __future__ import annotations

import contextlib
import ctypes
import warnings
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import _native
from .camera import Camera


def shard_bounds(n: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous balanced partition of range(n) into `world` slices (first n % world slices get one more)."""
    if world <= 0:
        raise ValueError("world size must be positive")
    base, extra = divmod(n, world)
    out, start = [], 0
    for r in range(world):
        size = base + (1 if r < extra else 0)
        out.append((start, start + size))
        start += size
    return out


def my_shard(n: int, rank: Optional[int] = None, world: Optional[int] = None) -> Tuple[int, int]:
    if rank is None or world is None:
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
        else:
            rank, world = 0, 1
    return shard_bounds(n, world)[rank]


def shard_slice(n: int, rank: Optional[int] = None, world: Optional[int] = None, interleave: bool = False) -> slice:
    """This rank's share of range(n) as a slice: a contiguous block (`shard_bounds`), or every world-th item
    starting at `rank`.  Interleaving is the better split for the views of a camera ring: the cost of a view depends
    on where it looks from, and neighbouring views cost alike, so contiguous blocks leave the ranks unevenly loaded
    (config E on 8 GPUs: slowest rank 1.36 ms contiguous, 1.21 ms interleaved, mean 1.2 ms)."""
    if rank is None or world is None:
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
        else:
            rank, world = 0, 1
    if interleave:
        return slice(rank, n, world)
    lo, hi = shard_bounds(n, world)[rank]
    return slice(lo, hi)


def shard_camera(cam: Camera, rank: Optional[int] = None, world: Optional[int] = None, interleave: bool = False) -> Camera:
    """The views of `cam` owned by this rank (possibly an empty camera batch)."""
    return cam[shard_slice(cam.mvp_mtx.shape[0], rank, world, interleave)]


def all_reduce_accumulators(accum: torch.Tensor, group=None) -> torch.Tensor:
    """SUM all-reduce of the packed bake accumulators, in place.  No-op outside a process group."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(accum, op=dist.ReduceOp.SUM, group=group)
    return accum


def finalize_accumulators_reference(accum: torch.Tensor, old_attr: Optional[torch.Tensor]):
    """Plain torch statement of wr_uv_finalize (uv.py:452-455), used by the CPU tests of the decomposition."""
    den = accum[..., 3:4].clamp(min=1e-5)
    any_ = accum[..., 4] > 0.5
    va = any_[..., None].to(accum.dtype)
    old = torch.zeros_like(accum[..., :3]) if old_attr is None else old_attr
    return (accum[..., :3] / den) * va + old * (1.0 - va), any_


def render_mesh_shard(ctx, meshes: Sequence, cam: Camera, height: int, width: int, rank: Optional[int] = None,
                      world: Optional[int] = None, **render_kwargs):
    """Config D: every rank renders its contiguous slice of `meshes` (all views each).  Returns
    (first mesh index, [RenderOutput, ...]).  No communication."""
    from .render import render
    lo, hi = my_shard(len(meshes), rank, world)
    return lo, [render(ctx, meshes[i], cam, height, width, **render_kwargs) for i in range(lo, hi)]


class P2PBakeWorkspace:
    """Peer-mapped (torch symmetric memory) buffers of the multi-GPU bake: every rank's accumulators, atlas and
    mask are addressable from every GPU of the node over NVLink / NVSwitch, which is what
    wr_uv_reduce_finalize_p2p reads and writes.  Creating one is a collective call."""

    def __init__(self, uv_h: int, uv_w: int, device: torch.device, group=None):
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if self.world > _native.MAX_P2P_RANKS:
            raise RuntimeError(f"at most {_native.MAX_P2P_RANKS} ranks share a peer-memory bake")
        T = uv_h * uv_w
        if T % 4 != 0:
            raise RuntimeError("peer-memory bake needs uv_h * uv_w to be a multiple of 4")
        self.uv_h, self.uv_w, self.T = uv_h, uv_w, T
        self._off_accum, self._off_attr, self._off_valid = 0, 20 * T, 32 * T  # byte offsets, all 16-byte aligned
        self.buf = symm_mem.empty(33 * T, dtype=torch.uint8, device=device)
        self.hdl = symm_mem.rendezvous(self.buf, self.group)
        self.base_ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        try:  # NVSwitch multicast window over the same allocation (0 / absent when NVLS is not available)
            self.mc_ptr = int(getattr(self.hdl, "multicast_ptr", 0) or 0)
        except Exception:
            self.mc_ptr = 0
        self.accum = self.buf[0:20 * T].view(torch.float32).view(uv_h, uv_w, 5)
        self.attr = self.buf[20 * T:32 * T].view(torch.float32).view(uv_h, uv_w, 3)
        self.valid = self.buf[32 * T:33 * T].view(uv_h, uv_w)

    def barrier(self, channel: int) -> None:
        self.hdl.barrier(channel=channel)  # device-side, ordered on the current stream

    def reduce_finalize(self, ctx, old_attr: Optional[torch.Tensor], multicast: Optional[bool] = None,
                        max_blocks: int = 0, tex_range: Optional[Tuple[int, int]] = None, last: bool = True):
        """multicast: True / False force the NVSwitch multicast (multimem) or the peer load / store kernel; None
        picks multicast from 4 ranks up when the window exists (measured on 8 x B200, 4096^2 atlas: multicast
        0.64 ms, peer 1.19 ms, NCCL all_reduce + finalize 1.09 ms; on 2 ranks peer 0.52 ms, multicast 0.79 ms)."""
        a = _native.P2PReduceArgs()
        if multicast is None:
            multicast = bool(self.mc_ptr) and self.world >= 4
        if multicast and self.mc_ptr:
            a.mc_accum = self.mc_ptr + self._off_accum
            a.mc_attr = self.mc_ptr + self._off_attr
            a.mc_valid = self.mc_ptr + self._off_valid
        elif multicast:
            raise RuntimeError("no multicast window for this workspace")
        for r in range(self.world):
            a.accum[r] = self.base_ptrs[r] + self._off_accum
            a.out_attr[r] = self.base_ptrs[r] + self._off_attr
            a.out_valid[r] = self.base_ptrs[r] + self._off_valid
        old = None
        if old_attr is not None:
            old = old_attr.to(torch.float32).contiguous()
            a.old_attr = _native.ptr(old)
        a.world, a.rank, a.Hu, a.Wu = self.world, self.rank, self.uv_h, self.uv_w
        a.max_blocks = int(max_blocks)
        if tex_range is not None:   # one chunk of the atlas: every rank owns 1/N of it
            a.tex_lo, a.tex_hi = int(tex_range[0]), int(tex_range[1])
        self.barrier(0)  # every rank's accumulators (of this chunk) are complete
        c = ctx.ctx
        c.check(_native.lib().wr_uv_reduce_finalize_p2p(c.handle, ctypes.byref(a), c.stream()),
                "wr_uv_reduce_finalize_p2p")
        if last:
            self.barrier(1)  # every rank's share of this atlas has landed
        del old
        return self.attr, self.valid.view(torch.bool)


_P2P_WORKSPACES: Dict[tuple, "P2PBakeWorkspace"] = {}
_P2P_DISABLED = False


def _p2p_workspace(uv_h: int, uv_w: int, device: torch.device, group, slot: int = 0) -> Optional["P2PBakeWorkspace"]:
    """Workspace `slot` for (size, group), created on first use; None when peer memory is not usable (then NCCL).
    A collective call the first time: every rank must ask for the same (size, group, slot) in the same order."""
    global _P2P_DISABLED
    if _P2P_DISABLED or not (dist.is_available() and dist.is_initialized()):
        return None
    if dist.get_backend(group) != "nccl" or dist.get_world_size(group) < 2 or (uv_h * uv_w) % 4 != 0:
        return None
    key = (uv_h, uv_w, device.index, id(group), int(slot))
    ws = _P2P_WORKSPACES.get(key)
    if ws is None:
        ws = _agreed_workspace(lambda: P2PBakeWorkspace(uv_h, uv_w, device, group), device, group,
                               "peer-memory bake unavailable", "using NCCL all_reduce")
        if ws is None:
            _P2P_DISABLED = True
            return None
        _P2P_WORKSPACES[key] = ws
    return ws


def _agreed_workspace(make, device: torch.device, group, what: str, instead: str):
    """make() on every rank of `group`, or None on every rank if it failed on any (a collective call)."""
    err = None
    try:
        ws = make()
    except Exception as e:
        ws, err = None, e
    # symm_mem.empty is a LOCAL allocation: it can fail on one rank only (out of memory).  Agree on the outcome
    # before anyone commits to a path, or that rank would sit in all_reduce while the others wait on the
    # symmetric-memory barrier.
    ok = torch.tensor([0 if ws is None else 1], dtype=torch.int32, device=device)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
    if int(ok.item()) == 0:
        why = f"{type(err).__name__}: {err}" if err is not None else "another rank could not set it up"
        warnings.warn(f"{what} ({why}); {instead}")
        return None
    return ws


class PoissonBandLayout(NamedTuple):
    plane_bytes: int   # one [C, band rows + 16, padded width] float plane (0: no tile row in this band)
    mask_bytes: int    # the region plane, one byte per plane point
    steps: int         # sweep launches S = ceil(num_iters / 8)
    row_lo: int        # image rows [row_lo, row_hi) this rank finishes
    row_hi: int


def poisson_band_layout(H: int, W: int, C: int, world: int, rank: int, num_iters: int = 0) -> PoissonBandLayout:
    """Plane sizes and band of `rank` in the banded Poisson solve (wr_poisson_band_layout)."""
    plane, mask = ctypes.c_uint64(), ctypes.c_uint64()
    steps, lo, hi = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    st = _native.lib().wr_poisson_band_layout(H, W, C, world, rank, num_iters, ctypes.byref(plane), ctypes.byref(mask),
                                              ctypes.byref(steps), ctypes.byref(lo), ctypes.byref(hi))
    if st != 0:
        raise ValueError(f"wr_poisson_band_layout({H}, {W}, {C}, world={world}, rank={rank}, num_iters={num_iters}): "
                         f"{_native.lib().wr_status_string(st).decode()}")
    return PoissonBandLayout(plane.value, mask.value, steps.value, lo.value, hi.value)


def _poisson_band_args(src, mask, tgt, num_iters: int, grad_mode: int, world: int, rank: int, xa, xb, out, b, m):
    """wr_poisson_band_args of one rank: src / tgt [H,W,C] float32 and mask [H,W] u8 local tensors; xa, xb, out the
    `world` device addresses of every rank's iterate planes and output atlas; b, m this rank's local planes."""
    H, W, C = tgt.shape
    a = _native.PoissonBandArgs()
    a.src, a.mask, a.tgt = _native.ptr(src), _native.ptr(mask), _native.ptr(tgt)
    a.H, a.W, a.C, a.num_iters, a.grad_mode, a.world, a.rank = H, W, C, int(num_iters), int(grad_mode), world, rank
    for r in range(world):
        a.xa[r], a.xb[r], a.out[r] = xa[r], xb[r], out[r]
    a.b, a.m = _native.ptr(b), _native.ptr(m)
    return a


def _poisson_band_stages(c: "_native.NativeContext", a: "_native.PoissonBandArgs"):
    """Launches the steps of one rank's share of a banded Poisson solve on the current stream and yields wherever a
    barrier across the ranks belongs: after every sweep launch (the next one pulls its halo rows from what the
    neighbours' launch wrote), before the finish (it stores into every rank's output, which the previous solve's
    readers may still hold) and after it (every output is complete).  The caller puts the barrier there; every
    rank yields the same number of times, a rank without a tile row included."""
    steps = poisson_band_layout(a.H, a.W, a.C, a.world, a.rank, a.num_iters).steps
    for step in range(steps + 2):
        a.step = step
        c.check(_native.lib().wr_poisson_band_step(c.handle, ctypes.byref(a), c.stream()), "wr_poisson_band_step")
        if step > 0 or steps == 0:
            yield


class PoissonBandWorkspace:
    """Buffers of the banded Poisson solve of a multi-GPU bake: every rank's two iterate planes and output atlas in
    torch symmetric memory (the halo rows are pulled from the neighbours' planes and the finished rows stored into
    every rank's atlas over NVLink / NVSwitch), the right-hand side and region planes local.  Creating one is a
    collective call."""

    def __init__(self, H: int, W: int, C: int, device: torch.device, group=None):
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if self.world > _native.MAX_P2P_RANKS:
            raise RuntimeError(f"at most {_native.MAX_P2P_RANKS} ranks share a banded Poisson solve")
        self.shape = (H, W, C)
        lay = [poisson_band_layout(H, W, C, self.world, r) for r in range(self.world)]
        plane = (max(l.plane_bytes for l in lay) + 255) & ~255   # every rank maps the same symmetric size
        self._off_xb, self._off_out = plane, 2 * plane
        self.buf = symm_mem.empty(2 * plane + H * W * C * 4, dtype=torch.uint8, device=device)
        self.hdl = symm_mem.rendezvous(self.buf, self.group)
        self.base_ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        own = lay[self.rank]
        self.b = torch.empty(own.plane_bytes, dtype=torch.uint8, device=device)
        self.m = torch.empty(own.mask_bytes, dtype=torch.uint8, device=device)
        self.out = self.buf[2 * plane:].view(torch.float32).view(H, W, C)

    def barrier(self, channel: int) -> None:
        self.hdl.barrier(channel=channel)  # device-side, ordered on the current stream

    def solve(self, c: "_native.NativeContext", src, mask, tgt, num_iters: int, grad_mode: int) -> torch.Tensor:
        """wr_poisson_blend(src, mask, tgt) of the whole atlas on every rank, each rank sweeping its band; the result is
        `out`, a view of the workspace (valid until the next solve).  Every rank of the group must call it alike."""
        if tuple(tgt.shape) != self.shape:
            raise ValueError(f"workspace is for {self.shape}, got {tuple(tgt.shape)}")
        a = _poisson_band_args(src, mask, tgt, num_iters, grad_mode, self.world, self.rank,
                               [p for p in self.base_ptrs], [p + self._off_xb for p in self.base_ptrs],
                               [p + self._off_out for p in self.base_ptrs], self.b, self.m)
        for _ in _poisson_band_stages(c, a):
            self.barrier(0)
        return self.out


_PB_WORKSPACES: Dict[tuple, "PoissonBandWorkspace"] = {}
_PB_DISABLED = False


def _poisson_workspace(H: int, W: int, C: int, device: torch.device, group, slot: int = 0) -> Optional[PoissonBandWorkspace]:
    """Banded-solve workspace `slot` for (atlas size, group), created on first use; None when peer memory is not usable
    (then every rank runs the whole solve).  A collective call the first time, like _p2p_workspace."""
    global _PB_DISABLED
    if _PB_DISABLED or not (dist.is_available() and dist.is_initialized()):
        return None
    if dist.get_backend(group) != "nccl" or dist.get_world_size(group) < 2:
        return None
    key = (H, W, C, device.index, id(group), int(slot))
    ws = _PB_WORKSPACES.get(key)
    if ws is None:
        ws = _agreed_workspace(lambda: PoissonBandWorkspace(H, W, C, device, group), device, group,
                               "banded Poisson solve unavailable", "every rank solves the whole atlas")
        if ws is None:
            _PB_DISABLED = True
            return None
        _PB_WORKSPACES[key] = ws
    return ws


class _BandPoissonSolver:
    """Stands in for a PoissonBlendingSolver in atlas_postprocess: the same inputs and sweep count, solved by
    `run(src, mask_u8, tgt, sweeps, grad_mode)` (the banded solve), which returns the blended atlas."""

    def __init__(self, solver, run):
        self.solver, self.run = solver, run

    def __call__(self, src, mask, tgt, num_iters, inplace=True, grad_mode="src"):
        assert not inplace   # sharded_bake's tail writes a fresh atlas
        src_c, mask_c, tgt_c, gm = self.solver._inputs(src, mask, tgt, inplace, grad_mode)
        return self.run(src_c, mask_c, tgt_c, self.solver._sweeps(num_iters), gm)


def _bake_tail(atlas, valid_any, pre, *, uv_padding: bool, poisson_blending: bool, pb_solver, pb_num_iters: int,
               pb_keep_original_border: bool, from_scratch: bool, band_run=None, native_ctx=None):
    """The post-processing tail of uv_blend (uv.py:426-461) on the exchanged atlas, on the current stream.  Every
    padding runs on every rank; with `band_run` (see _BandPoissonSolver) the Poisson solve of a PoissonBlendingSolver
    is split into row bands across the ranks instead.  Either way the result is identical on every rank."""
    from .blend import PoissonBlendingSolver
    from .uv import atlas_postprocess
    if band_run is not None and poisson_blending and isinstance(pb_solver, PoissonBlendingSolver):
        pb_solver = _BandPoissonSolver(pb_solver, band_run)
    return atlas_postprocess(None, atlas, valid_any, pre, do_uv_padding=uv_padding, pad_unseen_area=from_scratch,
                             poisson_blending=poisson_blending, pb_solver=pb_solver, pb_num_iters=pb_num_iters,
                             pb_keep_original_border=pb_keep_original_border, native_ctx=native_ctx)


_PRE_CACHE: Dict[tuple, tuple] = {}
_PRE_CACHE_SLOTS = 4


def _uv_precompute_cached(ctx, mesh, uv_size: int):
    """uv_precompute is replicated on every rank and depends on the mesh and atlas size only: the last few
    (device, mesh tensors, size) results are kept while the mesh tensors are unchanged (same storage and version;
    the entry holds the tensors themselves, so their addresses cannot be recycled), like CameraProjection does."""
    from .uv import UVPrecomputeOutput, uv_precompute
    srcs = (mesh.v_pos, mesh.t_pos_idx, mesh.v_tex, mesh.t_tex_idx)
    key = (ctx.device.index, int(uv_size)) + tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in srcs)
    hit = _PRE_CACHE.pop(key, None)
    if hit is None or any(a is not b for a, b in zip(hit[0], srcs)):
        pre = uv_precompute(ctx, mesh, uv_size, uv_size)
        hit = (srcs, pre.uv_mask, pre.uv_pos)
    _PRE_CACHE[key] = hit                       # most recently used last
    while len(_PRE_CACHE) > _PRE_CACHE_SLOTS:
        _PRE_CACHE.pop(next(iter(_PRE_CACHE)))
    return UVPrecomputeOutput(height=uv_size, width=uv_size, uv_attr=mesh.texture, uv_mask=hit[1], uv_pos=hit[2])


def sharded_bake(ctx, mesh, cam_local: Camera, images_local: torch.Tensor, uv_size: int, *, view_masks_local=None,
                 aoi_cos_valid_threshold: float = 0.3, depth_grad_dilation: int = 5,
                 depth_grad_threshold: Optional[float] = 0.1, uv_exp_blend_alpha: float = 6.0,
                 uv_exp_blend_view_weight_local=None, group=None, exchange: str = "auto",
                 uv_padding: bool = False, poisson_blending: bool = False, pb_solver=None, pb_num_iters: int = 1000,
                 pb_keep_original_border: bool = True, from_scratch: bool = False, chunks: int = 8,
                 chunk_shape: str = "equal", _slot: int = 0,
                 _exchange_stream: Optional["torch.cuda.Stream"] = None, _exchange_blocks: int = 0,
                 _tail_ctx: Optional["_native.NativeContext"] = None):
    """Config E: this rank holds `cam_local` / `images_local` (its share of the views, possibly none);
    the mesh is replicated.  Returns (atlas [uv,uv,3], valid_any [uv,uv] bool), identical on all ranks.

    exchange: "p2p"  -- one fused kernel over NVLink peer memory (reduce-scatter + finalise + all-gather);
              "nccl" -- all_reduce(SUM) of the accumulators, then wr_uv_finalize on every rank;
              "auto" -- p2p when symmetric memory is available for the group, else nccl.
    With "p2p" / "auto" the returned tensors are views of the workspace: valid until the next bake of that size.

    chunks: with peer memory the atlas is unprojected and exchanged in this many chunks, the exchange of chunk k on a
    side stream under the unprojection of chunk k + 1 (1 = unproject everything, then exchange); chunk_shape "equal"
    or "falling" (sizes K : K-1 : ... : 1).

    uv_padding / poisson_blending: the post-processing tail of uv_blend (uv.py:426-461) applied to the exchanged
    atlas; the returned atlas is then a fresh tensor, still identical on all ranks.  Every rank runs each seam
    padding on its own copy.  With peer memory and a PoissonBlendingSolver the Poisson solve is split into row bands,
    one per rank, that trade 8 halo rows per 8 sweeps and gather the result into every rank's atlas over NVLink; the
    result is bit-identical to every rank solving the whole atlas, which is what the NCCL path does."""
    from .blend import PoissonBlendingSolver
    from .uv import fused_unproject, fused_view_maps, uv_finalize
    if exchange not in ("auto", "p2p", "nccl"):
        raise ValueError(f"exchange={exchange!r}")
    pre = _uv_precompute_cached(ctx, mesh, uv_size)
    ws = _p2p_workspace(uv_size, uv_size, ctx.device, group, _slot) if exchange != "nccl" else None
    if exchange == "p2p" and ws is None:
        raise RuntimeError("exchange='p2p' requested but peer memory is not available for this process group")
    pws = None
    if ws is not None and poisson_blending and isinstance(pb_solver, PoissonBlendingSolver):
        pws = _poisson_workspace(uv_size, uv_size, 3, ctx.device, group, _slot)
    n_local = cam_local.mvp_mtx.shape[0]
    accum = ws.accum if ws is not None else None
    geo = att = None
    if n_local > 0:
        H, W = int(images_local.shape[1]), int(images_local.shape[2])
        _, geo, att = fused_view_maps(ctx, mesh, cam_local, images_local, H, W, int(depth_grad_dilation))

    def unproject(tex_range=None):
        nonlocal accum
        if n_local > 0:
            _, _, accum, _, _ = fused_unproject(
                ctx, pre, cam_local, H, W, geo, att, view_masks=view_masks_local, aoi_cos_thresh=aoi_cos_valid_threshold,
                depth_grad_thresh=depth_grad_threshold, alpha=uv_exp_blend_alpha,
                view_weight=uv_exp_blend_view_weight_local, accumulate_only=True, accum=accum, add_to_accum=False,
                tex_range=tex_range)

    cur = torch.cuda.current_stream(ctx.device)
    xs = _exchange_stream
    ntex = uv_size * uv_size
    nchunks = max(1, min(int(chunks), ntex // (1 << 16))) if ws is not None else 1
    if nchunks > 1:
        # The atlas in chunks: the exchange of a finished chunk runs on the side stream under the unprojection of the
        # next one (every rank runs the same chunk loop: the barriers inside reduce_finalize pair up).
        if n_local == 0:
            accum.zero_()
        side = xs if xs is not None else _side_stream(ctx.device)
        # Chunk sizes: equal by default.  Unprojection and exchange of a chunk take about the same time, so the bake
        # ends up as view passes + U(1) + sum of max(U(k + 1), X(k)) + X(K): falling sizes (K : K-1 : ... : 1, small
        # last exchange) put the large exchanges next to small unprojections and measured slower -- config E on
        # 8 x B200, chunks 4 / 6 / 8: falling 1.427 / 1.402 / 1.408 ms, equal 1.389 / 1.369 / 1.361 ms (one chunk: 1.703).
        # Boundaries on 1024 texels (the exchange kernels' blocks).
        bounds = chunk_bounds(ntex, nchunks, chunk_shape)
        # a small exchange grid leaves the SMs to the unprojection: one block per SM for the multicast kernel (its best
        # anyway), two for the peer-load kernel (it needs more loads in flight)
        sms = torch.cuda.get_device_properties(ctx.device).multi_processor_count
        blocks = _exchange_blocks or sms * (1 if (ws.mc_ptr and ws.world >= 4) else 2)
        for k, rng in enumerate(bounds):
            unproject(rng)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                atlas, valid_any = ws.reduce_finalize(ctx, pre.uv_attr, max_blocks=blocks, tex_range=rng,
                                                      last=k == len(bounds) - 1)
        if xs is None:
            cur.wait_stream(side)
    else:
        if n_local > 0:
            unproject()
        elif accum is not None:
            accum.zero_()
        else:
            accum = torch.zeros((uv_size, uv_size, 5), dtype=torch.float32, device=ctx.device)
        if xs is not None:  # BakePipeline: the exchange (and everything after it) runs on its own stream
            xs.wait_stream(cur)
            accum.record_stream(xs)
        with torch.cuda.stream(xs) if xs is not None else contextlib.nullcontext():
            if ws is not None:
                atlas, valid_any = ws.reduce_finalize(ctx, pre.uv_attr, max_blocks=_exchange_blocks)
            else:
                all_reduce_accumulators(accum, group)
                atlas, valid_any = uv_finalize(ctx, accum, pre.uv_attr)
    if uv_padding or poisson_blending:
        if xs is not None:   # BakePipeline: the tail follows the exchange on its stream
            for t in (pre.uv_mask, pre.uv_attr):
                if t is not None:
                    t.record_stream(xs)
        nctx = _tail_ctx if _tail_ctx is not None else _native.default_context(ctx.device)
        band_run = (lambda *a: pws.solve(nctx, *a)) if pws is not None else None
        with torch.cuda.stream(xs) if xs is not None else contextlib.nullcontext():
            atlas = _bake_tail(atlas, valid_any, pre, uv_padding=uv_padding, poisson_blending=poisson_blending,
                               pb_solver=pb_solver, pb_num_iters=pb_num_iters,
                               pb_keep_original_border=pb_keep_original_border, from_scratch=from_scratch,
                               band_run=band_run, native_ctx=_tail_ctx)
    return atlas, valid_any


def chunk_bounds(ntex: int, nchunks: int, shape: str = "equal") -> List[Tuple[int, int]]:
    """Texel ranges [lo, hi) of a chunked bake: a partition of range(ntex) into at most `nchunks` non-empty ranges whose
    inner boundaries are multiples of 1024 texels (the exchange kernels' blocks).  shape "equal": equal sizes;
    "falling": sizes K : K-1 : ... : 1 (a small last exchange)."""
    if shape not in ("falling", "equal"):
        raise ValueError("chunk_shape must be 'falling' or 'equal'")
    nchunks = max(1, int(nchunks))
    weights = [nchunks - k if shape == "falling" else 1 for k in range(nchunks)]
    total_w = sum(weights)
    bounds, lo = [], 0
    for k in range(nchunks):
        hi = ntex if k == nchunks - 1 else min(ntex, (lo + ntex * weights[k] // total_w + 1023) & ~1023)
        if hi > lo:
            bounds.append((lo, hi))
        lo = hi
    return bounds


_SIDE_STREAMS: Dict[int, "torch.cuda.Stream"] = {}


def _side_stream(device: torch.device) -> "torch.cuda.Stream":
    """High-priority stream for the exchange chunks of a single sharded_bake (one per device)."""
    s = _SIDE_STREAMS.get(device.index)
    if s is None:
        s = _SIDE_STREAMS[device.index] = torch.cuda.Stream(device, priority=-1)
    return s


_TAIL_FLAGS = ("uv_padding", "poisson_blending", "pb_solver", "pb_num_iters", "pb_keep_original_border", "from_scratch")


class BakeTicket:
    """Result of one `BakePipeline.submit`: `result()` makes the current stream wait for the exchange (and the
    post-processing tail, if asked for) and returns (atlas [uv,uv,3], valid_any [uv,uv] bool), identical on every
    rank.  With peer memory the tensors are views of a pipeline slot: valid until `depth` more bakes have been
    submitted (a post-processed atlas is a fresh tensor)."""

    def __init__(self, atlas, valid_any, done: "torch.cuda.Event", device):
        self._atlas, self._valid, self._done, self._device = atlas, valid_any, done, device

    def result(self):
        torch.cuda.current_stream(self._device).wait_event(self._done)
        return self._atlas, self._valid


class BakePipeline:
    """Batched multi-GPU baking (a stream of config-E bakes: SmartPainter rounds, a queue of meshes).

    One bake on N ranks is [render + unproject this rank's views] -> [exchange the accumulators, finalise]: the first
    part shrinks with N, the exchange does not (4096^2 x 20 B leave and 13 B reach every GPU over NVLink whatever N
    is), so a single bake cannot scale past compute / (compute + exchange).  A batch can: the exchange of bake k runs
    on its own stream, on pipeline slot k % depth (accumulators, atlas and barrier pads of its own in symmetric
    memory), while the compute stream already renders bake k + 1.  Throughput is then bounded by the longer of the two
    stages instead of their sum.  Every rank must submit the same bakes in the same order.

    postprocess: the post-processing tail every bake of the pipeline gets, as a dict of sharded_bake's tail flags
    (uv_padding, poisson_blending, pb_solver, pb_num_iters, pb_keep_original_border, from_scratch); None = the
    exchanged atlas.  The tail runs on the exchange stream behind the exchange of the same bake, with a native context
    of its own (the compute stream is already rendering the next bake with `ctx`).  With peer memory and a
    PoissonBlendingSolver the Poisson solve is banded across the ranks, with a workspace per slot set up here.  The
    tail is fixed per pipeline, not per bake: `submit` refuses these flags."""

    def __init__(self, ctx, uv_size: int, depth: int = 2, group=None, exchange: str = "auto", exchange_blocks_per_sm: int = 1,
                 postprocess: Optional[dict] = None):
        self.ctx, self.uv_size, self.depth, self.group, self.exchange = ctx, int(uv_size), max(1, int(depth)), group, exchange
        # the exchange kernel with its default grid (8 blocks per SM) takes every thread slot of the GPU and, at
        # high priority, simply runs INSTEAD of the next bake's view passes (measured: no overlap at all); it is bound
        # by NVLink, so a block or two per SM moves the same bytes in about the same time and leaves the SMs alone
        self._xblocks = max(1, int(exchange_blocks_per_sm)) * torch.cuda.get_device_properties(ctx.device).multi_processor_count
        self.device = ctx.device
        # high priority: the exchange kernel's blocks are placed as soon as SM slots free up instead of queueing
        # behind every block the compute stream has already launched (it is NVLink-bound and needs few of them)
        self._xs = torch.cuda.Stream(self.device, priority=-1)
        self._done: List[Optional[torch.cuda.Event]] = [None] * self.depth
        self._k = 0
        self._tail = dict(postprocess or {})
        unknown = set(self._tail) - set(_TAIL_FLAGS)
        if unknown:
            raise ValueError(f"postprocess: unknown flags {sorted(unknown)}")
        self._tail_ctx = _native.NativeContext(self.device) if self._tail else None
        if exchange != "nccl":   # collective set-up of every slot, up front and in the same order on all ranks
            from .blend import PoissonBlendingSolver
            banded = self._tail.get("poisson_blending") and isinstance(self._tail.get("pb_solver"), PoissonBlendingSolver)
            for slot in range(self.depth):
                if _p2p_workspace(self.uv_size, self.uv_size, self.device, group, slot) is not None and banded:
                    _poisson_workspace(self.uv_size, self.uv_size, 3, self.device, group, slot)

    def submit(self, mesh, cam_local: Camera, images_local: torch.Tensor, **bake_kwargs) -> BakeTicket:
        for k in _TAIL_FLAGS:
            if k in bake_kwargs:
                raise NotImplementedError("BakePipeline runs the post-processing tail given to its constructor "
                                          "(postprocess=...); it is not chosen per bake")
        slot = self._k % self.depth
        self._k += 1
        cur = torch.cuda.current_stream(self.device)
        if self._done[slot] is not None:   # the slot's previous exchange must have drained before its accumulators are rewritten
            cur.wait_event(self._done[slot])
        atlas, valid_any = sharded_bake(self.ctx, mesh, cam_local, images_local, self.uv_size, group=self.group,
                                        exchange=self.exchange, _slot=slot, _exchange_stream=self._xs,
                                        _exchange_blocks=self._xblocks, _tail_ctx=self._tail_ctx, **self._tail,
                                        **bake_kwargs)
        done = torch.cuda.Event()
        done.record(self._xs)
        self._done[slot] = done
        return BakeTicket(atlas, valid_any, done, self.device)
