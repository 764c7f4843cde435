"""The Poisson solve of a multi-GPU bake split into row bands (csrc/blend.cu wr_poisson_band_step, parallel.py), on ONE
device.

wr_poisson_band_step takes per-rank pointers to the iterate planes and output atlases: here they are N local buffer
sets standing in for the peer mappings, and the N ranks' stage generators (parallel._poisson_band_stages, the code the
real path runs with a symmetric-memory barrier at every yield) are stepped in lock step on one stream.  Every emulated
rank's output must equal wr_poisson_blend of the whole atlas bit for bit: each point gets the same float operations in
the same order."""
import ctypes

import pytest
import torch

import worldrenderer_b200 as wr
from worldrenderer_b200 import _native, parallel
from worldrenderer_b200.uv import atlas_postprocess

from test_gpu_bake_parity import _setup

GRAD_MODES = {"src": 0, "max": 1, "avg": 2}


def _lockstep(gens):
    """Runs every generator to its next yield, rank by rank, until all are exhausted (the barrier of the real path)."""
    end = object()
    while True:
        got = [next(g, end) for g in gens]
        if all(x is end for x in got):
            return
        assert not any(x is end for x in got), "the ranks yield a different number of times"


def _band_solve(c, src, mask, tgt, num_iters, grad_mode, world):
    """The banded solve over `world` emulated ranks; returns every rank's output atlas."""
    H, W, C = tgt.shape
    dev = tgt.device
    lay = [parallel.poisson_band_layout(H, W, C, world, r, num_iters) for r in range(world)]
    # stale values wherever a kernel reads what nobody wrote
    xa = [torch.full((max(l.plane_bytes // 4, 4),), float("nan"), device=dev) for l in lay]
    xb = [torch.full((max(l.plane_bytes // 4, 4),), float("nan"), device=dev) for l in lay]
    b = [torch.full((l.plane_bytes,), 0xFF, dtype=torch.uint8, device=dev) for l in lay]
    m = [torch.full((l.mask_bytes,), 0xFF, dtype=torch.uint8, device=dev) for l in lay]
    out = [torch.full((H, W, C), -5.0, device=dev) for _ in range(world)]
    ptrs = lambda ts: [t.data_ptr() for t in ts]
    args = [parallel._poisson_band_args(src, mask, tgt, num_iters, grad_mode, world, r, ptrs(xa), ptrs(xb), ptrs(out),
                                        b[r], m[r]) for r in range(world)]
    _lockstep([parallel._poisson_band_stages(c, a) for a in args])
    torch.cuda.synchronize()
    return out


def _emulated_band_run(c, world):
    """band_run of parallel._bake_tail over emulated ranks: checks that they agree, returns rank 0's atlas."""
    def run(src, mask, tgt, num_iters, grad_mode):
        outs = _band_solve(c, src, mask, tgt, num_iters, grad_mode, world)
        for r in range(1, world):
            assert torch.equal(outs[r], outs[0]), f"rank {r} holds another atlas than rank 0"
        return outs[0]
    return run


def _poisson_blend(c, src, mask, tgt, num_iters, grad_mode):
    H, W, C = tgt.shape
    out = torch.empty_like(tgt)
    c.check(_native.lib().wr_poisson_blend(c.handle, _native.ptr(src), _native.ptr(mask), _native.ptr(tgt), H, W, C,
                                           int(num_iters), int(grad_mode), _native.ptr(out), c.stream()),
            "wr_poisson_blend")
    torch.cuda.synchronize()
    return out


def _inputs(H, W, C, dev, seed, empty_mask=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    src = torch.rand((H, W, C), generator=g) * 1.4 - 0.2     # beyond [0, 1]: the finish clamps
    tgt = torch.rand((H, W, C), generator=g)
    mask = torch.zeros((H, W), dtype=torch.uint8)
    if not empty_mask:
        # the left half: touches the top, bottom and left border and crosses every band boundary; a ragged,
        # holed region on the right
        mask[:, : W // 2] = 1
        mask[H // 5:, W // 2:] = (torch.rand((H - H // 5, W - W // 2), generator=g) < 0.8).to(torch.uint8)
        mask[H // 3: H // 3 + 5, :] = 0
    return src.to(dev).contiguous(), mask.to(dev).contiguous(), tgt.to(dev).contiguous()


def _check(c, H, W, C, num_iters, mode, world, seed, empty_mask=False):
    src, mask, tgt = _inputs(H, W, C, torch.device(c.device), seed, empty_mask)
    want = _poisson_blend(c, src, mask, tgt, num_iters, GRAD_MODES[mode])
    outs = _band_solve(c, src, mask, tgt, num_iters, GRAD_MODES[mode], world)
    for r, o in enumerate(outs):
        assert torch.equal(o, want), f"rank {r}: {(o != want).sum().item()} values differ from wr_poisson_blend"


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 4, 8])
@pytest.mark.parametrize("mode", ["src", "max", "avg"])
@pytest.mark.parametrize("num_iters", [0, 1, 7, 8, 9, 64])
def test_band_small_atlas_every_iteration_count(wr_ctx, world, mode, num_iters):
    """96 x 172: two tile rows, so 4 and 8 ranks leave empty bands."""
    _check(wr_ctx.ctx, 96, 172, 3, num_iters, mode, world, seed=num_iters * 10 + world)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 4, 8])
@pytest.mark.parametrize("H,W,C,num_iters,mode", [
    (1030, 1024, 3, 64, "src"),    # ragged last tile row
    (1024, 1030, 3, 9, "max"),     # ragged last tile column
    (2048, 2048, 3, 64, "avg"),
    (1024, 1024, 3, 1000, "src"),  # the reference's default sweep count
    (200, 300, 1, 17, "avg"),
    (160, 500, 2, 64, "max"),
    (300, 260, 4, 9, "src"),
])
def test_band_equals_poisson_blend(wr_ctx, world, H, W, C, num_iters, mode):
    _check(wr_ctx.ctx, H, W, C, num_iters, mode, world, seed=H + W + C + world)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 8])
def test_band_empty_mask(wr_ctx, world):
    _check(wr_ctx.ctx, 500, 333, 3, 24, "src", world, seed=3, empty_mask=True)


def test_band_layout_follows_shard_bounds():
    """Bands are whole tile rows of the 112 x 48 tiling, dealt out by shard_bounds; S = ceil(num_iters / 8)."""
    for H, W, C, world in [(96, 172, 3, 8), (1030, 1024, 3, 3), (4096, 4096, 3, 8), (47, 5, 1, 2), (16384, 64, 4, 16)]:
        tiles_y, Wp = -(-H // 48), -(-W // 112) * 112 + 16
        for r, (t0, t1) in enumerate(parallel.shard_bounds(tiles_y, world)):
            lay = parallel.poisson_band_layout(H, W, C, world, r, 1001)
            assert (lay.row_lo, lay.row_hi) == (min(t0 * 48, H), min(t1 * 48, H))
            rows = (t1 - t0) * 48 + 16 if t1 > t0 else 0
            assert lay.plane_bytes == rows * Wp * C * 4 and lay.mask_bytes == rows * Wp
            assert lay.steps == 126
    for bad in [(0, 8, 3, 2, 0), (8, 8, 5, 2, 0), (8, 8, 3, 2, 2), (8, 8, 3, 17, 0), (8, 8, 3, 2, -1)]:
        with pytest.raises(ValueError):
            parallel.poisson_band_layout(*bad)


@pytest.mark.gpu
def test_band_step_rejects_bad_arguments(wr_ctx):
    c = wr_ctx.ctx
    dev = wr_ctx.device
    H, W, C, world = 100, 100, 3, 2
    src, mask, tgt = _inputs(H, W, C, dev, seed=1)
    lay = [parallel.poisson_band_layout(H, W, C, world, r) for r in range(world)]
    xs = [torch.zeros(l.plane_bytes // 4, device=dev) for l in lay for _ in range(2)]
    b = torch.zeros(lay[0].plane_bytes, dtype=torch.uint8, device=dev)
    m = torch.zeros(lay[0].mask_bytes, dtype=torch.uint8, device=dev)
    out = [torch.zeros((H, W, C), device=dev) for _ in range(world)]

    def args(**kw):
        a = parallel._poisson_band_args(src, mask, tgt, 16, 0, world, 0, [xs[0].data_ptr(), xs[2].data_ptr()],
                                        [xs[1].data_ptr(), xs[3].data_ptr()], [o.data_ptr() for o in out], b, m)
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    def status(a):
        return _native.lib().wr_poisson_band_step(c.handle, ctypes.byref(a), c.stream())

    assert status(args()) == 0
    for kw in [dict(rank=2), dict(rank=-1), dict(world=0), dict(world=17), dict(C=5), dict(C=0), dict(step=-1),
               dict(step=4), dict(grad_mode=3), dict(num_iters=-1), dict(src=None), dict(b=None), dict(m=None),
               dict(b=b.data_ptr() + 4)]:
        assert status(args(**kw)) != 0, kw
    for field, r in [("xa", 0), ("xb", 0), ("xa", 1), ("xb", 1), ("out", 1)]:   # rank 1 is rank 0's neighbour below
        a = args()
        getattr(a, field)[r] = None
        assert status(a) != 0, (field, r)
    assert _native.lib().wr_poisson_band_step(c.handle, None, c.stream()) != 0
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("keep_border,from_scratch", [(True, False), (False, False), (False, True)])
def test_banded_bake_tail_equals_atlas_postprocess(wr_ctx, world, keep_border, from_scratch):
    """parallel._bake_tail with the band solve (sharded_bake's peer-memory path) against the replicated tail."""
    mesh, cam, images = _setup(wr_ctx.device, uv_size=512)
    img = torch.from_numpy(images).to(wr_ctx.device)
    atlas, valid_any = parallel.sharded_bake(wr_ctx, mesh, cam, img, 512)
    atlas, valid_any = atlas.clone(), valid_any.clone()
    pre = parallel._uv_precompute_cached(wr_ctx, mesh, 512)
    solver = wr.PoissonBlendingSolver("torch-cuda", str(wr_ctx.device))
    kw = dict(pb_solver=solver, pb_num_iters=1000, pb_keep_original_border=keep_border)
    want = atlas_postprocess(None, atlas, valid_any, pre, do_uv_padding=True, pad_unseen_area=from_scratch,
                             poisson_blending=True, **kw)
    got = parallel._bake_tail(atlas, valid_any, pre, uv_padding=True, poisson_blending=True, from_scratch=from_scratch,
                              band_run=_emulated_band_run(wr_ctx.ctx, world), **kw)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    # and sharded_bake of one process (no peer memory: the replicated tail) gives the same atlas
    got1, _ = parallel.sharded_bake(wr_ctx, mesh, cam, img, 512, uv_padding=True, poisson_blending=True,
                                    from_scratch=from_scratch, **kw)
    assert torch.equal(got1, want)


@pytest.mark.gpu
@pytest.mark.parametrize("from_scratch", [False, True])
def test_bake_pipeline_tail_equals_sharded_bake(wr_ctx, from_scratch):
    """BakePipeline(postprocess=...): the tail on the pipeline's exchange stream, three bakes through two slots, equal
    sharded_bake with the same flags, also when more bakes are in flight than the pipeline has slots."""
    mesh, cam, images = _setup(wr_ctx.device, uv_size=256)
    img = torch.from_numpy(images).to(wr_ctx.device)
    imgs = [img, img.flip(0).contiguous(), (img * 0.5).contiguous()]
    solver = wr.PoissonBlendingSolver("torch-cuda", str(wr_ctx.device))
    tail = dict(uv_padding=True, poisson_blending=True, pb_solver=solver, pb_num_iters=200,
                pb_keep_original_border=not from_scratch, from_scratch=from_scratch)
    want = [tuple(t.clone() for t in parallel.sharded_bake(wr_ctx, mesh, cam, im, 256, **tail)) for im in imgs]
    pipe = parallel.BakePipeline(wr_ctx, 256, depth=2, postprocess=tail)
    got = []
    for im in imgs:
        got.append(pipe.submit(mesh, cam, im))
        if len(got) >= 2:   # consume with one bake in flight behind
            a, m = got[-2].result()
            got[-2] = (a.clone(), m.clone())
    a, m = got[-1].result()
    got[-1] = (a.clone(), m.clone())
    torch.cuda.synchronize()
    for (a, m), (wa, wm) in zip(got, want):
        assert torch.equal(m, wm) and torch.equal(a, wa)
    with pytest.raises(NotImplementedError):   # the tail is the pipeline's, not the bake's
        pipe.submit(mesh, cam, img, pb_num_iters=10)
    with pytest.raises(ValueError):
        parallel.BakePipeline(wr_ctx, 256, postprocess=dict(uv_padding=True, radius=4))
