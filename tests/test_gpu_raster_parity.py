"""GPU parity, operator level: wr_rasterize / wr_interpolate / wr_texture (through the
NVDiffRastContextWrapper methods, i.e. through the C ABI) against the CPU oracle on the same inputs.

Bar: triangle ids and coverage bit-exact; (u, v, z/w) and interpolated attributes within 1e-5 relative
(in practice they are bit-identical too, which the tests report and assert where it must hold).
"""
import numpy as np
import pytest
import torch

import cases
from oracle import shim

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6


def _gpu_rasterize(ctx, pos, tri, res):
    rast, ids = ctx.rasterize_with_ids(torch.from_numpy(pos).to(ctx.device), torch.from_numpy(tri).to(ctx.device), res)
    torch.cuda.synchronize()
    return rast.cpu().numpy(), ids.cpu().numpy()


def _check(ctx, pos, tri, res):
    ref_rast, ref_ids = shim.rasterize(pos, tri, res)
    rast, ids = _gpu_rasterize(ctx, pos, tri, res)
    assert ids.shape == ref_ids.shape
    bad = np.argwhere(ids != ref_ids)
    assert bad.size == 0, f"{len(bad)} pixels differ, first {bad[:5].tolist()}: gpu {ids[tuple(bad[0])]} ref {ref_ids[tuple(bad[0])]}"
    np.testing.assert_array_equal(rast[..., 3], ref_rast[..., 3])
    np.testing.assert_allclose(rast[..., :3], ref_rast[..., :3], rtol=RTOL, atol=ATOL)
    return rast, ids, ref_rast


def test_fullscreen_quad(wr_ctx):
    pos, tri = cases.quad_fullscreen()
    for res in [(8, 8), (16, 24), (33, 17), (768, 768)]:
        rast, ids, _ = _check(wr_ctx, pos, tri, res)
        assert (ids >= 0).all()  # every pixel covered exactly once by one of the two triangles
        assert set(np.unique(ids)) == {0, 1}


def test_empty_inputs(wr_ctx):
    pos = np.zeros((2, 0, 4), np.float32)
    tri = np.zeros((0, 3), np.int32)
    rast, ids = _gpu_rasterize(wr_ctx, pos, tri, (16, 16))
    assert (ids == -1).all() and (rast == 0).all()
    pos, _ = cases.quad_fullscreen()
    rast, ids = _gpu_rasterize(wr_ctx, pos, tri, (16, 16))
    assert (ids == -1).all() and (rast == 0).all()


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("res", [(64, 64), (97, 131), (512, 384)])
def test_random_soup(wr_ctx, seed, res):
    pos, tri = cases.random_soup(seed, 400, B=3)
    _check(wr_ctx, pos, tri, res)


@pytest.mark.parametrize("seed", [3, 4])
def test_random_soup_perspective(wr_ctx, seed):
    pos, tri = cases.random_soup(seed, 600, B=2, perspective=True)
    _check(wr_ctx, pos, tri, (256, 256))


@pytest.mark.parametrize("seed", [0, 1])
def test_fill_rule_ties(wr_ctx, seed):
    pos, tri = cases.snapped_grid_soup(seed, 300, 48, 40)
    _check(wr_ctx, pos, tri, (40, 48))


def test_shared_edges_watertight(wr_ctx):
    pos, tri = cases.shared_edge_fan(24)
    rast, ids, _ = _check(wr_ctx, pos, tri, (255, 255))
    # disc interior: no holes along the spokes
    yy, xx = np.mgrid[0:255, 0:255]
    r = np.hypot((2 * xx + 1) / 255 - 1, (2 * yy + 1) / 255 - 1)
    assert (ids[0][r < 0.85] >= 0).all()


def test_near_plane_and_negative_w(wr_ctx):
    pos, tri = cases.near_crossing_scene()
    _check(wr_ctx, pos, tri, (200, 320))


def test_guard_band_clipping(wr_ctx):
    pos, tri = cases.guard_band_scene()
    for res in [(128, 128), (600, 800)]:
        rast, ids, _ = _check(wr_ctx, pos, tri, res)
        assert (ids >= 0).mean() > 0.3


def test_big_small_degenerate_mix(wr_ctx):
    pos, tri = cases.big_and_small_mix()
    for res in [(300, 300), (1024, 1024)]:
        _check(wr_ctx, pos, tri, res)


@pytest.mark.parametrize("res", [(768, 1024), (333, 517), (2048, 2048)])
def test_tile_pass_huge_triangles(wr_ctx, res):
    """Hundreds of screen-sized triangles with depth ties, tiny triangles around them and clipped ones: the tile
    pass (binning, per-band lists in shared memory, register resolve) against the oracle, bit for bit."""
    pos, tri = cases.huge_triangle_scene()
    rast, ids, ref = _check(wr_ctx, pos, tri, res)
    np.testing.assert_array_equal(rast.view(np.uint32), ref.view(np.uint32))
    assert (ids >= 0).mean() > 0.9 and len(np.unique(ids)) > 100
    # only huge triangles, few of them (a single batch), and a box-like mesh through render()
    pos, tri = cases.huge_triangle_scene(seed=5, n_huge=9, n_small=0, n_clip=0, B=1)
    _check(wr_ctx, pos, tri, res)


def test_large_viewport_4096(wr_ctx):
    pos, tri = cases.random_soup(11, 64, B=1)
    rast, ids = _gpu_rasterize(wr_ctx, pos, tri, (4096, 4096))
    ref_rast, ref_ids = shim.rasterize(pos, tri, (4096, 4096))
    np.testing.assert_array_equal(ids, ref_ids)


def test_equal_depth_lowest_id_wins(wr_ctx):
    pos, tri = cases.quad_fullscreen()
    pos = np.concatenate([pos, pos], 1)
    tri = np.concatenate([tri + 4, tri], 0)  # duplicates: ids 0,1 and 2,3 cover the same pixels at the same depth
    rast, ids, _ = _check(wr_ctx, pos, tri, (32, 32))
    assert ids.max() <= 1


def test_range_mode(wr_ctx):
    pos, tri = cases.random_soup(21, 300, B=1)
    ranges = torch.tensor([[0, 100], [100, 150], [250, 50], [0, 0]], dtype=torch.int32)
    rast, ids = wr_ctx.rasterize_with_ids(torch.from_numpy(pos[0]).to(wr_ctx.device),
                                          torch.from_numpy(tri).to(wr_ctx.device), (96, 96), ranges=ranges)
    ids = ids.cpu().numpy()
    for b, (s, n) in enumerate(ranges.tolist()):
        _, ref = shim.rasterize(pos, tri[s:s + n], (96, 96))
        ref = np.where(ref >= 0, ref + s, -1)
        np.testing.assert_array_equal(ids[b], ref[0])


def test_interpolate_and_texture(wr_ctx):
    rng = np.random.default_rng(0)
    pos, tri = cases.random_soup(7, 500, B=2)
    rast, ids = _gpu_rasterize(wr_ctx, pos, tri, (128, 160))
    dev = wr_ctx.device
    for A, attr_B in [(3, 1), (2, 2), (7, 1)]:
        attr = rng.standard_normal((attr_B, pos.shape[1], A)).astype(np.float32)
        tri2 = rng.permutation(tri.reshape(-1)).reshape(-1, 3).astype(np.int32)  # a different index buffer
        out, empty = wr_ctx.interpolate(torch.from_numpy(attr).to(dev), torch.from_numpy(rast).to(dev),
                                        torch.from_numpy(tri2).to(dev))
        assert empty.shape == (2, 128, 160, 0)
        ref = shim.interpolate(attr, rast, tri2)
        np.testing.assert_array_equal(out.cpu().numpy(), ref)
    tex = rng.uniform(0, 1, (1, 37, 53, 3)).astype(np.float32)
    uv = rng.uniform(-1.5, 2.5, (2, 128, 160, 2)).astype(np.float32)
    for filt in ["nearest", "linear"]:
        for bnd in ["wrap", "clamp", "zero"]:
            out = wr_ctx.texture(torch.from_numpy(tex).to(dev), torch.from_numpy(uv).to(dev), filter_mode=filt,
                                 boundary_mode=bnd)
            ref = shim.texture(tex, uv, filt, bnd)
            np.testing.assert_array_equal(out.cpu().numpy(), ref, err_msg=f"{filt}/{bnd}")


def test_mesh_views_ids_bit_exact(wr_ctx):
    """Clip positions produced by the oracle's fixed-order transform, rasterised by both sides."""
    v, f = cases.icosphere_mesh(12)
    cam = cases.canonical_cameras()
    clip = shim.clip_positions(v, cam.mvp_mtx.numpy())
    _check(wr_ctx, clip, f, (256, 256))
    v, f = cases.terrain_mesh(96, 48)
    for cams in [cases.canonical_cameras(), cases.perspective_cameras(), cases.inside_cameras()]:
        clip = shim.clip_positions(v, cams.mvp_mtx.numpy())
        _check(wr_ctx, clip, f, (192, 256))


def test_maximum_viewport_8192(wr_ctx):
    pos, tri = cases.random_soup(17, 24, B=1)
    rast, ids = _gpu_rasterize(wr_ctx, pos, tri, (8192, 8192))
    _, ref_ids = shim.rasterize(pos, tri, (8192, 8192))
    np.testing.assert_array_equal(ids, ref_ids)
    with pytest.raises(RuntimeError):
        wr_ctx.rasterize_with_ids(torch.from_numpy(pos).to(wr_ctx.device), torch.from_numpy(tri).to(wr_ctx.device), (8193, 64))
    with pytest.raises(ValueError):
        wr_ctx.rasterize_with_ids(torch.from_numpy(pos[0, :, :3]).to(wr_ctx.device), torch.from_numpy(tri).to(wr_ctx.device), (64, 64))
