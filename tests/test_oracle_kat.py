"""Known-answer tests of the CPU oracle (oracle/wr_oracle.c) and its independent NumPy twin.

The reference holds no golden vectors for the rasterizer boundary (nvdiffrast is un-vendored), so these
hand-derivable cases pin the contract of DESIGN.md section 3: pixel-centre sampling, row 0 = NDC y -1,
top-left fill rule, id+1 / barycentric layout (render.py:53, warp.py:138-143), nearest depth wins with
lowest id on ties, z/w range rejection, geometric clipping with inherited ids."""
import numpy as np
import pytest

import cases
from oracle import raster_numpy, shim


def centre(k, n):
    return (2 * k + 1) / n - 1


def corner(k, n):
    return 2 * k / n - 1


def test_rect_through_pixel_centres_is_top_left_inclusive():
    W = H = 6
    x0, x1, y0, y1 = centre(1, W), centre(3, W), centre(1, H), centre(4, H)
    pos = np.array([[[x0, y0, 0, 1], [x1, y0, 0, 1], [x1, y1, 0, 1], [x0, y1, 0, 1]]], np.float32)
    want = -np.ones((H, W), np.int32)
    want[1:4, 1:3] = 0  # columns 1,2 (left edge in, right edge out), rows 1,2,3 (top edge in, bottom edge out)
    for tri in ([[0, 1, 2], [0, 2, 3]], [[0, 2, 1], [0, 3, 2]]):  # both windings are rasterised
        _, ids = shim.rasterize(pos, np.array(tri, np.int32), (H, W))
        assert ((ids[0] >= 0) == (want >= 0)).all()


def test_shared_diagonal_covers_every_pixel_once():
    W = H = 6
    pos = np.array([[[corner(0, W), corner(0, H), 0, 1], [corner(6, W), corner(0, H), 0, 1],
                     [corner(0, W), corner(6, H), 0, 1], [corner(6, W), corner(6, H), 0, 1]]], np.float32)
    rast, ids = shim.rasterize(pos, np.array([[0, 1, 2], [1, 3, 2]], np.int32), (H, W))
    yy, xx = np.mgrid[0:H, 0:W]
    want = np.where(xx + yy < W - 1, 0, 1)  # centres exactly on the diagonal go to exactly one triangle
    np.testing.assert_array_equal(ids[0], want)
    # layout (u, v, z/w, id+1): u weighs vertex 0, v vertex 1 (warp.py:140-143)
    np.testing.assert_allclose(rast[0, 0, 0], [1 - 1 / 6, 1 / 12, 0.0, 1.0], atol=1e-6)
    np.testing.assert_allclose(rast[0, 2, 1], [1 - 1.5 / 6 - 2.5 / 6, 1.5 / 6, 0.0, 1.0], atol=1e-6)
    assert rast[0, 5, 5, 3] == 2.0


def test_row_zero_is_ndc_y_minus_one():
    pos = np.array([[[-1, -1, 0, 1], [1, -1, 0, 1], [0, -0.5, 0, 1]]], np.float32)  # hugs the NDC y = -1 border
    _, ids = shim.rasterize(pos, np.array([[0, 1, 2]], np.int32), (8, 8))
    assert (ids[0, 0] >= 0).any() and (ids[0, 4:] == -1).all()


def test_nearest_depth_wins_then_lowest_id():
    q, t = cases.quad_fullscreen()
    near = q.copy(); near[..., 2] = -0.5
    far = q.copy(); far[..., 2] = 0.5
    pos = np.concatenate([far, near, near], 1)
    tri = np.concatenate([t, t + 4, t + 8], 0)
    rast, ids = shim.rasterize(pos, tri, (8, 8))
    assert set(np.unique(ids)) == {2, 3}  # the nearer copy with the lower ids
    np.testing.assert_allclose(rast[..., 2], -0.5)


def test_depth_range_and_offscreen_rejection():
    q, t = cases.quad_fullscreen()
    for z in (-1.5, 1.5):
        p = q.copy(); p[..., 2] = z
        _, ids = shim.rasterize(p, t, (8, 8))
        assert (ids == -1).all()
    p = q.copy(); p[..., 0] += 5.0
    assert (shim.rasterize(p, t, (8, 8))[1] == -1).all()
    p = q.copy(); p[..., 3] = -1.0  # behind the camera
    assert (shim.rasterize(p, t, (8, 8))[1] == -1).all()


def test_degenerate_subpixel_and_bad_indices():
    pos = np.array([[[0.1, 0.1, 0, 1], [0.1, 0.1, 0, 1], [0.3, 0.3, 0, 1],      # zero area
                     [0.01, 0.01, 0, 1], [0.012, 0.01, 0, 1], [0.01, 0.012, 0, 1],  # between sample points
                     [np.nan, 0, 0, 1], [1, 0, 0, 1], [0, 1, 0, 1]]], np.float32)
    tri = np.array([[0, 1, 2], [3, 4, 5], [6, 7, 8], [0, 1, 99], [-1, 0, 1]], np.int32)
    rast, ids = shim.rasterize(pos, tri, (16, 16))
    assert (ids == -1).all() and (rast == 0).all()


def test_near_plane_clip_keeps_parent_id_and_matches_unclipped_part():
    # a triangle reaching behind the camera: the visible part must be covered, with the parent's id
    pos = np.array([[[-0.5, -0.5, 0.0, 1.0], [0.5, -0.5, 0.0, 1.0], [0.0, 2.0, -3.0, -1.0]]], np.float32)
    _, ids = shim.rasterize(pos, np.array([[0, 1, 2]], np.int32), (32, 32))
    assert (ids >= 0).sum() > 20 and set(np.unique(ids)) <= {-1, 0}


def test_perspective_correct_barycentrics():
    # w differs per vertex: the barycentric of the pixel nearest to the screen-space centroid is NOT 1/3
    pos = np.array([[[-0.8, -0.8, 0.0, 1.0], [1.6, -1.6, 0.0, 2.0], [0.0, 3.2, 0.0, 4.0]]], np.float32)
    rast, ids = shim.rasterize(pos, np.array([[0, 1, 2]], np.int32), (64, 64))
    y, x = np.argwhere(ids[0] == 0)[len(np.argwhere(ids[0] == 0)) // 2]
    u, v = rast[0, y, x, 0], rast[0, y, x, 1]
    px, py = centre(x, 64), centre(y, 64)
    # reconstruct: sum_i b_i * clip_i, divided by its w, must land on the pixel centre
    b = np.array([u, v, 1 - u - v])
    clip = (b[:, None] * pos[0]).sum(0)
    np.testing.assert_allclose(clip[:2] / clip[3], [px, py], atol=1e-5)


@pytest.mark.parametrize("name", ["soup", "ties", "fan", "near", "mix", "guard"])
def test_c_oracle_equals_numpy_twin(name):
    pos, tri, res = {
        "soup": (*cases.random_soup(3, 60, B=2, perspective=True), (40, 56)),
        "ties": (*cases.snapped_grid_soup(0, 80, 24, 20), (20, 24)),
        "fan": (*cases.shared_edge_fan(12), (33, 33)),
        "near": (*cases.near_crossing_scene(5, 40), (32, 48)),
        "mix": (*cases.big_and_small_mix(9), (48, 48)),
        "guard": (*cases.guard_band_scene(13, 24), (40, 40)),
    }[name]
    if name == "mix":
        pos, tri = pos[:, :309], tri[:103]  # keep the pure-Python twin fast
    rast, ids = shim.rasterize(pos, tri, res)
    rast2, ids2 = raster_numpy.rasterize(pos, tri, res)
    np.testing.assert_array_equal(ids, ids2)
    np.testing.assert_array_equal(rast, rast2)
    attr = np.random.default_rng(0).standard_normal((1, pos.shape[1], 3)).astype(np.float32)
    np.testing.assert_array_equal(shim.interpolate(attr, rast, tri), raster_numpy.interpolate(attr, rast, tri))


def test_interpolate_zero_on_background_and_broadcast():
    pos, tri = cases.random_soup(1, 30, B=2)
    rast, ids = shim.rasterize(pos, tri, (24, 24))
    attr = np.ones((1, pos.shape[1], 2), np.float32)
    out = shim.interpolate(attr, rast, tri)
    assert (out[ids < 0] == 0).all()
    np.testing.assert_allclose(out[ids >= 0], 1.0, atol=1e-6)  # constant attribute -> partition of unity


def test_texture_nearest_linear_wrap():
    tex = np.arange(2 * 2 * 1, dtype=np.float32).reshape(1, 2, 2, 1)  # [[0,1],[2,3]]
    uv = np.array([[[[0.25, 0.25], [0.75, 0.25], [0.25, 0.75], [0.5, 0.5], [1.25, 0.25], [-0.25, 0.25]]]], np.float32)
    np.testing.assert_array_equal(shim.texture(tex, uv, "nearest")[0, 0, :, 0], [0, 1, 2, 3, 0, 1])
    lin = shim.texture(tex, uv, "linear")[0, 0, :, 0]
    np.testing.assert_allclose(lin[:4], [0, 1, 2, 1.5], atol=1e-6)  # texel centres exact, middle = mean
    np.testing.assert_allclose(lin[4], lin[0]) and np.testing.assert_allclose(lin[5], lin[1])


def test_sizes_and_empty():
    for res in [(1, 1), (3, 5), (17, 9)]:
        pos, tri = cases.quad_fullscreen()
        _, ids = shim.rasterize(pos, tri, res)
        assert (ids >= 0).all()
    r, i = shim.rasterize(np.zeros((1, 0, 4), np.float32), np.zeros((0, 3), np.int32), (4, 4))
    assert (i == -1).all() and (r == 0).all()


@pytest.mark.parametrize("H,W,C", [(1, 17, 1), (33, 20, 3), (64, 96, 4), (7, 5, 2)])
def test_grid_sample_matches_the_reference_operator(H, W, C):
    """render_oracle.grid_sample (the statement wr_grid_sample and the bake kernels follow bit for bit) against
    torch.nn.functional.grid_sample(bilinear, zeros, align_corners=False) itself, at non-square maps.

    Finite coordinates: not bit-exact, because torch forms the tap weights as (x0 + 1 - ix) where the oracle has
    1 - (ix - x0), and its pixel coordinate ix may round differently.  A shift of ix or iy by up to one ulp of the map
    extent moves the result by at most 2 * ulp(max(H, W)) * max |tap difference| <= 4 eps max(H, W) max |img|;
    measured up to 1.3e-5 on N(0, 1) maps of up to 64 x 96 (the bound there is 1.8e-4).

    Non-finite coordinates: torch returns NaN on CPU and 0 on CUDA; the oracle (and every kernel) returns 0 -- the
    sample adds nothing (DESIGN.md section 4)."""
    import torch
    import torch.nn.functional as F
    from oracle import render_oracle
    rng = np.random.default_rng(10 * H + W)
    img = rng.standard_normal((H, W, C)).astype(np.float32)
    ndc = rng.uniform(-1.3, 1.3, (23, 31, 2)).astype(np.float32)
    def edge(n):   # the borders, one pixel in / out of them, a pixel centre, -0
        return np.array([-1, 1, -1 - 1 / n, -1 + 1 / n, 1 - 1 / n, 1 + 1 / n, (2 * (n // 2) + 1) / n - 1, -0.0], np.float32)
    ndc[0, :8, 0] = edge(W)
    ndc[1, :8, 1] = edge(H)
    got = render_oracle.grid_sample(img, ndc)
    ref = F.grid_sample(torch.from_numpy(img).permute(2, 0, 1)[None], torch.from_numpy(ndc)[None], mode="bilinear",
                        padding_mode="zeros", align_corners=False)[0].permute(1, 2, 0).numpy()
    assert got.shape == (23, 31, C)
    tol = 4 * np.finfo(np.float32).eps * max(H, W) * np.abs(img).max()
    np.testing.assert_allclose(got, ref, rtol=0, atol=tol)
    assert np.abs(ref).max() > 0.5   # not a field of zeros

    bad = np.array([[np.nan, 0.0], [0.0, np.nan], [np.inf, 0.0], [-np.inf, 0.5], [0.25, np.inf], [0.0, -np.inf],
                    [np.inf, np.nan]], np.float32)[None]
    np.testing.assert_array_equal(render_oracle.grid_sample(img, bad), np.zeros((1, len(bad[0]), C), np.float32))
