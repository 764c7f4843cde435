"""Kernel output against the independent float64 geometry reference (oracle/geometry_f64.py), on the GPU.

The bit-exact parity tests hold the kernels to the C oracle, which restates the contract; these hold them to the
geometry, at the shapes and edges where the kernels have separate paths: the per-view queues, the coarse-lane set-up
(4 F <= H W) and the fine one, the tile pass (huge_triangle_scene), range mode, odd and large viewports, B = 1 / 9 /
40, render()'s multi-view switch, inside-the-mesh cameras on both render paths, stitched meshes, the attribute
and tangent maps and half-precision maps.  The UV bake is not held to this reference yet.  At every decided
pixel the id must be the float64 winner and every float within its a-priori float32 bound; a decided-fraction floor
keeps each case from going vacuous."""
import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import geometry_f64 as g
from worldrenderer_b200.render import render_geometry_raw
from test_oracle_f64 import adversarial_soup

pytestmark = pytest.mark.gpu

f32 = np.float32


def _rasterize(ctx, pos, tri, H, W):
    rast, ids = ctx.rasterize_with_ids(torch.from_numpy(np.ascontiguousarray(pos)).to(ctx.device),
                                       torch.from_numpy(tri).to(ctx.device), (H, W))
    return rast.cpu().numpy(), ids.cpu().numpy()


def _check(ctx, pos, tri, H, W, floor, max_pixels=1 << 16):
    rast, ids = _rasterize(ctx, pos, tri, H, W)
    rows, cols = g.pixel_sample(H, W, max_pixels)
    rep, _ = g.check_rasterize(pos, tri, H, W, rast, ids, rows, cols)
    print(f"{H}x{W} B={pos.shape[0]} F={tri.shape[0]}: {rep}")
    assert rep.fraction >= floor, rep
    return rep


# ---- operators ---------------------------------------------------------------------------------------------

SCENES = {
    "soup_ortho": (lambda: cases.random_soup(1, 400, B=2), (128, 160), 0.95),
    "soup_perspective": (lambda: cases.random_soup(3, 300, B=2, perspective=True), (128, 128), 0.95),
    "near_crossing": (cases.near_crossing_scene, (200, 320), 0.85),
    "guard_band": (cases.guard_band_scene, (600, 800), 0.98),
    "big_and_small_mix": (cases.big_and_small_mix, (1024, 1024), 0.98),
    "huge_triangles_tile_pass": (cases.huge_triangle_scene, (768, 1024), 0.92),
    "adversarial": (lambda: adversarial_soup(0, B=2), (256, 256), 0.6),
}


@pytest.mark.parametrize("name", list(SCENES))
def test_rasterize_scenes(wr_ctx, name):
    build, (H, W), floor = SCENES[name]
    pos, tri = build()
    _check(wr_ctx, pos, tri, H, W, floor)


@pytest.mark.parametrize("H,W", [(1, 300), (300, 1), (333, 517), (2048, 2048)])
def test_rasterize_viewports(wr_ctx, H, W):
    pos, tri = cases.random_soup(11, 200, B=1, perspective=True)
    if min(H, W) == 1:   # one row / column: few, large triangles, so that samples lie clear of the edges
        pos, tri = cases.random_soup(11, 6, B=1, scale=4.0, perspective=True)
    _check(wr_ctx, pos, tri, H, W, 0.8 if min(H, W) == 1 else 0.9)


def test_rasterize_1x1_viewport(wr_ctx):
    pos = np.array([[[-3, -3, 0.2, 1], [3, -2, 0.2, 1], [0, 3, 0.2, 1]]], f32)
    rep = _check(wr_ctx, pos, np.array([[0, 1, 2]], np.int32), 1, 1, 1.0)
    assert rep.covered == 1


def test_rasterize_8192_huge_triangles(wr_ctx):
    pos, tri = cases.huge_triangle_scene(seed=4, n_huge=300, n_small=500, n_clip=8, B=1)
    _check(wr_ctx, pos, tri, 8192, 8192, 0.9, max_pixels=1 << 15)


@pytest.mark.parametrize("B", [1, 9, 40])
def test_rasterize_batches_coarse_and_fine_setup(wr_ctx, B):
    # 4 F <= H W: the set-up pass runs four lanes per triangle; 4 F > H W (sub-pixel faces): one lane per triangle
    pos, tri = cases.random_soup(5, 120, B=B, perspective=True, scale=1.1)
    _check(wr_ctx, pos, tri, 64, 96, 0.9, max_pixels=1 << 14)
    pos, tri = cases.random_soup(6, 3000, B=B, scale=1.0)
    pos[..., :2] = pos[..., :2].reshape(B, -1, 3, 2).mean(2, keepdims=True).repeat(3, 2).reshape(B, -1, 2) \
        + np.random.default_rng(B).uniform(-0.03, 0.03, pos[..., :2].shape).astype(f32)
    _check(wr_ctx, pos, tri, 40, 48, 0.75, max_pixels=1 << 14)


def test_rasterize_range_mode(wr_ctx):
    pos, tri = cases.random_soup(8, 300, B=1, perspective=True)
    ranges = [[0, 100], [100, 150], [250, 50], [0, 0]]
    rast, _ = wr_ctx.rasterize(torch.from_numpy(pos[0]).to(wr_ctx.device), torch.from_numpy(tri).to(wr_ctx.device),
                               (96, 112), ranges=torch.tensor(ranges, dtype=torch.int32))
    rast = rast.cpu().numpy()
    for b, (s, n) in enumerate(ranges):
        sub = np.full_like(tri, -1)           # faces outside the range are dropped, ids stay global
        sub[s:s + n] = tri[s:s + n]
        rep, _ = g.check_rasterize(pos, sub, 96, 112, rast[b:b + 1])
        assert rep.fraction >= 0.9, (b, rep)


def test_interpolate_and_texture(wr_ctx):
    pos, tri = cases.random_soup(7, 150, B=2, perspective=True)
    H, W = 96, 112
    dev = wr_ctx.device
    rast_t, _ = wr_ctx.rasterize(torch.from_numpy(pos).to(dev), torch.from_numpy(tri).to(dev), (H, W))
    rast = rast_t.cpu().numpy()
    rng = np.random.default_rng(1)
    attr = rng.uniform(-2.0, 3.0, (pos.shape[1], 2)).astype(f32)
    uv_t, _ = wr_ctx.interpolate(torch.from_numpy(attr).to(dev), rast_t, torch.from_numpy(tri).to(dev))
    uv = uv_t.cpu().numpy()
    tex = rng.uniform(-1, 1, (13, 17, 3)).astype(f32)
    rows, cols = g.pixel_sample(H, W)
    _, views = g.check_rasterize(pos, tri, H, W, rast, None, rows, cols)
    for b, vr in enumerate(views):
        d = vr.decided & (vr.winner >= 0)
        r, c, face = rows[d], cols[d], vr.winner[d]
        bc = g.barycentrics(pos[b], np.zeros(pos[b].shape), tri, face, r, c, H, W)
        val, bound = g.interpolate(attr, tri, face, bc)
        assert np.all(np.abs(uv[b, r, c] - val) <= bound)
        q = uv[b, r, c]
        for filt in ("nearest", "linear"):
            for mode in ("wrap", "clamp", "zero"):
                got = wr_ctx.texture(torch.from_numpy(tex[None]).to(dev), torch.from_numpy(q[None, None]).to(dev),
                                     filter_mode=filt, boundary_mode=mode).cpu().numpy()[0, 0]
                want, tb, ok = g.texture(tex, q, filt, mode)
                assert ok.mean() > 0.99
                assert np.all(np.abs(got[ok] - want[ok]) <= tb[ok]), (filt, mode)


# ---- render() -----------------------------------------------------------------------------------------------

def _mesh(v, f, device):
    mesh = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32), t_pos_idx=torch.tensor(f, dtype=torch.int64))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    mesh.to(device)
    return mesh


def _render_check(ctx, mesh, cam, H, W, floor, dtype=torch.float32, max_pixels=1 << 16, tri_nrm=None):
    raw = render_geometry_raw(ctx, mesh, cam, H, W, depth_normalization_strategy=None, output_dtype=dtype)
    out = {k: raw[k].float().cpu().numpy() if k != "mask" else raw[k].cpu().numpy() for k in ("mask", "pos", "normal", "depth")}
    rows, cols = g.pixel_sample(H, W, max_pixels)
    rep = g.check_render(mesh.v_pos.cpu().numpy(), mesh.t_pos_idx.cpu().numpy(), cam.mvp_mtx.cpu().numpy(),
                         cam.w2c.cpu().numpy(), mesh.v_nrm.cpu().numpy(), H, W, out, rows, cols,
                         dtype=str(dtype).split(".")[-1], tri_nrm=tri_nrm)
    print(f"render {H}x{W} B={cam.mvp_mtx.shape[0]} F={mesh.t_pos_idx.shape[0]} {dtype}: {rep}")
    assert rep.fraction >= floor, rep
    return rep


@pytest.mark.parametrize("cam_name", ["canonical", "perspective", "inside"])
@pytest.mark.parametrize("mesh_name", ["icosphere", "terrain"])
def test_render_meshes(wr_ctx, mesh_name, cam_name):
    v, f = cases.icosphere_mesh(8) if mesh_name == "icosphere" else cases.terrain_mesh()
    cam = {"canonical": cases.canonical_cameras, "perspective": cases.perspective_cameras,
           "inside": cases.inside_cameras}[cam_name](device=wr_ctx.device)
    _render_check(wr_ctx, _mesh(v, f, wr_ctx.device), cam, 192, 224, 0.95)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_render_half_precision_maps(wr_ctx, dtype):
    v, f = cases.icosphere_mesh(8)
    _render_check(wr_ctx, _mesh(v, f, wr_ctx.device), cases.perspective_cameras(device=wr_ctx.device), 160, 176,
                  0.95, dtype=dtype)


def _fused_multiview(F, H, W):
    """render() rasterises with the multi-view kernels (k_snap_mv / k_setup_mv) when the faces are small for the
    viewport (4 F > H W) and the viewport fits their 16-bit records (H, W <= 2048); else with the per-view ones."""
    return 4 * F > H * W and H <= 2048 and W <= 2048


@pytest.mark.parametrize("H,W,nx,ny,fused", [
    (64, 64, 32, 16, False),     # F = 1024: 4 F = H W exactly, per-view side
    (64, 64, 32, 17, True),      # 4 F just above H W: multi-view side
    (128, 2048, 256, 160, True),  # F = 81920: 4 F > H W at both widths; 2048 is the widest multi-view viewport
    (128, 2049, 256, 160, False),
])
def test_render_multiview_switch(wr_ctx, H, W, nx, ny, fused):
    v, f = cases.terrain_mesh(nx, ny)
    assert _fused_multiview(f.shape[0], H, W) == fused
    _render_check(wr_ctx, _mesh(v, f, wr_ctx.device), cases.canonical_cameras(device=wr_ctx.device), H, W, 0.88,
                  max_pixels=1 << 15)


@pytest.mark.parametrize("mesh_name,H,W", [("terrain", 96, 128), ("icosphere", 128, 128)])
def test_render_inside_cameras_fused_multiview(wr_ctx, mesh_name, H, W):
    """Cameras inside the mesh on the multi-view path: faces cross the near plane there too."""
    v, f = cases.terrain_mesh(64, 32) if mesh_name == "terrain" else cases.icosphere_mesh(24)
    assert _fused_multiview(f.shape[0], H, W)
    _render_check(wr_ctx, _mesh(v, f, wr_ctx.device), cases.inside_cameras(device=wr_ctx.device), H, W, 0.85)


@pytest.mark.parametrize("H,W", [(64, 64), (128, 144)])
def test_render_attr_and_tangent(wr_ctx, H, W):
    """render_attr (UVs over their own faces, bilinear, wrap) and render_tangent (tangents over the stitched faces),
    with their backgrounds, on both raster paths."""
    d = cases.stitched_icosphere("permuted")    # tangents need one stitched vertex per position vertex
    F = d["t_pos_idx"].shape[0]
    assert _fused_multiview(F, H, W) == (H == 64)
    mesh = wr.TexturedMesh(v_pos=torch.from_numpy(d["v_pos"]), t_pos_idx=torch.from_numpy(d["t_pos_idx"]).long(),
                           v_tex=torch.from_numpy(d["v_tex"]), t_tex_idx=torch.from_numpy(d["t_tex_idx"]).long())
    mesh.set_stitched_mesh(torch.from_numpy(d["stitched_v_pos"]), torch.from_numpy(d["stitched_t_pos_idx"]).long())
    tex = np.random.default_rng(3).uniform(0, 1, (37, 53, 3)).astype(f32)
    mesh.texture = torch.from_numpy(tex)
    mesh.to(wr_ctx.device)
    cam = cases.perspective_cameras(device=wr_ctx.device)
    raw = render_geometry_raw(wr_ctx, mesh, cam, H, W, want_attr=True, want_tangent=True, tangent_background=0.25,
                              attr_background=0.5, depth_normalization_strategy=None)
    out = {k: raw[k].cpu().numpy() for k in ("mask", "pos", "normal", "depth", "attr", "tangent")}
    rep = g.check_render(d["v_pos"], d["t_pos_idx"], cam.mvp_mtx.cpu().numpy(), cam.w2c.cpu().numpy(),
                         mesh.v_nrm.cpu().numpy(), H, W, out, tri_nrm=d["stitched_t_pos_idx"],
                         v_tang=mesh.v_tang.cpu().numpy(), v_tex=d["v_tex"], tri_tex=d["t_tex_idx"], tex=tex,
                         tangent_background=0.25, attr_background=0.5)
    print(f"render attr + tangent {H}x{W}: {rep}")
    assert rep.fraction >= 0.9, rep
    assert {"attr", "tangent"} <= set(rep.ratio)


def test_render_mixed_40_view_rig(wr_ctx):
    v, f = cases.icosphere_mesh(10)
    _render_check(wr_ctx, _mesh(v, f, wr_ctx.device), cases.mixed_40_view_cameras(96, 80, device=wr_ctx.device),
                  96, 80, 0.93)


@pytest.mark.parametrize("form", cases.STITCHED_FORMS)
def test_render_stitched_mesh(wr_ctx, form):
    d = cases.stitched_icosphere(form)
    mesh = wr.TexturedMesh(v_pos=torch.from_numpy(d["v_pos"]), t_pos_idx=torch.from_numpy(d["t_pos_idx"]).long())
    mesh.set_stitched_mesh(torch.from_numpy(d["stitched_v_pos"]), torch.from_numpy(d["stitched_t_pos_idx"]).long())
    mesh.to(wr_ctx.device)
    _render_check(wr_ctx, mesh, cases.perspective_cameras(device=wr_ctx.device), 128, 144, 0.95,
                  tri_nrm=d["stitched_t_pos_idx"])


def test_render_config_b_terrain(wr_ctx):
    """The 1M-face terrain at 768^2 x 6 views (config B's size), on a pixel sample."""
    v, f = cases.terrain_mesh(1000, 500)
    _render_check(wr_ctx, _mesh(v, f, wr_ctx.device), cases.canonical_cameras(device=wr_ctx.device), 768, 768,
                  0.85, max_pixels=1 << 13)
