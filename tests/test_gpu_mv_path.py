"""GPU parity of the multi-view fast path of the fused render (k_snap_mv / k_setup_mv, csrc/raster.cu): dense
meshes at small viewports (4 F > H W selects it) against the oracle, ids bit-exact.

The path keeps 8-byte compact records per (vertex, view) and evaluates one-sample boxes by integer cross
products; everything it cannot represent must fall back to the contract's own classification (cold path) or
to the queues.  These cases aim at exactly those seams: samples on edges and vertices (fill rule), both
windings, depth ties, vertices behind the camera / beyond near and far / far off screen, large triangles among
small ones, odd view counts (padded record rows), more views than one compaction chunk, and the default
render() shading instantiation next to the generic one."""
import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import render_oracle
from oracle.render_oracle import DepthSpec
from worldrenderer_b200.render import render_geometry_raw

pytestmark = pytest.mark.gpu
f32 = np.float32


def _mesh(v, f, dev):
    m = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32), t_pos_idx=torch.tensor(f, dtype=torch.int64))
    m.set_stitched_mesh(m.v_pos, m.t_pos_idx)
    m.to(dev)
    m.v_nrm
    return m


def _cam(mvp, dev):
    """Camera whose mvp is given directly (w2c = identity-like so that view depth is defined)."""
    B = mvp.shape[0]
    eye = torch.eye(4, dtype=torch.float32).repeat(B, 1, 1)
    t = torch.tensor(mvp, dtype=torch.float32)
    return wr.Camera(c2w=eye.to(dev), w2c=eye.clone().to(dev), proj_mtx=t.to(dev), mvp_mtx=t.to(dev),
                     cam_pos=torch.zeros(B, 3, device=dev))


def _check(ctx, mesh, cam, H, W, atol=1e-6):
    """ids / mask / rast bit-exact through the generic shading instantiation, then the default render()
    (k_shade<kOutsRenderDefault, ·>) against the oracle's maps."""
    v = mesh.v_pos.cpu().numpy()
    f = mesh.t_pos_idx.cpu().numpy().astype(np.int32)
    ref = render_oracle.render(v, f, cam.mvp_mtx.cpu().numpy(), cam.w2c.cpu().numpy(), H, W,
                               v_nrm=mesh.v_nrm.cpu().numpy(), depth=DepthSpec("controlnet"))
    raw = render_geometry_raw(ctx, mesh, cam, H, W, want_tri_id=True, want_rast=True)
    np.testing.assert_array_equal(raw["tri_id"].cpu().numpy(), ref["tri_id"])
    np.testing.assert_array_equal(raw["mask"].cpu().numpy(), ref["mask"])
    np.testing.assert_array_equal(raw["rast"].cpu().numpy(), ref["rast"])
    out = wr.render(ctx, mesh, cam, H, W, render_attr=False)
    np.testing.assert_array_equal(out.mask.cpu().numpy(), ref["mask"])
    np.testing.assert_allclose(out.pos.cpu().numpy(), ref["pos"], rtol=1e-5, atol=atol)
    np.testing.assert_allclose(out.normal.cpu().numpy(), ref["normal"], rtol=1e-5, atol=atol)
    np.testing.assert_allclose(out.depth.cpu().numpy(), ref["depth"], rtol=1e-5, atol=atol)
    return ref


def _lattice_mesh(n, seed, jitter_z=True):
    """(n+1)^2 vertices on a regular lattice over [-1, 1]^2, two triangles per cell with alternating diagonals
    and windings; z from three values (depth ties between overlapping copies)."""
    rng = np.random.default_rng(seed)
    g = np.linspace(-1, 1, n + 1, dtype=np.float64)
    X, Y = np.meshgrid(g, g, indexing="xy")
    Z = rng.choice([-0.25, 0.0, 0.25], X.shape) if jitter_z else np.zeros_like(X)
    v = np.stack([X, Y, Z], -1).reshape(-1, 3).astype(f32)
    idx = lambda i, j: j * (n + 1) + i
    tris = []
    for j in range(n):
        for i in range(n):
            a, b, c, d = idx(i, j), idx(i + 1, j), idx(i + 1, j + 1), idx(i, j + 1)
            t = [(a, b, c), (a, c, d)] if (i + j) % 2 == 0 else [(a, b, d), (b, c, d)]
            if (i * 7 + j * 3) % 5 == 0:
                t = [(p, r, q) for (p, q, r) in t]  # flipped winding
            tris += t
    return v, np.array(tris, np.int32)


def _ortho(sx, sy, tx=0.0, ty=0.0, sz=0.5):
    m = np.eye(4, dtype=f32)
    m[0, 0], m[1, 1], m[2, 2], m[0, 3], m[1, 3] = sx, sy, sz, tx, ty
    return m


@pytest.mark.parametrize("H,W,n", [(32, 32, 32), (32, 32, 64), (48, 80, 80), (33, 47, 64)])
def test_samples_on_vertices_and_edges(wr_ctx, H, W, n):
    """Lattice vertices land exactly on pixel centres / corners / half-way points: every coverage decision of
    the single-sample path is a tie-break (mv_tie_break)."""
    v, f = _lattice_mesh(n, seed=n)
    assert 4 * f.shape[0] > H * W
    mesh = _mesh(v, f, wr_ctx.device)
    # view 0: cell == pixel (vertices on corners); view 1: shifted by half a pixel (vertices on centres);
    # view 2: 2x zoom, shifted; view 3: mirrored in x (all windings flip); view 4: anisotropic
    mvp = np.stack([_ortho(1, 1), _ortho(1, 1, 1.0 / W, 1.0 / H), _ortho(2, 2, 3.0 / W, -5.0 / H),
                    _ortho(-1, 1, 1.0 / W, 1.0 / H), _ortho(0.5, 1.5, -1.0 / W, 1.0 / H)])
    _check(wr_ctx, mesh, _cam(mvp, wr_ctx.device), H, W)


@pytest.mark.parametrize("B", [1, 2, 7, 9, 17])
def test_view_counts_pad_and_chunks(wr_ctx, B):
    """B odd (padded record rows), B > 8 (several compaction chunks), B = 1."""
    v, f = cases.terrain_mesh(96, 64, seed=3)
    H = W = 64
    assert 4 * f.shape[0] > H * W
    mesh = _mesh(v, f, wr_ctx.device)
    cam = wr.get_orthogonal_camera(elevation_deg=list(np.linspace(-80, 80, B)), distance=[1.0] * B, left=-0.55,
                                   right=0.55, bottom=-0.55, top=0.55, azimuth_deg=list(np.linspace(0, 300, B)),
                                   device=wr_ctx.device)
    _check(wr_ctx, mesh, cam, H, W)


def test_perspective_inside_the_mesh_cold_path(wr_ctx):
    """Cameras inside a dense sphere: many vertices behind the camera or beyond the near plane (records carry the
    sentinel, their triangles take the cold path and the clip queue), the rest goes through the fast path."""
    v, f = cases.icosphere_mesh(40)   # 32 000 faces
    H, W = 96, 128
    assert 4 * f.shape[0] > H * W
    mesh = _mesh(v, f, wr_ctx.device)
    _check(wr_ctx, mesh, cases.inside_cameras(device=wr_ctx.device), H, W, atol=2e-6)
    _check(wr_ctx, mesh, cases.perspective_cameras(device=wr_ctx.device), H, W)


def test_large_triangles_among_small_ones(wr_ctx):
    """A dense terrain plus a ground plane of two huge triangles, a far-off-screen sliver and a triangle spanning
    near to far: the fast path has to hand them to the medium / large / clip queues."""
    v, f = cases.terrain_mesh(128, 64, seed=5)
    n0 = v.shape[0]
    extra_v = np.array([[-0.7, -0.3, -0.7], [0.7, -0.3, -0.7], [0.7, -0.3, 0.7], [-0.7, -0.3, 0.7],   # ground plane
                        [40.0, 0.0, 0.0], [41.0, 0.0, 0.1], [0.0, 0.1, 0.0],                          # far off screen
                        [0.0, 0.0, -300.0], [0.1, 0.2, 300.0], [-0.2, 0.1, 0.0],                      # spans near..far
                        [0.05, 0.05, 0.0], [0.25, 0.06, 0.0], [0.1, 0.3, 0.0]], f32)                  # medium
    extra_f = np.array([[n0, n0 + 1, n0 + 2], [n0, n0 + 2, n0 + 3], [n0 + 4, n0 + 5, n0 + 6], [n0 + 7, n0 + 8, n0 + 9],
                        [n0 + 10, n0 + 11, n0 + 12]], np.int32)
    v = np.concatenate([v, extra_v]); f = np.concatenate([f, extra_f])
    H, W = 96, 96
    assert 4 * f.shape[0] > H * W
    mesh = _mesh(v, f, wr_ctx.device)
    _check(wr_ctx, mesh, cases.canonical_cameras(device=wr_ctx.device), H, W)
    _check(wr_ctx, mesh, cases.perspective_cameras(device=wr_ctx.device), H, W)


def test_bad_indices_and_non_finite_vertices(wr_ctx):
    v, f = cases.terrain_mesh(96, 48, seed=7)
    v = v.copy(); f = f.copy()
    v[100] = [np.nan, 0.0, 0.0]
    v[2000] = [np.inf, 0.1, 0.0]
    v[3000] = [0.0, 1e30, 0.0]
    f[50] = [0, 1, v.shape[0] + 3]
    f[51] = [-1, 2, 3]
    f[52] = [5, 5, 9]
    H = W = 64
    mesh = wr.TexturedMesh(v_pos=torch.tensor(v), t_pos_idx=torch.tensor(f.astype(np.int64)))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    mesh.to(wr_ctx.device)
    vn = np.zeros_like(v); vn[:, 1] = 1.0   # normals given: the reference's own normal pass is not the subject here
    mesh._v_nrm = torch.tensor(vn, device=wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    ref = render_oracle.render(v, f, cam.mvp_mtx.cpu().numpy(), cam.w2c.cpu().numpy(), H, W, v_nrm=vn,
                               depth=DepthSpec("controlnet"))
    raw = render_geometry_raw(wr_ctx, mesh, cam, H, W, want_tri_id=True)
    np.testing.assert_array_equal(raw["tri_id"].cpu().numpy(), ref["tri_id"])
    out = wr.render(wr_ctx, mesh, cam, H, W, render_attr=False)
    np.testing.assert_array_equal(out.mask.cpu().numpy(), ref["mask"])


def test_2048_viewport_uses_the_full_record_range(wr_ctx):
    """2048^2 is the largest viewport of the fast path (config E's view size): coordinates use the whole 16-bit
    record range; a mesh that also reaches beyond the viewport on every side."""
    v, f = cases.terrain_mesh(1536, 700, seed=11)   # 2.15 M faces > 2048^2 / 4
    v = (v * 2.6).astype(f32)                        # wider than the +-0.55 frustum
    H = W = 2048
    assert 4 * f.shape[0] > H * W
    mesh = _mesh(v, f, wr_ctx.device)
    cam = wr.get_orthogonal_camera(elevation_deg=[89.99, 20.0], distance=[1.0, 1.0], left=-0.55, right=0.55,
                                   bottom=-0.55, top=0.55, azimuth_deg=[90.0, 30.0], device=wr_ctx.device)
    ref = render_oracle.render(v, f, cam.mvp_mtx.cpu().numpy(), cam.w2c.cpu().numpy(), H, W,
                               v_nrm=mesh.v_nrm.cpu().numpy(), depth=DepthSpec("controlnet"))
    raw = render_geometry_raw(wr_ctx, mesh, cam, H, W, want_tri_id=True)
    np.testing.assert_array_equal(raw["tri_id"].cpu().numpy(), ref["tri_id"])
