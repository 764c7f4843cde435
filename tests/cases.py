"""Seeded inputs shared by the CPU (oracle) and GPU (parity) tests."""
from __future__ import annotations

import numpy as np

f32 = np.float32


def quad_fullscreen():
    pos = np.array([[[-1, -1, 0, 1], [1, -1, 0, 1], [1, 1, 0, 1], [-1, 1, 0, 1]]], f32)
    tri = np.array([[0, 1, 2], [0, 2, 3]], np.int32)
    return pos, tri


def random_soup(seed: int, n_tri: int, B: int = 1, scale: float = 1.2, perspective: bool = False):
    """Independent random triangles in clip space (w = 1, or w in [0.3, 3] when perspective)."""
    rng = np.random.default_rng(seed)
    V = 3 * n_tri
    pos = np.empty((B, V, 4), f32)
    pos[..., :2] = rng.uniform(-scale, scale, (B, V, 2))
    pos[..., 2] = rng.uniform(-1.1, 1.1, (B, V))
    pos[..., 3] = 1.0
    if perspective:
        w = rng.uniform(0.3, 3.0, (B, V)).astype(f32)
        pos[..., :3] *= w[..., None]
        pos[..., 3] = w
    tri = np.arange(V, dtype=np.int32).reshape(-1, 3)
    return pos, tri


def snapped_grid_soup(seed: int, n_tri: int, W: int, H: int):
    """Triangles whose vertices sit exactly on pixel centres / corners: maximises edge ties (fill rule)."""
    rng = np.random.default_rng(seed)
    V = 3 * n_tri
    # half-pixel lattice: NDC = k / W with integer k hits both centres (odd k) and corners (even k)
    kx = rng.integers(-W, W + 1, V)
    ky = rng.integers(-H, H + 1, V)
    pos = np.zeros((1, V, 4), f32)
    pos[0, :, 0] = kx / f32(W)
    pos[0, :, 1] = ky / f32(H)
    pos[0, :, 2] = rng.choice([-0.5, 0.0, 0.5], V)  # few distinct depths -> depth ties
    pos[0, :, 3] = 1.0
    tri = np.arange(V, dtype=np.int32).reshape(-1, 3)
    return pos, tri


def shared_edge_fan(n: int = 24):
    """A fan of triangles around the image centre: every spoke is an edge shared by two triangles."""
    ang = np.linspace(0, 2 * np.pi, n, endpoint=False)
    pos = np.zeros((1, n + 1, 4), f32)
    pos[0, 1:, 0] = 0.9 * np.cos(ang)
    pos[0, 1:, 1] = 0.9 * np.sin(ang)
    pos[0, :, 3] = 1.0
    tri = np.array([[0, 1 + i, 1 + (i + 1) % n] for i in range(n)], np.int32)
    tri[::2] = tri[::2][:, [0, 2, 1]]  # alternate winding
    return pos, tri


def near_crossing_scene(seed: int = 5, n_tri: int = 200):
    """Perspective-like clip coordinates with vertices behind the camera (w <= 0) and across z = +-w."""
    rng = np.random.default_rng(seed)
    V = 3 * n_tri
    pos = np.empty((1, V, 4), f32)
    pos[0, :, 0] = rng.uniform(-3, 3, V)
    pos[0, :, 1] = rng.uniform(-3, 3, V)
    pos[0, :, 3] = rng.uniform(-1.0, 3.0, V)
    pos[0, :, 2] = pos[0, :, 3] * rng.uniform(-1.3, 1.3, V) + rng.uniform(-0.2, 0.2, V)
    tri = np.arange(V, dtype=np.int32).reshape(-1, 3)
    return pos, tri


def guard_band_scene(seed: int = 13, n_tri: int = 60):
    """Triangles with vertices far outside the viewport (|x|, |y| up to 1e5 w): the snap range is exceeded, so
    they take the geometric clip against the +-16 w guard planes (DESIGN.md 3.2c)."""
    rng = np.random.default_rng(seed)
    V = 3 * n_tri
    pos = np.empty((1, V, 4), f32)
    mag = 10.0 ** rng.uniform(0, 5, (V, 2))
    pos[0, :, :2] = rng.choice([-1.0, 1.0], (V, 2)) * mag * rng.uniform(0.0, 1.0, (V, 2))
    pos[0, :, 2] = rng.uniform(-0.9, 0.9, V)
    pos[0, :, 3] = 1.0
    pos[0, ::3, :2] = rng.uniform(-1, 1, (n_tri, 2))  # one vertex of every triangle inside the viewport
    tri = np.arange(V, dtype=np.int32).reshape(-1, 3)
    return pos, tri


def big_and_small_mix(seed: int = 9):
    """A few screen-filling triangles + many tiny ones + off-screen ones + degenerate / bad-index faces."""
    rng = np.random.default_rng(seed)
    big = np.array([[-3, -3, 0.9, 1], [3, -3, 0.9, 1], [0, 3, 0.9, 1],
                    [-1.5, 1.2, 0.5, 1], [1.5, 1.2, 0.5, 1], [0, -2.5, 0.5, 1],
                    [-0.9, -0.9, 0.2, 1], [0.9, -0.8, 0.2, 1], [0.0, 0.95, 0.2, 1]], f32)
    n_small = 3000
    c = rng.uniform(-1.05, 1.05, (n_small, 1, 2))
    small = np.zeros((n_small, 3, 4), f32)
    small[..., :2] = c + rng.uniform(-0.01, 0.01, (n_small, 3, 2))
    small[..., 2] = rng.uniform(-1, 1, (n_small, 1))
    small[..., 3] = 1
    off = np.array([[2, 2, 0, 1], [3, 2, 0, 1], [2, 3, 0, 1]], f32)
    degen = np.array([[0.1, 0.1, 0, 1], [0.1, 0.1, 0, 1], [0.3, 0.2, 0, 1]], f32)
    nan = np.array([[np.nan, 0, 0, 1], [0.5, 0.5, 0, 1], [0.2, 0.7, 0, 1]], f32)
    pos = np.concatenate([big, small.reshape(-1, 4), off, degen, nan], 0)[None]
    V = pos.shape[1]
    tri = np.arange((V // 3) * 3, dtype=np.int32).reshape(-1, 3)
    bad = np.array([[0, 1, V + 5], [-1, 2, 3]], np.int32)  # out-of-range indices are ignored
    tri = np.concatenate([tri, bad], 0)
    return pos.astype(f32), tri


def icosphere_mesh(frequency: int = 8):
    from worldrenderer_b200 import synth
    v, f = synth.icosphere(frequency, 0.5)
    return v.astype(f32), f.astype(np.int32)


def exact_vertex_normals(v, f):
    """Vertex normals as the GPU splats them: float face normals summed in float64 (the correctly rounded sum,
    whatever the order), rounded to float once, normalised in float."""
    ff = np.asarray(f, np.int64)
    e1 = (v[ff[:, 1]] - v[ff[:, 0]]).astype(f32)
    e2 = (v[ff[:, 2]] - v[ff[:, 0]]).astype(f32)
    fn = np.stack([e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1], e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2],
                   e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]], -1).astype(f32)
    acc = np.zeros((v.shape[0], 3), np.float64)
    for k in range(3):
        np.add.at(acc, ff[:, k], fn.astype(np.float64))
    s32 = acc.astype(f32)
    n = s32 / np.maximum(np.sqrt((s32[:, 0] * s32[:, 0] + s32[:, 1] * s32[:, 1]) + s32[:, 2] * s32[:, 2]), f32(1e-12))[:, None]
    return n.astype(f32)


STITCHED_FORMS = ("seams", "permuted", "flat")


def stitched_icosphere(form: str, frequency: int = 8, seed: int = 0):
    """icosphere_mesh(frequency) with one cell_atlas_uv corner per face corner (v_tex [3F,2], t_tex_idx = arange),
    in one of three forms of the (v_pos, t_pos_idx) / stitched (v, f) pair that TexturedMesh.set_stitched_mesh takes:

    - "seams": what load_mesh makes of a trimesh asset with merge_vertices=True -- v_pos split per face corner
      (V = 3F, t_pos_idx = arange, like t_tex_idx), the stitched mesh the merged icosphere (Vn < V);
    - "permuted": v_pos the merged icosphere, the stitched vertices the same points in a random order (Vn == V) and
      the stitched faces inv_perm[t_pos_idx]: in range, but not the position indices;
    - "flat": v_pos merged, the stitched mesh split per face corner (Vn = 3F > V): every normal is a face normal.

    Returns dict(v_pos, t_pos_idx, v_tex, t_tex_idx, stitched_v_pos, stitched_t_pos_idx) as float32 / int32."""
    from worldrenderer_b200 import synth
    v, f = icosphere_mesh(frequency)
    F = f.shape[0]
    corners = np.arange(3 * F, dtype=np.int32).reshape(-1, 3)
    vt, ft = synth.cell_atlas_uv(F)
    if form == "seams":
        v_pos, t_pos, sv, sf = v[f.reshape(-1)], corners, v, f
    elif form == "permuted":
        perm = np.random.default_rng(seed).permutation(v.shape[0])
        inv = np.argsort(perm).astype(np.int32)
        v_pos, t_pos, sv, sf = v, f, v[perm], inv[f]
    elif form == "flat":
        v_pos, t_pos, sv, sf = v, f, v[f.reshape(-1)], corners
    else:
        raise ValueError(form)
    return dict(v_pos=np.ascontiguousarray(v_pos, f32), t_pos_idx=np.ascontiguousarray(t_pos, np.int32),
                v_tex=vt.astype(f32), t_tex_idx=ft.astype(np.int32),
                stitched_v_pos=np.ascontiguousarray(sv, f32), stitched_t_pos_idx=np.ascontiguousarray(sf, np.int32))


def terrain_mesh(nx: int = 64, ny: int = 32, seed: int = 0):
    from worldrenderer_b200 import synth
    v, f = synth.terrain(nx, ny, seed)
    v = v / np.abs(v).max() * 0.5
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1)  # load_mesh axis remap (up=+y, front=+x)
    return v.astype(f32), f.astype(np.int32)


def canonical_cameras(device=None):
    import worldrenderer_b200 as wr
    from worldrenderer_b200 import synth
    return wr.get_orthogonal_camera(device=device, **synth.CANONICAL_RIG)


def perspective_cameras(n: int = 4, fovy: float = 40.0, distance: float = 1.8, device=None):
    import worldrenderer_b200 as wr
    return wr.get_camera(elevation_deg=[10.0, -20.0, 35.0, 60.0][:n], distance=[distance] * n, fovy_deg=[fovy] * n,
                         azimuth_deg=[0.0, 75.0, 160.0, 250.0][:n], device=device)


def concat_cameras(*cams):
    """One rig from parts (views in argument order)."""
    import torch
    import worldrenderer_b200 as wr
    return wr.Camera(**{k: torch.cat([getattr(c, k) for c in cams]).contiguous()
                        for k in ("c2w", "w2c", "proj_mtx", "mvp_mtx", "cam_pos")})


def bake_perspective_cameras(H: int, W: int, device=None):
    """perspective_cameras() with the image aspect of an H x W view, as CameraProjection(cam=None) builds it."""
    import worldrenderer_b200 as wr
    return wr.get_camera(elevation_deg=[10.0, -20.0, 35.0, 60.0], distance=[1.8] * 4, fovy_deg=[40.0] * 4,
                         azimuth_deg=[0.0, 75.0, 160.0, 250.0], aspect_wh=W / H, device=device)


def mixed_40_view_cameras(H: int, W: int, device=None):
    """40 views: 34 perspective and the 6 canonical orthographic ones.  Orthographic views sit at indices 1-3 (the
    unit-row fast path of the unprojection) and 37-39 (beyond the 32-view bitmask: the general path); the perspective
    views 33-35 would read the bits of views 1-3 from a bitmask indexed by v & 31 instead of tested for v < 32."""
    import worldrenderer_b200 as wr
    n = 34
    persp = wr.get_camera(elevation_deg=np.linspace(-60.0, 70.0, n).tolist(), distance=[1.8] * n,
                          fovy_deg=[40.0] * n, azimuth_deg=((np.arange(n) * 137.5) % 360.0).tolist(),
                          aspect_wh=W / H, device=device)
    ortho = canonical_cameras(device=device)
    return concat_cameras(persp[0:1], ortho[0:3], persp[1:34], ortho[3:6])


def low_terrain_cameras(H: int, W: int, device=None):
    """Two wide perspective cameras close over the terrain_mesh: much of the terrain lies behind them (clip w <= 0,
    NDC up to ~1e5), which the bake projects without a w > 0 guard."""
    import worldrenderer_b200 as wr
    return wr.get_camera(elevation_deg=[60.0, 60.0], distance=[0.25, 0.25], fovy_deg=[110.0, 110.0],
                         azimuth_deg=[0.0, 120.0], near=0.01, aspect_wh=W / H, device=device)


def inside_cameras(device=None):
    """Perspective cameras placed INSIDE the mesh's bounding sphere: triangles cross the near plane."""
    import worldrenderer_b200 as wr
    return wr.get_camera(elevation_deg=[5.0, 40.0], distance=[0.3, 0.45], fovy_deg=[70.0, 90.0],
                         azimuth_deg=[20.0, 200.0], near=0.05, far=10.0, device=device)


def huge_triangle_scene(seed: int = 31, n_huge: int = 300, n_small: int = 2000, n_clip: int = 12, B: int = 2):
    """The tile pass of the LARGE class (csrc/raster.cu raster_tiles): hundreds of overlapping screen-sized triangles
    (more than one 256-triangle batch per band, depth and id ties among them), a layer of tiny triangles in front of
    and behind them (the tile owner's atomicMin must merge with what the set-up kernel already resolved), and a few
    triangles that need geometric clipping (they stay with the stripe pass, concurrently)."""
    rng = np.random.default_rng(seed)
    huge = np.zeros((B, n_huge, 3, 4), f32)
    huge[..., :2] = rng.uniform(-1.6, 1.6, (B, n_huge, 3, 2))
    huge[..., 2] = rng.choice([-0.4, 0.0, 0.3, 0.6], (B, n_huge, 1))   # few distinct depths: ties decided by id
    huge[..., 2] += rng.uniform(-0.3, 0.3, (B, n_huge, 3)) * (rng.random((B, n_huge, 1)) < 0.5)
    huge[..., 3] = 1
    c = rng.uniform(-1.0, 1.0, (B, n_small, 1, 2))
    small = np.zeros((B, n_small, 3, 4), f32)
    small[..., :2] = c + rng.uniform(-0.02, 0.02, (B, n_small, 3, 2))
    small[..., 2] = rng.uniform(-0.9, 0.9, (B, n_small, 1))
    small[..., 3] = 1
    clip = np.zeros((B, n_clip, 3, 4), f32)
    clip[..., :2] = rng.uniform(-1, 1, (B, n_clip, 3, 2))
    clip[:, :, 1:, :2] *= 10.0 ** rng.uniform(2, 5, (B, n_clip, 2, 1))
    clip[..., 2] = rng.uniform(-0.8, 0.8, (B, n_clip, 1))
    clip[..., 3] = 1
    pos = np.concatenate([huge.reshape(B, -1, 4), small.reshape(B, -1, 4), clip.reshape(B, -1, 4)], 1)
    tri = np.arange(pos.shape[1], dtype=np.int32).reshape(-1, 3)
    return pos.astype(f32), tri
