"""The C oracle against the independent float64 geometry reference (oracle/geometry_f64.py), on CPU.

Every bit-exact parity test holds the kernels to the oracle; this file holds the oracle -- the contract of DESIGN.md
section 3 -- to the geometry itself: at every decided pixel the triangle id must be the float64 winner and (u, v, z/w)
and the render() maps must lie within their a-priori float32 bounds.  A floor on the decided fraction keeps each case
from going vacuous (measured fractions in DESIGN.md section 6)."""
import numpy as np
import pytest

import cases
from oracle import geometry_f64 as g
from oracle import render_oracle, shim

MAX_PIXELS = 1 << 16
f32 = np.float32


def adversarial_soup(seed=0, B=1):
    """Faces built to sit where a contract mistake would show: vertices behind the camera (w < 0) and at w -> 0+,
    faces straddling z = -w and z = +w, vertices just inside and just outside the 2^22 snap limit (the guard-band
    clip), interpenetrating pairs (depth order crosses inside a triangle), slivers and back-facing faces.  Many of its
    pixels are undecided by construction (depth crossings, slivers, faces through the eye), and how many depends on the
    seed: at 256 x 256 the oracle decides 0.66 of the pixels for seeds 0 and 1 and 0.31 for seed 2, so the floor of
    0.6 below belongs to seed 0."""
    rng = np.random.default_rng(seed)
    faces = []

    def tri(p):
        faces.append(np.asarray(p, np.float64))

    for _ in range(40):   # w < 0 and w -> 0+ vertices
        a = [rng.uniform(-0.8, 0.8), rng.uniform(-0.8, 0.8), rng.uniform(-0.5, 0.5), 1.0]
        b = [rng.uniform(-1, 1), rng.uniform(-1, 1), 0.0, rng.choice([-0.5, 1e-6, 1e-3])]
        c = [rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(-0.5, 0.5), rng.uniform(0.5, 2.0)]
        tri([a, b, c])
    for _ in range(40):   # across z = -w and z = +w
        w = rng.uniform(0.5, 2.0, 3)
        k = rng.choice([-1.0, 1.0])
        z = w * (k + rng.uniform(-0.4, 0.4, 3))
        xy = rng.uniform(-1.2, 1.2, (3, 2)) * w[:, None]
        tri(np.column_stack([xy, z, w]))
    for _ in range(30):   # near the snap limit: |x/w| * 8W around 2^22 for W = 256
        lim = 2.0 ** 22 / (8 * 256)
        s = lim * rng.choice([0.999, 1.001]) * rng.choice([-1, 1])
        a = [rng.uniform(-0.9, 0.9), rng.uniform(-0.9, 0.9), 0.1, 1.0]
        tri([a, [s, rng.uniform(-1, 1), 0.1, 1.0], [rng.uniform(-1, 1), s, -0.1, 1.0]])
    for _ in range(30):   # interpenetrating pairs
        c = rng.uniform(-0.6, 0.6, 2)
        p = np.column_stack([c + rng.uniform(-0.4, 0.4, (3, 2)), [-0.5, 0.5, 0.0], np.ones(3)])
        q = np.column_stack([c + rng.uniform(-0.4, 0.4, (3, 2)), [0.5, -0.5, 0.1], np.ones(3)])
        tri(p)
        tri(q[::-1])      # back-facing
    for _ in range(60):   # slivers
        a = rng.uniform(-0.9, 0.9, 2)
        d = rng.uniform(-0.5, 0.5, 2)
        n = np.array([-d[1], d[0]]) * rng.uniform(1e-4, 2e-2)
        tri(np.column_stack([np.stack([a, a + d, a + 0.5 * d + n]), rng.uniform(-0.5, 0.5, 3), np.ones(3)]))
    pos = np.concatenate(faces)[None].astype(f32)
    pos = np.repeat(pos, B, 0)
    return pos, np.arange(pos.shape[1], dtype=np.int32).reshape(-1, 3)


SCENES = {
    # name: (builder, (H, W), floor of the decided fraction)
    "soup_ortho": (lambda: cases.random_soup(1, 400, B=2), (128, 160), 0.95),
    "soup_perspective": (lambda: cases.random_soup(3, 300, B=2, perspective=True), (128, 128), 0.95),
    "near_crossing": (cases.near_crossing_scene, (200, 320), 0.85),
    "guard_band": (cases.guard_band_scene, (600, 800), 0.98),
    "big_and_small_mix": (cases.big_and_small_mix, (1024, 1024), 0.98),
    "huge_triangles": (lambda: cases.huge_triangle_scene(B=1), (768, 1024), 0.92),
    "adversarial": (lambda: adversarial_soup(0, B=1), (256, 256), 0.6),
}


@pytest.mark.parametrize("name", list(SCENES))
def test_oracle_rasterize_matches_float64_geometry(name):
    build, (H, W), floor = SCENES[name]
    pos, tri = build()
    rast, ids = shim.rasterize(pos, tri, (H, W))
    rows, cols = g.pixel_sample(H, W, MAX_PIXELS)
    rep, _ = g.check_rasterize(pos, tri, H, W, rast, ids, rows, cols)
    print(name, rep)
    assert rep.fraction >= floor, rep
    assert rep.covered > 0.3 * rep.samples


MESHES = {"icosphere": lambda: cases.icosphere_mesh(8), "terrain": lambda: cases.terrain_mesh()}
CAMERAS = {"canonical": cases.canonical_cameras, "perspective": cases.perspective_cameras,
           "inside": cases.inside_cameras}


@pytest.mark.parametrize("cam_name", list(CAMERAS))
@pytest.mark.parametrize("mesh_name", list(MESHES))
def test_oracle_render_maps_match_float64_geometry(mesh_name, cam_name):
    v, f = MESHES[mesh_name]()
    n = cases.exact_vertex_normals(v, f)
    cam = CAMERAS[cam_name]()
    mvp, w2c = cam.mvp_mtx.numpy(), cam.w2c.numpy()
    H, W = 192, 224
    ref = render_oracle.render(v, f, mvp, w2c, H, W, v_nrm=n, depth=render_oracle.DepthSpec("none"))
    out = dict(mask=ref["mask"], pos=ref["pos"], normal=ref["normal"], depth=ref["depth"])
    rep = g.check_render(v, f, mvp, w2c, n, H, W, out)
    print(mesh_name, cam_name, rep)
    assert rep.fraction >= 0.95, rep
    assert rep.covered > 0.1 * rep.samples


def test_oracle_interpolate_and_texture_match_float64():
    """dr.interpolate of a UV attribute, then dr.texture in every filter / boundary mode, at decided pixels."""
    pos, tri = cases.random_soup(7, 150, B=1, perspective=True)
    H, W = 96, 112
    rast, ids = shim.rasterize(pos, tri, (H, W))
    rng = np.random.default_rng(1)
    attr = rng.uniform(-2.0, 3.0, (pos.shape[1], 2)).astype(np.float32)
    uv = shim.interpolate(attr[None], rast, tri)
    rows, cols = g.pixel_sample(H, W)
    _, views = g.check_rasterize(pos, tri, H, W, rast, ids, rows, cols)
    d = views[0].decided & (views[0].winner >= 0)
    r, c, face = rows[d], cols[d], views[0].winner[d]
    bc = g.barycentrics(pos[0], np.zeros(pos[0].shape), tri, face, r, c, H, W)
    val, bound = g.interpolate(attr, tri, face, bc)
    err = np.abs(uv[0, r, c] - val)
    assert np.all(err <= bound), float(np.max(err / bound))
    tex = rng.uniform(-1, 1, (13, 17, 3)).astype(np.float32)
    q = uv[0, r, c]
    for filt in ("nearest", "linear"):
        for mode in ("wrap", "clamp", "zero"):
            got = shim.texture(tex[None], q[None, None], filt, mode)[0, 0]
            want, tb, ok = g.texture(tex, q, filt, mode)
            assert ok.mean() > 0.99
            e = np.abs(got[ok] - want[ok])
            assert np.all(e <= tb[ok]), (filt, mode, float(np.max(e - tb[ok])))


def test_oracle_render_attr_and_tangent_maps_match_float64_geometry():
    """render()'s textured attribute map (UVs over their own faces, bilinear, wrap) and tangent map (vertex tangents
    over the normal faces, normalised), with their backgrounds."""
    from worldrenderer_b200 import synth
    v, f = cases.icosphere_mesh(8)
    n = cases.exact_vertex_normals(v, f)
    vt, ft = synth.cell_atlas_uv(f.shape[0])
    vt, ft = vt.astype(f32), ft.astype(np.int32)
    tex = np.random.default_rng(3).uniform(0, 1, (37, 53, 3)).astype(f32)
    tang = render_oracle.vertex_tangents(v, f, vt, ft, n)
    cam = cases.perspective_cameras()
    mvp, w2c = cam.mvp_mtx.numpy(), cam.w2c.numpy()
    H, W = 128, 144
    ref = render_oracle.render(v, f, mvp, w2c, H, W, v_nrm=n, depth=render_oracle.DepthSpec("none"), v_tex=vt,
                               tri_tex=ft, texture=tex)
    t = shim.interpolate(tang[None], ref["rast"], f)
    ln = np.sqrt((t[..., 0] * t[..., 0] + t[..., 1] * t[..., 1]) + t[..., 2] * t[..., 2])
    t = (t / np.maximum(ln, f32(1e-12))[..., None]).astype(f32)
    t[~ref["mask"]] = f32(0.25)
    out = dict(mask=ref["mask"], pos=ref["pos"], normal=ref["normal"], depth=ref["depth"], attr=ref["attr"],
               tangent=t)
    rep = g.check_render(v, f, mvp, w2c, n, H, W, out, v_tang=tang, v_tex=vt, tri_tex=ft, tex=tex,
                         tangent_background=0.25)
    print(rep)
    assert rep.fraction >= 0.95, rep
    assert {"attr", "tangent"} <= set(rep.ratio)
