"""GPU parity, render() level: the fused wr_render pipeline against the oracle's restatement of
render.py:220-286 (oracle/render_oracle.py, pinned to the reference's own Python by tests/golden).

Bar: mask / triangle id bit-exact; pos, normal, depth within 1e-5 relative."""
import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import render_oracle
from oracle.render_oracle import DepthSpec
from worldrenderer_b200.render import render_geometry_raw

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6


def make_mesh(v, f, device, with_uv=False, tex_size=32, seed=0):
    mesh = wr.TexturedMesh(v_pos=torch.tensor(v, dtype=torch.float32), t_pos_idx=torch.tensor(f, dtype=torch.int64))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    if with_uv:
        from worldrenderer_b200 import synth
        vt, ft = synth.cell_atlas_uv(f.shape[0])
        mesh.v_tex = torch.tensor(vt, dtype=torch.float32)
        mesh.t_tex_idx = torch.tensor(ft, dtype=torch.int64)
        rng = np.random.default_rng(seed)
        mesh.texture = torch.tensor(rng.uniform(0, 1, (tex_size, tex_size, 3)), dtype=torch.float32)
    mesh.to(device)
    return mesh


STRATEGIES = [
    (wr.DepthControlNetNormalization(), DepthSpec("controlnet")),
    (wr.DepthControlNetNormalization(far_clip=0.1, near_clip=0.9, bg_value=0.3), DepthSpec("controlnet", far_clip=0.1, near_clip=0.9, bg_value=0.3)),
    (wr.Zero123PlusPlusNormalization(), DepthSpec("zero123pp")),
    (wr.SimpleNormalization(), DepthSpec("simple", scale=1.0, offset=-1.0, clamp=True)),
    (wr.SimpleNormalization(scale=1.0, offset=0.0, clamp=False, bg_value=1e2), DepthSpec("simple", scale=1.0, offset=0.0, clamp=False, bg_value=1e2)),
    (None, DepthSpec("none")),
]


def _oracle(mesh, cam, H, W, spec, with_attr=False, filt="linear"):
    kw = {}
    if with_attr:
        kw = dict(v_tex=mesh.v_tex.cpu().numpy(), tri_tex=mesh.t_tex_idx.cpu().numpy().astype(np.int32),
                  texture=mesh.texture.cpu().numpy(), texture_filter_mode=filt)
    return render_oracle.render(mesh.v_pos.cpu().numpy(), mesh.t_pos_idx.cpu().numpy().astype(np.int32),
                                cam.mvp_mtx.cpu().numpy(), cam.w2c.cpu().numpy(), H, W,
                                v_nrm=mesh.v_nrm.cpu().numpy(), depth=spec, **kw)


def _compare(out, ref, ids=None):
    np.testing.assert_array_equal(out.mask.cpu().numpy(), ref["mask"])
    if ids is not None:
        np.testing.assert_array_equal(ids.cpu().numpy(), ref["tri_id"])
    np.testing.assert_allclose(out.pos.cpu().numpy(), ref["pos"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(out.normal.cpu().numpy(), ref["normal"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(out.depth.cpu().numpy(), ref["depth"], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("strategy,spec", STRATEGIES)
def test_icosphere_canonical_rig(wr_ctx, strategy, spec):
    v, f = cases.icosphere_mesh(10)
    mesh = make_mesh(v, f, wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    out = wr.render(wr_ctx, mesh, cam, 160, 160, render_attr=False, depth_normalization_strategy=strategy)
    assert out.mask.dtype == torch.bool and out.depth.shape == (6, 160, 160) and out.pos.shape == (6, 160, 160, 3)
    _compare(out, _oracle(mesh, cam, 160, 160, spec))


@pytest.mark.parametrize("H,W", [(30, 34), (33, 31), (7, 5), (64, 36), (1, 16), (50, 50)])
@pytest.mark.parametrize("strategy,spec", [STRATEGIES[0], STRATEGIES[2], STRATEGIES[5]])
def test_viewport_shapes_take_every_store_and_finalize_path(wr_ctx, H, W, strategy, spec):
    """H*W a multiple of 16 / of 4 only / of neither, W a multiple of 4 or not: the second depth pass has a
    16-pixel, a 4-pixel and a scalar form, and the background rows of the shading kernel a 16-byte-store form."""
    v, f = cases.icosphere_mesh(6)
    mesh = make_mesh(v, f, wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    out = wr.render(wr_ctx, mesh, cam, H, W, render_attr=False, depth_normalization_strategy=strategy)
    ref = _oracle(mesh, cam, H, W, spec)
    _compare(out, ref)
    for k in ("pos", "normal", "depth"):
        np.testing.assert_array_equal(getattr(out, k).cpu().numpy(), ref[k], err_msg=k)


def test_tri_ids_and_rast_fused(wr_ctx):
    v, f = cases.terrain_mesh(128, 64)
    mesh = make_mesh(v, f, wr_ctx.device)
    for cam in [cases.canonical_cameras(device=wr_ctx.device), cases.perspective_cameras(device=wr_ctx.device),
                cases.inside_cameras(device=wr_ctx.device)]:
        raw = render_geometry_raw(wr_ctx, mesh, cam, 200, 264, want_tri_id=True, want_rast=True,
                                  depth_normalization_strategy=wr.DepthControlNetNormalization())
        ref = _oracle(mesh, cam, 200, 264, DepthSpec("controlnet"))
        np.testing.assert_array_equal(raw["tri_id"].cpu().numpy(), ref["tri_id"])
        np.testing.assert_array_equal(raw["mask"].cpu().numpy(), ref["mask"])
        np.testing.assert_allclose(raw["rast"].cpu().numpy(), ref["rast"], rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(raw["pos"].cpu().numpy(), ref["pos"], rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(raw["normal"].cpu().numpy(), ref["normal"], rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(raw["depth"].cpu().numpy(), ref["depth"], rtol=RTOL, atol=ATOL)
        # Stronger than the 1e-5 bar: the kernels issue the same individually rounded operations in the same order
        # as the oracle (-fmad=false, IEEE div / sqrt), so every float map is identical bit for bit.
        for k in ("rast", "pos", "normal", "depth"):
            np.testing.assert_array_equal(raw[k].cpu().numpy(), ref[k], err_msg=k)


def test_custom_strategy_and_backgrounds(wr_ctx):
    v, f = cases.icosphere_mesh(6)
    mesh = make_mesh(v, f, wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)

    class Halve(wr.DepthNormalizationStrategy):
        def __init__(self):
            pass

        def __call__(self, depth, mask):
            return depth * 0.5

    out = wr.render(wr_ctx, mesh, cam, 64, 80, render_attr=False, depth_normalization_strategy=Halve(),
                    normal_background=torch.tensor([0.5, 0.25, 1.0]))
    ref = _oracle(mesh, cam, 64, 80, DepthSpec("none"))
    np.testing.assert_allclose(out.depth.cpu().numpy(), ref["depth"] * np.float32(0.5), rtol=RTOL, atol=ATOL)
    n = out.normal.cpu().numpy()
    assert np.allclose(n[~ref["mask"]], [0.5, 0.25, 1.0])
    np.testing.assert_allclose(n[ref["mask"]], ref["normal"][ref["mask"]], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("filt", ["linear", "nearest"])
def test_render_attr(wr_ctx, filt):
    v, f = cases.icosphere_mesh(6)
    mesh = make_mesh(v, f, wr_ctx.device, with_uv=True)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    out = wr.render(wr_ctx, mesh, cam, 128, 128, render_attr=True, texture_filter_mode=filt, attr_background=0.25)
    ref = _oracle(mesh, cam, 128, 128, DepthSpec("controlnet"), with_attr=True, filt=filt)
    ref_attr = np.where(ref["mask"][..., None], ref["attr"], np.float32(0.25))
    np.testing.assert_allclose(out.attr.cpu().numpy(), ref_attr, rtol=RTOL, atol=ATOL)
    _compare(out, ref)


def test_vertex_normals_match_oracle(wr_ctx):
    v, f = cases.terrain_mesh(64, 48)
    mesh = make_mesh(v, f, wr_ctx.device)
    ref = render_oracle.vertex_normals(v, f)
    # float atomics: sum order differs from the CPU loop, so tolerance (not bit) parity
    np.testing.assert_allclose(mesh.v_nrm.cpu().numpy(), ref, rtol=1e-5, atol=1e-6)


def test_vertex_normals_are_exact_sums_independent_of_order(wr_ctx):
    """The face normals are splatted in 64-bit fixed point: the result is the correctly rounded sum, identical bit for
    bit whatever the order of the atomics -- rerun, and with the faces listed in a different order."""
    v, f = cases.terrain_mesh(300, 200, seed=3)
    dev = wr_ctx.device
    a = make_mesh(v, f, dev).v_nrm
    b = make_mesh(v, f, dev).v_nrm
    perm = np.random.default_rng(0).permutation(f.shape[0])
    c = make_mesh(v, f[perm], dev).v_nrm
    assert torch.equal(a, b) and torch.equal(a, c)
    # against the exact sum in float64
    np.testing.assert_allclose(a.cpu().numpy(), cases.exact_vertex_normals(v, f), rtol=0, atol=1.2e-7)


def test_single_view_indexing_and_no_cpu_path(wr_ctx):
    v, f = cases.icosphere_mesh(4)
    mesh = make_mesh(v, f, wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    full = wr.render(wr_ctx, mesh, cam, 48, 48, render_attr=False)
    one = wr.render(wr_ctx, mesh, cam[2], 48, 48, render_attr=False)
    assert one.mask.shape == (1, 48, 48)
    assert torch.equal(one.mask[0], full.mask[2]) and torch.equal(one.pos[0], full.pos[2])
    cpu_mesh = make_mesh(v, f, "cpu")
    with pytest.raises(RuntimeError):
        wr.render(wr_ctx, cpu_mesh, cam, 48, 48, render_attr=False)
    with pytest.raises(RuntimeError):
        wr.NVDiffRastContextWrapper("cpu", "cuda")
    with pytest.raises(NotImplementedError):
        wr.NVDiffRastContextWrapper(str(wr_ctx.device), "vulkan")


def test_full_size_properties_1m_faces(wr_ctx):
    """BASELINE config B at full size (1M faces, 6 views, 768^2): properties that need no oracle run."""
    from worldrenderer_b200 import synth
    v, f = synth.terrain(1000, 500, 0)
    v = v / np.abs(v).max() * 0.5
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1).astype(np.float32)
    mesh = make_mesh(v, f.astype(np.int32), wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    raw = render_geometry_raw(wr_ctx, mesh, cam, 768, 768, want_tri_id=True, want_rast=True,
                              depth_normalization_strategy=wr.DepthControlNetNormalization())
    raw2 = render_geometry_raw(wr_ctx, mesh, cam, 768, 768, want_tri_id=True, want_rast=True,
                               depth_normalization_strategy=wr.DepthControlNetNormalization())
    ids = raw["tri_id"]
    assert torch.equal(ids, raw2["tri_id"]) and torch.equal(raw["pos"], raw2["pos"])  # deterministic
    assert int(ids.max()) < f.shape[0] and int(ids.min()) == -1
    assert torch.equal(raw["mask"], ids >= 0)
    # the face-on view of a height field covers its whole footprint: a filled rectangle
    m = raw["mask"][0]  # view 0 looks along -y at the full face of the (x, z) height-field wall
    rows = m.any(1).nonzero().flatten()
    cols = m.any(0).nonzero().flatten()
    # (eroded by 3 px: at 89.99 degrees the relief shifts the silhouette by a fraction of a pixel)
    assert bool(m[rows.min() + 3:rows.max() - 2, cols.min() + 3:cols.max() - 2].all())
    assert int(m.sum()) > 0.3 * 768 * 768
    # face-on views (0, 2).  The triangles are ~0.3 px across, and coverage is decided on vertices snapped to
    # 1/16 px while (u, v) come from the unsnapped ones (DESIGN.md 3.4): a sample can sit a few percent outside
    # the unsnapped outline, so u + v may exceed 1 slightly; it must stay a small extrapolation.
    for b in (0, 2):
        r = raw["rast"][b][raw["mask"][b]]
        assert float((r[:, 0] + r[:, 1]).max()) <= 1.5
        assert float(((r[:, 0] + r[:, 1]) > 1.05).float().mean()) < 0.02
        p = raw["pos"][b][raw["mask"][b]]
        assert float(p.abs().max()) <= 0.5 + 1e-2
    n = raw["normal"][raw["mask"]]
    assert torch.allclose(n.norm(dim=-1), torch.ones_like(n[:, 0]), atol=1e-5)
    d = raw["depth"]
    assert float(d[raw["mask"]].min()) >= 0.25 - 1e-6 and float(d.max()) <= 1.0 + 1e-6
    assert float(d[~raw["mask"]].abs().max()) == 0.0


def test_config_e_scale_runs_and_is_consistent(wr_ctx):
    """Config E shapes on one GPU's share: 5M faces, 4 views at 2048^2 (memory sizing + large-F indexing)."""
    from worldrenderer_b200 import synth
    v, f = synth.terrain(2500, 1000, 3)
    assert f.shape[0] == 5_000_000
    v = v / np.abs(v).max() * 0.5
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1).astype(np.float32)
    mesh = make_mesh(v, f.astype(np.int32), wr_ctx.device)
    cam = wr.get_orthogonal_camera(elevation_deg=[20.0] * 4, distance=[1.0] * 4, left=-0.55, right=0.55, bottom=-0.55,
                                   top=0.55, azimuth_deg=[-90.0, -45.0, 0.0, 60.0], device=str(wr_ctx.device))
    raw = render_geometry_raw(wr_ctx, mesh, cam, 2048, 2048, want_tri_id=True,
                              depth_normalization_strategy=wr.SimpleNormalization(scale=1.0, offset=0.0, clamp=False, bg_value=1e2))
    ids = raw["tri_id"]
    assert int(ids.max()) < 5_000_000 and torch.equal(raw["mask"], ids >= 0)
    assert int(raw["mask"][0].sum()) > 0.2 * 2048 * 2048
    # a low-resolution render of the same scene must agree with the high-resolution one where both are interior
    lo = render_geometry_raw(wr_ctx, mesh, cam, 512, 512, depth_normalization_strategy=wr.SimpleNormalization(scale=1.0, offset=0.0, clamp=False, bg_value=1e2))
    hi_pos = raw["pos"][:, 2::4, 2::4]  # pixel centres do not coincide exactly: compare loosely
    both = raw["mask"][:, 2::4, 2::4] & lo["mask"]
    diff = (hi_pos[both] - lo["pos"][both]).abs().max(dim=-1).values
    assert float((diff < 5e-3).float().mean()) > 0.97  # the rest sit on occlusion edges of the relief
    assert wr_ctx.ctx.scratch_bytes() < 2 << 30


def test_config_b_full_size_bit_exact_ids_against_oracle(wr_ctx):
    """BASELINE config B at full size: 1M-face terrain, canonical 6-view rig, 768^2 -- triangle ids and masks
    bit-exact, position / normal / depth within 1e-5 against the CPU oracle (about 2 s of host time)."""
    from worldrenderer_b200 import synth
    v, f = synth.terrain(1000, 500, 0)
    v = v / np.abs(v).max() * 0.5
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1).astype(np.float32)
    mesh = make_mesh(v, f.astype(np.int32), wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    raw = render_geometry_raw(wr_ctx, mesh, cam, 768, 768, want_tri_id=True,
                              depth_normalization_strategy=wr.DepthControlNetNormalization())
    ref = _oracle(mesh, cam, 768, 768, DepthSpec("controlnet"))
    np.testing.assert_array_equal(raw["tri_id"].cpu().numpy(), ref["tri_id"])
    np.testing.assert_array_equal(raw["mask"].cpu().numpy(), ref["mask"])
    np.testing.assert_allclose(raw["pos"].cpu().numpy(), ref["pos"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(raw["normal"].cpu().numpy(), ref["normal"], rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(raw["depth"].cpu().numpy(), ref["depth"], rtol=RTOL, atol=ATOL)
    for k in ("pos", "normal", "depth"):  # bit-identical as well (see test_tri_ids_and_rast_fused)
        np.testing.assert_array_equal(raw[k].cpu().numpy(), ref[k], err_msg=k)
    assert ref["mask"].sum() > 700_000


def test_render_tangent_fused(wr_ctx):
    """render_tangent=True (render.py:280-284): interpolated + normalised v_tang, against the operator form."""
    v, f = cases.icosphere_mesh(6)
    mesh = make_mesh(v, f, wr_ctx.device, with_uv=True)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    out = wr.render(wr_ctx, mesh, cam, 96, 96, render_attr=False, render_tangent=True, tangent_background=0.25)
    raw = render_geometry_raw(wr_ctx, mesh, cam, 96, 96, want_rast=True)
    tang, _ = wr_ctx.interpolate(mesh.v_tang[None], raw["rast"], mesh.t_pos_idx)
    tang = torch.nn.functional.normalize(tang, dim=-1, p=2)
    tang[~raw["mask"]] = 0.25
    assert out.tangent.shape == (6, 96, 96, 3)
    torch.testing.assert_close(out.tangent, tang, rtol=1e-5, atol=1e-6)
    # and the interpolation itself against the oracle
    from oracle import shim
    ref = shim.interpolate(mesh.v_tang.cpu().numpy()[None], raw["rast"].cpu().numpy(), f)
    ln = np.sqrt((ref * ref).sum(-1, keepdims=True))
    ref = ref / np.maximum(ln, 1e-12)
    m = raw["mask"].cpu().numpy()
    np.testing.assert_allclose(out.tangent.cpu().numpy()[m], ref[m], rtol=1e-5, atol=1e-6)


def test_many_views_small_resolution_and_single_view(wr_ctx):
    """SmartPainter-style batch (smart_paint.py:102-111): many perspective views of a small mesh at low resolution."""
    v, f = cases.icosphere_mesh(5)
    mesh = make_mesh(v, f, wr_ctx.device)
    n = 36
    cam = wr.get_camera(elevation_deg=list(np.linspace(-60, 60, n)), distance=[1.6] * n, fovy_deg=[45.0] * n,
                        azimuth_deg=list(np.linspace(0, 350, n)), device=str(wr_ctx.device))
    out = wr.render(wr_ctx, mesh, cam, 40, 56, render_attr=False)
    ref = _oracle(mesh, cam, 40, 56, DepthSpec("controlnet"))
    _compare(out, ref)
    one = wr.render(wr_ctx, mesh, cam[17], 40, 56, render_attr=False)
    assert torch.equal(one.mask[0], out.mask[17]) and torch.equal(one.normal[0], out.normal[17])


def test_empty_mesh_renders_background(wr_ctx):
    mesh = wr.TexturedMesh(v_pos=torch.zeros((3, 3), device=wr_ctx.device),
                           t_pos_idx=torch.zeros((0, 3), dtype=torch.int64, device=wr_ctx.device))
    mesh.set_stitched_mesh(mesh.v_pos, mesh.t_pos_idx)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    out = wr.render(wr_ctx, mesh, cam, 32, 48, render_attr=False, normal_background=0.5)
    assert not bool(out.mask.any()) and float(out.pos.abs().max()) == 0.0
    assert float((out.normal - 0.5).abs().max()) == 0.0 and float(out.depth.abs().max()) == 0.0


def test_guards_autograd_face_count_and_rast_id_range(wr_ctx):
    """Forward-only kernels refuse inputs that require grad (the reference is differentiable through nvdiffrast);
    the normal / bake-view / tangent paths check that the stitched faces pair up with t_pos_idx; the float-encoded
    triangle id of the rast tensor is refused beyond 2^24 faces."""
    from worldrenderer_b200.render import render_geometry_raw
    dev = wr_ctx.device
    v, f = cases.icosphere_mesh(4)
    mesh = make_mesh(v, f, dev)
    cam = cases.canonical_cameras(device=dev)
    mesh.v_pos.requires_grad_(True)
    with pytest.raises(NotImplementedError):
        wr.render(wr_ctx, mesh, cam, 32, 32, render_attr=False)
    with torch.no_grad():
        out = wr.render(wr_ctx, mesh, cam, 32, 32, render_attr=False)
    assert out.mask.any()
    pos = torch.zeros(1, 4, 4, device=dev, requires_grad=True)
    with pytest.raises(NotImplementedError):
        wr_ctx.rasterize(pos, torch.zeros(1, 3, dtype=torch.int32, device=dev), (8, 8))
    mesh.v_pos.requires_grad_(False)
    mesh.v_nrm
    mesh._stitched_t_pos_idx = mesh.t_pos_idx[:-5].clone()   # fewer stitched faces than faces
    for kw in (dict(want_geo=True, want_normal=False, want_pos=False,
                    depth_normalization_strategy=wr.SimpleNormalization(scale=1.0, offset=0.0, clamp=False, bg_value=1e2)),
               dict(want_normal=True)):
        with pytest.raises(ValueError):
            render_geometry_raw(wr_ctx, mesh, cam, 32, 32, **kw)
    big = torch.zeros(((1 << 24) + 1, 3), dtype=torch.int32, device=dev)
    with pytest.raises(NotImplementedError):
        wr_ctx.rasterize(torch.zeros(1, 4, 4, device=dev), big, (8, 8))
    _, ids = wr_ctx.rasterize_with_ids(torch.zeros(1, 4, 4, device=dev), big[: 1 << 20], (8, 8))
    assert (ids == -1).all()


def test_config_a_full_size_bit_exact_against_oracle(wr_ctx):
    """BASELINE config A at full size: 50k-face icosphere, canonical 6-view rig, 768^2 (the coarse-mesh path:
    several lanes per triangle in the set-up kernel, 16-byte vertex records in the shading kernel)."""
    v, f = cases.icosphere_mesh(50)
    assert f.shape[0] == 50_000
    mesh = make_mesh(v, f, wr_ctx.device)
    cam = cases.canonical_cameras(device=wr_ctx.device)
    raw = render_geometry_raw(wr_ctx, mesh, cam, 768, 768, want_tri_id=True,
                              depth_normalization_strategy=wr.DepthControlNetNormalization())
    ref = _oracle(mesh, cam, 768, 768, DepthSpec("controlnet"))
    np.testing.assert_array_equal(raw["tri_id"].cpu().numpy(), ref["tri_id"])
    np.testing.assert_array_equal(raw["mask"].cpu().numpy(), ref["mask"])
    for k in ("pos", "normal", "depth"):
        np.testing.assert_array_equal(raw[k].cpu().numpy(), ref[k], err_msg=k)
    assert ref["mask"].sum() > 6 * 0.6 * 768 * 768   # a sphere of radius 0.5 in a 1.1-wide frame covers 65 %


def test_config_e_share_bit_exact_against_oracle(wr_ctx):
    """BASELINE config E, one GPU's share at full size: 5M-face terrain, 4 of the 32 ring views at 2048^2 -- triangle
    ids, coverage, position, normal and depth identical to the CPU oracle (a few seconds of host time)."""
    from worldrenderer_b200 import synth
    v, f = synth.terrain(2500, 1000, 3)
    assert f.shape[0] == 5_000_000
    v = v / np.abs(v).max() * 0.5
    v = np.stack([v[:, 0], -v[:, 2], v[:, 1]], -1).astype(np.float32)
    mesh = make_mesh(v, f.astype(np.int32), wr_ctx.device)
    az = [360.0 * k / 32 - 90.0 for k in (0, 9, 18, 27)]
    cam = wr.get_orthogonal_camera(elevation_deg=[20.0] * 4, distance=[1.0] * 4, left=-0.55, right=0.55, bottom=-0.55,
                                   top=0.55, azimuth_deg=az, device=str(wr_ctx.device))
    spec = wr.SimpleNormalization(scale=1.0, offset=0.0, clamp=False, bg_value=1e2)
    raw = render_geometry_raw(wr_ctx, mesh, cam, 2048, 2048, want_tri_id=True, depth_normalization_strategy=spec)
    ref = _oracle(mesh, cam, 2048, 2048, DepthSpec("simple", scale=1.0, offset=0.0, clamp=False, bg_value=1e2))
    np.testing.assert_array_equal(raw["tri_id"].cpu().numpy(), ref["tri_id"])
    np.testing.assert_array_equal(raw["mask"].cpu().numpy(), ref["mask"])
    for k in ("pos", "normal", "depth"):
        np.testing.assert_array_equal(raw[k].cpu().numpy(), ref[k], err_msg=k)
    assert ref["mask"].sum() > 4 * 0.2 * 2048 * 2048
