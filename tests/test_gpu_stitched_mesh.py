"""GPU parity of render() and the UV bake on stitched meshes: meshes whose normals come from a second, merged vertex
set with its own face indices (TexturedMesh.set_stitched_mesh), as load_mesh builds them for every trimesh asset.
The shading kernel then reads the normals -- and the tangents -- through `tri_nrm`, the stitched faces, and the
vertex pass writes Vn 16-byte normal records next to the V position records.  The three forms of
cases.stitched_icosphere (seams: Vn < V, permuted: Vn == V with other indices, flat: Vn > V) on both raster paths
(multi-view when 4 F > H W, per-view otherwise) and both vertex-record forms (packed when B H W >= 32 (V + Vn)).

The bar is the one of the plain-mesh tests: masks and triangle ids bit-exact, and every float map bit-exact too
(the kernels issue the oracle's individually rounded operations in its order); blended bake colours within 1e-5."""
import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import render_oracle, shim
from oracle.render_oracle import DepthSpec
from worldrenderer_b200 import synth
from worldrenderer_b200.render import render_geometry_raw
from worldrenderer_b200.uv import fused_view_maps

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
f32 = np.float32
BAKE_DEPTH = dict(scale=1.0, offset=0.0, clamp=False, bg_value=1e2)


def _np(t):
    return t.detach().cpu().numpy()


def stitched_mesh(form, device, tex_size=(37, 53, 3), seed=0):
    d = cases.stitched_icosphere(form)
    mesh = wr.TexturedMesh(v_pos=torch.from_numpy(d["v_pos"]), t_pos_idx=torch.from_numpy(d["t_pos_idx"]).long(),
                           v_tex=torch.from_numpy(d["v_tex"]), t_tex_idx=torch.from_numpy(d["t_tex_idx"]).long())
    mesh.set_stitched_mesh(torch.from_numpy(d["stitched_v_pos"]), torch.from_numpy(d["stitched_t_pos_idx"]).long())
    rng = np.random.default_rng(seed)
    mesh.texture = torch.tensor(rng.uniform(0, 1, tex_size), dtype=torch.float32)
    mesh.to(device)
    return mesh


def raster_path(mesh, B, H, W):
    """(raster path, vertex-record form) wr_render takes for this mesh and output set (raster.cu use_mv, render.cu
    use_pack; every output set here reads the normals, so Vn counts)."""
    F, V, Vn = mesh.t_pos_idx.shape[0], mesh.v_pos.shape[0], mesh.v_nrm.shape[0]
    return ("multi-view" if 4 * F > H * W else "per-view",
            "packed" if B * H * W >= 32 * (V + Vn) else "unpacked")


RIGS = {"canonical6": lambda H, W, dev: cases.canonical_cameras(device=dev),
        "perspective4": lambda H, W, dev: cases.bake_perspective_cameras(H, W, device=dev),
        "mixed40": cases.mixed_40_view_cameras}

# (rig, H, W, expected path) -- the same for the three forms (V + Vn is 3.5 F for seams and flat, F for permuted)
PATHS = [
    ("canonical6", 64, 64, ("multi-view", "unpacked")),
    ("mixed40", 64, 64, ("multi-view", "packed")),
    ("perspective4", 96, 96, ("per-view", "unpacked")),
    ("canonical6", 160, 160, ("per-view", "packed")),
]


def _oracle(mesh, cam, H, W, spec, texture=None, filt="linear"):
    kw = {}
    if texture is not None:
        kw = dict(v_tex=_np(mesh.v_tex), tri_tex=_np(mesh.t_tex_idx).astype(np.int32), texture=texture,
                  texture_filter_mode=filt)
    return render_oracle.render(_np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32), _np(cam.mvp_mtx),
                                _np(cam.w2c), H, W, v_nrm=_np(mesh.v_nrm),
                                tri_nrm=_np(mesh.stitched_t_pos_idx).astype(np.int32), depth=spec, **kw)


def _same(got, want, what):
    np.testing.assert_array_equal(_np(got), want, err_msg=what)


@pytest.mark.parametrize("form", cases.STITCHED_FORMS)
def test_vertex_normals_are_exact_sums_over_stitched_faces(wr_ctx, form):
    """mesh.v_nrm has one row per stitched vertex and is the float64 sum of the float face normals of the stitched
    faces, rounded once, then normalised."""
    d = cases.stitched_icosphere(form)
    mesh = stitched_mesh(form, wr_ctx.device)
    sv, sf = d["stitched_v_pos"], d["stitched_t_pos_idx"].astype(np.int64)
    assert mesh.v_nrm.shape == sv.shape
    assert (sv.shape[0] < d["v_pos"].shape[0], sv.shape[0] == d["v_pos"].shape[0], sv.shape[0] > d["v_pos"].shape[0]) \
        == (form == "seams", form == "permuted", form == "flat")
    np.testing.assert_allclose(_np(mesh.v_nrm), cases.exact_vertex_normals(sv, sf), rtol=0, atol=1.2e-7)


@pytest.mark.parametrize("rig,H,W,path", PATHS, ids=[f"{p[0]}-{p[1]}-{r}-{h}x{w}" for r, h, w, p in PATHS])
@pytest.mark.parametrize("form", cases.STITCHED_FORMS)
def test_render_output_sets_match_oracle(wr_ctx, form, rig, H, W, path):
    """Each shading instantiation that reads the normals: the default controlnet set, SimpleNormalization, the bake
    view map (want_geo alone) and the generic one (triangle ids, the textured attribute, and on the permuted form
    the tangents, which need Vn == V)."""
    dev = wr_ctx.device
    mesh = stitched_mesh(form, dev)
    cam = RIGS[rig](H, W, dev)
    B = cam.mvp_mtx.shape[0]
    assert raster_path(mesh, B, H, W) == path

    # kOutsRenderDefault: mask + pos + normal + controlnet depth
    out = wr.render(wr_ctx, mesh, cam, H, W, render_attr=False)
    ref = _oracle(mesh, cam, H, W, DepthSpec("controlnet"))
    assert ref["mask"].sum() > 0.1 * B * H * W
    _same(out.mask, ref["mask"], "mask")
    for k in ("pos", "normal", "depth"):
        _same(getattr(out, k), ref[k], k)

    # kOutsSimpleDepth
    out = wr.render(wr_ctx, mesh, cam, H, W, render_attr=False, depth_normalization_strategy=wr.SimpleNormalization(),
                    normal_background=0.5)
    ref_s = render_oracle.render(_np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32), _np(cam.mvp_mtx),
                                 _np(cam.w2c), H, W, v_nrm=_np(mesh.v_nrm),
                                 tri_nrm=_np(mesh.stitched_t_pos_idx).astype(np.int32),
                                 depth=DepthSpec("simple", scale=1.0, offset=-1.0, clamp=True), normal_background=0.5)
    _same(out.mask, ref_s["mask"], "mask")
    for k in ("pos", "normal", "depth"):
        _same(getattr(out, k), ref_s[k], k)

    # kOutsBakeView: mask + (pos, aoi_cos) + raw view depth, no position or normal map
    raw = render_geometry_raw(wr_ctx, mesh, cam, H, W, want_pos=False, want_depth=True, want_normal=False,
                              want_geo=True, depth_normalization_strategy=wr.SimpleNormalization(**BAKE_DEPTH))
    assert set(raw) == {"mask", "depth", "geo"}
    stub = {"uv_pos": np.zeros((1, 1, 3), f32)}   # view planes only
    rgeo = render_oracle.uv_render_geometry(_np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32), _np(mesh.v_nrm),
                                            _np(mesh.stitched_t_pos_idx).astype(np.int32), _np(cam.mvp_mtx),
                                            _np(cam.w2c), H, W, stub, False)
    _same(raw["mask"], rgeo["view_mask"], "mask")
    _same(raw["geo"][..., :3], rgeo["view_position"], "geo.xyz")
    _same(raw["geo"][..., 3], rgeo["view_aoi_cos"], "geo.w")
    _same(raw["depth"], rgeo["view_depth"], "depth")

    # generic instantiation
    tangent = form == "permuted"
    raw = render_geometry_raw(wr_ctx, mesh, cam, H, W, want_attr=True, want_tri_id=True, want_tangent=tangent,
                              tangent_background=0.25, depth_normalization_strategy=wr.DepthControlNetNormalization())
    ref = _oracle(mesh, cam, H, W, DepthSpec("controlnet"), texture=_np(mesh.texture))
    _same(raw["tri_id"], ref["tri_id"], "tri_id")
    _same(raw["mask"], ref["mask"], "mask")
    for k in ("pos", "normal", "depth", "attr"):
        _same(raw[k], ref[k], k)
    if tangent:
        # render.py:280-284: v_tang interpolated over the stitched faces, normalised, background outside
        def tangent_map(faces):
            t = shim.interpolate(_np(mesh.v_tang)[None], ref["rast"], faces)
            ln = np.sqrt((t[..., 0] * t[..., 0] + t[..., 1] * t[..., 1]) + t[..., 2] * t[..., 2])
            t = (t / np.maximum(ln, f32(1e-12))[..., None]).astype(f32)
            t[~ref["mask"]] = f32(0.25)
            return t
        want = tangent_map(_np(mesh.stitched_t_pos_idx))
        _same(raw["tangent"], want, "tangent")
        # the stitched faces are not the position faces: read through those, the map would differ
        assert not np.array_equal(tangent_map(_np(mesh.t_pos_idx)), want)


def _bake_oracle(mesh, cam, images, uv_size, **kw):
    return render_oracle.camera_projection(
        images, _np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32), _np(mesh.v_nrm),
        _np(mesh.stitched_t_pos_idx).astype(np.int32), _np(mesh.v_tex), _np(mesh.t_tex_idx).astype(np.int32),
        _np(mesh.texture), _np(cam.mvp_mtx), _np(cam.w2c), uv_size, **kw)


def test_bake_of_seams_mesh_matches_oracle(wr_ctx):
    """The load_mesh form through the whole bake: CameraProjection's fused kernels (view map written by the shading
    kernel from the stitched normals) and the step-by-step uv_render_geometry (normal map, then wr_view_prep),
    against the oracle's camera_projection with the stitched faces -- intermediates bit-exact, colours within 1e-5."""
    dev = wr_ctx.device
    Hu = Wu = 128
    mesh = stitched_mesh("seams", dev, tex_size=(Hu, Wu, 3), seed=1)
    cam = cases.canonical_cameras(device=dev)
    H = W = 96
    images = synth.view_images(6, H, W, seed=1)
    kw = dict(aoi_cos_valid_threshold=0.2, depth_grad_threshold=0.1, uv_exp_blend_alpha=3.0, depth_grad_dilation=5)
    proj = wr.CameraProjection(None, None, str(dev), "cuda")
    out = proj(torch.from_numpy(images), mesh, cam, uv_size=Hu, poisson_blending=False, uv_padding=False,
               iou_rejection_threshold=None, return_dict=True, **kw)
    ref = _bake_oracle(mesh, cam, images, Hu, iou_rejection_threshold=None, **kw)
    assert ref["uv_proj_mask"].sum() > 0.3 * ref["pre"]["uv_mask"].sum()
    _same(out.uv_aoi_cos, ref["uv_aoi_cos"], "uv_aoi_cos")
    _same(out.uv_depth_grad, ref["uv_depth_grad"], "uv_depth_grad")
    _same(out.uv_proj_mask, ref["uv_proj_mask"], "uv_proj_mask")
    np.testing.assert_allclose(_np(out.uv_proj), ref["uv_proj"], rtol=RTOL, atol=ATOL)

    # the fused view map itself
    mask, geo_map, _ = fused_view_maps(wr_ctx, mesh, cam, torch.from_numpy(images).to(dev), H, W, 5)
    rgeo = ref["geo"]
    _same(mask, rgeo["view_mask"], "view_mask")
    _same(geo_map[..., :3], rgeo["view_position"], "geo.xyz")
    _same(geo_map[..., 3], rgeo["view_aoi_cos"], "geo.w")

    pre = wr.uv_precompute(wr_ctx, mesh, Hu, Wu)
    geo = wr.uv_render_geometry(wr_ctx, mesh, cam, H, W, pre, compute_depth_grad=True, depth_grad_dilation=5)
    attr = wr.uv_render_attr(torch.from_numpy(images), geo)
    _same(pre.uv_mask, ref["pre"]["uv_mask"], "uv_mask")
    _same(pre.uv_pos, ref["pre"]["uv_pos"], "uv_pos")
    _same(geo.view_mask, rgeo["view_mask"], "view_mask")
    for name in ["view_aoi_cos", "view_position", "view_normal", "view_depth"]:
        _same(getattr(geo, name), rgeo[name], name)
    _same(geo.view_depth_grad[:, 0], rgeo["view_depth_grad"], "view_depth_grad")
    for name in ["uv_pos_ndc", "uv_pos_proj", "uv_pos_error", "uv_aoi_cos", "uv_depth_grad"]:
        _same(getattr(geo, name), rgeo[name], name)
    _same(attr.uv_attr_proj, ref["attr"]["uv_attr_proj"], "uv_attr_proj")
    blend = wr.uv_blend(pre, geo, attr,
                        uv_validity_strategy=wr.SimpleUVValidityStrategy(aoi_cos_thresh=0.2, depth_grad_thresh=0.1),
                        uv_blend_weight_strategy=wr.ExponentialBlend(alpha=3.0), do_uv_padding=False)
    _same(blend.uv_valid_mask, ref["blend"]["uv_valid_mask"], "uv_valid_mask")
    _same(blend.uv_valid_mask_blend, ref["uv_proj_mask"], "uv_valid_mask_blend")
    np.testing.assert_allclose(_np(blend.uv_attr_blend), ref["uv_proj"], rtol=RTOL, atol=ATOL)
