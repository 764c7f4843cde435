"""GPU parity of the UV bake beyond the square orthographic rig: perspective, mixed orthographic / perspective and
40-view rigs, cameras with much of the scene behind them (clip w <= 0, NDC up to ~1e5), non-square views and atlases,
every tile path of k_view_prep (TMA and hand-loaded depth tile, partial tiles, the unrolled and the generic max-pool
window), both view-pass paths of the fused bake, and wr_grid_sample on its own.

The bar is the one of tests/test_gpu_bake_parity.py: view planes, materialised per-view tensors, validity and the
valid-any mask bit for bit against the oracle (NaN equal to NaN), blended colours within 1e-5 relative.  The oracle
is always fed the camera matrices the GPU used (get_camera on CUDA and on CPU may differ in the last bit)."""
import ctypes

import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import render_oracle, shim
from test_gpu_render_parity import make_mesh
from worldrenderer_b200 import _native, parallel, synth
from worldrenderer_b200.uv import (UVPrecomputeOutput, _unproject_args, fused_unproject, fused_view_maps,
                                   grid_sample_nhwc, uv_finalize)

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6
f32 = np.float32

RIGS = {"perspective": cases.bake_perspective_cameras, "mixed40": cases.mixed_40_view_cameras,
        "terrain": cases.low_terrain_cameras}
SCENES = {"perspective": "sphere", "mixed40": "sphere", "terrain": "terrain"}


def _np(t):
    return t.detach().cpu().numpy()


def _mesh(scene, device, Hu, Wu, seed=3):
    """icosphere(8) on a one-cell-per-triangle-pair atlas, or terrain_mesh(48, 24) on its planar chart; the existing
    texture is random, of the atlas shape."""
    if scene == "terrain":
        v, f = cases.terrain_mesh(48, 24)
        mesh = make_mesh(v, f, device)
        mesh.v_tex = torch.tensor(synth.terrain_uv(48, 24), dtype=torch.float32, device=device)
        mesh.t_tex_idx = mesh.t_pos_idx.clone()
    else:
        v, f = cases.icosphere_mesh(8)
        mesh = make_mesh(v, f, device, with_uv=True)
    rng = np.random.default_rng(seed)
    mesh.texture = torch.tensor(rng.uniform(0, 1, (Hu, Wu, 3)), dtype=torch.float32, device=device)
    return mesh


def _masks(images):
    """Smooth view masks in [0, 1]: about half of every view passes the 0.9 threshold."""
    return np.clip(2.0 * images[..., 1], 0, 1).astype(f32)


_ORACLE = {}


def _oracle_geometry(key, mesh, cam, H, W, Hu, Wu, dilation):
    """(oracle uv_precompute, oracle uv_render_geometry), kept for the module: the 40-view rig is used twice."""
    if key not in _ORACLE:
        v, f = _np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32)
        rpre = render_oracle.uv_precompute(v, f, _np(mesh.v_tex), _np(mesh.t_tex_idx).astype(np.int32), Hu, Wu)
        rgeo = render_oracle.uv_render_geometry(v, f, _np(mesh.v_nrm), f, _np(cam.mvp_mtx), _np(cam.w2c), H, W, rpre,
                                                True, dilation)
        _ORACLE[key] = (rpre, rgeo)
    return _ORACLE[key]


def _materialise(ctx, pre, mvp, H, W, geo_map, attr_map, view_masks=None):
    """wr_uv_unproject in its materialising form on given view maps (what uv_render_geometry issues after its own
    view pass): every per-view tensor of the reference, [Nv,Hu,Wu,...]."""
    uv_pos = pre.uv_pos.float().contiguous()
    uv_mask = pre.uv_mask.contiguous().view(torch.uint8)
    mvp = mvp.float().contiguous()
    Nv, Hu, Wu = mvp.shape[0], uv_pos.shape[0], uv_pos.shape[1]
    a = _unproject_args(uv_pos, uv_mask, mvp, H, W, geo_map, attr_map)
    dev = uv_pos.device
    out = {name: torch.full((Nv, Hu, Wu, c), float("nan"), dtype=torch.float32, device=dev)
           for name, c in (("uv_pos_ndc", 2), ("uv_pos_proj", 3), ("uv_pos_error", 1), ("uv_aoi_cos", 1),
                           ("uv_depth_grad", 1), ("uv_attr_proj", 3), ("uv_mask_proj", 1))}
    out["uv_valid"] = torch.full((Nv, Hu, Wu, 1), 7, dtype=torch.uint8, device=dev)
    for name, t in out.items():
        setattr(a, name, _native.ptr(t))
    vm = None
    if view_masks is not None:
        vm = view_masks.float().contiguous()
        a.view_masks = _native.ptr(vm)
    c = ctx.ctx
    c.check(_native.lib().wr_uv_unproject(c.handle, ctypes.byref(a), c.stream()), "wr_uv_unproject")
    return {k: _np(v[..., 0] if v.shape[-1] == 1 else v) for k, v in out.items()}


# (rig, view H x W, atlas Hu x Wu, depth-gradient dilation).  Views: 97 x 131 and 131 x 97 have W % 4 != 0 (the
# hand-loaded depth tile) and partial 32 x 32 tiles on both axes; 72 x 100 and 20 x 36 take the TMA tile with
# partial tiles (20 x 36: one partial tile per direction); 64 x 80 a partial tile on one axis.  Dilation 5 is the
# unrolled max-pool window (covered by the fused tests below), all others the generic loop; 37 is the largest the
# 48 KiB of shared memory of k_view_prep holds, on both tile paths.
STEPWISE = [
    ("perspective", (97, 131), (96, 160), 1),
    ("perspective", (131, 97), (160, 96), 3),
    ("perspective", (72, 100), (128, 128), 7),
    ("perspective", (20, 36), (96, 160), 37),
    ("mixed40", (64, 80), (128, 128), 9),
    ("terrain", (72, 100), (128, 128), 9),
    ("terrain", (97, 131), (160, 96), 37),
    ("terrain", (131, 97), (96, 160), 1),
    ("terrain", (20, 36), (160, 96), 3),
]


@pytest.mark.parametrize("rig,view,atlas,dilation", STEPWISE,
                         ids=[f"{r}-{v[0]}x{v[1]}-uv{a[0]}x{a[1]}-d{d}" for r, v, a, d in STEPWISE])
def test_stepwise_bake_matches_oracle(wr_ctx, rig, view, atlas, dilation):
    """uv_precompute -> uv_render_geometry(compute_depth_grad=True) -> uv_render_attr (with and without view masks)
    -> uv_blend, and the fused kernel on the same view maps, against the oracle."""
    (H, W), (Hu, Wu) = view, atlas
    dev = wr_ctx.device
    mesh = _mesh(SCENES[rig], dev, Hu, Wu)
    cam = RIGS[rig](H, W, device=dev)
    B = cam.mvp_mtx.shape[0]
    images = synth.view_images(B, H, W, seed=2)
    masks = _masks(images)
    pre = wr.uv_precompute(wr_ctx, mesh, Hu, Wu)
    geo = wr.uv_render_geometry(wr_ctx, mesh, cam, H, W, pre, compute_depth_grad=True, depth_grad_dilation=dilation)
    attr = wr.uv_render_attr(torch.from_numpy(images), geo)
    attr_m = wr.uv_render_attr(torch.from_numpy(images), geo, masks=torch.from_numpy(masks))
    rpre, rgeo = _oracle_geometry((rig, view, atlas, dilation), mesh, cam, H, W, Hu, Wu, dilation)

    np.testing.assert_array_equal(_np(pre.uv_mask), rpre["uv_mask"])
    np.testing.assert_array_equal(_np(pre.uv_pos), rpre["uv_pos"])
    np.testing.assert_array_equal(_np(geo.view_mask), rgeo["view_mask"])
    for name in ["view_aoi_cos", "view_position", "view_normal", "view_depth"]:
        np.testing.assert_array_equal(_np(getattr(geo, name)), rgeo[name], err_msg=name)
    np.testing.assert_array_equal(_np(geo.view_depth_grad[:, 0]), rgeo["view_depth_grad"])
    # Every texel, inside the charts or not: a texel outside them has the interpolated position 0 on both sides and
    # is projected and sampled like any other (only its validity is forced off).
    for name in ["uv_pos_ndc", "uv_pos_proj", "uv_pos_error", "uv_aoi_cos", "uv_depth_grad"]:
        np.testing.assert_array_equal(_np(getattr(geo, name)), rgeo[name], err_msg=name)
    rattr = render_oracle.uv_render_attr(images, rgeo)
    rattr_m = render_oracle.uv_render_attr(images, rgeo, masks)
    np.testing.assert_array_equal(_np(attr.uv_attr_proj), rattr["uv_attr_proj"])
    np.testing.assert_array_equal(_np(attr_m.uv_attr_proj), rattr_m["uv_attr_proj"])
    np.testing.assert_array_equal(_np(attr_m.uv_mask_proj), rattr_m["uv_mask_proj"])

    # at dilation 37 every pixel of a small view lies within reach of a silhouette: no texel passes a 0.1 threshold
    kw = dict(aoi_cos_thresh=0.2, depth_grad_thresh=0.1 if dilation <= 9 else None)
    strategy = wr.SimpleUVValidityStrategy(**kw)
    img = torch.from_numpy(images).to(dev)
    _, geo_map, attr_map = fused_view_maps(wr_ctx, mesh, cam, img, H, W, dilation)
    for a, ra, vm in ((attr, rattr, None), (attr_m, rattr_m, masks)):
        blend = wr.uv_blend(pre, geo, a, uv_validity_strategy=strategy,
                            uv_blend_weight_strategy=wr.ExponentialBlend(alpha=3.0), do_uv_padding=False)
        rbl = render_oracle.uv_blend(rpre, rgeo, ra, uv_attr_old=_np(mesh.texture), alpha=3.0, **kw)
        np.testing.assert_array_equal(_np(blend.uv_valid_mask), rbl["uv_valid_mask"])
        np.testing.assert_array_equal(_np(blend.uv_valid_mask_blend), rbl["uv_valid_mask_blend"])
        np.testing.assert_allclose(_np(blend.uv_attr_blend), rbl["uv_attr_blend"], rtol=RTOL, atol=ATOL)
        assert rbl["uv_valid_mask_blend"].sum() > 50
        fused, fused_any, _, _, _ = fused_unproject(
            wr_ctx, pre, cam, H, W, geo_map, attr_map, None if vm is None else torch.from_numpy(vm).to(dev),
            alpha=3.0, **kw)
        np.testing.assert_array_equal(_np(fused_any), rbl["uv_valid_mask_blend"])
        np.testing.assert_allclose(_np(fused), rbl["uv_attr_blend"], rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("view", [(97, 131), (20, 36)], ids=["hand-loaded-tile", "tma-tile"])
def test_view_prep_dilation_limits(wr_ctx, view):
    """37 is the largest dilation whose tiles fit in 48 KiB of shared memory (46.8 KB hand-loaded, 47.4 KB with the
    TMA box); 39 needs 49.3 KB and is refused, as is an even window (max_pool2d would change the map size)."""
    H, W = view
    dev = wr_ctx.device
    mesh = _mesh("sphere", dev, 64, 64)
    cam = cases.bake_perspective_cameras(H, W, device=dev)
    img = torch.from_numpy(synth.view_images(4, H, W)).to(dev)
    pre = wr.uv_precompute(wr_ctx, mesh, 64, 64)
    fused_view_maps(wr_ctx, mesh, cam, img, H, W, 37)
    for d in (39, 36, 2):
        with pytest.raises(NotImplementedError):
            fused_view_maps(wr_ctx, mesh, cam, img, H, W, d)
        with pytest.raises(NotImplementedError):
            wr.uv_render_geometry(wr_ctx, mesh, cam, H, W, pre, compute_depth_grad=True, depth_grad_dilation=d)


def test_camera_projection_default_call(wr_ctx):
    """The reference's default call: no camera, CameraProjection builds a perspective rig with aspect W / H from
    elevation / azimuth / distance / fovy lists.  97 x 131 views, view masks, per-view weights that make the blend
    exponents non-integer (powf), in all three kernel forms -- return_dict (per-view aoi / depth gradient), the plain
    return (blend only) and the step-by-step API (every per-view tensor) -- and sharded_bake in one process."""
    H, W = 97, 131
    dev = wr_ctx.device
    mesh = _mesh("sphere", dev, 128, 128)
    el, az, dist, fovy = [10.0, -20.0, 35.0, 60.0], [0.0, 75.0, 160.0, 250.0], [1.8] * 4, [40.0] * 4
    images = synth.view_images(4, H, W, seed=4)
    masks = _masks(images)
    vw = torch.tensor([1.0, 0.7, 1.3, 2.0])
    proj = wr.CameraProjection(None, None, str(dev), "cuda")
    call = dict(elevation_deg=el, azimuth_deg=az, distance=dist, fovy_deg=fovy, masks=torch.from_numpy(masks),
                uv_size=128, poisson_blending=False, uv_padding=False, iou_rejection_threshold=None,
                aoi_cos_valid_threshold=0.2, depth_grad_dilation=5, depth_grad_threshold=0.1, uv_exp_blend_alpha=3.0,
                uv_exp_blend_view_weight=vw)
    out = proj(torch.from_numpy(images), mesh, return_dict=True, **call)
    plain = proj(torch.from_numpy(images), mesh, **call)
    cam = wr.get_camera(el, dist, fovy, az, aspect_wh=W / H, device=dev)   # the rig the call builds
    assert cam.proj_mtx[0, 3, 3] == 0   # perspective
    ref = render_oracle.camera_projection(
        images, _np(mesh.v_pos), _np(mesh.t_pos_idx).astype(np.int32), _np(mesh.v_nrm),
        _np(mesh.t_pos_idx).astype(np.int32), _np(mesh.v_tex), _np(mesh.t_tex_idx).astype(np.int32),
        _np(mesh.texture), _np(cam.mvp_mtx), _np(cam.w2c), 128, masks=masks, iou_rejection_threshold=None,
        aoi_cos_valid_threshold=0.2, depth_grad_dilation=5, depth_grad_threshold=0.1, uv_exp_blend_alpha=3.0,
        uv_exp_blend_view_weight=vw.numpy())
    assert ref["uv_proj_mask"].sum() > 1000
    np.testing.assert_array_equal(_np(out.uv_proj_mask), ref["uv_proj_mask"])
    np.testing.assert_allclose(_np(out.uv_proj), ref["uv_proj"], rtol=RTOL, atol=ATOL)
    np.testing.assert_array_equal(_np(out.uv_aoi_cos), ref["uv_aoi_cos"])
    np.testing.assert_array_equal(_np(out.uv_depth_grad), ref["uv_depth_grad"])
    assert torch.equal(plain, out.uv_proj)

    pre = wr.uv_precompute(wr_ctx, mesh, 128, 128)
    geo = wr.uv_render_geometry(wr_ctx, mesh, cam, H, W, pre, compute_depth_grad=True, depth_grad_dilation=5)
    attr = wr.uv_render_attr(torch.from_numpy(images), geo, masks=torch.from_numpy(masks))
    blend = wr.uv_blend(pre, geo, attr,
                        uv_validity_strategy=wr.SimpleUVValidityStrategy(aoi_cos_thresh=0.2, depth_grad_thresh=0.1),
                        uv_blend_weight_strategy=wr.ExponentialBlend(alpha=3.0, view_weight=vw.to(dev)),
                        do_uv_padding=False)
    for name in ["uv_pos_ndc", "uv_pos_proj", "uv_pos_error", "uv_aoi_cos", "uv_depth_grad"]:
        np.testing.assert_array_equal(_np(getattr(geo, name)), ref["geo"][name], err_msg=name)
    np.testing.assert_array_equal(_np(attr.uv_attr_proj), ref["attr"]["uv_attr_proj"])
    np.testing.assert_array_equal(_np(attr.uv_mask_proj), ref["attr"]["uv_mask_proj"])
    np.testing.assert_array_equal(_np(blend.uv_valid_mask), ref["blend"]["uv_valid_mask"])
    np.testing.assert_array_equal(_np(blend.uv_valid_mask_blend), ref["uv_proj_mask"])
    np.testing.assert_allclose(_np(blend.uv_attr_blend), ref["uv_proj"], rtol=RTOL, atol=ATOL)

    atlas, any_ = parallel.sharded_bake(wr_ctx, mesh, cam, torch.from_numpy(images).to(dev), 128,
                                        view_masks_local=torch.from_numpy(masks).to(dev), aoi_cos_valid_threshold=0.2,
                                        depth_grad_dilation=5, depth_grad_threshold=0.1, uv_exp_blend_alpha=3.0,
                                        uv_exp_blend_view_weight_local=vw)
    assert torch.equal(any_, out.uv_proj_mask)
    torch.testing.assert_close(atlas, out.uv_proj, rtol=RTOL, atol=ATOL)


@pytest.mark.parametrize("freq,view,queue", [(8, (97, 131), True), (50, (64, 80), False)],
                         ids=["sparse-queue-packed", "dense-multiview-unpacked"])
def test_fused_view_maps_match_oracle(wr_ctx, freq, view, queue):
    """The view pass of the fused bake (shading kernel writing the packed (position, aoi_cos) map, then wr_view_prep
    adding the depth gradient to (rgb, depth_grad)) against the oracle's view planes, bit for bit.  A sparse mesh at
    large views takes the queue raster path with packed vertex records; a dense one at small views the multi-view
    raster fast path without them."""
    H, W = view
    dev = wr_ctx.device
    mesh = make_mesh(*cases.icosphere_mesh(freq), dev)
    cam = cases.concat_cameras(cases.bake_perspective_cameras(H, W, device=dev), cases.canonical_cameras(device=dev)[0:2])
    B = cam.mvp_mtx.shape[0]
    F, V, Vn = mesh.t_pos_idx.shape[0], mesh.v_pos.shape[0], mesh.v_nrm.shape[0]
    assert (4 * F > H * W) == (not queue)                   # raster.cu: multi-view fast path
    assert (B * H * W >= 32 * (V + Vn)) == queue            # render.cu: 16-byte vertex records
    images = synth.view_images(B, H, W, seed=6)
    mask, geo_map, attr_map = fused_view_maps(wr_ctx, mesh, cam, torch.from_numpy(images).to(dev), H, W, 5)
    f = _np(mesh.t_pos_idx).astype(np.int32)
    stub = {"uv_pos": np.zeros((1, 1, 3), f32)}   # view planes only
    rgeo = render_oracle.uv_render_geometry(_np(mesh.v_pos), f, _np(mesh.v_nrm), f, _np(cam.mvp_mtx), _np(cam.w2c),
                                            H, W, stub, True, 5)
    assert rgeo["view_mask"].sum() > 0.1 * B * H * W
    np.testing.assert_array_equal(_np(mask), rgeo["view_mask"])
    geo_map, attr_map = _np(geo_map), _np(attr_map)
    np.testing.assert_array_equal(geo_map[..., :3], rgeo["view_position"])
    np.testing.assert_array_equal(geo_map[..., 3], rgeo["view_aoi_cos"])
    np.testing.assert_array_equal(attr_map[..., :3], images)
    np.testing.assert_array_equal(attr_map[..., 3], rgeo["view_depth_grad"])


def test_forty_view_mixed_rig(wr_ctx):
    """More views than the 32-bit orthographic bitmask: the fused kernel against the oracle, and the same views
    accumulated in two shards split at view 32 and finalised (the orthographic views 37-39 move to positions 5-7 of
    the second shard, inside its bitmask)."""
    H, W, Hu, Wu, d = 64, 80, 128, 128, 9
    dev = wr_ctx.device
    mesh = _mesh("sphere", dev, Hu, Wu)
    cam = cases.mixed_40_view_cameras(H, W, device=dev)
    ortho = (cam.mvp_mtx[:, 3] == torch.tensor([0.0, 0.0, 0.0, 1.0], device=dev)).all(-1).cpu()
    assert ortho.nonzero().flatten().tolist() == [1, 2, 3, 37, 38, 39]
    images = synth.view_images(40, H, W, seed=2)
    img = torch.from_numpy(images).to(dev)
    pre = wr.uv_precompute(wr_ctx, mesh, Hu, Wu)
    kw = dict(aoi_cos_thresh=0.2, depth_grad_thresh=0.1, alpha=3.0)
    _, geo_map, attr_map = fused_view_maps(wr_ctx, mesh, cam, img, H, W, d)
    full, full_any, _, udg, uaoi = fused_unproject(wr_ctx, pre, cam, H, W, geo_map, attr_map, want_per_view=True, **kw)
    rpre, rgeo = _oracle_geometry(("mixed40", (H, W), (Hu, Wu), d), mesh, cam, H, W, Hu, Wu, d)
    rbl = render_oracle.uv_blend(rpre, rgeo, render_oracle.uv_render_attr(images, rgeo), uv_attr_old=_np(mesh.texture),
                                 **kw)
    per_view = rbl["uv_valid_mask"].sum((1, 2))
    assert (per_view[[1, 2, 3, 32, 33, 34, 35, 36, 37, 38, 39]] > 0).all()   # the views that matter here take part
    np.testing.assert_array_equal(_np(uaoi), rgeo["uv_aoi_cos"])
    np.testing.assert_array_equal(_np(udg), rgeo["uv_depth_grad"])
    np.testing.assert_array_equal(_np(full_any), rbl["uv_valid_mask_blend"])
    np.testing.assert_allclose(_np(full), rbl["uv_attr_blend"], rtol=RTOL, atol=ATOL)
    accum = None
    for sl in [slice(0, 32), slice(32, 40)]:
        _, g, a = fused_view_maps(wr_ctx, mesh, cam[sl], img[sl], H, W, d)
        _, _, accum, _, _ = fused_unproject(wr_ctx, pre, cam[sl], H, W, g, a, accumulate_only=True, accum=accum, **kw)
    out, any_ = uv_finalize(wr_ctx, accum, pre.uv_attr)
    assert torch.equal(any_, full_any)
    torch.testing.assert_close(out, full, rtol=1e-5, atol=1e-6)


def test_view_with_zero_w_row_drops_out(wr_ctx):
    """A view whose mvp has a zero w row projects every texel to clip.xy / 0 (+-inf, or NaN at clip x = 0): nothing
    is sampled there, so the view adds nothing -- the bake with it appended is the bake without it, bit for bit."""
    H, W, Hu, Wu = 72, 100, 128, 128
    dev = wr_ctx.device
    mesh = _mesh("sphere", dev, Hu, Wu)
    cam = cases.bake_perspective_cameras(H, W, device=dev)
    images = synth.view_images(4, H, W, seed=7)
    img = torch.from_numpy(images).to(dev)
    masks = torch.from_numpy(_masks(images)).to(dev)
    pre = wr.uv_precompute(wr_ctx, mesh, Hu, Wu)
    _, geo_map, attr_map = fused_view_maps(wr_ctx, mesh, cam, img, H, W, 5)
    flat = cam[1]
    flat.mvp_mtx = flat.mvp_mtx.clone()
    flat.mvp_mtx[:, 3] = 0.0
    cam5 = cases.concat_cameras(cam, flat)
    geo5, attr5, masks5 = (torch.cat([t, t[1:2]]) for t in (geo_map, attr_map, masks))
    kw = dict(aoi_cos_thresh=0.2, depth_grad_thresh=0.1, alpha=3.0)
    want, want_any, _, _, _ = fused_unproject(wr_ctx, pre, cam, H, W, geo_map, attr_map, masks, **kw)
    got, got_any, _, _, _ = fused_unproject(wr_ctx, pre, cam5, H, W, geo5, attr5, masks5, **kw)
    assert bool(want_any.any())
    assert torch.equal(got_any, want_any) and torch.equal(got, want)

    m = _materialise(wr_ctx, pre, cam5.mvp_mtx, H, W, geo5, attr5, masks5)
    up, M = _np(pre.uv_pos), _np(flat.mvp_mtx[0])
    cx = ((M[0, 0] * up[..., 0] + M[0, 1] * up[..., 1]) + M[0, 2] * up[..., 2]) + M[0, 3]
    cy = ((M[1, 0] * up[..., 0] + M[1, 1] * up[..., 1]) + M[1, 2] * up[..., 2]) + M[1, 3]
    with np.errstate(all="ignore"):
        ndc = np.stack([cx / f32(0), cy / f32(0)], -1)
    assert not np.isfinite(ndc).any()
    np.testing.assert_array_equal(m["uv_pos_ndc"][4], ndc)
    for name in ["uv_pos_proj", "uv_aoi_cos", "uv_depth_grad", "uv_attr_proj", "uv_mask_proj", "uv_valid"]:
        assert not m[name][4].any(), name
    # view 1 itself is untouched by its degenerate copy
    assert m["uv_valid"][1].any()


def test_non_finite_texel_positions_are_invalid_everywhere(wr_ctx):
    """Texels whose interpolated position is NaN or +-inf, under orthographic and perspective views.  Their NDC is
    clip.xy / clip.w as the oracle computes it -- NaN at an orthographic view, whose w = 0 * inf + 1 is NaN, not the
    +-inf of clip x alone -- and they are valid in no view; every other texel bakes as before."""
    H, W, Hu, Wu = 72, 100, 128, 128
    dev = wr_ctx.device
    mesh = _mesh("sphere", dev, Hu, Wu)
    cam = cases.concat_cameras(cases.canonical_cameras(device=dev), cases.bake_perspective_cameras(H, W, device=dev))
    B = cam.mvp_mtx.shape[0]
    pre = wr.uv_precompute(wr_ctx, mesh, Hu, Wu)
    img = torch.from_numpy(synth.view_images(B, H, W, seed=8)).to(dev)
    _, geo_map, attr_map = fused_view_maps(wr_ctx, mesh, cam, img, H, W, 3)
    kw = dict(aoi_cos_thresh=-1.0, alpha=3.0)   # every sampled aoi passes: only the position test can reject
    want, want_any, _, _, _ = fused_unproject(wr_ctx, pre, cam, H, W, geo_map, attr_map, **kw)
    inf, nan = float("inf"), float("nan")
    bad = [(inf, 0.1, 0.2), (-inf, 0.0, 0.0), (nan, 0.1, 0.1), (0.1, nan, 0.0), (0.2, 0.1, inf), (0.0, -inf, 0.0),
           (inf, -inf, 0.0), (nan, nan, nan)]
    seen = np.flatnonzero(_np(want_any))   # texels some view bakes: the bad position is what rejects them
    p = seen[np.linspace(0, len(seen) - 1, len(bad)).astype(int)]
    pick = torch.from_numpy(p).to(dev)
    uv_pos = pre.uv_pos.clone()
    uv_pos.view(-1, 3)[pick] = torch.tensor(bad, dtype=torch.float32, device=dev)
    bad_pre = UVPrecomputeOutput(height=Hu, width=Wu, uv_attr=pre.uv_attr, uv_mask=pre.uv_mask, uv_pos=uv_pos)

    geo = wr.uv_render_geometry(wr_ctx, mesh, cam, H, W, bad_pre, compute_depth_grad=True, depth_grad_dilation=3)
    clip = shim.clip_positions(_np(uv_pos).reshape(-1, 3), _np(cam.mvp_mtx)).reshape(B, Hu, Wu, 4)
    with np.errstate(all="ignore"):
        ndc = (clip[..., :2] / clip[..., 3:4]).astype(f32)
    np.testing.assert_array_equal(_np(geo.uv_pos_ndc), ndc)
    assert np.isnan(ndc[:6].reshape(6, -1, 2)[:, p]).all()
    for name in ["uv_pos_proj", "uv_aoi_cos", "uv_depth_grad"]:
        assert not _np(getattr(geo, name)).reshape(B, Hu * Wu, -1)[:, p].any(), name

    m = _materialise(wr_ctx, bad_pre, cam.mvp_mtx, H, W, geo_map, attr_map)
    assert not m["uv_valid"].reshape(B, -1)[:, p].any()
    assert m["uv_valid"].any()
    got, got_any, _, _, _ = fused_unproject(wr_ctx, bad_pre, cam, H, W, geo_map, attr_map, **kw)
    keep = torch.ones(Hu * Wu, dtype=torch.bool, device=dev)
    keep[pick] = False
    keep = keep.view(Hu, Wu)
    assert not bool(got_any.view(-1)[pick].any())
    assert torch.equal(got_any[keep], want_any[keep]) and torch.equal(got[keep], want[keep])
    assert torch.equal(got.view(-1, 3)[pick], pre.uv_attr.view(-1, 3)[pick])   # the existing texture stays


def _coords(rng, shape, H, W):
    """Sample coordinates: uniform in [-1.3, 1.3], and at the front a grid of edge cases on each axis -- the
    borders +-1 and one pixel in / out of them, pixel centres, -0.0, far out of range and non-finite values."""
    def specials(n):
        c = [-1.0, 1.0, -1 - 1 / n, -1 + 1 / n, 1 - 1 / n, 1 + 1 / n, (2 * (n // 2) + 1) / n - 1, 0.3,
             -0.0, 0.0, 1e8, -1e8, 1e30, -1e30, np.inf, -np.inf, np.nan]
        return np.array(c, f32)
    sx, sy = specials(W), specials(H)
    grid = np.stack(np.meshgrid(sx, sy, indexing="ij"), -1).reshape(-1, 2)
    out = rng.uniform(-1.3, 1.3, shape + (2,)).astype(f32)
    flat = out.reshape(shape[0], -1, 2)
    for b in range(shape[0]):
        flat[b, :len(grid)] = grid[rng.permutation(len(grid))]
    return out


@pytest.mark.parametrize("C", [1, 2, 3, 4, 7])
@pytest.mark.parametrize("H,W", [(1, 17), (33, 20), (64, 96)])
def test_grid_sample_nhwc_matches_oracle(wr_ctx, H, W, C):
    """wr_grid_sample on its own (in the bake it only runs with C = 3 and C = 1 on square views): channel counts,
    non-square maps, 23 x 31 samples per map (not a multiple of the 256-thread block), edge and non-finite
    coordinates.  A non-finite coordinate samples nothing: 0 (torch.nn.functional.grid_sample: NaN on CPU, 0 on
    CUDA)."""
    rng = np.random.default_rng(100 * H + 10 * W + C)
    B, Hs, Ws = 3, 23, 31
    maps = rng.standard_normal((B, H, W, C)).astype(f32)
    ndc = _coords(rng, (B, Hs, Ws), H, W)
    dev = wr_ctx.device
    got = _np(grid_sample_nhwc(torch.from_numpy(maps).to(dev), torch.from_numpy(ndc).to(dev)))
    want = np.stack([render_oracle.grid_sample(maps[b], ndc[b]) for b in range(B)])
    assert got.shape == (B, Hs, Ws, C)
    np.testing.assert_array_equal(got, want)
    assert not np.isfinite(ndc).all() and np.isfinite(got).all()
    assert (np.abs(got) > 0).mean() > 0.4   # most samples land on the map


def test_grid_sample_nhwc_empty_batch_and_devices(wr_ctx):
    dev = wr_ctx.device
    out = grid_sample_nhwc(torch.zeros(0, 5, 6, 2, device=dev), torch.zeros(0, 3, 4, 2, device=dev))
    assert out.shape == (0, 3, 4, 2) and out.device.type == "cuda"
    with pytest.raises(RuntimeError):
        grid_sample_nhwc(torch.zeros(1, 5, 6, 2, device=dev), torch.zeros(1, 3, 4, 2))
    with pytest.raises(RuntimeError):
        grid_sample_nhwc(torch.zeros(1, 5, 6, 2), torch.zeros(1, 3, 4, 2))
