"""GPU parity, bake level: CameraProjection / uv_* against the oracle's restatement of uv.py and
projection.py.  Measured (tools/bake_exactness_probe.py, B200): every intermediate of the bake -- the per-view
maps, uv_pos_ndc, the projected positions / errors / cosines / depth gradients / colours -- is identical to
the oracle BIT FOR BIT, hence so are the validity booleans and uv_proj_mask; only the blended colours differ, by
the rounding of the weight power and of the view sum (max 4.2e-7 relative at config C).  The tests therefore
assert exact equality for the intermediates and the masks, and north_star's 1e-5 relative for the colours."""
import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from oracle import render_oracle
from test_gpu_render_parity import make_mesh
from worldrenderer_b200 import synth

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-5, 1e-6


def _setup(device, freq=8, views=(96, 96), seed=1, old_texture=True, uv_size=128):
    v, f = cases.icosphere_mesh(freq)
    mesh = make_mesh(v, f, device, with_uv=True, tex_size=uv_size, seed=seed)
    if not old_texture:
        mesh.texture = torch.zeros_like(mesh.texture)
    cam = cases.canonical_cameras(device=device)
    images = synth.view_images(6, views[0], views[1], seed=seed)
    return mesh, cam, images


def _oracle_bake(mesh, cam, images, uv_size, masks=None, **kw):
    return render_oracle.camera_projection(
        images, mesh.v_pos.cpu().numpy(), mesh.t_pos_idx.cpu().numpy().astype(np.int32), mesh.v_nrm.cpu().numpy(),
        mesh.t_pos_idx.cpu().numpy().astype(np.int32), mesh.v_tex.cpu().numpy(),
        mesh.t_tex_idx.cpu().numpy().astype(np.int32), mesh.texture.cpu().numpy(), cam.mvp_mtx.cpu().numpy(),
        cam.w2c.cpu().numpy(), uv_size, masks=masks, **kw)


def test_uv_precompute(wr_ctx):
    mesh, cam, images = _setup(wr_ctx.device)
    pre = wr.uv_precompute(wr_ctx, mesh, 128, 128)
    ref = render_oracle.uv_precompute(mesh.v_pos.cpu().numpy(), mesh.t_pos_idx.cpu().numpy(), mesh.v_tex.cpu().numpy(),
                                      mesh.t_tex_idx.cpu().numpy(), 128, 128)
    np.testing.assert_array_equal(pre.uv_mask.cpu().numpy(), ref["uv_mask"])
    np.testing.assert_array_equal(pre.uv_pos.cpu().numpy(), ref["uv_pos"])


@pytest.mark.parametrize("aoi_thr,dg_thr,alpha,use_vw", [(0.2, 0.1, 3.0, True), (-1.0, None, 3.0, True), (0.3, 0.1, 6.0, False)])
def test_camera_projection_fused(wr_ctx, aoi_thr, dg_thr, alpha, use_vw):
    mesh, cam, images = _setup(wr_ctx.device)
    proj = wr.CameraProjection(pb_backend=None, bg_remover=None, device=str(wr_ctx.device), context_type="cuda")
    vw = torch.tensor([1.0, 0.5, 1.0, 2.0, 1.0, 1.0]) if use_vw else None
    out = proj(torch.from_numpy(images), mesh, cam, uv_size=128, poisson_blending=False, uv_padding=False,
               depth_grad_dilation=5, uv_exp_blend_alpha=alpha, uv_exp_blend_view_weight=vw,
               aoi_cos_valid_threshold=aoi_thr, depth_grad_threshold=dg_thr, iou_rejection_threshold=None,
               return_dict=True)
    ref = _oracle_bake(mesh, cam, images, 128, aoi_cos_valid_threshold=aoi_thr, depth_grad_threshold=dg_thr,
                       uv_exp_blend_alpha=alpha, uv_exp_blend_view_weight=None if vw is None else vw.numpy(),
                       depth_grad_dilation=5)
    np.testing.assert_array_equal(out.uv_aoi_cos.cpu().numpy(), ref["uv_aoi_cos"])
    np.testing.assert_array_equal(out.uv_depth_grad.cpu().numpy(), ref["uv_depth_grad"])
    got_mask = out.uv_proj_mask.cpu().numpy()
    np.testing.assert_array_equal(got_mask, ref["uv_proj_mask"])
    got = out.uv_proj.cpu().numpy()
    np.testing.assert_allclose(got, ref["uv_proj"], rtol=RTOL, atol=ATOL)
    assert got_mask.sum() > 0.3 * ref["pre"]["uv_mask"].sum()
    # plain return forms (projection.py:190-204)
    t = proj(torch.from_numpy(images), mesh, cam, uv_size=128, poisson_blending=False, uv_padding=False,
             uv_exp_blend_alpha=alpha, uv_exp_blend_view_weight=vw, aoi_cos_valid_threshold=aoi_thr,
             depth_grad_threshold=dg_thr, iou_rejection_threshold=None)
    assert torch.equal(t, out.uv_proj)
    t2, m2 = proj(torch.from_numpy(images), mesh, cam, uv_size=128, poisson_blending=False, uv_padding=False,
                  uv_exp_blend_alpha=alpha, uv_exp_blend_view_weight=vw, aoi_cos_valid_threshold=aoi_thr,
                  depth_grad_threshold=dg_thr, iou_rejection_threshold=None, return_uv_projection_mask=True)
    assert torch.equal(m2, out.uv_proj_mask)


def test_masks_and_iou_rejection(wr_ctx):
    mesh, cam, images = _setup(wr_ctx.device)
    proj = wr.CameraProjection(None, None, str(wr_ctx.device), "cuda")
    rendered = wr.render(wr_ctx, mesh, cam, 96, 96, render_attr=False).mask.float()
    out = proj(torch.from_numpy(images), mesh, cam, masks=rendered, uv_size=128, poisson_blending=False,
               uv_padding=False, return_dict=True)
    ref = _oracle_bake(mesh, cam, images, 128, masks=rendered.cpu().numpy())
    assert out is not None and ref is not None
    np.testing.assert_array_equal(out.uv_proj_mask.cpu().numpy(), ref["uv_proj_mask"])
    np.testing.assert_allclose(out.uv_proj.cpu().numpy(), ref["uv_proj"], rtol=RTOL, atol=ATOL)
    bad = torch.zeros_like(rendered)
    bad[:, :10, :10] = 1
    assert proj(torch.from_numpy(images), mesh, cam, masks=bad, uv_size=128, poisson_blending=False,
                uv_padding=False) is None


def test_stepwise_api_matches_oracle(wr_ctx):
    mesh, cam, images = _setup(wr_ctx.device)
    pre = wr.uv_precompute(wr_ctx, mesh, 128, 128)
    geo = wr.uv_render_geometry(wr_ctx, mesh, cam, 96, 96, pre, compute_depth_grad=True, depth_grad_dilation=3)
    attr = wr.uv_render_attr(torch.from_numpy(images), geo)
    v, f = mesh.v_pos.cpu().numpy(), mesh.t_pos_idx.cpu().numpy().astype(np.int32)
    rpre = render_oracle.uv_precompute(v, f, mesh.v_tex.cpu().numpy(), mesh.t_tex_idx.cpu().numpy(), 128, 128)
    rgeo = render_oracle.uv_render_geometry(v, f, mesh.v_nrm.cpu().numpy(), f, cam.mvp_mtx.cpu().numpy(),
                                            cam.w2c.cpu().numpy(), 96, 96, rpre, True, 3)
    rattr = render_oracle.uv_render_attr(images, rgeo)
    np.testing.assert_array_equal(geo.view_mask.cpu().numpy(), rgeo["view_mask"])
    inside = rpre["uv_mask"]
    for name in ["uv_pos_proj", "uv_pos_error", "uv_aoi_cos", "uv_pos_ndc", "uv_depth_grad"]:
        np.testing.assert_array_equal(getattr(geo, name).cpu().numpy()[:, inside], rgeo[name][:, inside], err_msg=name)
    for name in ["view_aoi_cos", "view_position", "view_normal", "view_depth"]:
        np.testing.assert_array_equal(getattr(geo, name).cpu().numpy(), rgeo[name], err_msg=name)
    np.testing.assert_array_equal(geo.view_depth_grad[:, 0].cpu().numpy(), rgeo["view_depth_grad"])
    np.testing.assert_array_equal(attr.uv_attr_proj.cpu().numpy()[:, inside], rattr["uv_attr_proj"][:, inside])
    blend = wr.uv_blend(pre, geo, attr, uv_validity_strategy=wr.SimpleUVValidityStrategy(aoi_cos_thresh=0.2, depth_grad_thresh=0.1),
                        uv_blend_weight_strategy=wr.ExponentialBlend(alpha=3.0), do_uv_padding=False)
    # the step-by-step blend and the fused kernel agree with each other
    proj = wr.CameraProjection(None, None, str(wr_ctx.device), "cuda")
    fused = proj(torch.from_numpy(images), mesh, cam, uv_size=128, poisson_blending=False, uv_padding=False,
                 depth_grad_dilation=3, uv_exp_blend_alpha=3.0, aoi_cos_valid_threshold=0.2, depth_grad_threshold=0.1,
                 iou_rejection_threshold=None, return_dict=True)
    assert torch.equal(fused.uv_proj_mask, blend.uv_valid_mask_blend)
    torch.testing.assert_close(fused.uv_proj, blend.uv_attr_blend, rtol=RTOL, atol=ATOL)


def test_accumulate_then_finalize_equals_fused(wr_ctx):
    """The multi-GPU decomposition on one device: two view shards accumulated, then finalised."""
    from worldrenderer_b200.uv import fused_unproject, fused_view_maps, uv_finalize
    mesh, cam, images = _setup(wr_ctx.device)
    pre = wr.uv_precompute(wr_ctx, mesh, 128, 128)
    img = torch.from_numpy(images).to(wr_ctx.device)
    kw = dict(aoi_cos_thresh=0.2, depth_grad_thresh=0.1, alpha=3.0)
    _, geo, att = fused_view_maps(wr_ctx, mesh, cam, img, 96, 96, 5)
    full, full_any, _, _, _ = fused_unproject(wr_ctx, pre, cam, 96, 96, geo, att, **kw)
    accum = None
    for sl in [slice(0, 2), slice(2, 6)]:
        _, g, a = fused_view_maps(wr_ctx, mesh, cam[sl], img[sl], 96, 96, 5)
        _, _, accum, _, _ = fused_unproject(wr_ctx, pre, cam[sl], 96, 96, g, a, accumulate_only=True, accum=accum, **kw)
    out, any_ = uv_finalize(wr_ctx, accum, pre.uv_attr)
    assert torch.equal(any_, full_any)
    torch.testing.assert_close(out, full, rtol=1e-5, atol=1e-6)


def test_fused_unprojection_with_first_view_dominate_equals_stepwise(wr_ctx):
    """wr_unproject_args.first_view_dominate (SimpleUVValidityStrategy(first_view_dominate=True), uv.py:294-296): a
    texel the first view sees is taken from that view alone.  The fused kernel against the step-by-step API, whose
    strategy objects are pinned to the reference on CPU (tests/test_host_api.py)."""
    from worldrenderer_b200.uv import fused_unproject, fused_view_maps
    mesh, cam, images = _setup(wr_ctx.device)
    pre = wr.uv_precompute(wr_ctx, mesh, 128, 128)
    img = torch.from_numpy(images).to(wr_ctx.device)
    # no depth-gradient threshold: at 96^2 it confines every view of the six-view rig to a 45-degree cap and the
    # views would not overlap at all
    kw = dict(aoi_cos_thresh=0.2, depth_grad_thresh=None, alpha=3.0)
    _, geo_m, att_m = fused_view_maps(wr_ctx, mesh, cam, img, 96, 96, 5)
    fused, fused_any, _, _, _ = fused_unproject(wr_ctx, pre, cam, 96, 96, geo_m, att_m, first_view_dominate=True, **kw)
    plain, plain_any, _, _, _ = fused_unproject(wr_ctx, pre, cam, 96, 96, geo_m, att_m, **kw)
    geo = wr.uv_render_geometry(wr_ctx, mesh, cam, 96, 96, pre, compute_depth_grad=True, depth_grad_dilation=5)
    attr = wr.uv_render_attr(torch.from_numpy(images), geo)
    strategy = wr.SimpleUVValidityStrategy(aoi_cos_thresh=0.2, first_view_dominate=True)
    blend = wr.uv_blend(pre, geo, attr, uv_validity_strategy=strategy,
                        uv_blend_weight_strategy=wr.ExponentialBlend(alpha=3.0), do_uv_padding=False)
    assert torch.equal(fused_any, blend.uv_valid_mask_blend)
    torch.testing.assert_close(fused, blend.uv_attr_blend, rtol=RTOL, atol=ATOL)
    # the option is live: same coverage (a texel of view 0 is still covered), other colours where views overlap
    assert torch.equal(fused_any, plain_any)
    first = blend.uv_valid_mask[0]
    assert bool(first.any()) and not bool((blend.uv_valid_mask[1:] & first[None]).any())
    assert float((fused - plain).abs().max()) > 1e-3


def test_unprojection_in_texel_ranges_equals_one_pass(wr_ctx):
    """wr_uv_unproject over texel ranges (what the chunked multi-GPU bake issues) fills the same accumulators, on a
    square and on non-square atlases: range ends inside a row, a single texel, and a range ending at a row end."""
    from worldrenderer_b200.uv import fused_unproject, fused_view_maps
    mesh, cam, images = _setup(wr_ctx.device)
    img = torch.from_numpy(images).to(wr_ctx.device)
    kw = dict(aoi_cos_thresh=0.2, depth_grad_thresh=0.1, alpha=3.0, accumulate_only=True)
    _, geo, att = fused_view_maps(wr_ctx, mesh, cam, img, 96, 96, 5)
    for Hu, Wu in [(128, 128), (96, 160), (160, 96)]:
        pre = wr.uv_precompute(wr_ctx, mesh, Hu, Wu)
        _, _, full, _, _ = fused_unproject(wr_ctx, pre, cam, 96, 96, geo, att, **kw)
        assert full.shape == (Hu, Wu, 5) and float(full[..., 4].sum()) > 1000
        row_end = (5001 // Wu + 1) * Wu
        cuts = [0, 5000, 5001, row_end, row_end + 1, Hu * Wu]
        assert 5000 % Wu and 5001 % Wu
        part = torch.full_like(full, float("nan"))
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            fused_unproject(wr_ctx, pre, cam, 96, 96, geo, att, accum=part, add_to_accum=False, tex_range=(lo, hi),
                            **kw)
        assert torch.equal(part, full), (Hu, Wu)
    with pytest.raises(RuntimeError):
        fused_unproject(wr_ctx, pre, cam, 96, 96, geo, att, accum=part, add_to_accum=False, tex_range=(10, 5), **kw)


def test_view_weights_are_re_read_when_the_tensor_changes(wr_ctx):
    """The per-view blend weights arrive as a host tensor with every call; the device copy of an unchanged tensor is
    reused, an in-place update (version counter) or another tensor is uploaded again."""
    mesh, cam, images = _setup(wr_ctx.device)
    proj = wr.CameraProjection(None, None, str(wr_ctx.device), "cuda")
    img = torch.from_numpy(images).to(wr_ctx.device)
    kw = dict(uv_size=128, poisson_blending=False, uv_padding=False, uv_exp_blend_alpha=3.0, aoi_cos_valid_threshold=0.2,
              iou_rejection_threshold=None)
    vw = torch.tensor([1.0, 0.5, 1.0, 2.0, 1.0, 1.0])
    first = proj(img, mesh, cam, uv_exp_blend_view_weight=vw, **kw).clone()
    again = proj(img, mesh, cam, uv_exp_blend_view_weight=vw, **kw)
    assert torch.equal(first, again)
    vw.mul_(torch.tensor([3.0, 1.0, 0.25, 1.0, 2.0, 1.0]))   # in place: same object, new version
    changed = proj(img, mesh, cam, uv_exp_blend_view_weight=vw, **kw)
    fresh = proj(img, mesh, cam, uv_exp_blend_view_weight=vw.clone(), **kw)
    assert torch.equal(changed, fresh) and not torch.equal(changed, first)


def test_unsupported_options_raise(wr_ctx):
    mesh, cam, images = _setup(wr_ctx.device)
    proj = wr.CameraProjection(None, None, str(wr_ctx.device), "cuda")
    with pytest.raises(ValueError):
        proj(torch.from_numpy(images), mesh, cam, uv_size=64)  # defaults ask for Poisson blending: needs pb_backend
    with pytest.raises(AssertionError):
        proj(torch.from_numpy(images), mesh, cam, uv_size=64, poisson_blending=True, uv_padding=False)  # uv.py:427
    with pytest.raises(NotImplementedError):
        proj(torch.from_numpy(images), mesh, cam, uv_size=64, poisson_blending=False, uv_padding=False,
             warp_images=True, images_background=1.0)


def test_sharded_bake_single_process_equals_camera_projection(wr_ctx):
    from worldrenderer_b200 import parallel
    mesh, cam, images = _setup(wr_ctx.device)
    img = torch.from_numpy(images).to(wr_ctx.device)
    proj = wr.CameraProjection(None, None, str(wr_ctx.device), "cuda")
    want = proj(img, mesh, cam, uv_size=128, poisson_blending=False, uv_padding=False, iou_rejection_threshold=None,
                return_dict=True)
    atlas, any_ = parallel.sharded_bake(wr_ctx, mesh, cam, img, 128)
    assert torch.equal(any_, want.uv_proj_mask)
    torch.testing.assert_close(atlas, want.uv_proj, rtol=1e-5, atol=1e-6)
    # a rank that owns no view contributes zeros
    atlas0, any0 = parallel.sharded_bake(wr_ctx, mesh, cam[0:0], img[0:0], 128)
    assert not bool(any0.any()) and torch.equal(atlas0, mesh.texture)
    lo, outs = parallel.render_mesh_shard(wr_ctx, [mesh, mesh, mesh], cam, 64, 64, rank=1, world=2, render_attr=False)
    assert lo == 2 and len(outs) == 1 and outs[0].mask.shape == (6, 64, 64)


def test_bake_pipeline_single_process_equals_sharded_bake(wr_ctx):
    """parallel.BakePipeline (exchange stage on its own stream, double-buffered) gives the bakes of sharded_bake, in
    order, also when more bakes are in flight than the pipeline has slots."""
    from worldrenderer_b200 import parallel
    mesh, cam, images = _setup(wr_ctx.device)
    img = torch.from_numpy(images).to(wr_ctx.device)
    imgs = [img, img.flip(0).contiguous(), (img * 0.5).contiguous(), img.roll(1, 0).contiguous(), img]
    want = [tuple(t.clone() for t in parallel.sharded_bake(wr_ctx, mesh, cam, im, 128)) for im in imgs]
    pipe = parallel.BakePipeline(wr_ctx, 128, depth=2)
    got = []
    for im in imgs:
        tk = pipe.submit(mesh, cam, im)
        got.append(tk)
        if len(got) >= 2:   # consume with one bake in flight behind
            a, m = got[-2].result()
            got[-2] = (a.clone(), m.clone())
    a, m = got[-1].result()
    got[-1] = (a.clone(), m.clone())
    torch.cuda.synchronize()
    for (a, m), (wa, wm) in zip(got, want):
        assert torch.equal(m, wm) and torch.equal(a, wa)
    with pytest.raises(NotImplementedError):
        pipe.submit(mesh, cam, img, uv_padding=True)


def test_config_c_full_size_against_oracle(wr_ctx):
    """BASELINE config C at full size: 50k-face icosphere, 6 x 768^2 images -> 1024^2 atlas."""
    mesh, cam, images = _setup(wr_ctx.device, freq=50, views=(768, 768), uv_size=1024)
    proj = wr.CameraProjection(None, None, str(wr_ctx.device), "cuda")
    vw = torch.ones(6)
    out = proj(torch.from_numpy(images), mesh, cam, uv_size=1024, poisson_blending=False, uv_padding=False,
               depth_grad_dilation=5, uv_exp_blend_alpha=3, uv_exp_blend_view_weight=vw, aoi_cos_valid_threshold=0.2,
               depth_grad_threshold=0.1, iou_rejection_threshold=None, return_dict=True)
    ref = _oracle_bake(mesh, cam, images, 1024, aoi_cos_valid_threshold=0.2, depth_grad_threshold=0.1,
                       uv_exp_blend_alpha=3.0, uv_exp_blend_view_weight=vw.numpy(), depth_grad_dilation=5)
    np.testing.assert_array_equal(out.uv_proj_mask.cpu().numpy(), ref["uv_proj_mask"])
    np.testing.assert_allclose(out.uv_proj.cpu().numpy(), ref["uv_proj"], rtol=RTOL, atol=ATOL)
    np.testing.assert_array_equal(out.uv_aoi_cos.cpu().numpy(), ref["uv_aoi_cos"])
    np.testing.assert_array_equal(out.uv_depth_grad.cpu().numpy(), ref["uv_depth_grad"])
    assert ref["uv_proj_mask"].sum() > 200_000
