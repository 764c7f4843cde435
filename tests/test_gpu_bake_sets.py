"""CameraProjection.project_sets: up to four image sets of one rig baked in one pass.

The one-set bake (`__call__`) is held to the CPU oracle by tests/test_gpu_bake_parity.py, test_gpu_bake_geometry.py
and test_gpu_blend_parity.py.  Here every result of `project_sets` must equal, bit for bit (torch.equal), the
`__call__` on that set alone with the same keywords: atlas, mask and the per-view planes of return_dict.  Below that,
the two new entry points are checked at the C ABI: the K-set seam padding against K one-set paddings, and the refusals
of the K-set unprojection."""
import ctypes

import numpy as np
import pytest
import torch

import cases
import worldrenderer_b200 as wr
from test_gpu_render_parity import make_mesh
from worldrenderer_b200 import _native, synth
from worldrenderer_b200.uv import _unproject_args, fused_view_maps, uv_padding, uv_padding_sets

pytestmark = pytest.mark.gpu

RIGS = {"ortho": lambda H, W, device: cases.canonical_cameras(device=device),
        "perspective": cases.bake_perspective_cameras, "mixed40": cases.mixed_40_view_cameras}

# the texture pipeline's colour modalities (rgb, base_color, orm): SURVEY.md section 3.3
COLOUR_KW = dict(aoi_cos_valid_threshold=-1.0, depth_grad_threshold=None, uv_exp_blend_alpha=3,
                 iou_rejection_threshold=None, poisson_blending=False)


def _mesh(device, uv_size, seed=3):
    v, f = cases.icosphere_mesh(8)
    return make_mesh(v, f, device, with_uv=True, tex_size=uv_size, seed=seed)


def _image_sets(K, Nv, H, W, device, seed=1):
    """K distinct sets; the last of four reaches outside [0, 1] (the padding clamps it)."""
    sets = [torch.from_numpy(synth.view_images(Nv, H, W, seed=seed + 7 * k)).to(device) for k in range(K)]
    if K == 4:
        sets[3] = sets[3] * 1.6 - 0.3
    return sets


def _assert_same(got, want):
    if want is None:
        assert got is None
    elif isinstance(want, torch.Tensor):
        assert torch.equal(got, want)
    elif isinstance(want, tuple):
        assert len(got) == len(want) and all(torch.equal(g, w) for g, w in zip(got, want))
    else:
        for name in ("uv_proj", "uv_proj_mask", "uv_depth_grad", "uv_aoi_cos"):
            g, w = getattr(got, name), getattr(want, name)
            assert (g is None and w is None) or torch.equal(g, w), name


def _check_sets(proj, sets, mesh, cam, textures=None, **kw):
    """project_sets against one __call__ per set (set k on the mesh with texture textures[k])."""
    outs = proj.project_sets(sets, mesh, cam, textures=textures, **kw)
    assert isinstance(outs, list) and len(outs) == len(sets)
    own = mesh.texture
    try:
        for k, images in enumerate(sets):
            if textures is not None:
                mesh.texture = textures[k]
            _assert_same(outs[k], proj(images, mesh, cam, **kw))
    finally:
        mesh.texture = own
    if kw.get("return_dict"):   # documented: the image-independent outputs are shared
        assert all(o.uv_proj_mask is outs[0].uv_proj_mask and o.uv_aoi_cos is outs[0].uv_aoi_cos for o in outs)
    return outs


@pytest.mark.parametrize("K", [1, 2, 3, 4])
@pytest.mark.parametrize("rig", sorted(RIGS))
def test_sets_equal_separate_calls_on_every_rig(wr_ctx, rig, K):
    """Non-square views, an atlas that is not a multiple of the 1024-texel blocks, the colour keywords."""
    dev = wr_ctx.device
    H, W, uv = 64, 96, 200
    mesh, cam = _mesh(dev, uv), RIGS[rig](H, W, device=dev)
    sets = _image_sets(K, cam.mvp_mtx.shape[0], H, W, dev)
    proj = wr.CameraProjection(None, None, str(dev), "cuda")
    outs = _check_sets(proj, sets, mesh, cam, uv_size=uv, uv_padding=True, return_dict=True,
                       uv_exp_blend_view_weight=torch.ones(cam.mvp_mtx.shape[0]), **COLOUR_KW)
    assert outs[0].uv_proj_mask.sum() > 0
    if K > 1:
        assert not torch.equal(outs[0].uv_proj, outs[1].uv_proj)


KEYWORD_CASES = {
    "defaults_with_poisson": dict(iou_rejection_threshold=None, pb_num_iters=40),
    "poisson_new_border": dict(iou_rejection_threshold=None, pb_num_iters=40, pb_keep_original_border=False),
    "dilation_1": dict(COLOUR_KW, depth_grad_dilation=1, depth_grad_threshold=0.1, return_dict=True),
    "dilation_7": dict(COLOUR_KW, depth_grad_dilation=7, depth_grad_threshold=0.1, return_dict=True),
    "no_padding": dict(COLOUR_KW, uv_padding=False, return_dict=True),
    "from_scratch": dict(COLOUR_KW, from_scratch=True),
    "mask_tuple": dict(COLOUR_KW, aoi_cos_valid_threshold=0.2, return_uv_projection_mask=True),
    "view_masks_and_weights": dict(COLOUR_KW, aoi_cos_valid_threshold=0.2, depth_grad_threshold=0.1, masks="smooth",
                                   uv_exp_blend_view_weight=torch.tensor([1.0, 0.5, 1.0, 2.0, 1.0, 1.0]),
                                   uv_exp_blend_alpha=6, return_dict=True),
}


@pytest.mark.parametrize("case", sorted(KEYWORD_CASES))
def test_sets_equal_separate_calls_for_every_keyword(wr_ctx, case):
    dev = wr_ctx.device
    kw = dict(KEYWORD_CASES[case])
    mesh, cam = _mesh(dev, 128), cases.canonical_cameras(device=dev)
    sets = _image_sets(3, 6, 96, 96, dev, seed=5)
    if kw.get("masks") == "smooth":   # about half of every view passes the 0.9 threshold
        kw["masks"] = torch.clamp(2.0 * sets[0][..., 1], 0, 1)
    proj = wr.CameraProjection("torch-cuda", None, str(dev), "cuda")
    _check_sets(proj, sets, mesh, cam, uv_size=128, **kw)


@pytest.mark.parametrize("tail", ["padding", "poisson"])
def test_sets_with_their_own_textures(wr_ctx, tail):
    """Distinct existing atlases per set, a None entry (stitched with zeros) and a zero atlas."""
    dev = wr_ctx.device
    uv = 128
    mesh, cam = _mesh(dev, uv), cases.canonical_cameras(device=dev)
    sets = _image_sets(4, 6, 96, 96, dev, seed=9)
    g = torch.Generator(device="cpu").manual_seed(4)
    own = [torch.rand((uv, uv, 3), generator=g).to(dev) for _ in range(2)]
    if tail == "padding":
        textures, kw = [own[0], None, torch.zeros((uv, uv, 3), device=dev), own[1]], dict(COLOUR_KW, uv_padding=True)
    else:   # pb_keep_original_border solves towards each set's own atlas (a None one is refused by __call__ too)
        textures = [own[0], torch.zeros((uv, uv, 3), device=dev), own[1], mesh.texture]
        kw = dict(iou_rejection_threshold=None, pb_num_iters=24)
    proj = wr.CameraProjection("torch-cuda", None, str(dev), "cuda")
    outs = _check_sets(proj, sets, mesh, cam, textures=textures, uv_size=uv, **kw)
    assert not torch.equal(outs[0], outs[3])


def test_iou_rejection_rejects_every_set(wr_ctx):
    dev = wr_ctx.device
    mesh, cam = _mesh(dev, 64), cases.canonical_cameras(device=dev)
    sets = _image_sets(3, 6, 96, 96, dev)
    bad = torch.zeros((6, 96, 96), device=dev)
    bad[:, :10, :10] = 1
    proj = wr.CameraProjection(None, None, str(dev), "cuda")
    assert proj.project_sets(sets, mesh, cam, masks=bad, uv_size=64, poisson_blending=False) == [None] * 3


def test_invalid_sets_raise(wr_ctx):
    dev = wr_ctx.device
    mesh, cam = _mesh(dev, 64), cases.canonical_cameras(device=dev)
    sets = _image_sets(4, 6, 32, 32, dev)
    proj = wr.CameraProjection(None, None, str(dev), "cuda")
    kw = dict(uv_size=64, poisson_blending=False, iou_rejection_threshold=None)
    rgba = torch.cat([sets[1], sets[1][..., :1]], -1)
    for bad, textures in (([], None), (sets + sets[:1], None), ([sets[0], sets[1][:, :16]], None),
                          ([sets[0], sets[1][:5]], None), ([sets[0], rgba], None), (sets[:2], [None]),
                          (sets[:2], [None, None, None])):
        with pytest.raises(ValueError):
            proj.project_sets(bad, mesh, cam, textures=textures, **kw)


def test_view_maps_of_several_sets(wr_ctx):
    """attr_map [Nv,H,W,K,4]: set 0 is the one-set map, set k is (rgb_k, 0); the sets are read in place."""
    dev = wr_ctx.device
    H, W = 40, 72   # W % 4 == 0: the TMA depth tile
    mesh, cam = _mesh(dev, 64), cases.bake_perspective_cameras(H, W, device=dev)
    sets = _image_sets(4, 4, H, W, dev)
    for d in (0, 5):
        _, geo1, att1 = fused_view_maps(wr_ctx, mesh, cam, sets[0], H, W, d)
        for K in (1, 2, 4):
            _, geo, att = fused_view_maps(wr_ctx, mesh, cam, sets[:K], H, W, d)
            assert att.shape == (4, H, W, K, 4) and torch.equal(geo, geo1)
            assert torch.equal(att[..., 0, :], att1)
            for k in range(1, K):
                assert torch.equal(att[..., k, :3], sets[k]) and not att[..., k, 3].any()


# ---- C ABI ----------------------------------------------------------------------------------------------------------

def _pad_sets_raw(ctx, attrs, mask, radius=3):
    c = ctx.ctx
    out = [torch.full_like(a, -7.0) for a in attrs]
    st = _native.lib().wr_uv_padding_sets(c.handle, _native.ptr_array(attrs), _native.ptr(mask), mask.shape[0],
                                          mask.shape[1], len(attrs), radius, _native.ptr_array(out), c.stream())
    return st, out


def _pad_one_raw(ctx, attr, mask, radius=3):
    c = ctx.ctx
    out = torch.full_like(attr, -7.0)
    st = _native.lib().wr_uv_padding(c.handle, _native.ptr(attr), _native.ptr(mask), mask.shape[0], mask.shape[1], 3,
                                     radius, _native.ptr(out), c.stream())
    assert st == 0
    return out


@pytest.mark.parametrize("shape,mask_kind", [((97, 131), "blobs"), ((64, 64), "empty"), ((64, 48), "full"),
                                             ((4096, 4096), "blobs")])
def test_padding_sets_equal_one_set_paddings(wr_ctx, shape, mask_kind):
    dev = wr_ctx.device
    H, W = shape
    g = torch.Generator(device="cpu").manual_seed(H + W)
    if mask_kind == "blobs":   # charts of random rectangles, most of the atlas to fill
        mask = torch.zeros((H, W), dtype=torch.bool)
        for _ in range(24):
            y, x = torch.randint(0, H - 8, (1,), generator=g).item(), torch.randint(0, W - 8, (1,), generator=g).item()
            mask[y:y + max(2, H // 10), x:x + max(2, W // 12)] = True
    else:   # no known texel (every texel is filled, none has a seed) / nothing to fill
        mask = torch.full((H, W), mask_kind == "full", dtype=torch.bool)
    mask = mask.to(dev).view(torch.uint8)
    ks = (4,) if H >= 4096 else (1, 2, 3, 4)
    attrs = [(torch.rand((H, W, 3), generator=g) * 1.4 - 0.2).to(dev) for _ in range(max(ks))]
    want = [_pad_one_raw(wr_ctx, a, mask) for a in attrs]
    for K in ks:
        st, got = _pad_sets_raw(wr_ctx, attrs[:K], mask)
        assert st == 0
        for k in range(K):
            assert torch.equal(got[k], want[k]), (K, k)
    for k, o in enumerate(uv_padding_sets(attrs, mask.bool(), 3)):   # the Python wrapper
        assert torch.equal(o, uv_padding(attrs[k], mask.bool(), 3))


def test_padding_sets_refuses_bad_arguments(wr_ctx):
    dev = wr_ctx.device
    mask = torch.ones((16, 16), dtype=torch.uint8, device=dev)
    attrs = [torch.rand((16, 16, 3), device=dev) for _ in range(5)]
    assert _pad_sets_raw(wr_ctx, attrs, mask)[0] == -1          # K = 5
    assert _pad_sets_raw(wr_ctx, attrs[:0], mask)[0] == -1      # K = 0
    c = wr_ctx.ctx
    holes = (ctypes.c_void_p * 2)(_native.ptr(attrs[0]), None)
    outs = _native.ptr_array(attrs[2:4])
    assert _native.lib().wr_uv_padding_sets(c.handle, holes, _native.ptr(mask), 16, 16, 2, 3, outs, c.stream()) == -1
    with pytest.raises(ValueError):
        uv_padding_sets([torch.rand((16, 16, 4), device=dev)], mask, 3)


def test_unproject_sets_refusals(wr_ctx):
    dev = wr_ctx.device
    H = W = 32
    mesh, cam = _mesh(dev, 64), cases.canonical_cameras(device=dev)
    sets = _image_sets(2, 6, H, W, dev)
    pre = wr.uv_precompute(wr_ctx, mesh, 64, 64)
    uv_pos, uv_mask, mvp = pre.uv_pos.contiguous(), pre.uv_mask.contiguous().view(torch.uint8), cam.mvp_mtx.contiguous()
    _, geo, att = fused_view_maps(wr_ctx, mesh, cam, sets, H, W, 5)
    c = wr_ctx.ctx
    out = [torch.empty((64, 64, 3), device=dev) for _ in range(2)]
    any_ = torch.empty((64, 64), dtype=torch.uint8, device=dev)
    accum = torch.zeros((64, 64, 5), device=dev)
    per_view = torch.empty((6, 64, 64, 2), device=dev)

    def run(**fields):
        a = _unproject_args(uv_pos, uv_mask, mvp, H, W, geo, att)
        a.attr_sets = 2
        a.out_attr, a.out_valid_any, a.out_attr_more[0] = _native.ptr(out[0]), _native.ptr(any_), _native.ptr(out[1])
        for k, v in fields.items():
            setattr(a, k, v)
        st = _native.lib().wr_uv_unproject(c.handle, ctypes.byref(a), c.stream())
        torch.cuda.synchronize(dev)
        return st

    assert run() == 0
    assert run(accum=_native.ptr(accum), out_attr=None, out_valid_any=None) == -5      # accumulate mode
    assert run(accum=_native.ptr(accum)) == -5
    assert run(uv_pos_ndc=_native.ptr(per_view)) == -5                                # full materialisation
    assert run(attr_sets=5) == -1
    assert run(attr_sets=-1) == -1
    assert run(out_attr=None) == -1
    more = (ctypes.c_void_p * 3)()
    assert run(out_attr_more=more) == -1                                               # set 1 has no output
