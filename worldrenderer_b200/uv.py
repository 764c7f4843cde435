"""UV-space precompute, geometry projection, attribute projection and blending (the texture bake).

Drop-in for mvadapter/utils/mesh_utils/uv.py of the reference: `uv_precompute` (:24-53),
`uv_render_geometry` (:72-184), `uv_render_attr` (:193-222), `SimpleUVValidityStrategy` (:248-298),
`ExponentialBlend` (:317-348), `uv_blend` (:385-468) and their output dataclasses.

The step-by-step functions keep the reference's contract -- they return the same (large) per-view
tensors -- but every sampling / projection step is one CUDA kernel of libwr_b200 (wr_rasterize,
wr_interpolate, wr_render, wr_view_prep, wr_uv_unproject in "materialise" mode, wr_grid_sample).
`fused_bake` is what `CameraProjection` uses when the configuration allows it: one unprojection
kernel per call that walks the views per texel and never materialises an [Nv,Huv,Wuv,*] tensor
unless the caller asks for one.

Atlas post-processing (SURVEY.md section 8f-2,3): `uv_padding` (seam fill; the reference's cvcuda inpaint is
replaced by this package's own fill, cv_ops.py) and Poisson blending through `blend.PoissonBlendingSolver`.
"""
from __future__ import annotations

import ctypes
from abc import ABC, abstractmethod
from dataclasses import dataclass
from typing import Optional

import torch
import torch.nn.functional as F

from . import _native
from .camera import Camera
from .mesh import TexturedMesh
from .render import NVDiffRastContextWrapper, SimpleNormalization, render_geometry_raw
from .utils import IMAGE_TYPE, image_to_tensor


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.float32).contiguous()


@dataclass
class UVPrecomputeOutput:
    height: int
    width: int
    uv_attr: torch.Tensor
    uv_mask: torch.Tensor
    uv_pos: torch.Tensor


def uv_precompute(ctx: NVDiffRastContextWrapper, mesh: TexturedMesh, height: int, width: int,
                  clone_attr: bool = False) -> UVPrecomputeOutput:
    """Rasterises the mesh in UV space and interpolates world positions per texel (uv.py:24-53)."""
    v_tex = _f32c(mesh.v_tex)
    uv_clip = v_tex * 2.0 - 1.0
    uv_clip4 = torch.cat((uv_clip, torch.zeros_like(uv_clip[..., 0:1]), torch.ones_like(uv_clip[..., 0:1])), dim=-1)
    rast, _ = ctx.rasterize(uv_clip4[None], mesh.index_i32("t_tex_idx"), (height, width))
    uv_mask = rast[0, :, :, 3] > 0
    uv_pos, _ = ctx.interpolate(mesh.v_pos[None], rast, mesh.index_i32("t_pos_idx"))
    return UVPrecomputeOutput(height=height, width=width,
                              uv_attr=mesh.texture.clone() if clone_attr else mesh.texture,
                              uv_mask=uv_mask, uv_pos=uv_pos[0])


@dataclass
class UVRenderGeometryOutput:
    uv_pos_proj: torch.Tensor
    uv_pos_error: torch.Tensor
    uv_aoi_cos: torch.Tensor
    uv_pos_ndc: torch.Tensor
    view_mask: torch.Tensor
    view_normal: torch.Tensor
    view_aoi_cos: torch.Tensor
    view_position: torch.Tensor
    view_depth: torch.Tensor
    view_depth_grad: Optional[torch.Tensor] = None
    uv_depth_grad: Optional[torch.Tensor] = None
    view_attr: Optional[torch.Tensor] = None


# bake view pass: geometry render with the un-normalised view depth and background 1e2 (uv.py:92-104)
_BAKE_DEPTH = dict(scale=1.0, offset=0.0, clamp=False, bg_value=1e2)


def _view_pass(ctx, mesh, cam, H, W, dilation, images=None, want_attr=False, want_maps=True, want_planes=True):
    """Geometry render of all views + wr_view_prep.  Returns (raw render dict, aoi, depth_grad, geo_map, attr_map)."""
    dev = ctx.device
    raw = render_geometry_raw(ctx, mesh, cam, H, W, want_pos=True, want_depth=True, want_normal=True,
                              want_attr=want_attr, depth_normalization_strategy=SimpleNormalization(**_BAKE_DEPTH))
    B = raw["pos"].shape[0]
    w2c = _f32c(cam.w2c)
    mask_u8 = raw["mask"].view(torch.uint8)
    aoi = torch.empty((B, H, W), dtype=torch.float32, device=dev) if want_planes else None
    dgrad = torch.empty((B, H, W), dtype=torch.float32, device=dev) if (want_planes and dilation > 0) else None
    geo = torch.empty((B, H, W, 4), dtype=torch.float32, device=dev) if want_maps else None
    att = torch.empty((B, H, W, 4), dtype=torch.float32, device=dev) if want_maps else None
    if images is not None:
        images = _f32c(images)
        if images.shape != (B, H, W, 3):
            raise ValueError(f"images must have shape {(B, H, W, 3)}, got {tuple(images.shape)}")
    c = ctx.ctx
    status = _native.lib().wr_view_prep(
        c.handle, _native.ptr(raw["normal"]), _native.ptr(mask_u8), _native.ptr(raw["depth"]),
        _native.ptr(raw["pos"]), _native.ptr(w2c), _native.ptr(images), B, H, W, int(dilation),
        _native.ptr(aoi), _native.ptr(dgrad), _native.ptr(geo), _native.ptr(att), c.stream())
    c.check(status, "wr_view_prep")
    return raw, aoi, dgrad, geo, att


def _unproject_args(pre_pos, pre_mask_u8, mvp, H, W, geo, att) -> "_native.UnprojectArgs":
    a = _native.UnprojectArgs()
    a.uv_pos, a.uv_mask = _native.ptr(pre_pos), _native.ptr(pre_mask_u8)
    a.Hu, a.Wu = pre_pos.shape[0], pre_pos.shape[1]
    a.mvp, a.Nv, a.H, a.W = _native.ptr(mvp), mvp.shape[0], H, W
    a.geo_map, a.attr_map = _native.ptr(geo), _native.ptr(att)
    # neutral strategy parameters: materialisation does not depend on them
    a.pos_error_eps, a.aoi_cos_thresh, a.mask_thresh, a.depth_grad_thresh = 1e-3, 0.1, 0.9, 0.0
    a.alpha = 1.0
    return a


def uv_render_geometry(ctx: NVDiffRastContextWrapper, mesh: TexturedMesh, cam: Camera, view_height: int,
                       view_width: int, uv_precompute_output: UVPrecomputeOutput, grid_sample_mode="bilinear",
                       compute_depth_grad: bool = False, depth_grad_dilation: int = 1,
                       render_attr: bool = False) -> UVRenderGeometryOutput:
    """Projects every texel into every view and samples the view geometry there (uv.py:72-184)."""
    if grid_sample_mode != "bilinear":
        raise NotImplementedError("only grid_sample_mode='bilinear' (the reference default) is implemented")
    dev = ctx.device
    H, W = int(view_height), int(view_width)
    dilation = int(depth_grad_dilation) if compute_depth_grad else 0
    raw, aoi, dgrad, geo, att = _view_pass(ctx, mesh, cam, H, W, dilation, want_attr=render_attr)
    B = raw["pos"].shape[0]
    uv_pos = _f32c(uv_precompute_output.uv_pos)
    uv_mask = uv_precompute_output.uv_mask.contiguous().view(torch.uint8)
    Hu, Wu = uv_pos.shape[0], uv_pos.shape[1]
    mvp = _f32c(cam.mvp_mtx)
    a = _unproject_args(uv_pos, uv_mask, mvp, H, W, geo, att)
    ndc = torch.empty((B, Hu, Wu, 2), dtype=torch.float32, device=dev)
    proj = torch.empty((B, Hu, Wu, 3), dtype=torch.float32, device=dev)
    err = torch.empty((B, Hu, Wu), dtype=torch.float32, device=dev)
    uaoi = torch.empty((B, Hu, Wu), dtype=torch.float32, device=dev)
    udg = torch.empty((B, Hu, Wu), dtype=torch.float32, device=dev) if compute_depth_grad else None
    a.uv_pos_ndc, a.uv_pos_proj, a.uv_pos_error = _native.ptr(ndc), _native.ptr(proj), _native.ptr(err)
    a.uv_aoi_cos, a.uv_depth_grad = _native.ptr(uaoi), _native.ptr(udg)
    c = ctx.ctx
    c.check(_native.lib().wr_uv_unproject(c.handle, ctypes.byref(a), c.stream()), "wr_uv_unproject")
    return UVRenderGeometryOutput(
        uv_pos_proj=proj, uv_pos_error=err, uv_aoi_cos=uaoi, uv_pos_ndc=ndc, view_mask=raw["mask"],
        view_position=raw["pos"], view_normal=raw["normal"], view_aoi_cos=aoi, view_depth=raw["depth"],
        view_depth_grad=dgrad[:, None] if dgrad is not None else None,  # reference keeps the conv channel dim
        uv_depth_grad=udg, view_attr=raw.get("attr") if render_attr else None)


def grid_sample_nhwc(maps: torch.Tensor, ndc: torch.Tensor) -> torch.Tensor:
    """Bilinear, zero padded, align_corners=False sampling of channels-last maps [B,H,W,C] at ndc [B,Hs,Ws,2]."""
    maps, ndc = _f32c(maps), _f32c(ndc)
    if maps.device.type != "cuda" or ndc.device != maps.device:
        raise RuntimeError("grid_sample_nhwc: inputs must live on the same CUDA device (there is no CPU path)")
    B, H, W, C = maps.shape
    out = torch.empty((B, ndc.shape[1], ndc.shape[2], C), dtype=torch.float32, device=maps.device)
    from .mesh import _shared_context
    c = _shared_context(maps.device)
    c.check(_native.lib().wr_grid_sample(c.handle, _native.ptr(maps), B, H, W, C, _native.ptr(ndc), ndc.shape[1],
                                         ndc.shape[2], _native.ptr(out), c.stream()), "wr_grid_sample")
    return out


@dataclass
class UVRenderAttrOutput:
    uv_attr_proj: torch.Tensor
    uv_mask_proj: Optional[torch.Tensor]


def uv_render_attr(images: IMAGE_TYPE, uv_render_geometry_output: UVRenderGeometryOutput,
                   masks: Optional[IMAGE_TYPE] = None, grid_sample_mode: str = "bilinear") -> UVRenderAttrOutput:
    """Samples the view images (and masks) at the projected texel positions (uv.py:193-222)."""
    if grid_sample_mode != "bilinear":
        raise NotImplementedError("only grid_sample_mode='bilinear' (the reference default) is implemented")
    ndc = uv_render_geometry_output.uv_pos_ndc
    images = image_to_tensor(images, device=ndc.device)
    uv_attr_proj = grid_sample_nhwc(images, ndc)
    uv_mask_proj = None
    if masks is not None:
        masks = image_to_tensor(masks, device=ndc.device)
        if masks.ndim == 4:
            masks = masks.mean(-1)
        uv_mask_proj = grid_sample_nhwc(masks[..., None], ndc)[..., 0]
    return UVRenderAttrOutput(uv_attr_proj=uv_attr_proj, uv_mask_proj=uv_mask_proj)


@dataclass
class UVBlendOutput:
    uv_attr_blend: Optional[torch.Tensor]
    uv_valid_mask: torch.Tensor
    uv_valid_mask_blend: torch.Tensor
    uv_blend_weight: torch.Tensor


class UVValidityStrategy(ABC):
    @abstractmethod
    def __init__(self, *args, **kwargs):
        pass

    @abstractmethod
    def __call__(self, uv_precompute_output, uv_render_geometry_output, uv_render_attr_output) -> torch.Tensor:
        pass


class SimpleUVValidityStrategy(UVValidityStrategy):
    """A texel is valid in a view if it re-projects onto itself, faces the camera enough, is not on a depth
    discontinuity, lies inside a chart and (optionally) inside the view's foreground mask (uv.py:248-298)."""

    def __init__(self, pos_error_eps: float = 1e-3, aoi_cos_thresh: float = 0.1, mask_thresh: float = 0.9,
                 depth_grad_thresh: Optional[float] = None, first_view_dominate: bool = False):
        self.pos_error_eps = pos_error_eps
        self.aoi_cos_thresh = aoi_cos_thresh
        self.mask_thresh = mask_thresh
        self.depth_grad_thresh = depth_grad_thresh
        self.first_view_dominate = first_view_dominate

    def __call__(self, uv_precompute_output, uv_render_geometry_output, uv_render_attr_output) -> torch.Tensor:
        geo = uv_render_geometry_output
        valid = (geo.uv_pos_error < self.pos_error_eps) & (geo.uv_aoi_cos > self.aoi_cos_thresh)
        if self.depth_grad_thresh is not None:
            if geo.uv_depth_grad is None:
                print("Warning: Depth gradient is not computed, depth gradient threshold is ignored.")
            else:
                valid &= geo.uv_depth_grad < self.depth_grad_thresh
        valid &= uv_precompute_output.uv_mask
        if uv_render_attr_output is not None and uv_render_attr_output.uv_mask_proj is not None:
            valid &= uv_render_attr_output.uv_mask_proj > self.mask_thresh
        else:
            print("No view mask provided for UV blending, using all valid pixels")
        if self.first_view_dominate:
            valid[1:] &= ~valid[0:1]
        return valid


class UVBlendWeightStrategy(ABC):
    @abstractmethod
    def __init__(self, *args, **kwargs):
        pass

    @abstractmethod
    def __call__(self, uv_precompute_output, uv_render_geometry_output, uv_render_attr_output,
                 uv_valid_mask) -> torch.Tensor:
        pass


class ExponentialBlend(UVBlendWeightStrategy):
    """weight = (aoi_cos * valid) ** alpha (or ** (alpha / view_weight)), normalised over views (uv.py:317-348)."""

    def __init__(self, alpha: float = 1.0, normalization: str = "linear", view_weight: Optional[torch.Tensor] = None):
        self.alpha = alpha
        self.normalization = normalization
        self.view_weight = view_weight

    def __call__(self, uv_precompute_output, uv_render_geometry_output, uv_render_attr_output,
                 uv_valid_mask) -> torch.Tensor:
        w = uv_render_geometry_output.uv_aoi_cos * uv_valid_mask.float()
        if self.view_weight is not None:
            w = w ** (self.alpha / self.view_weight[:, None, None].to(w))
        else:
            w = w ** self.alpha
        if self.normalization == "linear":
            return (w / w.sum(axis=0, keepdim=True).clamp(1e-5)).clamp(0.0, 1.0)
        if self.normalization == "softmax":
            w[~uv_valid_mask] = -1e5
            return F.softmax(w, dim=0)
        raise ValueError(f"unknown normalization {self.normalization!r}")


class RandomChoiceBlend(UVBlendWeightStrategy):
    """One random valid view per texel (uv.py:351-370)."""

    def __init__(self, alpha):
        self.alpha = alpha

    def __call__(self, uv_precompute_output, uv_render_geometry_output, uv_render_attr_output,
                 uv_valid_mask) -> torch.Tensor:
        w = uv_render_geometry_output.uv_aoi_cos * uv_valid_mask.float()
        w[w > 0] = torch.rand_like(w[w > 0])
        return F.one_hot(w.max(dim=0).indices, num_classes=w.shape[0]).float().permute(2, 0, 1)


def uv_padding(attr: torch.Tensor, inside_mask: torch.Tensor, radius: int, native_ctx=None):
    """Seam padding (uv.py:373-382): clamp to [0,1], quantise like inpaint_cvc (cv_ops.py:23-35), fill the
    texels outside `inside_mask`.  One `wr_uv_padding` call (clamp + quantise + fill + /255 fused); the fill is
    this package's own (cv_ops.py docstring), not cvcuda's.  native_ctx: the _native.NativeContext whose scratch
    the call uses (default: the device's shared one); a caller that pads on a second stream while the first one
    still uses the shared context passes its own."""
    if attr.ndim != 3 or inside_mask.shape != attr.shape[:2]:
        raise ValueError(f"uv_padding: attr [H,W,C] and inside_mask [H,W] expected, got {tuple(attr.shape)}, "
                         f"{tuple(inside_mask.shape)}")
    a = _f32c(attr.detach())
    m = (inside_mask != 0).contiguous().view(torch.uint8)
    H, W, C = a.shape
    out = torch.empty_like(a)
    c = native_ctx if native_ctx is not None else _native.default_context(a.device)
    c.check(_native.lib().wr_uv_padding(c.handle, _native.ptr(a), _native.ptr(m), H, W, C, int(radius),
                                        _native.ptr(out), c.stream()), "wr_uv_padding")
    return out


def uv_padding_sets(attrs, inside_mask: torch.Tensor, radius: int, native_ctx=None):
    """`uv_padding` of up to four [H,W,3] atlases against one mask in one `wr_uv_padding_sets` call: the jump flood,
    most of a padding's cost, runs once for all of them.  Returns a list; entry k equals
    uv_padding(attrs[k], inside_mask, radius) bit for bit."""
    if not 1 <= len(attrs) <= _native.MAX_BAKE_SETS:
        raise ValueError(f"uv_padding_sets: 1 to {_native.MAX_BAKE_SETS} atlases, got {len(attrs)}")
    a = [_f32c(x.detach()) for x in attrs]
    for x in a:
        if x.ndim != 3 or x.shape[2] != 3 or x.shape[:2] != inside_mask.shape:
            raise ValueError(f"uv_padding_sets: atlases [H,W,3] and inside_mask [H,W] expected, got {tuple(x.shape)}, "
                             f"{tuple(inside_mask.shape)}")
    m = (inside_mask != 0).contiguous().view(torch.uint8)
    H, W = m.shape
    out = [torch.empty_like(x) for x in a]
    c = native_ctx if native_ctx is not None else _native.default_context(a[0].device)
    c.check(_native.lib().wr_uv_padding_sets(c.handle, _native.ptr_array(a), _native.ptr(m), H, W, len(a), int(radius),
                                             _native.ptr_array(out), c.stream()), "wr_uv_padding_sets")
    return out


def uv_blend(
    uv_precompute_output: UVPrecomputeOutput,
    uv_render_geometry_output: UVRenderGeometryOutput,
    uv_render_attr_output: Optional[UVRenderAttrOutput],
    uv_validity_strategy: UVValidityStrategy = SimpleUVValidityStrategy(),
    uv_blend_weight_strategy: UVBlendWeightStrategy = ExponentialBlend(),
    empty_value: float = 0.0,
    do_uv_padding: bool = True,
    uv_padding_radius: int = 3,
    pad_unseen_area: bool = False,
    poisson_blending: bool = False,
    pb_solver=None,
    pb_num_iters: int = 1000,
    pb_keep_original_border: bool = True,
    pb_inplace: bool = False,
    pb_grad_mode: str = "src",
) -> UVBlendOutput:
    """Step-by-step blend on the materialised tensors (uv.py:385-468).  Strategies are arbitrary callables
    here; the fused path used by CameraProjection is `fused_unproject` followed by `atlas_postprocess`."""
    valid = uv_validity_strategy(uv_precompute_output, uv_render_geometry_output, uv_render_attr_output)
    weight = uv_blend_weight_strategy(uv_precompute_output, uv_render_geometry_output, uv_render_attr_output, valid)
    valid_any = valid.any(dim=0)
    if uv_render_attr_output is None:
        return UVBlendOutput(uv_attr_blend=None, uv_valid_mask=valid, uv_valid_mask_blend=valid_any,
                             uv_blend_weight=weight)
    blend = (uv_render_attr_output.uv_attr_proj * weight[..., None]).sum(axis=0)
    stitched = blend * valid_any[..., None].float() + uv_precompute_output.uv_attr * (~valid_any)[..., None].float()
    blend = atlas_postprocess(blend, stitched, valid_any, uv_precompute_output, do_uv_padding=do_uv_padding,
                              uv_padding_radius=uv_padding_radius, pad_unseen_area=pad_unseen_area,
                              poisson_blending=poisson_blending, pb_solver=pb_solver, pb_num_iters=pb_num_iters,
                              pb_keep_original_border=pb_keep_original_border, pb_inplace=pb_inplace,
                              pb_grad_mode=pb_grad_mode)
    return UVBlendOutput(uv_attr_blend=blend, uv_valid_mask=valid, uv_valid_mask_blend=valid_any,
                         uv_blend_weight=weight)


def atlas_postprocess(blend, stitched, valid_any, pre: UVPrecomputeOutput, *, do_uv_padding=True,
                      uv_padding_radius=3, pad_unseen_area=False, poisson_blending=False, pb_solver=None,
                      pb_num_iters=1000, pb_keep_original_border=True, pb_inplace=False, pb_grad_mode="src",
                      native_ctx=None, old_attrs=None):
    """Tail of uv_blend (uv.py:426-461) shared by the step-by-step and the fused bake: optional Poisson blend of
    the projected colours into the existing texture, then seam padding.  `blend` is the weighted view sum,
    `stitched` the same with the existing texture where no view is valid.  Where only texels outside
    `valid_any` differ (they are refilled by the padding before anything reads them) either may stand in for
    `blend`, which is how the fused bake calls it with blend=None.  native_ctx: passed on to `uv_padding`.

    `stitched` (and `blend`) may also be lists of [H,W,3] atlases baked with the same masks (the image sets of
    CameraProjection.project_sets).  Each padding then fills all of them in one `uv_padding_sets` call, the Poisson
    solve runs per atlas, and a list is returned.  old_attrs: the existing texture of each set, which
    pb_keep_original_border keeps (default pre.uv_attr for every set)."""
    sets = not torch.is_tensor(stitched)

    def pad(x, mask):
        if sets:
            return uv_padding_sets(x, mask, uv_padding_radius, native_ctx)
        return uv_padding(x, mask, uv_padding_radius, native_ctx)

    if poisson_blending:
        assert do_uv_padding  # uv.py:427
        assert pb_solver is not None
        padded = pad(stitched if blend is None else blend, valid_any)
        if pb_keep_original_border:
            if sets:
                pb_tgt = [pre.uv_attr] * len(stitched) if old_attrs is None else old_attrs
            else:
                pb_tgt = pre.uv_attr
        else:
            pb_tgt = pad(stitched, pre.uv_mask)
        if sets:
            out = [pb_solver(p, valid_any, t, pb_num_iters, inplace=pb_inplace, grad_mode=pb_grad_mode)
                   for p, t in zip(padded, pb_tgt)]
        else:
            out = pb_solver(padded, valid_any, pb_tgt, pb_num_iters, inplace=pb_inplace, grad_mode=pb_grad_mode)
    else:
        out = stitched
    if do_uv_padding:
        content = valid_any if pad_unseen_area else pre.uv_mask
        out = pad(out, content)
    return out


# ------------------------------------------------------------------------------------------------
# fused bake
# ------------------------------------------------------------------------------------------------

@dataclass
class FusedBakeOutput:
    uv_attr_blend: Optional[torch.Tensor]        # [Huv,Wuv,3] stitched with the existing texture (None if accumulate_only)
    uv_valid_mask_blend: Optional[torch.Tensor]  # [Huv,Wuv] bool
    accum: Optional[torch.Tensor]                # [Huv,Wuv,5] (sum w*rgb, sum w, sum valid) when requested
    uv_depth_grad: Optional[torch.Tensor]        # [Nv,Huv,Wuv] when requested
    uv_aoi_cos: Optional[torch.Tensor]           # [Nv,Huv,Wuv] when requested
    view_mask: torch.Tensor                      # [Nv,H,W] bool (IoU rejection needs it)


def fused_view_maps(ctx, mesh, cam, images, H, W, dilation):
    """View pass of the fused bake: returns (view_mask bool [Nv,H,W], geo_map, attr_map).  The shading kernel
    writes the packed (pos, aoi_cos) map directly (no position / normal maps in HBM); wr_view_prep_sets then only
    adds the depth gradient and packs (rgb, depth_grad).

    `images` is one [Nv,H,W,3] tensor (attr_map [Nv,H,W,4]) or a list of 1 to 4 of them, image sets of the same rig
    baked together (attr_map [Nv,H,W,K,4]: set 0 is (rgb, depth_grad), set k is (rgb_k, 0)).  Float32 contiguous
    sets are read in place."""
    dev = ctx.device
    raw = render_geometry_raw(ctx, mesh, cam, H, W, want_pos=False, want_depth=True, want_normal=False, want_geo=True,
                              depth_normalization_strategy=SimpleNormalization(**_BAKE_DEPTH))
    B = raw["geo"].shape[0]
    sets = [images] if torch.is_tensor(images) else list(images)
    if not 1 <= len(sets) <= _native.MAX_BAKE_SETS:
        raise ValueError(f"1 to {_native.MAX_BAKE_SETS} image sets, got {len(sets)}")
    sets = [_f32c(x) for x in sets]
    for x in sets:
        if x.shape != (B, H, W, 3):
            raise ValueError(f"images must have shape {(B, H, W, 3)}, got {tuple(x.shape)}")
    shape = (B, H, W, 4) if torch.is_tensor(images) else (B, H, W, len(sets), 4)
    att = torch.empty(shape, dtype=torch.float32, device=dev)
    c = ctx.ctx
    status = _native.lib().wr_view_prep_sets(c.handle, _native.ptr(raw["depth"]), _native.ptr_array(sets), len(sets),
                                             B, H, W, int(dilation), None, _native.ptr(att), c.stream())
    c.check(status, "wr_view_prep_sets")
    return raw["mask"], raw["geo"], att


_VW_CACHE: list = []   # [(source tensor kept alive, version, device, device copy)], last four


def _view_weight_on(dev, view_weight) -> torch.Tensor:
    """The per-view blend weights as a flat float32 tensor on `dev`.  Callers pass a small HOST tensor with every bake
    (projection.py:87); uploading it is a synchronous pageable copy per call, so the copy of an unchanged tensor is
    reused (same object, same version counter)."""
    t = torch.as_tensor(view_weight)
    if t.device == dev:
        return _f32c(t).reshape(-1)
    for src, ver, d, out in _VW_CACHE:
        if src is t and ver == t._version and d == dev:
            return out
    out = _f32c(t.to(dev)).reshape(-1)
    _VW_CACHE.append((t, t._version, dev, out))
    del _VW_CACHE[:-4]
    return out


def fused_unproject(ctx, pre: UVPrecomputeOutput, cam: Camera, H: int, W: int, geo, att, view_masks=None, *,
                    pos_error_eps=1e-3, aoi_cos_thresh=0.1, mask_thresh=0.9, depth_grad_thresh=None,
                    first_view_dominate=False, alpha=1.0, view_weight=None, want_per_view=False,
                    accumulate_only=False, accum: Optional[torch.Tensor] = None, add_to_accum: bool = True,
                    tex_range: Optional[tuple] = None, old_attrs=None):
    """One wr_uv_unproject launch.  Returns (attr_blend, valid_any, accum, uv_depth_grad, uv_aoi_cos).
    With accumulate_only, a given `accum` is added to (add_to_accum=True) or overwritten (False).
    tex_range = (lo, hi): only these texels of the flattened atlas (the multi-GPU bake works chunk by chunk).
    A K-set `att` ([Nv,H,W,K,4] from fused_view_maps with a list of image sets) bakes every set in the same launch
    (not with accumulate_only) and attr_blend is a list of K atlases; old_attrs: the existing texture of each set,
    a tensor or None (default pre.uv_attr for every set)."""
    dev = ctx.device
    uv_pos = _f32c(pre.uv_pos)
    uv_mask = pre.uv_mask.contiguous().view(torch.uint8)
    Hu, Wu = uv_pos.shape[0], uv_pos.shape[1]
    mvp = _f32c(cam.mvp_mtx)
    Nv = mvp.shape[0]
    a = _unproject_args(uv_pos, uv_mask, mvp, H, W, geo, att)
    K = att.shape[3] if att.dim() == 5 else 1
    a.attr_sets = K
    keep = [uv_pos, uv_mask, mvp]
    a.pos_error_eps, a.aoi_cos_thresh, a.mask_thresh = float(pos_error_eps), float(aoi_cos_thresh), float(mask_thresh)
    a.use_depth_grad = 0 if depth_grad_thresh is None else 1
    a.depth_grad_thresh = 0.0 if depth_grad_thresh is None else float(depth_grad_thresh)
    a.first_view_dominate = int(bool(first_view_dominate))
    a.alpha = float(alpha)
    if view_weight is not None:
        vw = _view_weight_on(dev, view_weight)
        if vw.shape[0] != Nv:
            raise ValueError("view_weight must have one entry per view")
        keep.append(vw)
        a.view_weight = _native.ptr(vw)
    if view_masks is not None:
        vm = _f32c(view_masks)
        keep.append(vm)
        a.view_masks = _native.ptr(vm)
    udg = uaoi = None
    if want_per_view:
        udg = torch.empty((Nv, Hu, Wu), dtype=torch.float32, device=dev)
        uaoi = torch.empty((Nv, Hu, Wu), dtype=torch.float32, device=dev)
        a.uv_depth_grad, a.uv_aoi_cos = _native.ptr(udg), _native.ptr(uaoi)
    out_attr = out_any = None
    if accumulate_only:
        if accum is None:
            accum = torch.empty((Hu, Wu, 5), dtype=torch.float32, device=dev)
        else:
            if accum.shape != (Hu, Wu, 5) or accum.dtype != torch.float32 or not accum.is_contiguous():
                raise ValueError("accum must be a contiguous float32 tensor of shape [Huv, Wuv, 5]")
            a.accumulate = 1 if add_to_accum else 0
        a.accum = _native.ptr(accum)
    else:
        olds = [pre.uv_attr] * K if old_attrs is None else list(old_attrs)
        if len(olds) != K:
            raise ValueError(f"old_attrs must have one entry per image set ({K}), got {len(olds)}")
        outs = []
        for k, old in enumerate(olds):
            if old is not None:
                old = _f32c(old)
                if old.shape != (Hu, Wu, 3):
                    raise ValueError(f"existing texture must be {(Hu, Wu, 3)}, got {tuple(old.shape)}")
                keep.append(old)
            outs.append(torch.empty((Hu, Wu, 3), dtype=torch.float32, device=dev))
            if k == 0:
                a.old_attr, a.out_attr = _native.ptr(old), _native.ptr(outs[0])
            else:
                a.old_attr_more[k - 1], a.out_attr_more[k - 1] = _native.ptr(old), _native.ptr(outs[k])
        out_attr = outs if att.dim() == 5 else outs[0]
        out_any = torch.empty((Hu, Wu), dtype=torch.uint8, device=dev)
        a.out_valid_any = _native.ptr(out_any)
    if tex_range is not None:
        a.tex_lo, a.tex_hi = int(tex_range[0]), int(tex_range[1])
    c = ctx.ctx
    c.check(_native.lib().wr_uv_unproject(c.handle, ctypes.byref(a), c.stream()), "wr_uv_unproject")
    del keep
    return out_attr, (out_any.view(torch.bool) if out_any is not None else None), accum, udg, uaoi


def uv_finalize(ctx, accum: torch.Tensor, old_attr: Optional[torch.Tensor]):
    """accumulators (after an all-reduce) -> (stitched atlas [Huv,Wuv,3], valid_any [Huv,Wuv] bool)."""
    accum = _f32c(accum)
    Hu, Wu = accum.shape[0], accum.shape[1]
    old = _f32c(old_attr) if old_attr is not None else None
    out = torch.empty((Hu, Wu, 3), dtype=torch.float32, device=accum.device)
    any_ = torch.empty((Hu, Wu), dtype=torch.uint8, device=accum.device)
    c = ctx.ctx
    c.check(_native.lib().wr_uv_finalize(c.handle, _native.ptr(accum), _native.ptr(old), Hu, Wu, _native.ptr(out),
                                         _native.ptr(any_), c.stream()), "wr_uv_finalize")
    return out, any_.view(torch.bool)
