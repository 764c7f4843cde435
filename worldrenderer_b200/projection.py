"""CameraProjection: bake view images into the mesh's UV atlas.

Drop-in for mvadapter/utils/mesh_utils/projection.py of the reference (`CameraProjectionOutput`
:33-38, `CameraProjection.__init__` :42-52, `__call__` :54-204).  The call keeps the reference's
keyword surface; internally it is four launches groups on one stream:

    uv_precompute        wr_rasterize + wr_interpolate in UV space              (uv.py:24-53)
    view pass            wr_render (geometry, SimpleNormalization bg 1e2) + wr_view_prep
    unprojection         wr_uv_unproject: per texel, all views, validity, weights, blend, stitch
    (multi-GPU)          accumulators -> all_reduce(SUM) -> wr_uv_finalize      (parallel.py)

    post-processing      wr_uv_padding_sets / wr_poisson_blend (uv.py:426-461) when requested

`project_sets` bakes up to four image sets of one rig (rgb, base colour, ORM, ...) through the same launches; `__call__`
is its one-set case.

Options outside the path raise NotImplementedError instead of silently doing something else:
`warp_images=True`, `remove_bg=True` without a remover.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch

from .camera import Camera, get_camera
from .mesh import TexturedMesh
from .render import NVDiffRastContextWrapper
from .utils import IMAGE_TYPE, LIST_TYPE, image_to_tensor
from ._native import MAX_BAKE_SETS
from .blend import PoissonBlendingSolver
from .uv import UVPrecomputeOutput, atlas_postprocess, fused_unproject, fused_view_maps, uv_precompute


@dataclass
class CameraProjectionOutput:
    uv_proj: torch.Tensor
    uv_proj_mask: torch.Tensor
    uv_depth_grad: Optional[torch.Tensor]
    uv_aoi_cos: Optional[torch.Tensor]


class CameraProjection:
    def __init__(self, pb_backend: Optional[str] = None, bg_remover=None, device: str = "cuda",
                 context_type: str = "gl") -> None:
        # pb_backend names the reference's Poisson solver backend (blend.py:186-196); here every backend is the
        # native kernel.  None (not accepted by the reference) leaves the solver out for callers that never blend.
        self.pb_backend = pb_backend
        self.pb_solver = PoissonBlendingSolver(pb_backend, device) if pb_backend is not None else None
        self.ctx = NVDiffRastContextWrapper(device, context_type)
        self.bg_remover = bg_remover
        self.device = device
        self._pre_cache = None  # (key, tensors kept alive, uv_mask, uv_pos)

    def _uv_precompute(self, mesh: TexturedMesh, uv_size: int) -> UVPrecomputeOutput:
        """uv_precompute (uv.py:24-53) depends on the mesh and the atlas size only; the reference recomputes it on
        every call, here the last result is reused while the mesh tensors are unchanged (same storage, same
        version counter).  The texture is always taken fresh from the mesh."""
        srcs = (mesh.v_pos, mesh.t_pos_idx, mesh.v_tex, mesh.t_tex_idx)
        key = (int(uv_size),) + tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in srcs)
        if self._pre_cache is not None and self._pre_cache[0] == key:
            _, _, uv_mask, uv_pos = self._pre_cache
        else:
            pre = uv_precompute(self.ctx, mesh, height=uv_size, width=uv_size)
            uv_mask, uv_pos = pre.uv_mask, pre.uv_pos
            self._pre_cache = (key, srcs, uv_mask, uv_pos)  # srcs kept alive so a pointer cannot be recycled
        return UVPrecomputeOutput(height=uv_size, width=uv_size, uv_attr=mesh.texture, uv_mask=uv_mask, uv_pos=uv_pos)

    def __call__(
        self,
        images: IMAGE_TYPE,
        mesh: TexturedMesh,
        cam: Optional[Camera] = None,
        fovy_deg: Optional[LIST_TYPE] = None,
        masks: Optional[IMAGE_TYPE] = None,
        remove_bg: bool = False,
        c2w: Optional[torch.Tensor] = None,
        elevation_deg: Optional[LIST_TYPE] = None,
        distance: Optional[LIST_TYPE] = None,
        azimuth_deg: Optional[LIST_TYPE] = None,
        num_views: Optional[int] = None,
        uv_size: int = 2048,
        warp_images: bool = False,
        images_background: Optional[float] = None,
        iou_rejection_threshold: Optional[float] = 0.8,
        aoi_cos_valid_threshold: float = 0.3,
        depth_grad_dilation: int = 5,
        depth_grad_threshold: float = 0.1,
        uv_exp_blend_alpha: float = 6,
        uv_exp_blend_view_weight: Optional[torch.Tensor] = None,
        poisson_blending: bool = True,
        pb_num_iters: int = 1000,
        pb_keep_original_border: bool = True,
        from_scratch: bool = False,
        uv_padding: bool = True,
        return_uv_projection_mask: bool = False,
        return_dict: bool = False,
    ):
        return self.project_sets(
            [images], mesh, cam, fovy_deg=fovy_deg, masks=masks, remove_bg=remove_bg, c2w=c2w,
            elevation_deg=elevation_deg, distance=distance, azimuth_deg=azimuth_deg, num_views=num_views,
            uv_size=uv_size, warp_images=warp_images, images_background=images_background,
            iou_rejection_threshold=iou_rejection_threshold, aoi_cos_valid_threshold=aoi_cos_valid_threshold,
            depth_grad_dilation=depth_grad_dilation, depth_grad_threshold=depth_grad_threshold,
            uv_exp_blend_alpha=uv_exp_blend_alpha, uv_exp_blend_view_weight=uv_exp_blend_view_weight,
            poisson_blending=poisson_blending, pb_num_iters=pb_num_iters, pb_keep_original_border=pb_keep_original_border,
            from_scratch=from_scratch, uv_padding=uv_padding, return_uv_projection_mask=return_uv_projection_mask,
            return_dict=return_dict)[0]

    def project_sets(
        self,
        image_sets: Sequence[IMAGE_TYPE],
        mesh: TexturedMesh,
        cam: Optional[Camera] = None,
        fovy_deg: Optional[LIST_TYPE] = None,
        masks: Optional[IMAGE_TYPE] = None,
        remove_bg: bool = False,
        c2w: Optional[torch.Tensor] = None,
        elevation_deg: Optional[LIST_TYPE] = None,
        distance: Optional[LIST_TYPE] = None,
        azimuth_deg: Optional[LIST_TYPE] = None,
        num_views: Optional[int] = None,
        uv_size: int = 2048,
        warp_images: bool = False,
        images_background: Optional[float] = None,
        iou_rejection_threshold: Optional[float] = 0.8,
        aoi_cos_valid_threshold: float = 0.3,
        depth_grad_dilation: int = 5,
        depth_grad_threshold: float = 0.1,
        uv_exp_blend_alpha: float = 6,
        uv_exp_blend_view_weight: Optional[torch.Tensor] = None,
        poisson_blending: bool = True,
        pb_num_iters: int = 1000,
        pb_keep_original_border: bool = True,
        from_scratch: bool = False,
        uv_padding: bool = True,
        return_uv_projection_mask: bool = False,
        return_dict: bool = False,
        textures: Optional[Sequence[Optional[torch.Tensor]]] = None,
    ) -> List:
        """Bakes 1 to 4 image sets of one camera rig in one pass, e.g. the rgb, base colour and ORM views of a capture.

        Every set is what `__call__` takes as `images` and must come out as [Nv,H,W,3], all of the same shape.  The
        keywords are those of `__call__` and apply to every set; masks, cameras and thresholds are shared.  `textures`
        is None (every set is stitched with mesh.texture) or one entry per set: the existing [uv,uv,3] atlas of that
        set, or None.  The view pass, the geometry half of the unprojection and the jump flood of every seam padding
        run once for all sets; each set adds only its colour taps, its sums and the fills of its paddings.

        Returns a list of K results.  Result k is, bit for bit, what `__call__` returns for images `image_sets[k]` on
        a mesh whose texture is `textures[k]`: a tensor, a tuple or a CameraProjectionOutput.  The mask and the
        per-view `uv_depth_grad` / `uv_aoi_cos` of `return_dict` do not depend on the images: the K results share
        one tensor object for each.  The IoU rejection depends on the masks only: it returns [None] * K."""
        if poisson_blending:
            assert uv_padding  # uv.py:427
            if self.pb_solver is None:
                raise ValueError("poisson_blending=True needs a solver: construct CameraProjection with pb_backend")
        if warp_images:
            raise NotImplementedError("warp_images=True (reference warp.py) is outside the scope of worldrenderer_b200")

        image_sets = list(image_sets)
        K = len(image_sets)
        if not 1 <= K <= MAX_BAKE_SETS:
            raise ValueError(f"project_sets bakes 1 to {MAX_BAKE_SETS} image sets, got {K}")
        if textures is None:
            textures = [mesh.texture] * K
        elif len(textures) != K:
            raise ValueError(f"textures must have one entry per image set ({K}), got {len(textures)}")
        sets_pt = [image_to_tensor(images, device=self.device) for images in image_sets]
        images_pt = sets_pt[0]
        assert images_pt.ndim == 4
        Nv, H, W, C = images_pt.shape
        if C != 3:
            raise ValueError(f"images must have 3 channels to be baked into the RGB atlas, got {C}")
        for k, x in enumerate(sets_pt[1:], 1):
            if x.shape != images_pt.shape:
                raise ValueError(f"image set {k} has shape {tuple(x.shape)}, set 0 has {tuple(images_pt.shape)}")

        if masks is not None:
            masks_pt = image_to_tensor(masks, device=self.device)
        elif remove_bg:
            assert self.bg_remover is not None
            masks_pt = self.bg_remover(images_pt)
        else:
            masks_pt = None
        if masks_pt is not None and masks_pt.ndim == 4:
            masks_pt = masks_pt.mean(-1)

        if cam is None:
            cam = get_camera(elevation_deg, distance, fovy_deg, azimuth_deg, num_views, c2w, aspect_wh=W / H,
                             device=self.device)

        pre = self._uv_precompute(mesh, uv_size)
        view_mask, geo_map, attr_map = fused_view_maps(self.ctx, mesh, cam, sets_pt, H, W, int(depth_grad_dilation))

        if masks_pt is not None and iou_rejection_threshold is not None:  # projection.py:125-138
            given = (masks_pt > 0.5).float()
            rendered = view_mask.float()
            inter = given * rendered
            union = given + rendered - inter
            iou = inter.sum((1, 2)) / union.sum((1, 2))
            iou_min = iou.min()
            print(f"Debug: Per view IoU: {iou.tolist()}")
            if iou_min < iou_rejection_threshold:
                print(f"Warning: Minimum view IoU {iou_min} below threshold {iou_rejection_threshold}, "
                      "skipping camera projection!")
                return [None] * K

        if masks_pt is None:
            print("No view mask provided for UV blending, using all valid pixels")
        blends, valid_any, _, uv_depth_grad, uv_aoi_cos = fused_unproject(
            self.ctx, pre, cam, H, W, geo_map, attr_map, view_masks=masks_pt,
            aoi_cos_thresh=aoi_cos_valid_threshold, depth_grad_thresh=depth_grad_threshold,
            alpha=uv_exp_blend_alpha, view_weight=uv_exp_blend_view_weight, want_per_view=return_dict,
            old_attrs=textures)
        if poisson_blending or uv_padding:  # uv.py:426-461
            blends = atlas_postprocess(None, blends, valid_any, pre, do_uv_padding=uv_padding,
                                       pad_unseen_area=from_scratch, poisson_blending=poisson_blending,
                                       pb_solver=self.pb_solver, pb_num_iters=pb_num_iters,
                                       pb_keep_original_border=pb_keep_original_border, old_attrs=textures)

        if return_dict:
            return [CameraProjectionOutput(uv_proj=blend, uv_proj_mask=valid_any, uv_depth_grad=uv_depth_grad,
                                           uv_aoi_cos=uv_aoi_cos) for blend in blends]
        if return_uv_projection_mask:
            return [(blend, valid_any) for blend in blends]
        return blends
