"""render() and the rasterizer context of the geometry path, backed by libwr_b200 (sm_100a).

Drop-in for mvadapter/utils/mesh_utils/render.py of the reference: `RenderOutput` (:20-27),
`NVDiffRastContextWrapper` (:30-149, the operator boundary the reference fills with nvdiffrast),
the depth normalisers (:152-217) and `render` (:220-286).

`render()` does not compose the operators the way the reference does (clip transform -> rasterize ->
3-4 interpolate calls -> ~15 element-wise torch kernels); it issues ONE fused pipeline,
`wr_render` (csrc/raster.cu + csrc/shade.cu): vertices are transformed and snapped once per view,
triangles are set up / rasterised into an L2-resident packed depth+id buffer, and one shading pass
writes mask, position, view depth, normal (and optionally the textured attribute map) directly.
The operators remain available on the context for callers that use them one by one.
"""
from __future__ import annotations

import ctypes
from abc import ABC, abstractmethod
from dataclasses import dataclass
from typing import Optional, Union

import torch
import torch.nn.functional as F

from . import _native
from .camera import Camera
from .mesh import TexturedMesh

_FILTER_MODES = {"nearest": 0, "linear": 1, "auto": 1}
_BOUNDARY_MODES = {"wrap": 0, "clamp": 1, "zero": 2}
# render(output_dtype=...): element type of the pos / depth / normal / tangent / attr maps (wr_render_args.out_dtype)
_OUTPUT_DTYPES = {torch.float32: _native.DTYPE_F32, torch.float16: _native.DTYPE_F16,
                  torch.bfloat16: _native.DTYPE_BF16}


@dataclass
class RenderOutput:
    attr: Optional[torch.Tensor] = None
    mask: Optional[torch.Tensor] = None
    depth: Optional[torch.Tensor] = None
    normal: Optional[torch.Tensor] = None
    tangent: Optional[torch.Tensor] = None
    pos: Optional[torch.Tensor] = None


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.float32).contiguous()


def _i32c(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.int32).contiguous()


def _no_autograd(what: str, *tensors) -> None:
    """The reference is differentiable through nvdiffrast; these kernels are forward-only.  A caller that optimises
    through the result must hear about it instead of silently getting no gradient."""
    if torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad for t in tensors):
        raise NotImplementedError(
            f"{what}: an input requires grad, but worldrenderer_b200 is forward-only (no backward kernels). "
            "Detach the inputs or call under torch.no_grad().")


class NVDiffRastContextWrapper:
    """Same constructor and methods as the reference wrapper (render.py:30-149).

    `context_type` "gl" and "cuda" both select the sm_100a software rasterizer of this package (there is
    no OpenGL path); anything else raises NotImplementedError like the reference.  `.ctx` is the native
    context object (the reference passes `ctx.ctx` around, projection.py:152-153).
    """

    def __init__(self, device: str, context_type: str = "gl"):
        if context_type not in ("gl", "cuda"):
            raise NotImplementedError
        self.ctx = _native.NativeContext(device)
        self.device = self.ctx.device
        self.context_type = context_type

    # ---- helpers -------------------------------------------------------------------------------
    def _check_device(self, *tensors: torch.Tensor) -> None:
        for t in tensors:
            if t is not None and t.device != self.device:
                raise RuntimeError(f"tensor on {t.device}, context on {self.device}: all inputs must live on the "
                                   "context's CUDA device (there is no CPU path)")

    # ---- dr.rasterize --------------------------------------------------------------------------
    def rasterize(self, pos, tri, resolution, ranges=None, grad_db=True):
        """pos [B,V,4] (instanced) or [V,4] + ranges [B,2] on the CPU (range mode); tri [F,3];
        resolution (H, W).  Returns (rast [B,H,W,4] = (u, v, z/w, triangle_id + 1), rast_db [B,H,W,0]).
        Image-space derivatives are not produced (the geometry path never reads them)."""
        rast, _ = self.rasterize_with_ids(pos, tri, resolution, ranges, want_ids=False)
        return rast, rast.new_zeros(*rast.shape[:-1], 0)

    def rasterize_with_ids(self, pos, tri, resolution, ranges=None, want_ids=True):
        _no_autograd("rasterize()", pos)
        pos = _f32c(pos)
        tri = _i32c(tri)
        self._check_device(pos, tri)
        H, W = int(resolution[0]), int(resolution[1])
        if tri.ndim != 2 or tri.shape[1] != 3:
            raise ValueError("tri must have shape [num_triangles, 3]")
        ranges_host = None
        if pos.ndim == 3:
            if pos.shape[2] != 4:
                raise ValueError("pos must have shape [minibatch_size, num_vertices, 4]")
            B, V, batched = pos.shape[0], pos.shape[1], 1
        elif pos.ndim == 2:
            if pos.shape[1] != 4:
                raise ValueError("pos must have shape [num_vertices, 4]")
            if ranges is None:
                raise ValueError("range mode (2-D pos) needs a ranges tensor")
            if ranges.device.type != "cpu":
                raise ValueError("ranges must reside in CPU memory")
            ranges_host = ranges.to(torch.int32).contiguous()
            if ranges_host.ndim != 2 or ranges_host.shape[1] != 2:
                raise ValueError("ranges must have shape [minibatch_size, 2]")
            B, V, batched = ranges_host.shape[0], pos.shape[0], 0
        else:
            raise ValueError("pos must be 2-D (range mode) or 3-D (instanced mode)")
        rast = torch.empty((B, H, W, 4), dtype=torch.float32, device=self.device)
        ids = torch.empty((B, H, W), dtype=torch.int32, device=self.device) if want_ids else None
        c = self.ctx
        status = _native.lib().wr_rasterize(
            c.handle, _native.ptr(pos), B, V, batched, _native.ptr(tri), tri.shape[0],
            ranges_host.data_ptr() if ranges_host is not None else None, H, W,
            _native.ptr(rast), _native.ptr(ids), c.stream())
        c.check(status, "wr_rasterize")
        return rast, ids

    # ---- dr.interpolate ------------------------------------------------------------------------
    def interpolate(self, attr, rast, tri, rast_db=None, diff_attrs=None):
        """attr [1|B,V,A] or [V,A]; rast from rasterize(); tri [F,3] -> ([B,H,W,A], empty [B,H,W,0])."""
        if rast_db is not None and diff_attrs is not None:
            raise NotImplementedError("attribute derivatives (rast_db / diff_attrs) are outside the geometry path")
        _no_autograd("interpolate()", attr, rast)
        attr = _f32c(attr)
        tri = _i32c(tri)
        rast = _f32c(rast)
        self._check_device(attr, rast, tri)
        if attr.ndim == 2:
            attr = attr[None]
        B, H, W, _ = rast.shape
        if attr.shape[0] not in (1, B):
            raise ValueError("attr minibatch must be 1 or match rast")
        A = attr.shape[2]
        out = torch.empty((B, H, W, A), dtype=torch.float32, device=self.device)
        c = self.ctx
        status = _native.lib().wr_interpolate(c.handle, _native.ptr(attr), attr.shape[0], attr.shape[1], A,
                                              _native.ptr(rast), B, H, W, _native.ptr(tri), tri.shape[0],
                                              _native.ptr(out), c.stream())
        c.check(status, "wr_interpolate")
        return out, out.new_zeros(B, H, W, 0)

    # ---- dr.texture ----------------------------------------------------------------------------
    def texture(self, tex, uv, uv_da=None, mip_level_bias=None, mip=None, filter_mode="auto",
                boundary_mode="wrap", max_mip_level=None):
        """2-D texture fetch, 'nearest' / 'linear' ('auto' = 'linear' without derivatives), boundary
        'wrap' / 'clamp' / 'zero'.  Mip-mapped modes and cube maps are not part of the geometry path."""
        if uv_da is not None or mip_level_bias is not None or mip is not None:
            raise NotImplementedError("mip-mapped texture sampling is outside the geometry path")
        if filter_mode not in _FILTER_MODES or boundary_mode not in _BOUNDARY_MODES:
            raise NotImplementedError(f"texture: filter_mode={filter_mode!r}, boundary_mode={boundary_mode!r}")
        _no_autograd("texture()", tex, uv)
        tex = _f32c(tex)
        uv = _f32c(uv)
        self._check_device(tex, uv)
        if tex.ndim != 4 or uv.ndim != 4 or uv.shape[-1] != 2:
            raise ValueError("tex must be [minibatch, height, width, channels] and uv [minibatch, height, width, 2]")
        B, H, W, _ = uv.shape
        if tex.shape[0] not in (1, B):
            raise ValueError("tex minibatch must be 1 or match uv")
        out = torch.empty((B, H, W, tex.shape[3]), dtype=torch.float32, device=self.device)
        c = self.ctx
        status = _native.lib().wr_texture(c.handle, _native.ptr(tex), tex.shape[0], tex.shape[1], tex.shape[2],
                                          tex.shape[3], _native.ptr(uv), B, H, W, _FILTER_MODES[filter_mode],
                                          _BOUNDARY_MODES[boundary_mode], _native.ptr(out), c.stream())
        c.check(status, "wr_texture")
        return out

    def antialias(self, color, rast, pos, tri, topology_hash=None, pos_gradient_boost=1.0):
        raise NotImplementedError("antialias (render.py:122-149, off by default in render()) is outside the "
                                  "geometry path")


# ------------------------------------------------------------------------------------------------
# depth normalisation strategies (render.py:152-217).  Callable on tensors like the reference; the
# three known classes are also recognised by render() and folded into the shading kernels.
# ------------------------------------------------------------------------------------------------

class DepthNormalizationStrategy(ABC):
    @abstractmethod
    def __init__(self, *args, **kwargs):
        pass

    @abstractmethod
    def __call__(self, depth: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        pass


def _minmax_per_view(depth: torch.Tensor):
    flat = depth.reshape(depth.shape[0], -1)
    return flat.min(dim=-1)[0][:, None, None], flat.max(dim=-1)[0][:, None, None]


class DepthControlNetNormalization(DepthNormalizationStrategy):
    def __init__(self, far_clip: float = 0.25, near_clip: float = 1.0, bg_value: float = 0.0):
        self.far_clip = far_clip
        self.near_clip = near_clip
        self.bg_value = bg_value

    def __call__(self, depth: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        lo, hi = _minmax_per_view(depth)
        depth = 1.0 - ((depth - lo) / (hi - lo + 1e-5)).clamp(0.0, 1.0)
        depth = depth * (self.near_clip - self.far_clip) + self.far_clip
        depth[~mask] = self.bg_value
        return depth


class Zero123PlusPlusNormalization(DepthNormalizationStrategy):
    def __init__(self, bg_value: float = 0.8):
        self.bg_value = bg_value

    def __call__(self, depth: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        lo, hi = _minmax_per_view(depth)
        depth = ((depth - lo) / (hi - lo + 1e-5)).clamp(0.0, 1.0)
        depth[~mask] = self.bg_value
        return depth


class SimpleNormalization(DepthNormalizationStrategy):
    def __init__(self, scale: float = 1.0, offset: float = -1.0, clamp: bool = True, bg_value: float = 1.0):
        self.scale = scale
        self.offset = offset
        self.clamp = clamp
        self.bg_value = bg_value

    def __call__(self, depth: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
        depth = depth * self.scale + self.offset
        if self.clamp:
            depth = depth.clamp(0.0, 1.0)
        depth[~mask] = self.bg_value
        return depth


def _depth_kernel_params(strategy):
    """(mode, p0, p1, clamp, bg, post) -- `post` is a callable to run on tensors for unknown strategies."""
    if strategy is None:
        return _native.DEPTH_NONE, 0.0, 0.0, 0, 0.0, None
    kind = type(strategy)
    if kind is DepthControlNetNormalization:
        return (_native.DEPTH_CONTROLNET, float(strategy.far_clip), float(strategy.near_clip - strategy.far_clip),
                0, float(strategy.bg_value), None)
    if kind is Zero123PlusPlusNormalization:
        return _native.DEPTH_ZERO123PP, 0.0, 0.0, 0, float(strategy.bg_value), None
    if kind is SimpleNormalization:
        return (_native.DEPTH_SIMPLE, float(strategy.scale), float(strategy.offset), int(bool(strategy.clamp)),
                float(strategy.bg_value), None)
    # user-defined strategy (or a subclass that may override __call__): kernel fills the background with the
    # per-view minimum (render.py:250-255) and the strategy runs on the tensors
    return _native.DEPTH_NONE, 0.0, 0.0, 0, 0.0, strategy


def _background_triplet(value, what: str):
    if isinstance(value, torch.Tensor):
        flat = value.detach().reshape(-1).to("cpu", torch.float32)
        if flat.numel() == 1:
            return [float(flat[0])] * 3
        if flat.numel() == 3:
            return [float(x) for x in flat]
        return None  # per-pixel background tensor: handled with torch indexing by the caller
    return [float(value)] * 3


def render_geometry_raw(ctx: NVDiffRastContextWrapper, mesh: TexturedMesh, cam: Camera, height: int, width: int, *,
                        want_pos=True, want_depth=True, want_normal=True, want_attr=False, want_tri_id=False,
                        want_rast=False, want_tangent=False, tangent_background=0.0, want_geo=False,
                        depth_normalization_strategy=None, normal_background=0.0,
                        attr_background=0.5, texture_override=None, texture_filter_mode="linear", out_buffers=None,
                        raster_done_event=None, output_dtype=torch.float32):
    """One wr_render call.  Returns a dict of tensors; `mask` is uint8 0/1 (callers view it as bool).
    out_buffers: optional {name: preallocated contiguous tensor} written instead of fresh allocations (RenderGraph
    renders groups of views into slices of one output).  raster_done_event: a recorded-at-least-once torch.cuda.Event,
    re-recorded by the library between the raster passes and the shading pass (wr_render_args.raster_done_event).
    output_dtype: float32, float16 or bfloat16 for pos / depth / normal / tangent / attr (geo stays float32); the
    result equals the float32 maps cast to it."""
    if output_dtype not in _OUTPUT_DTYPES:
        raise ValueError(f"output_dtype must be torch.float32, torch.float16 or torch.bfloat16, got {output_dtype!r}")
    dev = ctx.device

    def _new(name, shape, dtype):
        buf = None if out_buffers is None else out_buffers.get(name)
        if buf is None:
            return torch.empty(shape, dtype=dtype, device=dev)
        if buf.dtype == torch.bool and dtype == torch.uint8:
            buf = buf.view(torch.uint8)
        if tuple(buf.shape) != tuple(shape) or buf.dtype != dtype or buf.device != dev or not buf.is_contiguous():
            raise ValueError(f"out_buffers[{name!r}]: expected a contiguous {dtype} tensor of shape {tuple(shape)} on {dev}")
        return buf

    _no_autograd("render()", mesh.v_pos, cam.mvp_mtx, cam.w2c, mesh.texture if want_attr else None, texture_override)
    v_pos = _f32c(mesh.v_pos)
    tri = mesh.index_i32("t_pos_idx")
    mvp = _f32c(cam.mvp_mtx)
    w2c = _f32c(cam.w2c)
    ctx._check_device(v_pos, tri, mvp, w2c)
    B, H, W = mvp.shape[0], int(height), int(width)
    post = _depth_kernel_params(depth_normalization_strategy)[5] if want_depth else None
    nbg = _background_triplet(normal_background, "normal_background") if (want_normal or want_geo) else None
    tbg = _background_triplet(tangent_background, "tangent_background") if want_tangent else None
    abg_is_tensor = want_attr and isinstance(attr_background, torch.Tensor) and attr_background.numel() != 1
    # A map that torch post-processes (user-defined depth strategy, per-pixel background tensor) is computed in float32
    # and cast once at the end, so that the result still equals the float32 render cast to output_dtype.
    torch_tail = post is not None or (want_normal and nbg is None) or (want_tangent and tbg is None) or abg_is_tensor
    map_dtype = torch.float32 if torch_tail else output_dtype

    def _map(name, shape):
        if map_dtype != output_dtype:   # not the caller's buffer: the cast at the end allocates the result
            return torch.empty(shape, dtype=map_dtype, device=dev)
        return _new(name, shape, map_dtype)

    a = _native.RenderArgs()
    a.out_dtype = _OUTPUT_DTYPES[map_dtype]
    keep = [v_pos, tri, mvp, w2c]
    a.v_pos, a.tri, a.V, a.F = _native.ptr(v_pos), _native.ptr(tri), v_pos.shape[0], tri.shape[0]
    a.mvp, a.w2c, a.B, a.H, a.W = _native.ptr(mvp), _native.ptr(w2c), B, H, W
    out = {}
    out["mask"] = _new("mask", (B, H, W), torch.uint8)
    a.out_mask = _native.ptr(out["mask"])
    if want_pos:
        out["pos"] = _map("pos", (B, H, W, 3))
        a.out_pos = _native.ptr(out["pos"])
    if want_depth:
        mode, p0, p1, clamp, bg, _ = _depth_kernel_params(depth_normalization_strategy)
        a.depth_mode, a.depth_p0, a.depth_p1, a.depth_clamp, a.depth_bg = mode, p0, p1, clamp, bg
        out["depth"] = _map("depth", (B, H, W))
        a.out_depth = _native.ptr(out["depth"])
    if want_geo or want_normal or want_tangent:
        # the kernel reads tri_nrm[3 * id] for every covered pixel: one row per face of t_pos_idx, or an
        # out-of-bounds device read
        if mesh.index_i32("stitched_t_pos_idx").shape[0] != tri.shape[0]:
            raise ValueError("stitched_t_pos_idx must have one row per face of t_pos_idx")
    if want_geo:  # bake view map (pos.xyz, aoi_cos): needs the vertex normals but writes no normal map
        v_nrm = _f32c(mesh.v_nrm)
        tri_n = mesh.index_i32("stitched_t_pos_idx")
        ctx._check_device(v_nrm, tri_n)
        keep += [v_nrm, tri_n]
        same_faces = mesh._stitched_t_pos_idx is None or mesh._stitched_t_pos_idx is mesh.t_pos_idx
        a.v_nrm, a.Vn = _native.ptr(v_nrm), v_nrm.shape[0]
        a.tri_nrm = None if same_faces else _native.ptr(tri_n)
        a.normal_bg = (ctypes.c_float * 3)(*(nbg or [0.0, 0.0, 0.0]))
        out["geo"] = _new("geo", (B, H, W, 4), torch.float32)
        a.out_geo = _native.ptr(out["geo"])
    nbg_tensor = None
    if want_normal:
        v_nrm = _f32c(mesh.v_nrm)
        tri_n = mesh.index_i32("stitched_t_pos_idx")
        ctx._check_device(v_nrm, tri_n)
        keep += [v_nrm, tri_n]
        # a mesh that was not stitched shares one index tensor: the kernel then reuses the position indices
        same_faces = mesh._stitched_t_pos_idx is None or mesh._stitched_t_pos_idx is mesh.t_pos_idx
        a.v_nrm, a.Vn = _native.ptr(v_nrm), v_nrm.shape[0]
        a.tri_nrm = None if same_faces else _native.ptr(tri_n)
        if nbg is None:
            nbg_tensor, nbg = normal_background, [0.0, 0.0, 0.0]
        a.normal_bg = (ctypes.c_float * 3)(*nbg)
        out["normal"] = _map("normal", (B, H, W, 3))
        a.out_normal = _native.ptr(out["normal"])
    tbg_tensor = None
    if want_tangent:
        v_tang = _f32c(mesh.v_tang)
        tri_n = mesh.index_i32("stitched_t_pos_idx")
        v_nrm_for_count = _f32c(mesh.v_nrm)
        if v_tang.shape != v_nrm_for_count.shape:
            raise ValueError("v_tang must have one row per (stitched) vertex, like v_nrm")
        ctx._check_device(v_tang, tri_n)
        keep += [v_tang, tri_n]
        same_faces = mesh._stitched_t_pos_idx is None or mesh._stitched_t_pos_idx is mesh.t_pos_idx
        a.v_tang, a.Vn = _native.ptr(v_tang), v_tang.shape[0]
        a.tri_nrm = None if same_faces else _native.ptr(tri_n)
        if tbg is None:
            tbg_tensor, tbg = tangent_background, [0.0, 0.0, 0.0]
        a.tangent_bg = (ctypes.c_float * 3)(*tbg)
        out["tangent"] = _map("tangent", (B, H, W, 3))
        a.out_tangent = _native.ptr(out["tangent"])
    abg_tensor = None
    if want_attr:
        tex = texture_override if texture_override is not None else mesh.texture
        if tex is None or mesh.v_tex is None or mesh.t_tex_idx is None:
            raise ValueError("render_attr=True needs mesh.v_tex, mesh.t_tex_idx and a texture")
        if texture_filter_mode not in _FILTER_MODES:
            raise NotImplementedError(f"texture_filter_mode={texture_filter_mode!r}")
        tex = _f32c(tex)
        v_tex = _f32c(mesh.v_tex)
        tri_t = mesh.index_i32("t_tex_idx")
        ctx._check_device(tex, v_tex, tri_t)
        keep += [tex, v_tex, tri_t]
        a.v_tex, a.tri_tex, a.Vt = _native.ptr(v_tex), _native.ptr(tri_t), v_tex.shape[0]
        a.texture, a.TH, a.TW, a.TC = _native.ptr(tex), tex.shape[0], tex.shape[1], tex.shape[2]
        a.tex_filter = _FILTER_MODES[texture_filter_mode]
        if abg_is_tensor:
            abg_tensor, a.attr_bg = attr_background, 0.0
        else:
            a.attr_bg = float(attr_background)
        out["attr"] = _map("attr", (B, H, W, tex.shape[2]))
        a.out_attr = _native.ptr(out["attr"])
    if want_tri_id:
        out["tri_id"] = _new("tri_id", (B, H, W), torch.int32)
        a.out_tri_id = _native.ptr(out["tri_id"])
    if want_rast:
        out["rast"] = _new("rast", (B, H, W, 4), torch.float32)
        a.out_rast = _native.ptr(out["rast"])
    if raster_done_event is not None:
        handle = int(raster_done_event.cuda_event)
        if not handle:
            raise ValueError("raster_done_event must have been recorded once (torch creates the CUDA event lazily)")
        a.raster_done_event = handle
    c = ctx.ctx
    c.check(_native.lib().wr_render(c.handle, ctypes.byref(a), c.stream()), "wr_render")
    del keep
    mask_bool = out["mask"].view(torch.bool)
    if post is not None:
        out["depth"] = post(out["depth"], mask_bool)
    if tbg_tensor is not None:
        out["tangent"][~mask_bool] = tbg_tensor.to(out["tangent"])
    if nbg_tensor is not None:  # tensor-valued background, torch indexing like the reference (render.py:277)
        out["normal"][~mask_bool] = nbg_tensor.to(out["normal"])
    if abg_tensor is not None:
        bgv = torch.ones_like(out["attr"]) * abg_tensor.to(out["attr"])
        out["attr"] = torch.where(mask_bool[..., None], out["attr"], bgv)
    if map_dtype != output_dtype:
        for name in ("pos", "depth", "normal", "tangent", "attr"):
            if name in out:
                out[name] = out[name].to(output_dtype)
    out["mask"] = mask_bool
    return out


def render(
    ctx: NVDiffRastContextWrapper,
    mesh: TexturedMesh,
    cam: Camera,
    height: int,
    width: int,
    render_attr: bool = True,
    render_depth: bool = True,
    render_normal: bool = True,
    render_tangent: bool = False,
    depth_normalization_strategy: DepthNormalizationStrategy = DepthControlNetNormalization(),
    attr_background: Union[float, torch.Tensor] = 0.5,
    antialias_attr=False,
    normal_background: Union[float, torch.Tensor] = 0.0,
    tangent_background: Union[float, torch.Tensor] = 0.0,
    texture_override=None,
    texture_filter_mode: str = "linear",
    output_dtype: torch.dtype = torch.float32,
    _out_buffers=None,
    _raster_done_event=None,
) -> RenderOutput:
    """Same signature and outputs as the reference render() (render.py:220-286), plus `output_dtype`.

    output_dtype: torch.float32 (default), torch.float16 or torch.bfloat16 -- element type of pos, depth, normal,
    tangent and attr (mask stays bool).  Everything is computed in float32 and rounded to nearest even when stored,
    so the maps equal `render(...)` with each float map cast by `.to(output_dtype)` (NaN tangents stay NaN; their bit
    pattern may differ).  Half the bytes of float32 to write, keep and copy.  Anything else raises ValueError."""
    if antialias_attr:
        raise NotImplementedError("antialias_attr=True (dr.antialias) is outside the geometry path")
    raw = render_geometry_raw(
        ctx, mesh, cam, height, width, want_pos=True, want_depth=render_depth, want_normal=render_normal,
        want_attr=render_attr, want_tangent=render_tangent, tangent_background=tangent_background,
        depth_normalization_strategy=depth_normalization_strategy,
        normal_background=normal_background, attr_background=attr_background, texture_override=texture_override,
        texture_filter_mode=texture_filter_mode, out_buffers=_out_buffers,
        raster_done_event=_raster_done_event, output_dtype=output_dtype)
    out = RenderOutput(mask=raw["mask"], pos=raw["pos"], depth=raw.get("depth"), attr=raw.get("attr"),
                       normal=raw.get("normal"))
    out.tangent = raw.get("tangent")
    return out
