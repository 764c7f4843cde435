"""ctypes binding of libwr_b200.so (include/wr_b200.h).

This is the only door from Python to the CUDA kernels.  There is no fallback of any kind: if the
library is missing, was built for another architecture, or a call returns a non-zero status, a
RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# WR_B200_LIB: measurement aid only (time two builds of this library side by side, e.g. before and after a change);
# it must still point at a build of this library -- there is no other implementation.
LIB_PATH = os.environ.get("WR_B200_LIB") or os.path.join(_HERE, "lib", "libwr_b200.so")

_c_f32p = ctypes.c_void_p
_LIB: Optional[ctypes.CDLL] = None

# every symbol include/wr_b200.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "wr_status_string", "wr_ctx_last_error", "wr_version", "wr_ctx_create", "wr_ctx_destroy",
    "wr_ctx_scratch_bytes", "wr_ctx_profile", "wr_ctx_profile_read", "wr_ctx_profile_stage_name", "wr_rasterize", "wr_interpolate", "wr_texture", "wr_vertex_normals",
    "wr_vertex_tangents", "wr_tangent_space_normals",
    "wr_render", "wr_view_prep", "wr_uv_unproject", "wr_uv_finalize", "wr_grid_sample", "wr_uv_reduce_finalize_p2p",
    "wr_poisson_blend", "wr_poisson_band_layout", "wr_poisson_band_step", "wr_inpaint_u8", "wr_uv_padding", "wr_view_scores",
]

DEPTH_NONE, DEPTH_CONTROLNET, DEPTH_ZERO123PP, DEPTH_SIMPLE = 0, 1, 2, 3


class RenderArgs(ctypes.Structure):
    _fields_ = [
        ("v_pos", ctypes.c_void_p), ("tri", ctypes.c_void_p), ("V", ctypes.c_int), ("F", ctypes.c_int),
        ("v_nrm", ctypes.c_void_p), ("tri_nrm", ctypes.c_void_p), ("Vn", ctypes.c_int),
        ("v_tang", ctypes.c_void_p),
        ("v_tex", ctypes.c_void_p), ("tri_tex", ctypes.c_void_p), ("Vt", ctypes.c_int),
        ("texture", ctypes.c_void_p), ("TH", ctypes.c_int), ("TW", ctypes.c_int), ("TC", ctypes.c_int),
        ("tex_filter", ctypes.c_int),
        ("mvp", ctypes.c_void_p), ("w2c", ctypes.c_void_p),
        ("B", ctypes.c_int), ("H", ctypes.c_int), ("W", ctypes.c_int),
        ("depth_mode", ctypes.c_int), ("depth_p0", ctypes.c_float), ("depth_p1", ctypes.c_float),
        ("depth_clamp", ctypes.c_int), ("depth_bg", ctypes.c_float),
        ("normal_bg", ctypes.c_float * 3), ("tangent_bg", ctypes.c_float * 3), ("attr_bg", ctypes.c_float),
        ("out_mask", ctypes.c_void_p), ("out_pos", ctypes.c_void_p), ("out_depth", ctypes.c_void_p),
        ("out_normal", ctypes.c_void_p), ("out_tangent", ctypes.c_void_p), ("out_geo", ctypes.c_void_p), ("out_attr", ctypes.c_void_p), ("out_tri_id", ctypes.c_void_p),
        ("out_rast", ctypes.c_void_p),
        ("raster_done_event", ctypes.c_void_p),
    ]


class UnprojectArgs(ctypes.Structure):
    _fields_ = [
        ("uv_pos", ctypes.c_void_p), ("uv_mask", ctypes.c_void_p), ("Hu", ctypes.c_int), ("Wu", ctypes.c_int),
        ("mvp", ctypes.c_void_p), ("Nv", ctypes.c_int), ("H", ctypes.c_int), ("W", ctypes.c_int),
        ("geo_map", ctypes.c_void_p), ("attr_map", ctypes.c_void_p), ("view_masks", ctypes.c_void_p),
        ("pos_error_eps", ctypes.c_float), ("aoi_cos_thresh", ctypes.c_float), ("mask_thresh", ctypes.c_float),
        ("depth_grad_thresh", ctypes.c_float), ("use_depth_grad", ctypes.c_int),
        ("first_view_dominate", ctypes.c_int),
        ("alpha", ctypes.c_float), ("view_weight", ctypes.c_void_p),
        ("accum", ctypes.c_void_p), ("accumulate", ctypes.c_int),
        ("uv_pos_ndc", ctypes.c_void_p), ("uv_pos_proj", ctypes.c_void_p), ("uv_pos_error", ctypes.c_void_p),
        ("uv_aoi_cos", ctypes.c_void_p), ("uv_depth_grad", ctypes.c_void_p), ("uv_attr_proj", ctypes.c_void_p),
        ("uv_mask_proj", ctypes.c_void_p), ("uv_valid", ctypes.c_void_p), ("uv_weight", ctypes.c_void_p),
        ("old_attr", ctypes.c_void_p), ("out_attr", ctypes.c_void_p), ("out_valid_any", ctypes.c_void_p),
        ("tex_lo", ctypes.c_longlong), ("tex_hi", ctypes.c_longlong),
    ]


ABI_VERSION = 103   # include/wr_b200.h WR_B200_ABI_VERSION (the ctypes structures below mirror that header)
MAX_P2P_RANKS = 16


class P2PReduceArgs(ctypes.Structure):
    _fields_ = [
        ("accum", ctypes.c_void_p * MAX_P2P_RANKS), ("out_attr", ctypes.c_void_p * MAX_P2P_RANKS),
        ("out_valid", ctypes.c_void_p * MAX_P2P_RANKS), ("old_attr", ctypes.c_void_p),
        ("world", ctypes.c_int), ("rank", ctypes.c_int), ("Hu", ctypes.c_int), ("Wu", ctypes.c_int),
        ("mc_accum", ctypes.c_void_p), ("mc_attr", ctypes.c_void_p), ("mc_valid", ctypes.c_void_p),
        ("max_blocks", ctypes.c_int),
        ("tex_lo", ctypes.c_longlong), ("tex_hi", ctypes.c_longlong),
    ]


class PoissonBandArgs(ctypes.Structure):
    _fields_ = [
        ("src", ctypes.c_void_p), ("mask", ctypes.c_void_p), ("tgt", ctypes.c_void_p),
        ("H", ctypes.c_int), ("W", ctypes.c_int), ("C", ctypes.c_int),
        ("num_iters", ctypes.c_int), ("grad_mode", ctypes.c_int), ("world", ctypes.c_int), ("rank", ctypes.c_int),
        ("xa", ctypes.c_void_p * MAX_P2P_RANKS), ("xb", ctypes.c_void_p * MAX_P2P_RANKS),
        ("out", ctypes.c_void_p * MAX_P2P_RANKS), ("b", ctypes.c_void_p), ("m", ctypes.c_void_p),
        ("step", ctypes.c_int),
    ]


def lib() -> ctypes.CDLL:
    """Loads libwr_b200.so; raises if it has not been built (python -m worldrenderer_b200.build_native)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m worldrenderer_b200.build_native` "
            "(nvcc, sm_100a). worldrenderer_b200 has no CPU or PyTorch fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, ci = ctypes.c_void_p, ctypes.c_int
    L.wr_status_string.restype = ctypes.c_char_p
    L.wr_status_string.argtypes = [ci]
    L.wr_ctx_last_error.restype = ctypes.c_char_p
    L.wr_ctx_last_error.argtypes = [vp]
    L.wr_version.restype = ci
    L.wr_ctx_create.restype = ci
    L.wr_ctx_create.argtypes = [ci, ctypes.POINTER(vp)]
    L.wr_ctx_destroy.restype = None
    L.wr_ctx_destroy.argtypes = [vp]
    L.wr_ctx_scratch_bytes.restype = ctypes.c_uint64
    L.wr_ctx_scratch_bytes.argtypes = [vp]
    L.wr_ctx_profile.restype = ci
    L.wr_ctx_profile.argtypes = [vp, ci]
    L.wr_ctx_profile_read.restype = ci
    L.wr_ctx_profile_read.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ci]
    L.wr_ctx_profile_stage_name.restype = ctypes.c_char_p
    L.wr_ctx_profile_stage_name.argtypes = [vp, ci]
    L.wr_rasterize.restype = ci
    L.wr_rasterize.argtypes = [vp, vp, ci, ci, ci, vp, ci, vp, ci, ci, vp, vp, vp]
    L.wr_interpolate.restype = ci
    L.wr_interpolate.argtypes = [vp, vp, ci, ci, ci, vp, ci, ci, ci, vp, ci, vp, vp]
    L.wr_texture.restype = ci
    L.wr_texture.argtypes = [vp, vp, ci, ci, ci, ci, vp, ci, ci, ci, ci, ci, vp, vp]
    L.wr_vertex_normals.restype = ci
    L.wr_vertex_normals.argtypes = [vp, vp, ci, vp, ci, vp, vp]
    L.wr_vertex_tangents.restype = ci
    L.wr_vertex_tangents.argtypes = [vp, vp, ci, vp, vp, ci, vp, ci, vp, vp, vp]
    L.wr_tangent_space_normals.restype = ci
    L.wr_tangent_space_normals.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, vp, vp]
    L.wr_render.restype = ci
    L.wr_render.argtypes = [vp, ctypes.POINTER(RenderArgs), vp]
    L.wr_view_prep.restype = ci
    L.wr_view_prep.argtypes = [vp, vp, vp, vp, vp, vp, vp, ci, ci, ci, ci, vp, vp, vp, vp, vp]
    L.wr_uv_unproject.restype = ci
    L.wr_uv_unproject.argtypes = [vp, ctypes.POINTER(UnprojectArgs), vp]
    L.wr_uv_finalize.restype = ci
    L.wr_uv_finalize.argtypes = [vp, vp, vp, ci, ci, vp, vp, vp]
    L.wr_uv_reduce_finalize_p2p.restype = ci
    L.wr_uv_reduce_finalize_p2p.argtypes = [vp, ctypes.POINTER(P2PReduceArgs), vp]
    L.wr_grid_sample.restype = ci
    L.wr_grid_sample.argtypes = [vp, vp, ci, ci, ci, ci, vp, ci, ci, vp, vp]
    L.wr_poisson_blend.restype = ci
    L.wr_poisson_blend.argtypes = [vp, vp, vp, vp, ci, ci, ci, ci, ci, vp, vp]
    L.wr_poisson_band_layout.restype = ci
    u64p = ctypes.POINTER(ctypes.c_uint64)
    cip = ctypes.POINTER(ci)
    L.wr_poisson_band_layout.argtypes = [ci, ci, ci, ci, ci, ci, u64p, u64p, cip, cip, cip]
    L.wr_poisson_band_step.restype = ci
    L.wr_poisson_band_step.argtypes = [vp, ctypes.POINTER(PoissonBandArgs), vp]
    L.wr_inpaint_u8.restype = ci
    L.wr_inpaint_u8.argtypes = [vp, vp, vp, ci, ci, ci, ci, vp, vp]
    L.wr_view_scores.restype = ci
    L.wr_view_scores.argtypes = [vp, vp, ci, vp, ci, ci, ci, ctypes.c_float, ctypes.c_float, ctypes.c_float, vp, vp, vp]
    L.wr_uv_padding.restype = ci
    L.wr_uv_padding.argtypes = [vp, vp, vp, ci, ci, ci, ci, vp, vp]
    if L.wr_version() != ABI_VERSION:   # a stale library: its argument structs differ from the ones declared here
        raise RuntimeError(f"{LIB_PATH} has ABI version {L.wr_version()}, this package expects {ABI_VERSION}: rebuild it "
                           "with `python -m worldrenderer_b200.build_native --force`")
    _LIB = L
    return L


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a tensor (None stays NULL).  Empty tensors map to NULL as well."""
    if t is None or t.numel() == 0:
        return None
    return t.data_ptr()


def stream_ptr(device: torch.device) -> int:
    """cudaStream_t of torch's current stream on `device` (the raw-handle query: ~10x cheaper than building a
    torch.cuda.Stream object per call, which showed in the host time of an eager render())."""
    index = device.index if device.index is not None else torch.cuda.current_device()
    try:
        return torch._C._cuda_getCurrentRawStream(index)
    except AttributeError:  # pragma: no cover -- older / newer torch without the private hook
        return torch.cuda.current_stream(device).cuda_stream


class NativeContext:
    """Owns one wr_ctx (per-device scratch).  Replaces dr.RasterizeCudaContext / RasterizeGLContext."""

    def __init__(self, device) -> None:
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError(
                f"worldrenderer_b200 runs on CUDA devices only (got {self.device}); there is no CPU path")
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA is not available: worldrenderer_b200 has no CPU fallback")
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", index)
        self._lib = lib()
        handle = ctypes.c_void_p()
        status = self._lib.wr_ctx_create(index, ctypes.byref(handle))
        if status != 0:
            raise RuntimeError(f"wr_ctx_create(device={index}) failed: {self._lib.wr_status_string(status).decode()}")
        self._h = handle

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.wr_ctx_destroy(h)
            except Exception:
                pass
            self._h = None

    @property
    def handle(self):
        return self._h

    def check(self, status: int, what: str) -> None:
        if status != 0:
            msg = self._lib.wr_status_string(status).decode()
            detail = self._lib.wr_ctx_last_error(self._h).decode()
            if status == -5:
                raise NotImplementedError(f"{what}: {msg}")
            raise RuntimeError(f"{what} failed: {msg}" + (f" ({detail})" if detail else ""))

    def stream(self) -> int:
        return stream_ptr(self.device)

    def scratch_bytes(self) -> int:
        return int(self._lib.wr_ctx_scratch_bytes(self._h))

    def profile(self, enable: bool) -> None:
        """Per-kernel CUDA-event timing of the following calls (measurement aid for bench.py)."""
        self.check(self._lib.wr_ctx_profile(self._h, int(bool(enable))), "wr_ctx_profile")

    def profile_read(self):
        """[(stage name, ms)] of the most recent native call; waits for it to finish."""
        buf = (ctypes.c_float * 17)()
        n = self._lib.wr_ctx_profile_read(self._h, buf, 17)
        if n < 0:
            self.check(n, "wr_ctx_profile_read")
        return [(self._lib.wr_ctx_profile_stage_name(self._h, i).decode(), float(buf[i])) for i in range(n)]


_DEFAULT_CTX: dict = {}


def default_context(device) -> NativeContext:
    """One shared NativeContext per device for the operators whose reference form takes no context object
    (cv_ops.inpaint_cvc, uv.uv_padding).  Same rule as everywhere: one stream at a time per context."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"worldrenderer_b200 runs on CUDA devices only (got {dev}); there is no CPU path")
    index = dev.index if dev.index is not None else torch.cuda.current_device()
    ctx = _DEFAULT_CTX.get(index)
    if ctx is None:
        ctx = _DEFAULT_CTX[index] = NativeContext(torch.device("cuda", index))
    return ctx
