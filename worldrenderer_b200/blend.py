"""Poisson blending of the baked atlas.

Drop-in for mvadapter/utils/mesh_utils/blend.py of the reference: `PoissonBlendingSolver(backend, device)`
(:186-212) and its `__call__(src, mask, tgt, num_iters, inplace=True, grad_mode="src")` (:214-324).

The reference flattens the solve region into gathered index lists and runs one Jacobi kernel per sweep with
a device synchronisation after each (torch-cuda backend, :60-100), or a Triton / eager-PyTorch equivalent.
Here the whole call is `wr_poisson_blend` (csrc/blend.cu): the region stays a 2-D image and a temporally
blocked stencil kernel runs eight sweeps per launch out of registers.  `backend` keeps its meaning only in one
respect -- how many sweeps an odd `num_iters` yields (see `_sweeps`).
"""
from __future__ import annotations

import torch

from . import _native
from .utils import SINGLE_IMAGE_TYPE, image_to_tensor

_BACKENDS = ("torch-native", "torch-cuda", "triton")
_GRAD_MODES = {"src": 0, "max": 1, "avg": 2}


class PoissonBlendingSolver:
    def __init__(self, backend: str, device: str):
        if backend not in _BACKENDS:
            raise ValueError(f"Unknown backend: {backend}")  # blend.py:195-196
        self.backend = backend
        self.device = device
        self._ctx = _native.NativeContext(device)

    def _sweeps(self, num_iters: int) -> int:
        # "torch-native" applies every sweep in place (blend.py:176-183).  The other two backends swap LOCAL
        # buffer handles (blend.py:88-100, 166-169) while the caller keeps reading the original X: after an odd
        # number of sweeps the newest iterate sits in the scratch buffer, so the caller sees sweep num_iters - 1.
        n = int(num_iters)
        return n if self.backend == "torch-native" else n - (n & 1)

    def _inputs(self, src: SINGLE_IMAGE_TYPE, mask: SINGLE_IMAGE_TYPE, tgt: SINGLE_IMAGE_TYPE, inplace: bool,
                grad_mode: str):
        """(src, mask as u8, tgt, grad-mode index) in the form the kernels take: [H,W,C] float32 on the device,
        C <= 4, the mask thresholded as in blend.py:229-232."""
        if grad_mode not in _GRAD_MODES:
            raise ValueError(f"Unknown grad_mode: {grad_mode}")
        dev = self._ctx.device
        src = image_to_tensor(src, device=dev)
        mask = image_to_tensor(mask, device=dev)
        tgt = image_to_tensor(tgt, device=dev)
        assert src.ndim == 3 and tgt.ndim == 3 and mask.ndim in [2, 3]
        if src.shape != tgt.shape or mask.shape[:2] != tgt.shape[:2]:
            raise ValueError(f"src {tuple(src.shape)}, mask {tuple(mask.shape)} and tgt {tuple(tgt.shape)} must agree")
        mask = (mask.mean(-1) > 0.5) if mask.ndim == 3 else (mask > 0.5)  # blend.py:229-232
        if tgt.shape[2] > 4:
            raise NotImplementedError("PoissonBlendingSolver: more than 4 channels")
        if inplace and not tgt.is_contiguous():
            raise ValueError("inplace=True needs a contiguous target")
        return src.contiguous(), mask.contiguous().view(torch.uint8), tgt.contiguous(), _GRAD_MODES[grad_mode]

    def __call__(self, src: SINGLE_IMAGE_TYPE, mask: SINGLE_IMAGE_TYPE, tgt: SINGLE_IMAGE_TYPE, num_iters: int,
                 inplace: bool = True, grad_mode: str = "src"):
        src_c, mask_c, tgt_c, gm = self._inputs(src, mask, tgt, inplace, grad_mode)
        H, W, C = tgt_c.shape
        out = tgt_c if inplace else torch.empty_like(tgt_c)
        c = self._ctx
        c.check(_native.lib().wr_poisson_blend(c.handle, _native.ptr(src_c), _native.ptr(mask_c), _native.ptr(tgt_c),
                                               H, W, C, self._sweeps(num_iters), gm,
                                               _native.ptr(out), c.stream()), "wr_poisson_blend")
        return out
