"""Python wrappers for the sampler kernels of libpww_b200 (csrc/sampler.cuh): the UNet-input prepare, the fused CFG +
sampler-step update and the per-image device noise.  CUDA only; a non-zero status raises.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _native

COEF_ROW = 12   # floats in a device coefficient row (layout in include/pww_b200.h)


def _stream(t: torch.Tensor):
    return torch.cuda.current_stream(t.device).cuda_stream


def _check_latent(name: str, t: torch.Tensor) -> None:
    if not (t.is_cuda and t.dtype == torch.float32 and t.dim() == 4 and t.is_contiguous()):
        raise ValueError(f"{name} must be a contiguous CUDA float32 [m, C, H, W] tensor")


def _check_coef(coef: torch.Tensor) -> None:
    if not (coef.is_cuda and coef.dtype == torch.float32 and coef.is_contiguous() and coef.numel() >= COEF_ROW):
        raise ValueError(f"coef must be a contiguous CUDA float32 row of {COEF_ROW} values")


def prepare_unet_input(latents: torch.Tensor, extra: Optional[torch.Tensor], coef: torch.Tensor,
                       out: torch.Tensor) -> torch.Tensor:
    """out [2m, C+Ce, H, W] fp16 channels-last <- both copies of cat(coef[1] * latents, extra)."""
    _check_latent("latents", latents)
    _check_coef(coef)
    m, C, H, W = latents.shape
    Ce = 0
    if extra is not None:
        _check_latent("extra", extra)
        Ce = extra.shape[1]
        if extra.shape[0] != m or tuple(extra.shape[2:]) != (H, W):
            raise ValueError(f"extra {tuple(extra.shape)} does not match latents {tuple(latents.shape)}")
    if (out.dtype != torch.float16 or out.shape != (2 * m, C + Ce, H, W) or
            not out.is_contiguous(memory_format=torch.channels_last)):
        raise ValueError("out must be a channels-last float16 [2m, C+Ce, H, W] tensor")
    with torch.cuda.device(latents.device):
        rc = _native.lib().pww_sampler_prepare_f16(latents.data_ptr(), None if extra is None else extra.data_ptr(),
                                                   coef.data_ptr(), out.data_ptr(), m, C, Ce, H, W, _stream(latents))
    _native.check(rc, "pww_sampler_prepare_f16")
    _native.launch_count += 1
    return out


def sampler_step(eps: torch.Tensor, latents: torch.Tensor, x0_prev: torch.Tensor, coef: torch.Tensor,
                 seeds: torch.Tensor, guidance_scale: float) -> None:
    """In place: latents <- a*x + b*eps_hat + c*x0 + d*x0_prev + s*noise, x0_prev <- x0 (coefficients from `coef`).
    eps: [2m, C, H, W] fp16 in any layout (cond rows first); seeds: int64 [m] on the device."""
    _check_latent("latents", latents)
    _check_latent("x0_prev", x0_prev)
    _check_coef(coef)
    m, C, H, W = latents.shape
    if eps.dtype != torch.float16 or tuple(eps.shape) != (2 * m, C, H, W) or not eps.is_cuda:
        raise ValueError(f"eps must be a CUDA float16 [{2 * m}, {C}, {H}, {W}] tensor, got {eps.dtype} {tuple(eps.shape)}")
    if x0_prev.shape != latents.shape or seeds.dtype != torch.int64 or seeds.numel() != m or not seeds.is_contiguous():
        raise ValueError("x0_prev must match latents and seeds must be a contiguous int64 tensor of one seed per image")
    with torch.cuda.device(latents.device):
        rc = _native.lib().pww_sampler_step_f32(eps.data_ptr(), *eps.stride(), latents.data_ptr(), x0_prev.data_ptr(),
                                                coef.data_ptr(), seeds.data_ptr(), float(guidance_scale), m, C, H, W,
                                                _stream(latents))
    _native.check(rc, "pww_sampler_step_f32")
    _native.launch_count += 1


def randn(shape, seed: int, step: int, device="cuda") -> torch.Tensor:
    """The noise the step kernel adds for one image with this seed at this absolute step index (shape = the image's
    [C, H, W] latent, or a leading batch dim of 1)."""
    out = torch.empty(shape, dtype=torch.float32, device=device)
    with torch.cuda.device(out.device):
        rc = _native.lib().pww_randn_f32(out.data_ptr(), out.numel(), int(seed) & 0xFFFFFFFFFFFFFFFF, int(step),
                                         _stream(out))
    _native.check(rc, "pww_randn_f32")
    _native.launch_count += 1
    return out
