"""Float64 restatement of the Euler, Euler-ancestral and DPM-Solver++(2M) updates -- TEST INFRASTRUCTURE.

Written independently of `paint_with_words_sd_b200.scheduler` (which tabulates one coefficient row per step):
  * Euler and Euler ancestral as diffusers 0.10 writes them (derivative (x - x0)/sigma times dt);
  * DPM-Solver++(2M) in the paper's form (Lu et al. 2022, Algorithm 2): VP state x_vp = alpha_t x_ve with
    alpha_t = 1/sqrt(1 + sigma^2), sigma_t = sigma/sqrt(1 + sigma^2), lambda_t = log(alpha_t/sigma_t), data
    prediction x0, and the result scaled back to the sigma (VE) state.
So agreement with the VE-form classes checks the conversion, not just the arithmetic.  All inputs are upcast to float64.
"""
from __future__ import annotations

import math
from typing import Optional

import torch


def _f64(t):
    return t.to(torch.float64) if isinstance(t, torch.Tensor) else torch.tensor(t, dtype=torch.float64)


def guided_eps(eps_cond, eps_uncond, guidance_scale: float):
    ec, eu = _f64(eps_cond), _f64(eps_uncond)
    return eu + guidance_scale * (ec - eu)


def euler_step(x, eps, sigma: float, sigma_next: float):
    """diffusers 0.10 EulerDiscreteScheduler.step with s_churn = 0 (gamma = 0, sigma_hat = sigma)."""
    x, eps = _f64(x), _f64(eps)
    x0 = x - sigma * eps
    derivative = (x - x0) / sigma
    return x + derivative * (sigma_next - sigma)


def euler_ancestral_step(x, eps, sigma: float, sigma_next: float, noise):
    """diffusers 0.10 EulerAncestralDiscreteScheduler.step."""
    x, eps = _f64(x), _f64(eps)
    x0 = x - sigma * eps
    sigma_up = (sigma_next ** 2 * (sigma ** 2 - sigma_next ** 2) / sigma ** 2) ** 0.5
    sigma_down = (sigma_next ** 2 - sigma_up ** 2) ** 0.5
    derivative = (x - x0) / sigma
    return x + derivative * (sigma_down - sigma) + _f64(noise) * sigma_up


def _vp(sigma: float):
    """(alpha_t, sigma_t, lambda_t) of the VP process whose noise-to-signal ratio is `sigma`."""
    alpha = 1.0 / math.sqrt(1.0 + sigma * sigma)
    s = sigma * alpha
    return alpha, s, (math.log(alpha / s) if s > 0 else math.inf)


def dpmpp_2m_step(x, eps, sigma: float, sigma_next: float, sigma_prev: Optional[float] = None, x0_prev=None):
    """One DPM-Solver++(2M) step; first order when `sigma_prev` is None (first step of a run) or sigma_next == 0.
    Returns (x_next, x0) in the VE state."""
    x, eps = _f64(x), _f64(eps)
    x0 = x - sigma * eps
    a_s, s_s, lam_s = _vp(sigma)
    a_t, s_t, lam_t = _vp(sigma_next)
    x_vp = a_s * x
    if sigma_next == 0.0:
        return x0.clone(), x0          # lambda_t = inf: the solver lands on the data prediction
    h = lam_t - lam_s
    if sigma_prev is None:
        d = x0
    else:
        _, _, lam_prev = _vp(sigma_prev)
        r = (lam_s - lam_prev) / h
        d = (1.0 + 1.0 / (2.0 * r)) * x0 - (1.0 / (2.0 * r)) * _f64(x0_prev)
    x_t = (s_t / s_s) * x_vp - a_t * math.expm1(-h) * d
    return x_t / a_t, x0


def karras_sigmas(sigma_min: float, sigma_max: float, n: int, rho: float = 7.0):
    """Karras et al. (2022) eq. 5, n values from sigma_max down to sigma_min (float64, no trailing zero)."""
    i = torch.arange(n, dtype=torch.float64)
    ramp = i / (n - 1) if n > 1 else i
    return (sigma_max ** (1 / rho) + ramp * (sigma_min ** (1 / rho) - sigma_max ** (1 / rho))) ** rho


def run(kind: str, sigmas, start: int, x, eps_fn, noise_fn=None):
    """Drive one sampler over sigmas[start:] (sigmas ends with 0).  eps_fn(i, x) -> guided eps at schedule index i;
    noise_fn(i) -> the ancestral noise of step i.  Returns the final x (float64)."""
    sig = [float(s) for s in sigmas]
    x = _f64(x)
    x0_prev = None
    for k, i in enumerate(range(start, len(sig) - 1)):
        eps = eps_fn(i, x)
        if kind == "euler":
            x = euler_step(x, eps, sig[i], sig[i + 1])
        elif kind == "euler_a":
            x = euler_ancestral_step(x, eps, sig[i], sig[i + 1], noise_fn(i))
        elif kind == "dpmpp_2m":
            x, x0_prev = dpmpp_2m_step(x, eps, sig[i], sig[i + 1], None if k == 0 else sig[i - 1], x0_prev)
        else:
            raise ValueError(kind)
    return x
