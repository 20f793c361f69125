"""Euler, Euler-ancestral and DPM-Solver++(2M) schedulers on the host: schedules, per-step agreement with the float64
oracle (oracle/samplers.py), analytic properties, the public-API surface and ABI argument validation (no GPU)."""
import ctypes
import math

import numpy as np
import pytest
import torch

import paint_with_words_sd_b200 as P
from oracle import loop as oracle_loop
from oracle import samplers as O
from paint_with_words_sd_b200 import _native
from paint_with_words_sd_b200.scheduler import (DPMSolverMultistepScheduler, EulerAncestralDiscreteScheduler,
                                                EulerDiscreteScheduler, LMSDiscreteScheduler)

SD = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
CLASSES = {"euler": EulerDiscreteScheduler, "euler_a": EulerAncestralDiscreteScheduler,
           "dpmpp_2m": DPMSolverMultistepScheduler}


def _make(kind, steps, karras=False):
    s = CLASSES[kind](use_karras_sigmas=karras, **SD)
    s.set_timesteps(steps)
    return s


@pytest.mark.parametrize("steps", [1, 2, 15, 25])
def test_euler_sigmas_equal_lms_sigmas(steps):
    lms = LMSDiscreteScheduler(**SD)
    lms.set_timesteps(steps)
    for kind in CLASSES:
        s = _make(kind, steps)
        assert torch.equal(s.sigmas, lms.sigmas) and torch.equal(s.timesteps, lms.timesteps)
        assert float(s.init_noise_sigma) == float(lms.init_noise_sigma)


@pytest.mark.parametrize("steps", [2, 15, 25])
def test_karras_schedule(steps):
    s = _make("dpmpp_2m", steps, karras=True)
    ac = s.alphas_cumprod.double()
    train = ((1 - ac) / ac).sqrt()
    smin, smax = float(train[0]), float(train[-1])
    ref = O.karras_sigmas(smin, smax, steps)
    assert s.sigmas.shape == (steps + 1,) and float(s.sigmas[-1]) == 0.0
    np.testing.assert_allclose(s.sigmas[:-1].double().numpy(), ref.numpy(), rtol=2e-6)
    np.testing.assert_allclose(float(s.sigmas[0]), smax, rtol=1e-6)
    np.testing.assert_allclose(float(s.sigmas[steps - 1]), smin, rtol=1e-6)
    t = s.timesteps.double()
    assert abs(float(t[0]) - 999.0) < 1e-3 and abs(float(t[-1])) < 1e-3
    assert bool((t[1:] < t[:-1]).all())
    # the timestep of a sigma is its position on the train schedule: interpolating back gives the sigma
    back = np.exp(np.interp(t.numpy(), np.arange(1000), np.log(train.numpy())))
    np.testing.assert_allclose(back, s.sigmas[:-1].double().numpy(), rtol=1e-5)


def _host_run(kind, steps, t_start, karras, seed=0):
    """The host scheduler and the oracle over the same eps sequence; returns (host, oracle) final latents."""
    s = _make(kind, steps, karras)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64) * float(s.sigmas[t_start])
    epss = [torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64) for _ in range(steps)]
    noises = [torch.randn(1, 4, 8, 8, generator=g, dtype=torch.float64) for _ in range(steps)]
    xh = x.clone()
    for i in range(t_start, steps):
        xh = s.step(epss[i], s.timesteps[i], xh, noise=noises[i]).prev_sample
    xo = O.run(kind, s.sigmas.double(), t_start, x, lambda i, _x: epss[i], lambda i: noises[i])
    return xh, xo


@pytest.mark.parametrize("kind", list(CLASSES))
@pytest.mark.parametrize("steps", [1, 2, 15, 25])
@pytest.mark.parametrize("karras", [False, True])
def test_host_classes_match_oracle(kind, steps, karras):
    for t_start in sorted({0, steps // 2, steps - 1}):
        xh, xo = _host_run(kind, steps, t_start, karras)
        assert torch.isfinite(xh).all()
        np.testing.assert_allclose(xh.numpy(), xo.numpy(), rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("karras", [False, True])
def test_euler_exact_for_constant_eps(karras):
    """dx/dsigma = eps is integrated exactly when eps is constant: x_end = x_start + (0 - sigma_start) * eps."""
    s = _make("euler", 10, karras)
    eps = torch.randn(1, 4, 8, 8, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    x = torch.randn(1, 4, 8, 8, dtype=torch.float64) * float(s.sigmas[0])
    x_end = x.clone()
    for t in s.timesteps:
        x_end = s.step(eps, t, x_end).prev_sample
    np.testing.assert_allclose(x_end.numpy(), (x - float(s.sigmas[0]) * eps).numpy(), rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("karras", [False, True])
@pytest.mark.parametrize("t_start", [0, 4])
def test_dpmpp_exact_for_constant_x0(karras, t_start):
    """With a constant data prediction x0 the exact solution is x(sigma) = x0 + (sigma/sigma_s)(x_s - x0); both the
    first- and the second-order update reproduce it at every step."""
    s = _make("dpmpp_2m", 12, karras)
    g = torch.Generator().manual_seed(2)
    x0 = torch.randn(1, 4, 8, 8, dtype=torch.float64, generator=g)
    s0 = float(s.sigmas[t_start])
    x_s = x0 + s0 * torch.randn(1, 4, 8, 8, dtype=torch.float64, generator=g)
    x = x_s.clone()
    for i in range(t_start, 12):
        sigma = float(s.sigmas[i])
        eps = (x - x0) / sigma                   # the model predicts exactly x0
        x = s.step(eps, s.timesteps[i], x).prev_sample
        expect = x0 + (float(s.sigmas[i + 1]) / s0) * (x_s - x0)
        np.testing.assert_allclose(x.numpy(), expect.numpy(), rtol=1e-9, atol=1e-9)


@pytest.mark.parametrize("karras", [False, True])
def test_euler_ancestral_preserves_marginal(karras):
    """With x0 = 0, x ~ N(0, sigma^2) maps to sigma_down/sigma * x + sigma_up * xi ~ N(0, sigma_down^2 + sigma_up^2),
    and sigma_down^2 + sigma_up^2 = sigma'^2 at every step."""
    s = _make("euler_a", 20, karras)
    for i in range(20):
        sig, nxt = float(s.sigmas[i]), float(s.sigmas[i + 1])
        a, b, c, d, up = s.coefficients(i, i == 0)
        down = b + sig                            # b = sigma_down - sigma
        assert (a, c, d) == (1.0, 0.0, 0.0) and down >= 0.0 and up >= 0.0
        assert math.isclose(down * down + up * up, nxt * nxt, rel_tol=1e-12, abs_tol=1e-15)
    # and the same through `step` on samples (x0 = 0 means eps = x / sigma)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(200000, dtype=torch.float64, generator=g) * float(s.sigmas[5])
    out = s.step(x / float(s.sigmas[5]), s.timesteps[5], x,
                 noise=torch.randn(200000, dtype=torch.float64, generator=g)).prev_sample
    assert abs(out.std().item() / float(s.sigmas[6]) - 1) < 1e-2


@pytest.mark.parametrize("kind", list(CLASSES))
@pytest.mark.parametrize("karras", [False, True])
def test_last_step_is_finite(kind, karras):
    s = _make(kind, 5, karras)
    assert float(s.sigmas[-1]) == 0.0
    for first in (False, True):
        row = s.coefficients(4, first)
        assert all(math.isfinite(v) for v in row), row
    xh, _ = _host_run(kind, 5, 0, karras)
    assert torch.isfinite(xh).all()


def test_dpmpp_rejects_unimplemented_variants():
    with pytest.raises(ValueError):
        DPMSolverMultistepScheduler(algorithm_type="dpmsolver", **SD)
    with pytest.raises(ValueError):
        DPMSolverMultistepScheduler(solver_order=3, **SD)
    with pytest.raises(ValueError):
        DPMSolverMultistepScheduler.from_config(dict(SD), algorithm_type="sde-dpmsolver++")


@pytest.mark.parametrize("cls", [EulerDiscreteScheduler, EulerAncestralDiscreteScheduler, DPMSolverMultistepScheduler])
def test_load_tools_and_from_config(cls):
    vae, unet, enc, tok, sch = P.pww_load_tools("cpu", scheduler_type=cls, hf_model_path="synthetic:tiny")
    assert type(sch) is cls and sch.config["beta_schedule"] == "scaled_linear"
    lms = LMSDiscreteScheduler(**SD)
    new = cls.from_config(lms.config)
    assert type(new) is cls and all(new.config[k] == v for k, v in lms.config.items())
    again = cls.from_config(new.config)
    assert again.config == new.config
    k = cls.from_config(new.config, use_karras_sigmas=True)
    assert k.config["use_karras_sigmas"] is True and cls.from_config(k.config).use_karras_sigmas
    back = LMSDiscreteScheduler(**{kk: new.config[kk] for kk in lms.config})
    assert back.config == lms.config
    for s in (new, k):
        s.set_timesteps(4)
        x = torch.randn(1, 4, 8, 8)
        assert torch.equal(s.scale_model_input(x, s.timesteps[1]), x / ((float(s.sigmas[1]) ** 2 + 1) ** 0.5))
        noisy = s.add_noise(x, torch.ones_like(x), s.timesteps[2:3])
        assert torch.allclose(noisy, x + float(s.sigmas[2]))


def test_sampler_rejects_unknown_scheduler():
    class Other:
        timesteps = torch.tensor([999.0])
    with pytest.raises(TypeError, match="EulerAncestralDiscreteScheduler"):
        P.PwWSampler(None, Other(), [{}], [{}], torch.zeros(1, 4, 8, 8), lambda w, s, q: 0.0)


@pytest.mark.parametrize("kind", list(CLASSES))
def test_oracle_loop_runs_each_sampler(kind):
    from paint_with_words_sd_b200 import conditioning as C
    from paint_with_words_sd_b200.synthetic import RandomTextEncoder, SimpleWordTokenizer
    from paint_with_words_sd_b200.unet import UNetConfig, attention_modules, build_unet
    from tests.fixtures import SETTINGS, color_map_image
    cfg = UNetConfig.tiny()
    unet = build_unet(cfg, seed=0)
    s = SETTINGS["aurora"]
    _, _, cond, uncond = C._encode_text_color_inputs(RandomTextEncoder(cfg.cross_attention_dim), SimpleWordTokenizer(),
                                                     "cpu", color_map_image("aurora", 64), dict(s["ctx"]), s["prompt"], "")
    sch = _make(kind, 3)
    lat = torch.randn(1, 4, 8, 8, generator=torch.manual_seed(0)) * sch.init_noise_sigma
    try:
        oracle_loop.patch_with_oracle(unet)
        out = oracle_loop.reference_denoise_loop(unet, sch, cond, uncond, lat,
                                                 lambda w, sigma, qk: 0.4 * w * math.log(1 + sigma) * qk.max())
    finally:
        cls = attention_modules(unet)[0].__class__
        if "__call__" in cls.__dict__:
            delattr(cls, "__call__")
    assert out.shape == lat.shape and torch.isfinite(out).all() and not torch.equal(out, lat)


def test_sampler_abi_validation_without_gpu():
    """Null / misaligned pointers, non-positive sizes and bad strides return before any CUDA call."""
    L = _native.lib()
    buf = (ctypes.c_char * 4096)()
    p = (ctypes.addressof(buf) + 15) // 16 * 16
    # prepare: null latents, null coef, non-positive sizes, extra without channels, misaligned, too many channels
    assert L.pww_sampler_prepare_f16(None, None, p, p, 1, 4, 0, 8, 8, None) == -1
    assert L.pww_sampler_prepare_f16(p, None, None, p, 1, 4, 0, 8, 8, None) == -1
    assert L.pww_sampler_prepare_f16(p, None, p, p, 0, 4, 0, 8, 8, None) == -1
    assert L.pww_sampler_prepare_f16(p, None, p, p, 1, 4, 0, 8, -8, None) == -1
    assert L.pww_sampler_prepare_f16(p, p, p, p, 1, 4, 0, 8, 8, None) == -1
    assert L.pww_sampler_prepare_f16(p, None, p, p, 1, 4, 5, 8, 8, None) == -1
    assert L.pww_sampler_prepare_f16(p + 2, None, p, p, 1, 4, 0, 8, 8, None) == -1
    assert L.pww_sampler_prepare_f16(p, None, p, p + 1, 1, 4, 0, 8, 8, None) == -1
    assert L.pww_sampler_prepare_f16(p, p, p, p, 1, 4, 13, 8, 8, None) == -2
    # step: null pointers, misaligned, non-positive sizes / strides
    ok = (p, 256, 64, 8, 1, p, p, p, p, 7.5, 1, 4, 8, 8, None)
    for i in (0, 5, 6, 7, 8):
        args = list(ok)
        args[i] = None
        assert L.pww_sampler_step_f32(*args) == -1, i
    for i, v in ((0, p + 1), (5, p + 2), (6, p + 1), (7, p + 3), (8, p + 4)):
        args = list(ok)
        args[i] = v
        assert L.pww_sampler_step_f32(*args) == -1, i
    for i in (1, 2, 3, 4, 10, 11, 12, 13):
        args = list(ok)
        args[i] = 0
        assert L.pww_sampler_step_f32(*args) == -1, i
    # randn: null / misaligned output, non-positive count, negative step
    assert L.pww_randn_f32(None, 16, 0, 0, None) == -1
    assert L.pww_randn_f32(p + 2, 16, 0, 0, None) == -1
    assert L.pww_randn_f32(p, 0, 0, 0, None) == -1
    assert L.pww_randn_f32(p, 16, 0, -1, None) == -1
