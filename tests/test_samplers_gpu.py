"""The Euler / Euler-ancestral / DPM-Solver++(2M) kernels on the GPU: the fused step against the float64 oracle, the
UNet-input prepare against the torch expression it replaces, the device noise, and loop-level parity of PwWSampler
against the restated reference loop driving the host schedulers."""
import math

import numpy as np
import pytest
import torch

import paint_with_words_sd_b200 as P
from oracle import loop as oracle_loop
from oracle import samplers as O
from paint_with_words_sd_b200 import conditioning as C
from paint_with_words_sd_b200 import sampler_ops
from paint_with_words_sd_b200.pipeline import PwWSampler
from paint_with_words_sd_b200.scheduler import (DPMSolverMultistepScheduler, EulerAncestralDiscreteScheduler,
                                                EulerDiscreteScheduler, LMSDiscreteScheduler)
from paint_with_words_sd_b200.synthetic import RandomTextEncoder, SimpleWordTokenizer
from paint_with_words_sd_b200.unet import UNetConfig, attention_modules, build_unet
from tests.fixtures import SETTINGS, color_map_image, moon_mask_image

pytestmark = pytest.mark.gpu
SD = dict(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
CLASSES = {"euler": EulerDiscreteScheduler, "euler_a": EulerAncestralDiscreteScheduler,
           "dpmpp_2m": DPMSolverMultistepScheduler}
WF = lambda w, sigma, qk: 0.4 * w * math.log(1 + sigma) * qk.max()   # noqa: E731
DEV = "cuda"


def _row(sch, i, first):
    a, b, c, d, s = sch.coefficients(i, first)
    sig = float(sch.sigmas[i])
    return torch.tensor([sig, 1 / math.sqrt(sig * sig + 1), float(sch.timesteps[i]), a, b, c, d, s, 0.0, float(i), 0, 0],
                        dtype=torch.float32, device=DEV)


@pytest.mark.parametrize("kind", list(CLASSES))
@pytest.mark.parametrize("m", [1, 3])
@pytest.mark.parametrize("channels_last", [False, True])
def test_step_kernel_matches_oracle(kind, m, channels_last):
    sch = CLASSES[kind](**SD)
    sch.set_timesteps(20)
    g = torch.Generator().manual_seed(11)
    h = w = 16
    seeds = [101 + 7 * i for i in range(m)]
    for i in (0, 1, 9, 19):                       # first, second-order, middle, sigma' = 0
        first = i == 0
        x = torch.randn(m, 4, h, w, generator=g) * float(sch.sigmas[0]) * 5 / 3
        x0p = torch.randn(m, 4, h, w, generator=g) * 3
        eps = torch.randn(2 * m, 4, h, w, generator=g).half()
        eps_d = eps.to(DEV)
        if channels_last:
            eps_d = eps_d.contiguous(memory_format=torch.channels_last)
        lat, x0p_d = x.to(DEV), x0p.to(DEV)
        seeds_d = torch.tensor(seeds, dtype=torch.int64, device=DEV)
        sampler_ops.sampler_step(eps_d, lat, x0p_d, _row(sch, i, first), seeds_d, 7.5)
        ehat = O.guided_eps(eps[:m], eps[m:], 7.5)
        s0, s1 = float(sch.sigmas[i]), float(sch.sigmas[i + 1])
        if kind == "euler":
            ref = O.euler_step(x, ehat, s0, s1)
        elif kind == "euler_a":
            noise = torch.stack([sampler_ops.randn((4, h, w), sd, i).cpu() for sd in seeds])
            ref = O.euler_ancestral_step(x, ehat, s0, s1, noise)
        else:
            ref, _ = O.dpmpp_2m_step(x, ehat, s0, s1, None if first else float(sch.sigmas[i - 1]), x0p)
        ref_x0 = x.double() - s0 * ehat
        np.testing.assert_allclose(lat.cpu().double().numpy(), ref.numpy(), rtol=1e-5, atol=1e-4)
        np.testing.assert_allclose(x0p_d.cpu().double().numpy(), ref_x0.numpy(), rtol=1e-5, atol=1e-4)
        assert torch.isfinite(lat).all()


@pytest.mark.parametrize("extra_ch", [0, 5])
@pytest.mark.parametrize("m", [1, 2])
@pytest.mark.parametrize("hw", [(16, 16), (5, 7)])
def test_prepare_kernel_bit_exact(extra_ch, m, hw):
    g = torch.Generator().manual_seed(5)
    h, w = hw
    lat = (torch.randn(m, 4, h, w, generator=g) * 14.6).to(DEV)
    extra = (torch.randn(m, extra_ch, h, w, generator=g)).to(DEV) if extra_ch else None
    coef = torch.zeros(12, dtype=torch.float32, device=DEV)
    coef[1] = 1 / math.sqrt(14.6 ** 2 + 1)
    out = torch.empty(2 * m, 4 + extra_ch, h, w, dtype=torch.float16, device=DEV, memory_format=torch.channels_last)
    sampler_ops.prepare_unet_input(lat, extra, coef, out)
    x = lat * coef[1]
    if extra is not None:
        x = torch.cat([x, extra], dim=1)
    ref = torch.cat([x, x], 0).to(torch.float16).contiguous(memory_format=torch.channels_last)
    assert out.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))


def test_randn_statistics_and_determinism():
    n = 1 << 21
    a = sampler_ops.randn((n,), 1234, 7)
    b = sampler_ops.randn((n,), 1234, 7)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    a64 = a.double()
    assert abs(a64.mean().item()) < 3e-3 and abs(a64.var().item() - 1) < 1e-2
    for other in (sampler_ops.randn((n,), 1235, 7), sampler_ops.randn((n,), 1234, 8)):
        corr = ((a64 - a64.mean()) * (other.double() - other.double().mean())).mean() / (a64.std() * other.double().std())
        assert abs(corr.item()) < 3e-3
    # odd counts and offsets: element e of a shorter draw equals element e of a longer one
    short = sampler_ops.randn((1001,), 1234, 7)
    assert torch.equal(short, a[:1001])


def test_step_kernel_noise_is_randn():
    """Euler a with x = 0, eps = 0: x' = sigma_up * noise, so the kernel's noise is recovered exactly."""
    sch = EulerAncestralDiscreteScheduler(**SD)
    sch.set_timesteps(20)
    m, h, w, i = 3, 16, 16, 6
    seeds = [5, 99, 2 ** 40 + 3]
    lat = torch.zeros(m, 4, h, w, device=DEV)
    x0p = torch.zeros_like(lat)
    eps = torch.zeros(2 * m, 4, h, w, dtype=torch.float16, device=DEV)
    row = _row(sch, i, False)
    row[4] = 0.0                                  # b = 0 and s = 1 isolate the noise term
    row[7] = 1.0
    sampler_ops.sampler_step(eps, lat, x0p, row, torch.tensor(seeds, dtype=torch.int64, device=DEV), 7.5)
    for k, sd in enumerate(seeds):
        assert torch.equal(lat[k], sampler_ops.randn((4, h, w), sd, i))


# ---- loop parity -------------------------------------------------------------------------------------------------
def _setup(cfg, size, sch, device, seed=0):
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(cfg.cross_attention_dim)
    s = SETTINGS["aurora"]
    _, _, cond, uncond = C._encode_text_color_inputs(enc.to(device), tok, device, color_map_image("aurora", size),
                                                     dict(s["ctx"]), s["prompt"], "")
    lat = torch.randn(1, 4, size // 8, size // 8, generator=torch.manual_seed(seed)) * sch.init_noise_sigma
    return cond, uncond, lat


def _device_noise_scheduler(cls, seed):
    """The host class with the ancestral noise taken from the device generator (what PwWSampler adds)."""
    class Injected(cls):
        def step(self, model_output, timestep, sample, **kw):
            i = self.step_index_of(timestep)
            noise = sampler_ops.randn(tuple(sample.shape), seed, i).cpu() if self.ancestral else None
            return super().step(model_output, timestep, sample, noise=noise)
    return Injected


def _reference(cfg, size, sch, timesteps=None, extra=None, lat=None):
    unet = build_unet(cfg, seed=0)
    cond, uncond, lat0 = _setup(cfg, size, sch, "cpu")
    lat = lat0 if lat is None else lat
    try:
        oracle_loop.patch_with_oracle(unet)
        return oracle_loop.reference_denoise_loop(unet, sch, cond, uncond, lat, WF, timesteps=timesteps,
                                                  extra_input=extra)
    finally:
        cls = attention_modules(unet)[0].__class__
        if "__call__" in cls.__dict__:
            delattr(cls, "__call__")


def _rel_rmse(out, ref):
    return ((out - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt()).item()


@pytest.mark.parametrize("kind", list(CLASSES))
@pytest.mark.parametrize("use_graph", [False, True])
def test_sampler_loop_matches_reference_loop(kind, use_graph):
    cfg, size, steps, seed = UNetConfig.tiny(), 128, 4, 3
    sch = _device_noise_scheduler(CLASSES[kind], seed)(**SD)
    sch.set_timesteps(steps)
    ref = _reference(cfg, size, sch)
    sch.set_timesteps(steps)
    unet = build_unet(cfg, seed=0, dtype=torch.float16, device=DEV)
    cond, uncond, lat = _setup(cfg, size, sch, DEV)
    try:
        P.patch_unet(unet)
        out = PwWSampler(unet, sch, [cond], [uncond], lat.to(DEV), WF, 7.5, use_graph=use_graph,
                         noise_seeds=[seed]).run().float().cpu()
    finally:
        P.unpatch_all()
    r = _rel_rmse(out, ref)
    assert torch.isfinite(out).all() and r < 3e-2, r


@pytest.mark.parametrize("mode", ["inpaint", "img2img"])
def test_dpmpp_inpaint_and_img2img_match_reference_loop(mode):
    size, steps = 128, 6
    cfg = UNetConfig.tiny(in_channels=9 if mode == "inpaint" else 4)
    sch = DPMSolverMultistepScheduler(**SD)
    sch.set_timesteps(steps)
    g = torch.Generator().manual_seed(5)
    extra, timesteps, lat = None, None, None
    if mode == "inpaint":
        mask = (torch.rand(1, 1, size // 8, size // 8, generator=g) > 0.5).float()
        extra = torch.cat([mask, torch.randn(1, 4, size // 8, size // 8, generator=g) * 0.18215 * (1 - mask)], 1)
    else:                                          # strength 0.5: start mid-schedule from noised "image" latents
        t_start = steps - int(steps * 0.5)
        timesteps = sch.timesteps[t_start:]
        init = torch.randn(1, 4, size // 8, size // 8, generator=g) * 0.8
        lat = sch.add_noise(init, torch.randn(init.shape, generator=g), timesteps[:1])
    ref = _reference(cfg, size, sch, timesteps=timesteps, extra=extra, lat=lat)
    sch.set_timesteps(steps)
    unet = build_unet(cfg, seed=0, dtype=torch.float16, device=DEV)
    cond, uncond, lat0 = _setup(cfg, size, sch, DEV)
    lat = lat0 if lat is None else lat
    try:
        P.patch_unet(unet)
        out = PwWSampler(unet, sch, [cond], [uncond], lat.to(DEV), WF, 7.5, timesteps=timesteps,
                         extra_input=None if extra is None else extra.to(DEV)).run().float().cpu()
    finally:
        P.unpatch_all()
    r = _rel_rmse(out, ref)
    assert torch.isfinite(out).all() and r < 3e-2, r


def test_euler_a_batched_images_match_solo_runs():
    cfg, size, steps = UNetConfig.tiny(), 128, 3
    unet = build_unet(cfg, seed=0, dtype=torch.float16, device=DEV)
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(cfg.cross_attention_dim).to(DEV)
    sch = EulerAncestralDiscreteScheduler(**SD)
    sch.set_timesteps(steps)
    conds, unconds, lats, seeds = [], [], [], [17, 4242]
    for i, name in enumerate(("aurora", "cat_dog")):
        s = SETTINGS[name]
        _, _, c, u = C._encode_text_color_inputs(enc, tok, DEV, color_map_image(name, size), dict(s["ctx"]),
                                                 s["prompt"], "")
        conds.append(c); unconds.append(u)
        lats.append(torch.randn(1, 4, size // 8, size // 8, generator=torch.manual_seed(i)) * sch.init_noise_sigma)
    try:
        P.patch_unet(unet)
        both = PwWSampler(unet, sch, conds, unconds, torch.cat(lats, 0).to(DEV), WF, 7.5, use_graph=False,
                          noise_seeds=seeds).run().clone()
        solo = [PwWSampler(unet, sch, [conds[i]], [unconds[i]], lats[i].to(DEV), WF, 7.5, use_graph=False,
                           noise_seeds=[seeds[i]]).run().clone() for i in range(2)]
    finally:
        P.unpatch_all()
    for i in range(2):
        d = (both[i] - solo[i][0]).abs().max().item()
        assert d <= 2e-2 * solo[i].abs().max().item(), (i, d)


@pytest.mark.parametrize("karras", [False, True])
def test_public_api_and_pipelines_with_every_sampler(karras):
    s = SETTINGS["aurora"]
    vae, unet, enc, tok, _ = P.pww_load_tools("cuda:0", hf_model_path="synthetic:tiny")
    unet9 = build_unet(UNetConfig.tiny(in_channels=9), seed=0, dtype=torch.float16, device=DEV)
    try:
        cfg = UNetConfig.tiny()
        lms = LMSDiscreteScheduler(**SD)
        lms.set_timesteps(2)
        cond, uncond, lat = _setup(cfg, 128, lms, DEV)
        base = PwWSampler(unet, lms, [cond], [uncond], lat.to(DEV), WF, 7.5)
        base.run()
        for cls in CLASSES.values():
            sch = cls(use_karras_sigmas=karras, **SD)
            img = P.paint_with_words(color_context=dict(s["ctx"]), color_map_image=color_map_image("aurora", 128),
                                     input_prompt=s["prompt"], num_inference_steps=3, device="cuda:0",
                                     weight_function=WF, preloaded_utils=(vae, unet, enc, tok, sch))
            assert img.size == (128, 128)
            img = P.paint_with_words_inpaint(color_context=dict(s["ctx"]), color_map_image=color_map_image("aurora", 128),
                                             mask_image=moon_mask_image(128), init_image=color_map_image("aurora", 128),
                                             input_prompt=s["prompt"], num_inference_steps=3, device="cuda:0",
                                             weight_function=WF, preloaded_utils=(vae, unet9, enc, tok, sch))
            assert img.size == (128, 128)
            pipe = P.PaintWithWord_StableDiffusionPipeline(vae=vae, text_encoder=enc, tokenizer=tok, unet=unet)
            pipe.scheduler = cls.from_config(pipe.scheduler.config, use_karras_sigmas=karras)
            out = pipe(s["prompt"], color_map_image=color_map_image("aurora", 128), color_context=dict(s["ctx"]),
                       weight_function=WF, num_inference_steps=3, seed=3, output_type="latent")
            ref = P.paint_with_words(color_context=dict(s["ctx"]), color_map_image=color_map_image("aurora", 128),
                                     input_prompt=s["prompt"], num_inference_steps=3, seed=3, device="cuda:0",
                                     weight_function=WF, preloaded_utils=(vae, unet, enc, tok, pipe.scheduler),
                                     return_latents=True)
            assert torch.equal(out.images, ref) and torch.isfinite(ref).all()
            ipipe = P.PaintWithWord_StableDiffusionInpaintPipeline(vae=vae, text_encoder=enc, tokenizer=tok, unet=unet9)
            ipipe.scheduler = cls.from_config(ipipe.scheduler.config, use_karras_sigmas=karras)
            res = ipipe(s["prompt"], image=color_map_image("aurora", 128), mask_image=moon_mask_image(128),
                        color_map_image=color_map_image("aurora", 128), color_context=dict(s["ctx"]), weight_function=WF,
                        num_inference_steps=2, return_dict=False)
            assert res[0][0].size == (128, 128)
            sch.set_timesteps(2)
            fused = PwWSampler(unet, sch, [cond], [uncond], lat.to(DEV), WF, 7.5)
            fused.run()
            assert fused.native_launches_per_step == base.native_launches_per_step + 2
    finally:
        P.unpatch_all()
