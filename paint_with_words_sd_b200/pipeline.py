"""Public API: `paint_with_words()`, `paint_with_words_inpaint()`, `pww_load_tools()` -- same keyword
arguments, defaults and return type as the reference (paint_with_words/paint_with_words.py:128-204,
391-510; paint_with_words_inpaint.py:137-270) -- plus `PwWSampler`, the B200-first engine behind them.

What is different underneath (results equal within the stated fp16 tolerance):
  * the attention of every UNet block runs in libpww_b200.so (see attention.py);
  * cond and uncond are ONE batch-2 UNet forward with per-image bias enable and per-image score
    statistic instead of two batch-1 forwards (paint_with_words.py:483-499);
  * the whole step (UNet, CFG combine, LMS update) is captured in a CUDA graph; sigma, G(sigma) and the
    LMS coefficients are device scalars refreshed by tiny copies, so a replay does no host math;
  * with the Euler, Euler-ancestral and DPM-Solver++(2M) schedulers the CFG combine and update are one native kernel;
  * K/V of the text context are step-invariant, so the context tensors are staged once per image.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F
from PIL import Image

from . import attention as _attention
from .conditioning import _encode_text_color_inputs, _get_binary_mask, pack_weight_map, packed_key
from . import sampler_ops as _sampler_ops
from .scheduler import SIGMA_SAMPLERS, LMSDiscreteScheduler, _CoefficientScheduler
from .synthetic import IdentityVAE, RandomTextEncoder, SimpleWordTokenizer
from .unet import UNet2DConditionModel, UNetConfig, build_unet
from .weight_function import g_of_sigma, probe_weight_function


def default_weight_function(w, sigma, qk):
    """paint_with_words.py:402-405."""
    return 0.1 * w * math.log(sigma + 1) * qk.max()


def _zero_weight_function(w, sigma, qk):
    """The uncond branch's `lambda w, sigma, qk: 0.0` (paint_with_words.py:493)."""
    return 0.0


_SYNTHETIC_CONFIGS = {
    "synthetic:sd15": UNetConfig.sd15,
    "synthetic:sd15-inpaint": UNetConfig.sd15_inpaint,
    "synthetic:sd21": UNetConfig.sd21,
    "synthetic:tiny": UNetConfig.tiny,
    "synthetic:tiny-inpaint": lambda: UNetConfig.tiny(in_channels=9),
}


def pww_load_tools(device: str = "cuda:0", scheduler_type=LMSDiscreteScheduler,
                   local_model_path: Optional[str] = None, hf_model_path: Optional[str] = None,
                   model_token: Optional[str] = None, seed: int = 0):
    """paint_with_words.py:128-204: returns (vae, unet, text_encoder, tokenizer, scheduler) with the
    attention of `unet` patched.  `"synthetic:<sd15|sd15-inpaint|sd21|tiny>"` model paths build seeded
    random-weight stand-ins (no weights or network exist in this environment); any other path is
    loaded with diffusers/transformers when those are installed."""
    assert local_model_path or hf_model_path, "either local_model_path or hf_model_path must be provided"
    model_path = local_model_path if local_model_path is not None else hf_model_path
    dtype = torch.float16 if device != "mps" else torch.float32
    if model_path in _SYNTHETIC_CONFIGS:
        cfg = _SYNTHETIC_CONFIGS[model_path]()
        unet = build_unet(cfg, seed=seed, dtype=dtype, device=device)
        text_encoder = RandomTextEncoder(cfg.cross_attention_dim).to(device)
        tokenizer, vae = SimpleWordTokenizer(), IdentityVAE().to(device)
    else:
        try:
            from diffusers import AutoencoderKL, UNet2DConditionModel as _HFUNet
            from transformers import CLIPTextModel, CLIPTokenizer
        except ImportError as e:
            raise ImportError(f"loading '{model_path}' needs diffusers + transformers, which are not installed; "
                              "use a 'synthetic:*' model path or pass preloaded_utils") from e
        local_only = local_model_path is not None
        vae = AutoencoderKL.from_pretrained(model_path, subfolder="vae", torch_dtype=dtype,
                                            local_files_only=local_only).to(device)
        tokenizer = CLIPTokenizer.from_pretrained(model_path, subfolder="tokenizer")
        text_encoder = CLIPTextModel.from_pretrained(model_path, subfolder="text_encoder").to(device)
        unet = _HFUNet.from_pretrained(model_path, subfolder="unet", torch_dtype=dtype,
                                       local_files_only=local_only).to(device)
    _attention.patch_unet(unet)
    scheduler = scheduler_type(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                               num_train_timesteps=1000)
    return vae, unet, text_encoder, tokenizer, scheduler


def _module_dtype(module, default=torch.float32):
    p = next(iter(module.parameters()), None) if hasattr(module, "parameters") else None
    return p.dtype if p is not None else default


def _pil_from_latents(vae, latents):
    """paint_with_words.py:48-57.  (The reference runs under torch.autocast; here the VAE gets its own dtype.)"""
    image = vae.decode((1 / 0.18215 * latents.clone()).to(_module_dtype(vae, latents.dtype))).sample
    image = (image / 2 + 0.5).clamp(0, 1).detach().cpu().permute(0, 2, 3, 1).float().numpy()
    return [Image.fromarray(a) for a in (image * 255).round().astype("uint8")]


def preprocess(image):
    """paint_with_words.py:28-35."""
    w, h = image.size
    w, h = w - w % 32, h - h % 32
    arr = np.array(image.resize((w, h), resample=Image.LANCZOS)).astype(np.float32) / 255.0
    return 2.0 * torch.from_numpy(arr[None].transpose(0, 3, 1, 2)) - 1.0


def initial_latents(latent_size, seed: int, extra_seeds: Dict[int, int], seperated_word_contexts) -> torch.Tensor:
    """paint_with_words.py:445-455: host-side seeded noise, optionally re-seeded per region."""
    latents = torch.randn(latent_size, generator=torch.manual_seed(seed))
    if len(extra_seeds) > 0:
        print("Use region based seeding: ", extra_seeds)
        per_seed = [torch.randn(latent_size, generator=torch.manual_seed(s)) for s in extra_seeds.values()]
        masks = _get_binary_mask(seperated_word_contexts, extra_seeds, dtype=latents[0].dtype, size=latent_size[-2:])
        foreground = (sum(masks) > 0).squeeze()
        mixed = sum(l * m for l, m in zip(per_seed, masks))
        latents[:, :, foreground] = mixed[:, :, foreground]
    return latents


# ---------------------------------------------------------------------------------------------
# the engine
# ---------------------------------------------------------------------------------------------
class PwWSampler:
    """Denoising loop for a group of images on ONE GPU (paint_with_words.py:471-506 semantics per image).

    Each image i has a cond context dict, an uncond context dict and latents; a step runs one UNet
    forward over the batch [cond_0..cond_{m-1}, uncond_0..uncond_{m-1}], the CFG combine and the sampler
    update.  `use_graph=True` captures the step in a CUDA graph.

    With `LMSDiscreteScheduler` the update is the LMS step below in PyTorch.  With the Euler, Euler-ancestral and
    DPM-Solver++(2M) schedulers a step is "prepare -> UNet -> step": one native launch writes the fp16 channels-last
    UNet input, one applies the CFG combine and the update (sampler_ops.py).  `noise_seeds` (one per image, default
    0..m-1) key the ancestral noise, so an image's result does not depend on how images are batched.
    """

    def __init__(self, unet, scheduler: LMSDiscreteScheduler, cond_ctxs: Sequence[dict], uncond_ctxs: Sequence[dict],
                 latents: torch.Tensor, weight_function: Callable, guidance_scale: float = 7.5,
                 extra_input: Optional[torch.Tensor] = None, use_graph: bool = True, timesteps=None,
                 noise_seeds: Optional[Sequence[int]] = None):
        if isinstance(scheduler, LMSDiscreteScheduler):
            self._fused = False
        elif isinstance(scheduler, _CoefficientScheduler):
            self._fused = True
        else:
            names = ", ".join(c.__name__ for c in (LMSDiscreteScheduler,) + SIGMA_SAMPLERS)
            raise TypeError(f"PwWSampler does not support {type(scheduler).__name__}; supported schedulers: {names}")
        self.unet, self.scheduler = unet, scheduler
        self.m = len(cond_ctxs)
        self.device = latents.device
        self.guidance_scale = float(guidance_scale)
        self.weight_function = weight_function
        self.timesteps = list((scheduler.timesteps if timesteps is None else timesteps).tolist())
        self.latents = latents.clone().float()
        self.extra_input = extra_input            # inpaint: [m,5,h,w] (mask + masked-image latents)
        self.use_graph = use_graph and latents.is_cuda
        self._graph = None
        self._kv_graph = None
        self.native_launches_per_step = None
        self._probed = probe_weight_function(weight_function, 1.0)
        up = next(iter(unet.parameters()), None)
        self._unet_dtype = up.dtype if up is not None else torch.float32
        self._ctx = self._merge_contexts(cond_ctxs, uncond_ctxs)
        dev = self.device
        # Per-step scalars (sigma, 1/sqrt(sigma^2+1), t, 4 LMS coefficients, G(sigma)) are tabulated
        # once on the host and uploaded; a step copies its row into `_params` (one 32-byte D2D copy), so
        # a captured graph sees new values and the host never feeds the stream mid-loop.
        if self._fused:
            self._init_fused(noise_seeds)
        else:
            self._table = self._build_step_table().to(dev)
            self._params = torch.zeros(8, dtype=torch.float32, device=dev)
            self._derivs = torch.zeros((4,) + tuple(self.latents.shape), dtype=torch.float32, device=dev)
            self._ctx["G_SIGMA"] = self._params[7:8]
        self._step_no = 0

    def _init_fused(self, noise_seeds):
        if not self.latents.is_cuda:
            raise ValueError(f"{type(self.scheduler).__name__} runs its step on the GPU; latents are on {self.device}")
        if self._unet_dtype != torch.float16:
            raise ValueError(f"{type(self.scheduler).__name__} feeds the UNet fp16; this UNet is {self._unet_dtype}")
        dev, m = self.device, self.m
        self.latents = self.latents.contiguous()
        seeds = list(range(m)) if noise_seeds is None else [int(v) for v in noise_seeds]
        if len(seeds) != m:
            raise ValueError(f"noise_seeds has {len(seeds)} entries for {m} images")
        self._seeds = torch.tensor(seeds, dtype=torch.int64, device=dev)
        self._extra = None if self.extra_input is None else self.extra_input.to(dev, torch.float32).contiguous()
        _, c, h, w = self.latents.shape
        ce = 0 if self._extra is None else self._extra.shape[1]
        self._unet_in = torch.empty((2 * m, c + ce, h, w), dtype=torch.float16, device=dev,
                                    memory_format=torch.channels_last)
        self._x0_prev = torch.zeros_like(self.latents)
        self._table = self._build_coefficient_table().to(dev)
        self._params = torch.zeros(_sampler_ops.COEF_ROW, dtype=torch.float32, device=dev)
        self._ctx["G_SIGMA"] = self._params[8:9]

    def _build_coefficient_table(self) -> torch.Tensor:
        """Row k (run step k): sigma, c_in, t, a, b, c, d, s, G(sigma), absolute step index, 0, 0
        (layout in include/pww_b200.h)."""
        sch = self.scheduler
        rows = []
        for k, t in enumerate(self.timesteps):
            si = sch.step_index_of(t)
            sigma = float(sch.sigmas[si])
            a, b, c, d, s = sch.coefficients(si, first=(k == 0))
            g = g_of_sigma(self.weight_function, self._probed, sch.sigmas[si])
            rows.append([sigma, 1.0 / math.sqrt(sigma * sigma + 1.0), float(t), a, b, c, d, s, g, float(si), 0.0, 0.0])
        return torch.tensor(rows, dtype=torch.float32)

    def _build_step_table(self) -> torch.Tensor:
        sch = self.scheduler
        rows = []
        for t in self.timesteps:
            si = sch.step_index_of(t)
            sigma = float(sch.sigmas[si])
            # paint_with_words.py:506 -> LMS order = min(step_index+1, 4) on the ABSOLUTE schedule index;
            # missing history (img2img starts mid-schedule) simply contributes nothing (zip truncation).
            coeffs = list(sch._coeffs[si]) if sch._coeffs is not None else sch._lms_coeffs(si, min(si + 1, 4))
            coeffs = (coeffs + [0.0] * 4)[:4]
            g = g_of_sigma(self.weight_function, self._probed, sch.sigmas[si])
            rows.append([sigma, 1.0 / math.sqrt(sigma * sigma + 1.0), float(t), *coeffs, g])
        return torch.tensor(rows, dtype=torch.float32)

    def _merge_contexts(self, conds, unconds) -> dict:
        """Batch the per-image dicts: CONTEXT_TENSOR -> [2m,77,Dc]; weight maps -> [m,N,77] stacks;
        WMAP_INDEX = [0..m-1, -1 x m]."""
        m = self.m
        ctx = {"CONTEXT_TENSOR": torch.cat([c["CONTEXT_TENSOR"] for c in conds] +
                                           [u["CONTEXT_TENSOR"] for u in unconds], 0).to(self.device)}
        for key in conds[0]:
            if not key.startswith("CROSS_ATTENTION_WEIGHT_"):
                continue
            vals = [c[key] for c in conds]
            if key == "CROSS_ATTENTION_WEIGHT_ORIG":
                ctx[key] = vals[0] if m == 1 else 0   # ORIG fallback is a single-image path ...
                if m > 1 and any(isinstance(v, torch.Tensor) for v in vals):
                    ctx["ORIG_FALLBACK_DROPPED"] = True   # ... and a level that would need it raises instead of losing its bias
                continue
            if all(isinstance(v, torch.Tensor) for v in vals):
                dense = torch.stack([v.detach().to("cpu", torch.float32) for v in vals], 0).contiguous()
                ctx[key] = dense.to(self.device)
                packed = pack_weight_map(dense)      # host-side set-up, like the map builder itself
                if packed is not None:
                    n = int(key.rsplit("_", 1)[1])
                    ctx[packed_key(n)] = (packed[0].to(self.device), packed[1].to(self.device))
            else:
                ctx[key] = 0
        ctx["WMAP_INDEX"] = torch.tensor(list(range(m)) + [-1] * m, dtype=torch.int32, device=self.device)
        ctx["WEIGHT_FUNCTION"] = self.weight_function
        ctx["SIGMA"] = None
        ctx["KV_CACHE"] = {}       # to_k/to_v of the text context are step-invariant: computed at the first step
        # scratch of the attention launches, owned by this sampler: its captured graphs never see a buffer that another
        # sampler or a later, larger call replaced
        from . import _native
        ctx["PWW_SCRATCH"] = (torch.zeros(max(64, 2 * m), dtype=torch.float32, device=self.device),
                              torch.zeros(_native.lib().pww_xattn_fused_workspace_bytes(), dtype=torch.uint8,
                                          device=self.device))
        return ctx

    # -- one step, expressed only with device tensors / device scalars --------------------------
    def _step_body(self):
        if self._fused:
            self._fused_step_body()
            return
        m = self.m
        x = self.latents * self._params[1]
        if self.extra_input is not None:
            x = torch.cat([x, self.extra_input], dim=1)
        x2 = torch.cat([x, x], 0).to(self._unet_dtype)      # the reference runs under autocast: feed the UNet its own dtype
        eps = self.unet(x2, self._params[2:3], encoder_hidden_states=self._ctx).sample.float()
        eps_c, eps_u = eps[:m], eps[m:]
        noise_pred = eps_u + self.guidance_scale * (eps_c - eps_u)
        # LMS (epsilon prediction): derivative == noise_pred; history kept in a rolling device buffer
        self._derivs.copy_(torch.roll(self._derivs, 1, 0))
        self._derivs[0].copy_(noise_pred)
        upd = (self._params[3:7].view(4, 1, 1, 1, 1) * self._derivs).sum(0)
        self.latents.add_(upd)

    def _fused_step_body(self):
        _sampler_ops.prepare_unet_input(self.latents, self._extra, self._params, self._unet_in)
        eps = self.unet(self._unet_in, self._params[2:3], encoder_hidden_states=self._ctx).sample
        _sampler_ops.sampler_step(eps, self.latents, self._x0_prev, self._params, self._seeds, self.guidance_scale)

    def _state(self) -> List[torch.Tensor]:
        """Device tensors a step updates in place (what warm-up and capture must restore)."""
        return [self.latents, self._x0_prev] if self._fused else [self.latents, self._derivs]

    def _set_step_scalars(self, i: int, step_index: int):
        self._params.copy_(self._table[i])
        self._ctx["SIGMA"] = self.scheduler.sigmas[step_index]

    # -- host-buffer interface (what bench.py's e2e leg drives) -----------------------------------
    def device_inputs(self) -> Dict[str, torch.Tensor]:
        """Persistent device tensors a step reads: latents, the text context and the stacked weight maps.
        Copying new values INTO them (same addresses) is valid between graph replays."""
        d = {"latents": self.latents, "CONTEXT_TENSOR": self._ctx["CONTEXT_TENSOR"]}
        for k, v in self._ctx.items():
            if k.startswith("CROSS_ATTENTION_PACKED_"):
                d[k + "_M"], d[k + "_C"] = v                       # packed map + token column index
            elif k.startswith("CROSS_ATTENTION_WEIGHT_") and isinstance(v, torch.Tensor) and v.is_cuda:
                n = k.rsplit("_", 1)[1]
                if n.isdigit() and packed_key(int(n)) not in self._ctx:
                    d[k] = v                                       # dense map (only when it could not be packed)
        return d

    def stage_from_host(self, pinned: Dict[str, torch.Tensor]) -> int:
        """Async H2D copy of this step's inputs from pinned host buffers; returns bytes copied."""
        dev = self.device_inputs()
        n = 0
        for k, h in pinned.items():
            dev[k].copy_(h, non_blocking=True)
            n += h.numel() * h.element_size()
        if "CONTEXT_TENSOR" in pinned and self._ctx.get("KV_CACHE"):
            # the cached K/V follow the new context: 16 small GEMMs, replayed as one CUDA graph
            if not self.use_graph:
                _attention.refresh_kv_cache(self._ctx)
            else:
                if self._kv_graph is None:
                    s = torch.cuda.Stream(device=self.device)
                    s.wait_stream(torch.cuda.current_stream(self.device))
                    with torch.cuda.stream(s):
                        _attention.refresh_kv_cache(self._ctx)
                    torch.cuda.current_stream(self.device).wait_stream(s)
                    self._kv_graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self._kv_graph):
                        _attention.refresh_kv_cache(self._ctx)
                self._kv_graph.replay()
        return n

    def restart(self, latents: Optional[torch.Tensor] = None):
        """Rewind to step 0 (fresh LMS / multistep history), optionally with new latents."""
        self._step_no = 0
        self._state()[1].zero_()
        if latents is not None:
            self.latents.copy_(latents)

    def step(self):
        i = self._step_no
        step_index = self.scheduler.step_index_of(self.timesteps[i])
        self._set_step_scalars(i, step_index)
        if not self.use_graph:
            self._step_body()
        elif self._graph is None:
            # warm-up on a side stream (allocator + cuDNN/cuBLAS autotune), then capture
            self._capture()
            self._graph.replay()
        else:
            self._graph.replay()
        self._step_no += 1

    def _capture(self):
        state = self._state()
        snap = [t.clone() for t in state]
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            for _ in range(2):
                self._step_body()
        torch.cuda.current_stream(self.device).wait_stream(s)
        for t, v in zip(state, snap):
            t.copy_(v)
        g = torch.cuda.CUDAGraph()
        from . import _native
        before = _native.launch_count
        with torch.cuda.graph(g):
            self._step_body()
        self.native_launches_per_step = _native.launch_count - before
        for t, v in zip(state, snap):
            t.copy_(v)
        self._graph = g

    def run(self, num_steps: Optional[int] = None) -> torch.Tensor:
        n = len(self.timesteps) - self._step_no if num_steps is None else num_steps
        with torch.no_grad():
            for _ in range(n):
                self.step()
        return self.latents


@torch.no_grad()
def paint_with_words(
    color_context: Dict[Tuple[int, int, int], str] = {},
    color_map_image: Optional[Image.Image] = None,
    input_prompt: str = "",
    num_inference_steps: int = 30,
    guidance_scale: float = 7.5,
    seed: int = 0,
    scheduler_type=LMSDiscreteScheduler,
    device: str = "cuda:0",
    weight_function: Callable = default_weight_function,
    local_model_path: Optional[str] = None,
    hf_model_path: Optional[str] = "synthetic:sd15",
    preloaded_utils: Optional[Tuple] = None,
    unconditional_input_prompt: str = "",
    model_token: Optional[str] = None,
    init_image: Optional[Image.Image] = None,
    strength: float = 0.5,
    return_latents: bool = False,
):
    """paint_with_words.py:391-510.  Returns one PIL.Image (or the final latents with return_latents)."""
    width, height = color_map_image.size
    vae, unet, text_encoder, tokenizer, scheduler = (
        pww_load_tools(device, scheduler_type, local_model_path=local_model_path, hf_model_path=hf_model_path,
                       model_token=model_token)
        if preloaded_utils is None else preloaded_utils)
    extra_seeds, seperated_word_contexts, cond, uncond = _encode_text_color_inputs(
        text_encoder, tokenizer, device, color_map_image, color_context, input_prompt, unconditional_input_prompt)

    scheduler.set_timesteps(num_inference_steps)
    timesteps = scheduler.timesteps
    if init_image is None:
        latents = initial_latents((1, unet.in_channels, height // 8, width // 8), seed, extra_seeds,
                                  seperated_word_contexts).to(device)
        latents = latents * scheduler.init_noise_sigma
    else:
        init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
        t_start = max(num_inference_steps - init_timestep, 0)
        timesteps = scheduler.timesteps[t_start:]
        image = preprocess(init_image).to(device=device)
        init_latents = 0.18215 * vae.encode(image.to(_module_dtype(vae, image.dtype))).latent_dist.sample().float()
        noise = torch.randn(init_latents.shape).to(device)
        latents = scheduler.add_noise(init_latents, noise, timesteps[:1])

    sampler = PwWSampler(unet, scheduler, [cond], [uncond], latents, weight_function, guidance_scale,
                         timesteps=timesteps, noise_seeds=[seed])
    latents = sampler.run()
    if return_latents:
        return latents
    return _pil_from_latents(vae, latents)[0]


def prepare_mask_and_masked_image(image, mask):
    """paint_with_words_inpaint.py:20-106 (PIL / ndarray inputs): mask binarised at 0.5, image in [-1,1],
    masked_image = image * (mask < 0.5)."""
    if isinstance(image, torch.Tensor) or isinstance(mask, torch.Tensor):
        if not (isinstance(image, torch.Tensor) and isinstance(mask, torch.Tensor)):
            raise TypeError("`image` and `mask` must both be tensors or both be PIL/ndarray")
        if image.ndim == 3:
            image = image.unsqueeze(0)
        if mask.ndim == 2:
            mask = mask[None, None]
        elif mask.ndim == 3:
            mask = mask.unsqueeze(0) if mask.shape[0] == 1 else mask.unsqueeze(1)
        if image.min() < -1 or image.max() > 1:
            raise ValueError("Image should be in [-1, 1] range")
        if mask.min() < 0 or mask.max() > 1:
            raise ValueError("Mask should be in [0, 1] range")
        mask = (mask >= 0.5).to(torch.float32)
        image = image.to(torch.float32)
    else:
        if isinstance(image, Image.Image):
            image = np.array(image.convert("RGB"))
        image = torch.from_numpy(image[None].transpose(0, 3, 1, 2)).to(torch.float32) / 127.5 - 1.0
        if isinstance(mask, Image.Image):
            mask = np.array(mask.convert("L")).astype(np.float32) / 255.0
        mask = torch.from_numpy((mask[None, None] >= 0.5).astype(np.float32))
    return mask, image * (mask < 0.5)


@torch.no_grad()
def paint_with_words_inpaint(
    color_context: Dict[Tuple[int, int, int], str] = {},
    color_map_image: Optional[Image.Image] = None,
    mask_image: Optional[Image.Image] = None,
    init_image: Image.Image = None,
    input_prompt: str = "",
    num_inference_steps: int = 150,
    guidance_scale: float = 7.5,
    seed: int = 0,
    scheduler_type=LMSDiscreteScheduler,
    device: str = "cuda:0",
    weight_function: Callable = default_weight_function,
    local_model_path: Optional[str] = None,
    hf_model_path: Optional[str] = "synthetic:sd15-inpaint",
    preloaded_utils: Optional[Tuple] = None,
    unconditional_input_prompt: str = "",
    model_token: Optional[str] = None,
    strength: float = 1.0,
    return_latents: bool = False,
):
    """paint_with_words_inpaint.py:137-270: 9-channel UNet input cat[latents, mask, masked-image latents]."""
    vae, unet, text_encoder, tokenizer, scheduler = (
        pww_load_tools(device, scheduler_type, local_model_path=local_model_path, hf_model_path=hf_model_path,
                       model_token=model_token)
        if preloaded_utils is None else preloaded_utils)
    width, height = init_image.size
    color_map_image = color_map_image.resize((width, height), Image.NEAREST)
    mask_image = mask_image.resize((width, height), Image.NEAREST)
    _, _, cond, uncond = _encode_text_color_inputs(
        text_encoder, tokenizer, device, color_map_image, color_context, input_prompt, unconditional_input_prompt)
    mask, masked_image = prepare_mask_and_masked_image(init_image, mask_image)

    scheduler.set_timesteps(num_inference_steps)
    init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
    t_start = max(num_inference_steps - init_timestep, 0)
    timesteps = scheduler.timesteps[t_start:]

    generator = torch.manual_seed(seed)
    image = preprocess(init_image).to(device=device)
    init_latents = 0.18215 * vae.encode(image.to(_module_dtype(vae, image.dtype))).latent_dist.sample().float()
    noise = torch.randn(init_latents.shape, generator=generator).to(device)
    latents = scheduler.add_noise(init_latents, noise, timesteps[:1])

    mask = F.interpolate(mask, size=(height // 8, width // 8)).to(device=device, dtype=latents.dtype)
    masked_image_latents = 0.18215 * vae.encode(masked_image.to(device=device, dtype=_module_dtype(vae, latents.dtype))).latent_dist.sample().float()
    mask = F.interpolate(mask, size=latents.shape[-2:], mode="nearest")
    masked_image_latents = F.interpolate(masked_image_latents, size=latents.shape[-2:], mode="nearest")
    total = latents.shape[1] + mask.shape[1] + masked_image_latents.shape[1]
    if total != unet.in_channels:
        raise ValueError(
            f"Incorrect configuration settings! The unet expects {unet.in_channels} input channels but received "
            f"num_channels_latents: {latents.shape[1]} + num_channels_mask: {mask.shape[1]} + "
            f"num_channels_masked_image: {masked_image_latents.shape[1]} = {total}.")
    sampler = PwWSampler(unet, scheduler, [cond], [uncond], latents, weight_function, guidance_scale,
                         extra_input=torch.cat([mask, masked_image_latents], 1).float(), timesteps=timesteps,
                         noise_seeds=[seed])
    latents = sampler.run()
    if return_latents:
        return latents
    return _pil_from_latents(vae, latents)[0]


# ---------------------------------------------------------------------------------------------
# pipeline classes (paint_with_words.py:513-842, paint_with_words_inpaint.py:273-575): API surface only
# ---------------------------------------------------------------------------------------------
class PipelineOutput:
    """Stand-in for diffusers' StableDiffusionPipelineOutput: `.images`, `.nsfw_content_detected`."""

    def __init__(self, images, nsfw_content_detected=False):
        self.images, self.nsfw_content_detected = images, nsfw_content_detected


class PaintWithWord_StableDiffusionPipeline:
    """Same constructor / `from_pretrained` / `plugin_cross_attention` / `__call__` surface as the reference class
    (paint_with_words.py:513-842); the work is `paint_with_words()` above (one `PwWSampler`).  Like the reference class
    it always uses its own LMS scheduler (paint_with_words.py:534-539) and has no regional blur (:574)."""

    def __init__(self, vae, text_encoder, tokenizer, unet, scheduler=None, safety_checker=None, feature_extractor=None,
                 requires_safety_checker: bool = False):
        self.vae, self.text_encoder, self.tokenizer, self.unet = vae, text_encoder, tokenizer, unet
        self.safety_checker, self.feature_extractor = safety_checker, feature_extractor
        self.scheduler = LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                                              num_train_timesteps=1000)
        self.plugin_cross_attention()

    @classmethod
    def from_pretrained(cls, save_dir, device: str = "cuda:0", **kwargs):
        vae, unet, text_encoder, tokenizer, scheduler = pww_load_tools(device, local_model_path=save_dir)
        return cls(vae=vae, text_encoder=text_encoder, tokenizer=tokenizer, unet=unet, scheduler=scheduler)

    def plugin_cross_attention(self):
        """paint_with_words.py:556-559."""
        return _attention.patch_unet(self.unet)

    @property
    def device(self):
        return next(iter(self.unet.parameters())).device

    def _run(self, fn, prompt, color_map_image, color_context, weight_function, num_inference_steps, guidance_scale,
             negative_prompt, seed, output_type, return_dict, callback, callback_steps, **extra):
        if isinstance(prompt, (list, tuple)):
            if len(prompt) != 1:
                raise ValueError("the Paint-with-Words pipelines take one prompt per call (batch size 1, paint_with_words.py:445)")
            prompt = prompt[0]
        if isinstance(negative_prompt, (list, tuple)):
            negative_prompt = negative_prompt[0]
        tools = (self.vae, self.unet, self.text_encoder, self.tokenizer, self.scheduler)
        latents = fn(color_context=color_context, color_map_image=color_map_image, input_prompt=prompt,
                     num_inference_steps=num_inference_steps, guidance_scale=guidance_scale, seed=seed,
                     device=str(self.device), weight_function=weight_function, preloaded_utils=tools,
                     unconditional_input_prompt=negative_prompt or "", return_latents=True, **extra)
        if callback is not None:
            callback(num_inference_steps - 1, int(self.scheduler.timesteps[-1]), latents)
        if output_type == "latent":
            images = latents
        else:
            images = _pil_from_latents(self.vae, latents)
            if output_type != "pil":
                images = np.stack([np.asarray(im, dtype=np.float32) / 255.0 for im in images])
        return PipelineOutput(images, False) if return_dict else (images, False)

    @torch.no_grad()
    def __call__(self, prompt, color_map_image=None, color_context={}, weight_function: Callable = default_weight_function,
                 height=None, width=None, num_inference_steps: int = 30, guidance_scale: float = 7.5, negative_prompt="",
                 num_images_per_prompt: int = 1, eta: float = 0.5, seed: int = 0, generator=None, image=None, latents=None,
                 output_type: str = "pil", return_dict: bool = True, callback=None, callback_steps: int = 1):
        extra = {} if image is None else {"init_image": image, "strength": eta}
        return self._run(paint_with_words, prompt, color_map_image, dict(color_context), weight_function,
                         num_inference_steps, guidance_scale, negative_prompt, seed, output_type, return_dict, callback,
                         callback_steps, **extra)


class PaintWithWord_StableDiffusionInpaintPipeline(PaintWithWord_StableDiffusionPipeline):
    """paint_with_words_inpaint.py:273-575: `__call__(prompt, image, mask_image, color_map_image, color_context, ...)`."""

    @classmethod
    def from_pretrained(cls, save_dir, device: str = "cuda:0", **kwargs):
        vae, unet, text_encoder, tokenizer, scheduler = pww_load_tools(device, local_model_path=save_dir)
        return cls(vae=vae, text_encoder=text_encoder, tokenizer=tokenizer, unet=unet, scheduler=scheduler)

    @torch.no_grad()
    def __call__(self, prompt, image=None, mask_image=None, color_map_image=None, color_context={},
                 weight_function: Callable = default_weight_function, height=None, width=None,
                 num_inference_steps: int = 30, guidance_scale: float = 7.5, negative_prompt="",
                 num_images_per_prompt: int = 1, eta: float = 1.0, seed: int = 0, generator=None, latents=None,
                 output_type: str = "pil", return_dict: bool = True, callback=None, callback_steps: int = 1):
        return self._run(paint_with_words_inpaint, prompt, color_map_image, dict(color_context), weight_function,
                         num_inference_steps, guidance_scale, negative_prompt, seed, output_type, return_dict, callback,
                         callback_steps, mask_image=mask_image, init_image=image, strength=eta)
