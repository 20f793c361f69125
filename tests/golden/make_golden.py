"""Generate the committed golden fixtures by running the UNMODIFIED reference functions.

    python tests/golden/make_golden.py          (build container only: needs /root/reference)

The reference has no tests or golden vectors for the Paint-with-Words path (SURVEY.md section 4), so the
oracle (oracle/pww_oracle.py) is pinned against the reference's own code executed here through
oracle/ref_loader.py.  Outputs (all under tests/golden/, all small):

  color_maps.npz     region-index maps derived from contents/example_input.png, contents/aurora_1.png
                     (0 = pixel matches no context colour, i+1 = i-th colour of the runner.py setting) and
                     the binarised contents/moon_mask.png -- the only inputs the mask builder looks at, so
                     the GPU box (which has no /root/reference) can rebuild equivalent PIL images.
  mask_builder.npz   reference outputs of always_round, _extract_seed_and_sigma_from_context,
                     _image_context_seperator, _tokens_img_attention_weight (ratios 8/16/32/64 and ORIG
                     digests), _get_binary_mask, _blur_image_mask for the runner.py settings.
  attention.npz      reference `inj_forward` (CPU fp32) inputs and outputs: dict context with max / std /
                     sigma^2 weight functions, uncond dict, tensor context, self-attention, ORIG fallback.
"""
from __future__ import annotations

import math
import os
import sys

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.ref_loader import REFERENCE_ROOT, load_reference  # noqa: E402
from paint_with_words_sd_b200.synthetic import SimpleWordTokenizer  # noqa: E402
from paint_with_words_sd_b200.unet import CrossAttention  # noqa: E402
from tests.fixtures import digest  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))

# settings restated from runner.py:9-72 (colour -> "label,strength[,seed]") -- data, not code
SETTINGS = {
    "cat_dog": dict(
        png="example_input.png",
        ctx={(0, 0, 0): "cat,1.0", (255, 255, 255): "dog,1.0", (13, 255, 0): "tree,1.5",
             (90, 206, 255): "sky,0.2", (74, 18, 1): "ground,0.2"},
        prompt="realistic photo of a dog, cat, tree, with beautiful sky, on sandy ground"),
    "aurora": dict(
        png="aurora_1.png",
        ctx={(7, 9, 182): "aurora,0.5", (136, 178, 92): "full moon,1.5", (51, 193, 217): "mountains,0.4",
             (61, 163, 35): "a half-frozen lake,0.3", (89, 102, 255): "boat,2.0"},
        prompt="A digital painting of a half-frozen lake near mountains under a full moon and aurora. "
               "A boat is in the middle of the lake. Highly detailed."),
}
AURORA_SEED_CTX = {(7, 9, 182): "aurora,0.5,-1", (136, 178, 92): "full moon,1.5,-1",
                   (51, 193, 217): "mountains,0.4,-1", (61, 163, 35): "a half-frozen lake,0.3,-1",
                   (89, 102, 255): "boat,2.0,2077"}


def region_index_map(img: Image.Image, colors) -> np.ndarray:
    a = np.array(img.convert("RGB"))
    idx = np.zeros(a.shape[:2], dtype=np.uint8)
    for i, c in enumerate(colors):
        idx[(a == np.array(c, dtype=np.uint8)).all(-1)] = i + 1
    return idx


def main():
    ref = load_reference()
    tok = SimpleWordTokenizer()
    contents = os.path.join(REFERENCE_ROOT, "contents")

    # ---- colour maps ----------------------------------------------------------------------
    cm = {}
    for name, s in SETTINGS.items():
        img = Image.open(os.path.join(contents, s["png"])).convert("RGB")
        cm[f"{name}_index"] = region_index_map(img, list(s["ctx"].keys()))
        cm[f"{name}_palette"] = np.array(list(s["ctx"].keys()), dtype=np.uint8)
    moon = np.array(Image.open(os.path.join(contents, "moon_mask.png")).convert("L"))
    cm["moon_mask"] = (moon.astype(np.float32) / 255.0 >= 0.5).astype(np.uint8)
    np.savez_compressed(os.path.join(OUT, "color_maps.npz"), **cm)

    # ---- mask builder -----------------------------------------------------------------------
    mb = {}
    xs = [0.5, 1.5, 2.5, 3.5, 4.5, 8.5, 16.25, 31.5, 32.5, 33.5, 63.5, 64.0, 12.49, 12.51, 95.5, 96.5]
    mb["always_round_x"] = np.array(xs)
    mb["always_round_y"] = np.array([ref.always_round(x) for x in xs])

    seed_in = {"a": "boat,2.0,2077", "b": "sky,0.5,-1", "c": "x,1.0,5,3.0", "d": "cat,1.0", "e": "a, b,0.3,7"}
    cc, seeds, sigmas = ref._extract_seed_and_sigma_from_context(dict(seed_in))
    mb["seed_ctx_out"] = np.array([cc[k] for k in seed_in])
    mb["seed_keys"], mb["seed_vals"] = np.array(list(seeds.keys())), np.array(list(seeds.values()))
    mb["sigma_keys"], mb["sigma_vals"] = np.array(list(sigmas.keys())), np.array(list(sigmas.values()))

    for name, s in SETTINGS.items():
        for size in (512, 256):
            img = Image.open(os.path.join(contents, s["png"])).convert("RGB")
            if size != 512:
                img = img.resize((size, size), Image.NEAREST)     # gradio_pww.py:17
            text_input = tok([s["prompt"]], padding="max_length", max_length=tok.model_max_length,
                             truncation=True, return_tensors="pt")
            sep, w, h = ref._image_context_seperator(img, dict(s["ctx"]), tok)
            tag = f"{name}_{size}"
            mb[f"{tag}_ids"] = text_input["input_ids"][0].numpy()
            mb[f"{tag}_region_pixels"] = np.array([int((m > 0).sum()) for _, m in sep])
            mb[f"{tag}_region_sum"] = np.array([float(m.double().sum()) for _, m in sep])
            for r in (8, 16, 32, 64):
                wt = ref._tokens_img_attention_weight(sep, text_input, ratio=r)
                mb[f"{tag}_w{r}"] = wt.numpy()
            orig = ref._tokens_img_attention_weight(sep, text_input, ratio=1, original_shape=True)
            mb[f"{tag}_orig_shape"] = np.array(orig.shape)
            mb[f"{tag}_orig_digest"] = digest(orig)
            if size == 512 and name == "aurora":
                # regional seeding + blur (runner.py:61-72 style context)
                ctx2 = dict(AURORA_SEED_CTX)
                ctx2[(136, 178, 92)] = "full moon,1.5,-1,4.0"
                cc2, seeds2, sigmas2 = ref._extract_seed_and_sigma_from_context(ctx2)
                sep2, _, _ = ref._image_context_seperator(img, cc2, tok)
                masks = ref._get_binary_mask(sep2, seeds2, dtype=torch.float32, size=(64, 64))
                mb["aurora_binary_mask"] = torch.cat(masks, 0).numpy()
                blurred = ref._blur_image_mask(list(sep2), sigmas2)
                bm = blurred[1][1]
                mb["aurora_blur_sub"] = bm[::8, ::8].numpy()
                mb["aurora_blur_digest"] = digest(bm)
                # region-seeded latents exactly as paint_with_words.py:445-455
                latent_size = (1, 4, 64, 64)
                latents = torch.randn(latent_size, generator=torch.manual_seed(0))
                multi = [torch.randn(latent_size, generator=torch.manual_seed(s_)) for s_ in seeds2.values()]
                fg = (sum(masks) > 0).squeeze()
                summed = sum(l * m for l, m in zip(multi, masks))
                latents[:, :, fg] = summed[:, :, fg]
                mb["aurora_seeded_latents"] = latents.numpy()
    np.savez_compressed(os.path.join(OUT, "mask_builder.npz"), **mb)

    # ---- attention (reference inj_forward, CPU fp32) -------------------------------------------
    at = {}
    g = torch.Generator().manual_seed(20260922)
    heads, d, n_side, dc, T = 2, 40, 8, 32, 77
    C, N = heads * d, n_side * n_side
    attn = CrossAttention(C, dc, heads, d)
    attn_self = CrossAttention(C, None, heads, d)
    for m in (attn, attn_self):
        for p in m.parameters():
            p.data = torch.randn(p.shape, generator=g) * (0.3 if p.dim() > 1 else 0.05)
    x = torch.randn(1, N, C, generator=g)
    ctx = torch.randn(1, T, dc, generator=g)
    w = torch.zeros(N, T)
    w[:, 3] = (torch.rand(N, generator=g) > 0.5).float() * 1.5
    w[:, 7:9] = (torch.rand(N, 1, generator=g) > 0.7).float() * 0.4
    w_orig = torch.zeros(24, 24, T)                      # ORIG map for the KeyError path (N=64 -> ratio 3)
    w_orig[4:14, 6:20, 5] = 2.0
    w_orig[10:24, 0:9, 11:13] = 0.7
    sigma = torch.tensor(7.25)
    fns = {
        "max": lambda w, sigma, qk: 0.4 * w * math.log(1 + sigma) * qk.max(),
        "std": lambda w, sigma, qk: 0.5 * w * math.log(1 + sigma) * qk.std(),
        "std_sig2": lambda w, sigma, qk: 0.5 * w * math.log(1 + sigma ** 2) * qk.std(),
        "zero": lambda w, sigma, qk: 0.0,
    }
    for name, p in list(attn.named_parameters()):
        at[f"attn.{name}"] = p.detach().numpy()
    for name, p in list(attn_self.named_parameters()):
        at[f"attn_self.{name}"] = p.detach().numpy()
    at.update(x=x.numpy(), ctx=ctx.numpy(), w=w.numpy(), w_orig=w_orig.numpy(), sigma=np.float32(sigma.item()),
              heads=np.int64(heads))
    with torch.no_grad():
        for fname, f in fns.items():
            c = {"CONTEXT_TENSOR": ctx, f"CROSS_ATTENTION_WEIGHT_{N}": w, "CROSS_ATTENTION_WEIGHT_ORIG": w_orig,
                 "SIGMA": sigma, "WEIGHT_FUNCTION": f}
            at[f"out_dict_{fname}"] = ref.inj_forward(attn, x, c).numpy()
        c = {"CONTEXT_TENSOR": ctx, "CROSS_ATTENTION_WEIGHT_4096": w, "CROSS_ATTENTION_WEIGHT_ORIG": 0,
             "SIGMA": sigma, "WEIGHT_FUNCTION": fns["max"]}
        at["out_dict_uncond_int0"] = ref.inj_forward(attn, x, c).numpy()
        c = {"CONTEXT_TENSOR": ctx, "CROSS_ATTENTION_WEIGHT_ORIG": w_orig, "SIGMA": sigma,
             "WEIGHT_FUNCTION": fns["max"]}
        at["out_dict_orig_fallback"] = ref.inj_forward(attn, x, c).numpy()
        at["out_tensor_ctx"] = ref.inj_forward(attn, x, ctx).numpy()
        at["out_self"] = ref.inj_forward(attn_self, x, None).numpy()
    np.savez_compressed(os.path.join(OUT, "attention.npz"), **at)
    for f in ("color_maps.npz", "mask_builder.npz", "attention.npz"):
        print(f, os.path.getsize(os.path.join(OUT, f)), "bytes")


if __name__ == "__main__":
    main()
