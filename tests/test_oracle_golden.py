"""Pin the oracle (oracle/pww_oracle.py) against outputs of the UNMODIFIED reference captured in
tests/golden/*.npz by tests/golden/make_golden.py (the reference ships no tests for this path)."""
import math

import numpy as np
import pytest
import torch

from oracle import pww_oracle as O
from paint_with_words_sd_b200.synthetic import SimpleWordTokenizer
from paint_with_words_sd_b200.unet import CrossAttention
from tests.fixtures import SETTINGS, color_map_image, digest


def test_always_round(golden):
    mb = golden["mask_builder"]
    got = [O.always_round(float(x)) for x in mb["always_round_x"]]
    assert got == mb["always_round_y"].tolist()


def test_seed_sigma_parser(golden):
    mb = golden["mask_builder"]
    seed_in = {"a": "boat,2.0,2077", "b": "sky,0.5,-1", "c": "x,1.0,5,3.0", "d": "cat,1.0", "e": "a, b,0.3,7"}
    cc, seeds, sigmas = O.extract_seed_and_sigma_from_context(dict(seed_in))
    assert [cc[k] for k in seed_in] == mb["seed_ctx_out"].tolist()
    assert list(seeds.keys()) == mb["seed_keys"].tolist() and list(seeds.values()) == mb["seed_vals"].tolist()
    assert list(sigmas.keys()) == mb["sigma_keys"].tolist() and list(sigmas.values()) == mb["sigma_vals"].tolist()


@pytest.mark.parametrize("name", ["cat_dog", "aurora"])
@pytest.mark.parametrize("size", [512, 256])
def test_weight_maps_bit_exact(golden, name, size):
    mb = golden["mask_builder"]
    tok = SimpleWordTokenizer()
    s = SETTINGS[name]
    img = color_map_image(name, size)
    ids = tok([s["prompt"]], padding="max_length", max_length=77, truncation=True, return_tensors="pt")["input_ids"][0]
    tag = f"{name}_{size}"
    assert ids.tolist() == mb[f"{tag}_ids"].tolist()
    sep, w, h = O.image_context_separator(np.array(img), dict(s["ctx"]), tok)
    assert (w, h) == (size, size)
    assert [int((m > 0).sum()) for _, m in sep] == mb[f"{tag}_region_pixels"].tolist()
    for r in (8, 16, 32, 64):
        got = O.tokens_img_attention_weight(sep, ids.tolist(), ratio=r)
        assert torch.equal(got, torch.from_numpy(mb[f"{tag}_w{r}"])), f"ratio {r} not bit-exact"
    orig = O.tokens_img_attention_weight(sep, ids.tolist(), ratio=1, original_shape=True)
    assert list(orig.shape) == mb[f"{tag}_orig_shape"].tolist()
    assert np.array_equal(digest(orig), mb[f"{tag}_orig_digest"])


def test_binary_mask_blur_and_seeded_latents(golden):
    mb = golden["mask_builder"]
    tok = SimpleWordTokenizer()
    ctx = {(7, 9, 182): "aurora,0.5,-1", (136, 178, 92): "full moon,1.5,-1,4.0", (51, 193, 217): "mountains,0.4,-1",
           (61, 163, 35): "a half-frozen lake,0.3,-1", (89, 102, 255): "boat,2.0,2077"}
    cc, seeds, sigmas = O.extract_seed_and_sigma_from_context(ctx)
    assert seeds == {4: 2077} and sigmas == {1: 4.0}
    sep, _, _ = O.image_context_separator(np.array(color_map_image("aurora")), cc, tok)
    masks = O.get_binary_mask(sep, seeds, torch.float32, (64, 64))
    assert torch.equal(torch.cat(masks, 0), torch.from_numpy(mb["aurora_binary_mask"]))
    blurred = O.gaussian_blur_39(sep[1][1], 4.0)
    assert torch.allclose(blurred[::8, ::8], torch.from_numpy(mb["aurora_blur_sub"]), atol=1e-6, rtol=1e-5)
    lat = O.regional_seed_latents((1, 4, 64, 64), 0, seeds, sep)
    assert torch.equal(lat, torch.from_numpy(mb["aurora_seeded_latents"]))


def _modules(at):
    heads = int(at["heads"])
    C = at["x"].shape[-1]
    dc = at["ctx"].shape[-1]
    attn = CrossAttention(C, dc, heads, C // heads)
    attn_self = CrossAttention(C, None, heads, C // heads)
    for name, p in attn.named_parameters():
        p.data = torch.from_numpy(at[f"attn.{name}"])
    for name, p in attn_self.named_parameters():
        p.data = torch.from_numpy(at[f"attn_self.{name}"])
    return attn, attn_self


FNS = {
    "max": lambda w, sigma, qk: 0.4 * w * math.log(1 + sigma) * qk.max(),
    "std": lambda w, sigma, qk: 0.5 * w * math.log(1 + sigma) * qk.std(),
    "std_sig2": lambda w, sigma, qk: 0.5 * w * math.log(1 + sigma ** 2) * qk.std(),
    "zero": lambda w, sigma, qk: 0.0,
}


@torch.no_grad()
def test_inj_forward_matches_reference(golden):
    at = golden["attention"]
    attn, attn_self = _modules(at)
    x, ctx, w = (torch.from_numpy(at[k]) for k in ("x", "ctx", "w"))
    w_orig, sigma = torch.from_numpy(at["w_orig"]), torch.tensor(float(at["sigma"]))
    N = x.shape[1]
    tol = dict(atol=2e-6, rtol=1e-5)
    for name, f in FNS.items():
        c = {"CONTEXT_TENSOR": ctx, f"CROSS_ATTENTION_WEIGHT_{N}": w, "CROSS_ATTENTION_WEIGHT_ORIG": w_orig,
             "SIGMA": sigma, "WEIGHT_FUNCTION": f}
        assert torch.allclose(O.inj_forward(attn, x, c), torch.from_numpy(at[f"out_dict_{name}"]), **tol), name
    c = {"CONTEXT_TENSOR": ctx, "CROSS_ATTENTION_WEIGHT_4096": w, "CROSS_ATTENTION_WEIGHT_ORIG": 0, "SIGMA": sigma,
         "WEIGHT_FUNCTION": FNS["max"]}
    assert torch.allclose(O.inj_forward(attn, x, c), torch.from_numpy(at["out_dict_uncond_int0"]), **tol)
    c = {"CONTEXT_TENSOR": ctx, "CROSS_ATTENTION_WEIGHT_ORIG": w_orig, "SIGMA": sigma, "WEIGHT_FUNCTION": FNS["max"]}
    assert torch.allclose(O.inj_forward(attn, x, c), torch.from_numpy(at["out_dict_orig_fallback"]), **tol)
    assert torch.allclose(O.inj_forward(attn, x, ctx), torch.from_numpy(at["out_tensor_ctx"]), **tol)
    assert torch.allclose(O.inj_forward(attn_self, x, None), torch.from_numpy(at["out_self"]), **tol)


@torch.no_grad()
def test_f64_form_agrees_with_torch_form(golden):
    """Second, independent statement of the fused region (numpy float64) against the torch form."""
    at = golden["attention"]
    attn, _ = _modules(at)
    x, ctx, w = (torch.from_numpy(at[k]) for k in ("x", "ctx", "w"))
    q, k, v = attn.to_q(x), attn.to_k(ctx), attn.to_v(ctx)
    sigma = float(at["sigma"])
    for stat, coef in (("max", 0.4), ("std", 0.5)):
        g = coef * math.log(1 + sigma)
        ref = O.attention_core(q, k, v, attn.heads, attn.scale,
                               lambda s: g * w * (s.max() if stat == "max" else s.std()))
        got = O.attention_core_f64(q[0].numpy(), k[0].numpy(), v[0].numpy(), attn.heads, attn.scale, w.numpy(), g, stat)
        assert np.allclose(got, ref[0].numpy(), atol=5e-6, rtol=1e-5)
