"""Host side of the product (conditioning builder, weight-function probe, scheduler, UNet contract) on CPU."""
import math

import numpy as np
import pytest
import torch

import paint_with_words_sd_b200 as P
from paint_with_words_sd_b200 import conditioning as C
from paint_with_words_sd_b200.scheduler import LMSDiscreteScheduler
from paint_with_words_sd_b200.synthetic import RandomTextEncoder, SimpleWordTokenizer
from paint_with_words_sd_b200.unet import UNetConfig, attention_modules, build_unet
from paint_with_words_sd_b200.weight_function import (STAT_MAX, STAT_STD, UnsupportedWeightFunction, WeightFunction,
                                                      g_of_sigma, probe_weight_function)
from oracle import loop as oracle_loop
from oracle import pww_oracle as O
from tests.fixtures import SETTINGS, color_map_image, digest


def test_always_round_matches_golden(golden):
    mb = golden["mask_builder"]
    assert [C.always_round(float(x)) for x in mb["always_round_x"]] == mb["always_round_y"].tolist()


def test_seed_parser_matches_golden_and_mutates(golden):
    mb = golden["mask_builder"]
    d = {"a": "boat,2.0,2077", "b": "sky,0.5,-1", "c": "x,1.0,5,3.0", "d": "cat,1.0", "e": "a, b,0.3,7"}
    out, seeds, sigmas = C._extract_seed_and_sigma_from_context(d)
    assert out is d                                    # in-place, like the reference (pww.py:296)
    assert [d[k] for k in d] == mb["seed_ctx_out"].tolist()
    assert list(seeds.items()) == list(zip(mb["seed_keys"].tolist(), mb["seed_vals"].tolist()))
    assert list(sigmas.items()) == list(zip(mb["sigma_keys"].tolist(), mb["sigma_vals"].tolist()))


@pytest.mark.parametrize("name,size", [("cat_dog", 256), ("aurora", 512), ("cat_dog", 512), ("aurora", 256)])
def test_encode_text_color_inputs_bit_exact(golden, name, size):
    mb = golden["mask_builder"]
    s = SETTINGS[name]
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(32)
    ctx = dict(s["ctx"])
    extra_seeds, sep, cond, uncond = C._encode_text_color_inputs(enc, tok, "cpu", color_map_image(name, size), ctx,
                                                                 s["prompt"], "")
    assert extra_seeds == {}
    tag = f"{name}_{size}"
    for r in (8, 16, 32, 64):
        n = (size // r) ** 2
        key = f"CROSS_ATTENTION_WEIGHT_{n}"
        assert torch.equal(cond[key], torch.from_numpy(mb[f"{tag}_w{r}"])), key   # bit-exact mask step
        assert uncond[key] == 0
    assert uncond["CROSS_ATTENTION_WEIGHT_ORIG"] == 0
    assert list(cond["CROSS_ATTENTION_WEIGHT_ORIG"].shape) == mb[f"{tag}_orig_shape"].tolist()
    assert cond["CONTEXT_TENSOR"].shape == (1, 77, 32) and uncond["CONTEXT_TENSOR"].shape == (1, 77, 32)


def test_hex_color_keys_and_missing_color(capsys):
    tok = SimpleWordTokenizer()
    img = color_map_image("aurora", 256)
    sep, w, h = C._image_context_seperator(img, {"#0709b6": "aurora,1.0", "#010203": "ghost,2.0", (9, 9, 9): "nothing,1"}, tok)
    assert int((sep[0][1] > 0).sum()) > 0 and float(sep[1][1].max()) == 2.0
    assert float(sep[2][1].sum()) == 0.0
    assert "not found in image" in capsys.readouterr().out
    sep, w, h = C._image_context_seperator(None, {}, tok)
    assert sep[0][0] == [-1] and (w, h) == (512, 512)


def test_repeated_and_missing_labels_accumulate():
    tok = SimpleWordTokenizer()
    prompt = "a cat and a cat on a mat"
    ids = tok([prompt], padding="max_length", max_length=77, truncation=True, return_tensors="pt")
    m = torch.zeros(64, 64); m[:32] = 1.5
    sep = [(tok("cat")["input_ids"][1:-1], m), (tok("a cat")["input_ids"][1:-1], m), (tok("dog")["input_ids"][1:-1], m)]
    w = C._tokens_img_attention_weight(sep, ids, ratio=8)
    ref = O.tokens_img_attention_weight(sep, ids["input_ids"][0].tolist(), ratio=8)
    assert torch.equal(w, ref)
    cat_cols = [i for i, t in enumerate(ids["input_ids"][0].tolist()) if t == sep[0][0][0]]
    assert len(cat_cols) == 2 and float(w[0, cat_cols[0]]) == 3.0      # "cat" + "a cat" both hit the column


@pytest.mark.parametrize("name,size", [("aurora", 512), ("cat_dog", 256)])
def test_factored_weight_map_reproduces_the_dense_one(name, size):
    """W = M C^T (SURVEY 8f-4 packed mask format): bit-exact where every token belongs to one region (the reference's
    own examples), and the factors are tiny compared with the dense map."""
    tok = SimpleWordTokenizer()
    s = SETTINGS[name]
    ctx, _, _ = C._extract_seed_and_sigma_from_context(dict(s["ctx"]))
    sep, _, _ = C._image_context_seperator(color_map_image(name, size), ctx, tok)
    ids = tok([s["prompt"]], padding="max_length", max_length=77, truncation=True, return_tensors="pt")
    for ratio in (8, 16, 32, 64):
        w = C._tokens_img_attention_weight(sep, ids, ratio=ratio)
        m, c = C._tokens_img_attention_factors(sep, ids, ratio=ratio)
        assert m.shape[0] == w.shape[0] and c.shape[0] == 77 and m.shape[1] == c.shape[1] <= len(sep)
        assert torch.equal(m @ c.T, w)
        if w.shape[0] >= 1024:
            assert m.numel() + c.numel() < w.numel() / 5
        # fp16 storage of the factors (what a UMMA operand would hold) stays far inside the attention tolerance
        w16 = m.half().float() @ c.T
        assert (w16 - w).abs().max().item() <= 2 ** -11 * w.abs().max().item()


def test_factored_weight_map_with_repeats_and_missing_labels():
    tok = SimpleWordTokenizer()
    ids = tok(["a cat and a cat on a mat"], padding="max_length", max_length=77, truncation=True, return_tensors="pt")
    m1 = torch.zeros(64, 64); m1[:32] = 1.5
    m2 = torch.zeros(64, 64); m2[16:48, 8:40] = 0.7
    sep = [(tok("cat")["input_ids"][1:-1], m1), (tok("a cat")["input_ids"][1:-1], m2), (tok("dog")["input_ids"][1:-1], m1)]
    w = C._tokens_img_attention_weight(sep, ids, ratio=8)
    m, c = C._tokens_img_attention_factors(sep, ids, ratio=8)
    assert m.shape[1] == 2                                   # "dog" is not in the prompt: dropped like the reference does
    assert float(c.max()) == 2.0 or float(c.sum()) == 6.0    # "cat" twice (1 token), "a cat" twice (2 tokens)
    assert torch.allclose(m @ c.T, w, rtol=0, atol=1e-6)


def test_orig_fallback_matches_oracle(golden):
    w_orig = torch.from_numpy(golden["attention"]["w_orig"])
    assert torch.equal(C.expand_orig_weight_map(w_orig, 64), O.orig_map_fallback(w_orig, 64))


# ---- weight function probe ------------------------------------------------------------------------
def test_probe_family():
    sig = torch.tensor(3.0)
    f1 = lambda w, sigma, qk: 0.4 * w * math.log(1 + sigma) * qk.max()
    f2 = lambda w, sigma, qk: 0.5 * w * math.log(1 + sigma ** 2) * qk.std()
    f0 = lambda w, sigma, qk: 0.0
    p1, p2, p0 = (probe_weight_function(f, sig) for f in (f1, f2, f0))
    assert p1.stat == STAT_MAX and p2.stat == STAT_STD and p0.is_zero
    assert g_of_sigma(f1, p1, sig) == pytest.approx(0.4 * math.log(4.0), rel=1e-6)
    assert g_of_sigma(f2, p2, sig) == pytest.approx(0.5 * math.log(10.0), rel=1e-6)
    assert g_of_sigma(f0, p0, sig) == 0.0
    wf = WeightFunction(0.4, 1.0, "max")
    assert probe_weight_function(wf).stat == STAT_MAX and wf.g(3.0) == pytest.approx(0.4 * math.log(4.0))
    # a WeightFunction is also a valid reference-style callable
    qk = torch.randn(2, 5, 7)
    w = torch.rand(5, 7)
    assert torch.allclose(wf(w, sig, qk), f1(w, sig, qk))


def test_probe_rejects_unfusable():
    for bad in (lambda w, s, qk: w * qk.mean(), lambda w, s, qk: w * qk.max() * qk.std(),
                lambda w, s, qk: w * w * qk.max(), lambda w, s, qk: w * qk.max() ** 2,
                lambda w, s, qk: (w + 1.0) * qk.max()):
        with pytest.raises(UnsupportedWeightFunction):
            probe_weight_function(bad, 2.0)


# ---- scheduler -------------------------------------------------------------------------------------
def test_lms_schedule_values():
    s = LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear", num_train_timesteps=1000)
    assert float(s.init_noise_sigma) == pytest.approx(14.6146, rel=1e-4)
    s.set_timesteps(30)
    assert len(s.timesteps) == 30 and len(s.sigmas) == 31 and float(s.sigmas[-1]) == 0.0
    assert float(s.sigmas[0]) == pytest.approx(14.6146, rel=1e-4) and float(s.sigmas[29]) == pytest.approx(0.0292, rel=2e-2)
    assert float(s.timesteps[0]) == 999.0 and float(s.timesteps[-1]) == 0.0
    # first step is Euler: coefficient = sigma_next - sigma
    assert s._coeffs[0][0] == pytest.approx(float(s.sigmas[1] - s.sigmas[0]), rel=1e-4)
    x = torch.randn(1, 4, 8, 8)
    assert torch.allclose(s.scale_model_input(x, s.timesteps[3]), x / (float(s.sigmas[3]) ** 2 + 1) ** 0.5)
    # order-4 coefficients integrate the Lagrange basis: they sum to the interval length
    assert sum(s._coeffs[10]) == pytest.approx(float(s.sigmas[11] - s.sigmas[10]), rel=1e-3)


def test_lms_step_exact_for_linear_ode():
    """dx/dsigma = const is integrated exactly by any LMS order."""
    s = LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    s.set_timesteps(12)
    x = torch.full((1, 1, 2, 2), 5.0)
    eps = torch.full_like(x, 0.25)
    x0 = x.clone()
    for t in s.timesteps:
        x = s.step(eps, t, x).prev_sample
    assert torch.allclose(x, x0 + 0.25 * (0.0 - float(s.sigmas[0])), atol=1e-4)


# ---- UNet contract + CPU loop with the oracle attention ----------------------------------------------
def test_unet_contract_and_reference_loop_runs():
    unet = build_unet(UNetConfig.tiny(), seed=0)
    mods = attention_modules(unet)
    assert len(mods) == 32 and all(hasattr(m, a) for m in mods for a in ("to_q", "to_k", "to_v", "to_out", "heads", "scale"))
    tok, enc = SimpleWordTokenizer(), RandomTextEncoder(64)
    s = SETTINGS["cat_dog"]
    _, _, cond, uncond = C._encode_text_color_inputs(enc, tok, "cpu", color_map_image("cat_dog", 128), dict(s["ctx"]),
                                                     s["prompt"], "")
    sch = LMSDiscreteScheduler(beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear")
    sch.set_timesteps(3)
    lat = torch.randn(1, 4, 16, 16, generator=torch.manual_seed(0)) * sch.init_noise_sigma
    try:
        assert oracle_loop.patch_with_oracle(unet) == 32
        f = lambda w, sigma, qk: 0.4 * w * math.log(1 + sigma) * qk.max()
        out = oracle_loop.reference_denoise_loop(unet, sch, cond, uncond, lat, f)
        sch.set_timesteps(3)
        out0 = oracle_loop.reference_denoise_loop(unet, sch, cond, uncond, lat, lambda w, sigma, qk: 0.0)
    finally:
        P.unpatch_all()
        for m in mods[:1]:
            if "__call__" in m.__class__.__dict__:
                delattr(m.__class__, "__call__")
    assert out.shape == lat.shape and torch.isfinite(out).all()
    assert (out - out0).abs().max() > 1e-4          # the bias changes the result


def test_product_attention_refuses_cpu():
    unet = build_unet(UNetConfig.tiny(), seed=0)
    m = attention_modules(unet)[0]
    with pytest.raises(RuntimeError):
        P.inj_forward(m, torch.randn(1, 16, 32))


# ------------------------------------------------------------------------------------------------------------------
# packed weight maps (SURVEY 8f-4): the column dictionary the one-launch kernel consumes
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["aurora_512", "cat_dog_512", "aurora_256", "cat_dog_256"])
@pytest.mark.parametrize("ratio", [8, 16, 32, 64])
def test_pack_weight_map_reproduces_the_reference_maps(golden, name, ratio):
    """pack -> unpack gives back the map the REFERENCE built (tests/golden/mask_builder.npz) to hi+lo fp16 precision:
    relative 2^-21 (two fp16 mantissas) or the fp16 subnormal step 2^-25 absolute, whichever is larger; the zero
    pattern and the column sharing are exact."""
    from paint_with_words_sd_b200.conditioning import PACK_CAPACITY, pack_weight_map, unpack_weight_map
    w = torch.from_numpy(golden["mask_builder"][f"{name}_w{ratio}"])
    packed = pack_weight_map(w)
    assert packed is not None
    mpack, cidx = packed
    assert mpack.shape == (1, w.shape[0], 32) and mpack.dtype == torch.float16 and cidx.shape == (1, 80)
    assert int(cidx.max()) < PACK_CAPACITY and (cidx[0, 77:] == -1).all()
    rec = unpack_weight_map(mpack, cidx)[0]
    assert torch.equal(rec == 0, w == 0)
    assert ((rec - w).abs() <= torch.clamp(2.0 ** -21 * w.abs(), min=2.0 ** -25)).all()
    # tokens of one label share a dictionary entry: as many entries as distinct non-zero columns
    nz = [tuple(w[:, t].tolist()) for t in range(77) if (w[:, t] != 0).any()]
    assert len(set(nz)) == int(cidx.max()) + 1
    assert (mpack[0, :, :10] == mpack[0, :, 20:30]).all() and (mpack[0, :, 30:] == 0).all()


def test_pack_weight_map_limits():
    from paint_with_words_sd_b200.conditioning import pack_weight_map
    n = 64
    w = torch.zeros(2, n, 77)
    mp, ci = pack_weight_map(w)                                   # all-zero maps pack to nothing
    assert (mp == 0).all() and (ci == -1).all()
    g = torch.Generator().manual_seed(0)
    w[1, :, :11] = torch.rand(n, 11, generator=g)                 # 11 distinct columns: over capacity
    assert pack_weight_map(w) is None
    w[1, :, 10] = w[1, :, 9]                                      # ... 10 distinct: fits
    assert pack_weight_map(w) is not None
    w[0, 0, 0] = 1.0e5                                            # outside fp16 range
    assert pack_weight_map(w) is None


def test_product_binary_mask_blur_and_seeded_latents_match_reference_fixtures(golden):
    """The PRODUCT's `_get_binary_mask`, `_blur_image_mask` and `initial_latents` (paint_with_words.py:300-312, 445-455)
    against the fixtures the unmodified reference produced (tests/golden/make_golden.py): bit-exact for the binary
    masks and the regionally seeded latents, 1e-6 for the 39x39 Gaussian blur."""
    from paint_with_words_sd_b200.pipeline import initial_latents
    mb = golden["mask_builder"]
    tok = SimpleWordTokenizer()
    ctx = {(7, 9, 182): "aurora,0.5,-1", (136, 178, 92): "full moon,1.5,-1,4.0", (51, 193, 217): "mountains,0.4,-1",
           (61, 163, 35): "a half-frozen lake,0.3,-1", (89, 102, 255): "boat,2.0,2077"}
    ctx, seeds, sigmas = C._extract_seed_and_sigma_from_context(ctx)
    assert seeds == {4: 2077} and sigmas == {1: 4.0}
    sep, w, h = C._image_context_seperator(color_map_image("aurora"), ctx, tok)
    masks = C._get_binary_mask(sep, seeds, torch.float32, (64, 64))
    assert torch.equal(torch.cat(masks, 0), torch.from_numpy(mb["aurora_binary_mask"]))
    lat = initial_latents((1, 4, 64, 64), 0, seeds, sep)
    assert torch.equal(lat, torch.from_numpy(mb["aurora_seeded_latents"]))
    blurred = C._blur_image_mask(list(sep), sigmas)[1][1]
    assert torch.allclose(blurred[::8, ::8], torch.from_numpy(mb["aurora_blur_sub"]), atol=1e-6, rtol=1e-5)
    assert np.allclose(digest(blurred), mb["aurora_blur_digest"], rtol=1e-6)
