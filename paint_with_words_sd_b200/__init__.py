"""paint_with_words_sd_b200 -- B200-native Paint-with-Words attention path.

Same public names as the reference package (paint_with_words/__init__.py:1-3) plus the native pieces.
The repo root also carries the hyphenated alias `paint-with-words-sd_b200` (a symlink to this
directory) because the canonical project name is not an importable identifier.
"""
from .attention import PwWAttnProcessor, inj_forward, patch_unet, unpatch_all  # noqa: F401
from .conditioning import (  # noqa: F401
    _blur_image_mask, _encode_text_color_inputs, _extract_seed_and_sigma_from_context, _get_binary_mask,
    _image_context_seperator, _img_importance_flatten, _tokens_img_attention_weight, always_round,
)
from .pipeline import (  # noqa: F401
    PaintWithWord_StableDiffusionInpaintPipeline, PaintWithWord_StableDiffusionPipeline, PwWSampler, paint_with_words,
    paint_with_words_inpaint, preprocess, prepare_mask_and_masked_image, pww_load_tools,
)
from .scheduler import (  # noqa: F401
    DPMSolverMultistepScheduler, EulerAncestralDiscreteScheduler, EulerDiscreteScheduler, LMSDiscreteScheduler,
)
from .weight_function import UnsupportedWeightFunction, WeightFunction, probe_weight_function  # noqa: F401

__version__ = "0.1.0"
