"""Shared test/bench inputs rebuilt from the committed golden fixtures (no /root/reference needed)."""
import math
import os

import numpy as np
import torch
from PIL import Image

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

SETTINGS = {
    "cat_dog": dict(
        ctx={(0, 0, 0): "cat,1.0", (255, 255, 255): "dog,1.0", (13, 255, 0): "tree,1.5",
             (90, 206, 255): "sky,0.2", (74, 18, 1): "ground,0.2"},
        prompt="realistic photo of a dog, cat, tree, with beautiful sky, on sandy ground"),
    "aurora": dict(
        ctx={(7, 9, 182): "aurora,0.5", (136, 178, 92): "full moon,1.5", (51, 193, 217): "mountains,0.4",
             (61, 163, 35): "a half-frozen lake,0.3", (89, 102, 255): "boat,2.0"},
        prompt="A digital painting of a half-frozen lake near mountains under a full moon and aurora. "
               "A boat is in the middle of the lake. Highly detailed."),
}
UNMATCHED_RGB = (1, 2, 3)   # stands for every antialiased pixel that matches no context colour


def color_map_image(name: str, size: int = 512) -> Image.Image:
    """PIL RGB image equivalent (for the mask builder) to the reference's contents/*.png colour map."""
    cm = np.load(os.path.join(GOLDEN, "color_maps.npz"))
    idx, pal = cm[f"{name}_index"], cm[f"{name}_palette"]
    lut = np.concatenate([np.array([UNMATCHED_RGB], dtype=np.uint8), pal], 0)
    img = Image.fromarray(lut[idx])
    if size != img.size[0]:
        img = img.resize((size, size), Image.NEAREST)   # gradio_pww.py:17 behaviour
    return img


def digest(t: torch.Tensor) -> np.ndarray:
    """[sum, sum of squares, weighted checksum] in float64 -- for tensors too big to commit.  Each sum is exactly
    rounded (math.fsum over the non-zero entries), so the digest of the same tensor is the same on every CPU, whatever
    its vector width or thread count."""
    x = t.double().flatten()
    nz = torch.nonzero(x).flatten()
    v, w = x[nz], (nz + 1).double() % 9973
    return np.array([math.fsum(v.tolist()), math.fsum((v * v).tolist()), math.fsum((v * w).tolist())])


def moon_mask_image(size: int = 512) -> Image.Image:
    cm = np.load(os.path.join(GOLDEN, "color_maps.npz"))
    img = Image.fromarray((cm["moon_mask"] * 255).astype(np.uint8), mode="L")
    return img if size == 512 else img.resize((size, size), Image.NEAREST)
