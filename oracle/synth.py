"""Deterministic synthetic weights/inputs for parity tests (TEST INFRASTRUCTURE).

The reference initialises 61 weight tensors to zero (zero_module: openaimodel.py:306-314, attention.py:699-704,
video_model.py:439), which makes a fresh VideoUNet output exactly 0 (SURVEY.md §0.6).  Parity tests therefore
fill EVERY tensor from a per-name seeded generator, independent of module construction order, so the
reference module (in make_golden.py), the oracle and the CUDA path (on the GPU box) see identical weights
without shipping a 6 GB state_dict.
"""
from __future__ import annotations

import zlib
from typing import Dict, Iterable, Tuple

import torch


def _gen(name: str, seed: int) -> torch.Generator:
    g = torch.Generator(device="cpu")
    g.manual_seed((zlib.crc32(name.encode("utf-8")) ^ (seed * 0x9E3779B1)) & 0x7FFFFFFF)
    return g


def synth_tensor(name: str, shape: Tuple[int, ...], seed: int = 0, gain: float = 1.0) -> torch.Tensor:
    """Value distribution by role (decided from the key name and rank):
    conv/linear weights ~ N(0, gain^2 / fan_in); biases ~ N(0, 0.05^2); norm weights ~ 1 + N(0, 0.1^2);
    mix_factor ~ N(0, 1) (sigmoid -> blend weights away from 0/1)."""
    g = _gen(name, seed)
    shape = tuple(shape)
    if name.endswith("mix_factor"):
        return torch.randn(shape, generator=g)
    if len(shape) >= 2:
        fan_in = 1
        for d in shape[1:]:
            fan_in *= d
        return torch.randn(shape, generator=g) * (gain / fan_in ** 0.5)
    if name.endswith(".weight"):
        # every rank-1 ".weight" on this path is a GroupNorm / LayerNorm scale
        return 1.0 + 0.1 * torch.randn(shape, generator=g)
    return 0.05 * torch.randn(shape, generator=g)


def synth_state_dict(shapes: Dict[str, Iterable[int]], seed: int = 0, gain: float = 1.0) -> Dict[str, torch.Tensor]:
    return {k: synth_tensor(k, tuple(v), seed, gain) for k, v in shapes.items()}


def synth_inputs(T: int, latent_hw: int, seed: int = 23, ctx_dim: int = 1024, adm: int = 768):
    """Synthetic conditioning in the shape sample_one builds (scripts/pub/V3D_512.py:247-269; BASELINE.md §3):
    c = {crossattn [T,1,1024], concat [T,4,h,w], vector [T,768]}, uc = zeros / zeros / same vector."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    x = torch.randn(T, 4, latent_hw, latent_hw, generator=g)
    # sample_one repeats ONE image's embedding over the T frames (V3D_512.py:263-267)
    cross = torch.randn(1, 1, ctx_dim, generator=g).repeat(T, 1, 1)
    concat = torch.randn(1, 4, latent_hw, latent_hw, generator=g).repeat(T, 1, 1, 1)
    vector = torch.randn(T, adm, generator=g)
    c = {"crossattn": cross, "concat": concat, "vector": vector}
    uc = {"crossattn": torch.zeros_like(cross), "concat": torch.zeros_like(concat), "vector": vector.clone()}
    return x, c, uc


def synth_latents(B: int, latent_hw: int, seed: int = 77) -> torch.Tensor:
    """Latents [B, 4, h, w] ~ N(0, 1) for the decode fixtures."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    return torch.randn(B, 4, latent_hw, latent_hw, generator=g)
