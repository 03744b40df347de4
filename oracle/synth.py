"""Deterministic synthetic weights / inputs shared by the golden generator and the tests.

TEST INFRASTRUCTURE (see oracle/lvdm_oracle.py header).  There is no checkpoint on disk and no
network, so every parity test runs on seeded synthetic weights.  Weights are regenerated from
(name, shape, seed) instead of being stored, so golden fixtures only hold inputs and outputs.
"""
from __future__ import annotations

import math
import zlib
from typing import Dict, Iterable, Tuple

import torch


def synth_tensor(name: str, shape: Tuple[int, ...], seed: int = 0) -> torch.Tensor:
    """One tensor, independent of every other (seeded by crc32(name)): N(0,1/fan_in) for matrices and
    conv kernels, 1+0.1*N for norm scales, 0.05*N for biases."""
    g = torch.Generator().manual_seed((zlib.crc32(name.encode()) + 7919 * seed) & 0x7FFFFFFF)
    shape = tuple(int(s) for s in shape)
    r = torch.randn(shape, generator=g)
    if len(shape) >= 2:
        fan_in = 1
        for s in shape[1:]:
            fan_in *= s
        return r / math.sqrt(fan_in)
    if name.endswith(".weight"):
        return 1.0 + 0.1 * r
    return 0.05 * r


def synth_state_dict(shapes: Iterable[Tuple[str, Tuple[int, ...]]], seed: int = 0) -> Dict[str, torch.Tensor]:
    return {n: synth_tensor(n, s, seed) for n, s in shapes}


def module_shapes(module: torch.nn.Module):
    return [(k, tuple(v.shape)) for k, v in module.state_dict().items()]


class ToyText(torch.nn.Module):
    """Stands in for FrozenOpenCLIPEmbedder (condition.py:174-234): "" and any other prompt map to two fixed 77-token contexts."""

    def __init__(self):
        super().__init__()
        self.register_buffer("tab", torch.randn(2, 77, 1024, generator=torch.Generator().manual_seed(5)))

    def forward(self, prompts):
        return torch.cat([self.tab[0:1] if p == "" else self.tab[1:2] for p in prompts], 0)

    def encode(self, prompts):
        return self(prompts)


class ToyImage(torch.nn.Module):
    """Stands in for FrozenOpenCLIPImageEmbedderV2 (condition.py:295-372): a fixed projection of a 4x4 pooled image."""

    def __init__(self, tokens=9, dim=64):
        super().__init__()
        self.register_buffer("w", torch.randn(48, tokens * dim, generator=torch.Generator().manual_seed(6)) * 0.2)
        self.tokens, self.dim = tokens, dim

    def forward(self, img):
        return (torch.nn.functional.adaptive_avg_pool2d(img.float(), 4).flatten(1) @ self.w).reshape(img.shape[0], self.tokens, self.dim)
