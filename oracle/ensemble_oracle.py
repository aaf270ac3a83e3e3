"""ORACLE (test infrastructure, not product): the x8 geometric self-ensemble restated with torch ops.

For k = 0..7 on [B, C, H, W]:
    T_k(x)    = rot90(x if k < 4 else flip(x, [3]), k % 4, [2, 3])
    T_k^-1(y) = rot90(y, -(k % 4), [2, 3]), then flip(., [3]) if k >= 4
    out       = (((y_0 + y_1) + y_2) + ... + y_7) * 0.125   in fp32, adds in k order, y_k = T_k^-1(f(T_k(x)))

The transformed batch is two groups of 4B images (include/b200dn.h): the even k at H x W and the odd k at W x H;
image (k >> 1) * B + b of group k & 1 holds T_k(x[b]).
"""
from __future__ import annotations

from typing import Callable

import torch

Tensor = torch.Tensor


def transform(x: Tensor, k: int) -> Tensor:
    return torch.rot90(x if k < 4 else torch.flip(x, dims=[3]), k % 4, dims=[2, 3])


def inverse(y: Tensor, k: int) -> Tensor:
    y = torch.rot90(y, -(k % 4), dims=[2, 3])
    return torch.flip(y, dims=[3]) if k >= 4 else y


def group(k: int) -> int:
    return k & 1


def index(k: int, b: int, B: int) -> int:
    return (k >> 1) * B + b


def expand(x: Tensor) -> tuple[Tensor, Tensor]:
    """(even [4B, C, H, W], odd [4B, C, W, H])"""
    even = torch.cat([transform(x, k) for k in (0, 2, 4, 6)]).contiguous()
    odd = torch.cat([transform(x, k) for k in (1, 3, 5, 7)]).contiguous()
    return even, odd


def _mean_in_k_order(ys) -> Tensor:
    acc = ys[0]
    for y in ys[1:]:
        acc = acc + y
    return acc * 0.125


def reduce(even: Tensor, odd: Tensor) -> Tensor:
    B = even.shape[0] // 4
    groups = (even, odd)
    return _mean_in_k_order([inverse(groups[group(k)][index(k, 0, B):index(k, B, B)], k) for k in range(8)])


def self_ensemble(f: Callable[[Tensor], Tensor], x: Tensor) -> Tensor:
    """Eight calls f(T_k(x)) at batch B, each transformed back, averaged in k order."""
    return _mean_in_k_order([inverse(f(transform(x, k)), k) for k in range(8)])
