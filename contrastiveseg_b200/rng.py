"""Host-side replay of the reference's sampling RNG (lib/loss/loss_contrast.py:79-82,
segmentor/trainer_contrastive.py:127): torch.randperm on the CPU generator, drawn in the reference's
data-dependent order.  Used by the 'torch_cpu' RNG mode (bit-identical samples to the reference for the
same torch seed, at the price of one small D2H copy per step) and by the parity tests (injected
permutations).  The default 'device' mode needs none of this."""
from __future__ import annotations

from typing import Callable, List, Tuple

import numpy as np
import torch


def host_plan(counts: np.ndarray, max_samples: int, max_views: int):
    """counts (B, 2K) int: [b, 2c] = hard pixels, [b, 2c+1] = easy pixels of class c in image b.
    Mirrors k_plan (csrc/pcl_select.cu) / loss_contrast.py:37-48,63-77.
    Returns (pairs [(b, c, n_hard, n_easy, keep_hard, keep_easy)], TC, V)."""
    B, NK = counts.shape
    K = NK // 2
    tot = counts[:, 0::2] + counts[:, 1::2]
    kept = [(b, c) for b in range(B) for c in range(K) if tot[b, c] > max_views]
    TC = len(kept)
    if TC == 0:
        return [], 0, 0
    V = min(max_samples // TC, max_views)
    pairs = []
    for b, c in kept:
        nh, ne = int(counts[b, 2 * c]), int(counts[b, 2 * c + 1])
        if 2 * nh >= V and 2 * ne >= V:
            kh = V // 2
            ke = V - kh
        elif 2 * nh >= V:
            ke = ne
            kh = V - ke
        elif 2 * ne >= V:
            kh = nh
            ke = V - kh
        else:
            raise RuntimeError(f"hard/easy split impossible: {nh} {ne} {V}")
        pairs.append((b, c, nh, ne, kh, ke))
    return pairs, TC, V


def anchor_rank_table(pairs, V: int, perm_fn: Callable[[int], torch.Tensor]) -> torch.Tensor:
    """(TC, V) int32: for every pair, the first keep_hard values of perm(n_hard) then the first keep_easy
    values of perm(n_easy) — both permutations are always drawn, in that order (loss_contrast.py:79-82)."""
    table = torch.zeros((max(len(pairs), 1), max(V, 1)), dtype=torch.int32)
    for t, (_, _, nh, ne, kh, ke) in enumerate(pairs):
        ph = perm_fn(nh)
        pe = perm_fn(ne)
        if V > 0:
            table[t, :kh] = ph[:kh].to(torch.int32)
            table[t, kh:kh + ke] = pe[:ke].to(torch.int32)
    return table


def bank_rank_table(counts: np.ndarray, F: int, perm_fn: Callable[[int], torch.Tensor]) -> torch.Tensor:
    """counts (B, K) pixels per (image, class) in the sub-sampled label grid.  One randperm(n) per
    (image asc, class asc, class > 0, n > 0) slot (trainer_contrastive.py:113-127); returns (B*K, F) int32."""
    B, K = counts.shape
    table = torch.zeros((B * K, max(F, 1)), dtype=torch.int32)
    for b in range(B):
        for c in range(1, K):
            n = int(counts[b, c])
            if n > 0:
                p = perm_fn(n)
                k = min(n, F)
                table[b * K + c, :k] = p[:k].to(torch.int32)
    return table


# ---------------------------------------------------------------------------------------------------------------
# Host model of the DEVICE sampling RNG (csrc/pcl_common.cuh: mix64, keyed_perm) — diagnostics and tests only (which
# pixels will a given seed pick, statistical quality of the draw); the product never samples on the host in this mode.
# ---------------------------------------------------------------------------------------------------------------
_M64 = (1 << 64) - 1


def mix64(z: int) -> int:
    z = (z + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def keyed_perm(j: int, n: int, key: int) -> int:
    """Element that view j of an n-element group takes: 8-round balanced Feistel bijection with cycle walking."""
    if n <= 1:
        return 0
    bits = (n - 1).bit_length()
    hb = (bits + 1) >> 1
    hmask = (1 << hb) - 1
    x = j
    while True:
        L, R = x >> hb, x & hmask
        for r in range(8):
            f = mix64((key + r * 0x9E3779B97F4A7C15 + R) & _M64) & hmask
            L, R = R, L ^ f
        x = (L << hb) | R
        if x < n:
            return x


def device_step_seed(seed: int, step_counter: int) -> int:
    """pcl_step_desc.seed of the eager call number `step_counter` (functional._step_counter after the increment)."""
    return (int(seed) * 0x9E3779B97F4A7C15 + step_counter) & _M64


def device_rank(step_seed: int, image: int, cls: int, num_classes: int, easy: bool, j: int, n: int) -> int:
    """Rank (within the hard or easy pixel list of (image, cls), ascending pixel order) of the j-th sampled view."""
    return keyed_perm(j, n, mix64(step_seed ^ (((image * num_classes + cls) << 1) | (1 if easy else 0))))


def device_bank_rank(enqueue_seed: int, slot: int, j: int, n: int) -> int:
    """Pixel column of the j-th row that the bank enqueue (csrc/pcl_bank.cu k_bank_rows) takes from the n pixels of
    slot = image * num_classes + class, for the seed the packet kernel receives (bank.enqueue_seed(seed) + call counter)."""
    return keyed_perm(j, n, mix64((enqueue_seed ^ (0xB5 << 56) ^ slot) & _M64))
