"""The kernels' dropout masks restated in numpy, and the engine's choice of mask per dropout site.

No mask is stored anywhere: every kernel recomputes its keep bits from a counter-based hash of
(seed + device step counter, site, element index) (csrc/tt_common.cuh: mix32, drop_key, drop_keep_k;
the host drop_threshold of each .cu file). A backward often recomputes the mask in another kernel
than the one that applied it in the forward, so the tests compare every kernel with this one
restatement, and the fp64 oracle takes the masks built here (``engine_masks``) to follow a dropout
training step of the engine.

All arithmetic is uint64 holding 32-bit values, masked with 0xFFFFFFFF after every product: a 32 x
32-bit product overflows int64 (and torch has no uint64 arithmetic).

Element indices are 64-bit. drop_keep_k here folds the high word into the hash as the kernels'
drop_keep_k and their 64-bit quad / pair forms do (the tiled attention kernels, the single-query
kernels), so it is right above 2^32 too: the long-history tests compare masks there. The 32-bit
quad / pair forms of the kernels that keep a sequence on chip agree with it below 2^32 only, and
tt_attn_causal_fwd / _bwd refuse dropout on those kernels once B*H*L*L passes 2^32.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import torch

from mrm_b200.engine import SITE_EMB, SITE_ITEM, _site

BASE_SEED = 0x5EED          # TwoTowerEngine.base_seed
COUNTER_STEP = 0x9E3779B97F4A7C15   # what tt_step_counters_advance adds to engine.seed_dev every optimizer step
ITEM_P = 0.1                # the item tower's dropout, fixed whatever cfg.dropout is (engine.item_forward)

_M32 = np.uint64(0xFFFFFFFF)
_MULS = np.array([1, 0x9E3779B1, 0x85EBCA6B, 0xC2B2AE35], dtype=np.uint64)   # kDropMul1..3 (word 0: h itself)


def _u64(x) -> np.ndarray:
    return np.asarray(x, dtype=np.uint64)


def mix32(x) -> np.ndarray:
    x = _u64(x) & _M32
    x = x ^ (x >> np.uint64(16))
    x = (x * np.uint64(0x7FEB352D)) & _M32
    x = x ^ (x >> np.uint64(15))
    x = (x * np.uint64(0x846CA68B)) & _M32
    x = x ^ (x >> np.uint64(16))
    return x


def drop_key(seed: int, site: int) -> int:
    seed &= (1 << 64) - 1
    lo, hi = seed & 0xFFFFFFFF, seed >> 32
    inner = int(mix32((hi + site * 0x9E3779B9) & 0xFFFFFFFF))
    return int(mix32(lo ^ inner))


def drop_keep_k(key: int, idx, thresh: int) -> np.ndarray:
    """Keep bit of every (64-bit) element index in ``idx``."""
    idx = _u64(idx)
    quad = idx >> np.uint64(2)
    x = (quad & _M32) ^ (((quad >> np.uint64(32)) * np.uint64(0x85EBCA6B)) & _M32)
    h = mix32(x ^ np.uint64(key))
    word = (h * _MULS[(idx & np.uint64(3)).astype(np.intp)]) & _M32
    return word >= np.uint64(thresh)


def drop_threshold(p: float) -> int:
    """Host-side threshold: p rounded to float32, times 2^32 in double, truncated, clamped, at least 1."""
    p32 = float(np.float32(p))
    if p32 <= 0.0:
        return 0
    t = p32 * 4294967296.0
    v = 0xFFFFFFFF if t >= 4294967295.0 else int(t)
    return max(v, 1)


def drop_scale(p: float) -> np.float32:
    """1 / (1 - p) in float32, as the host computes it."""
    return np.float32(1.0) / (np.float32(1.0) - np.float32(p)) if p > 0 else np.float32(1.0)


def keep_bits(seed: int, site: int, n: int, p: float, start: int = 0) -> np.ndarray:
    """Keep bits of the element indices start .. start+n-1 at (seed, site) and rate p."""
    assert 0 <= start and start + n <= 1 << 64
    thresh = drop_threshold(p)
    if thresh == 0:
        return np.ones(n, dtype=bool)
    return drop_keep_k(drop_key(seed, site), np.arange(start, start + n, dtype=np.uint64), thresh)


def scaled_mask(seed: int, site: int, shape, p: float) -> np.ndarray:
    """float32 keep * 1/(1-p) over a row-major tensor of ``shape`` whose flat index is the hash index."""
    n = int(np.prod(shape))
    return np.where(keep_bits(seed, site, n, p), drop_scale(p), np.float32(0.0)).astype(np.float32).reshape(shape)


def last_index(batch) -> np.ndarray:
    """The row each sequence's user embedding is read from (ops.last_index / the oracle's ``lengths``)."""
    m = batch.get("history_mask")
    valid = (batch["history_ids"] != 0) if m is None else (m != 0)
    return (valid.sum(dim=1).long() - 1).clamp(min=0).numpy()


def counter_after(steps: int) -> int:
    """engine.seed_dev (as uint64) after ``steps`` optimizer steps from a fresh engine."""
    return steps * COUNTER_STEP % (1 << 64)


def engine_masks(cfg, batch, counter: int, prune_last_layer: bool = True,
                 base_seed: int = BASE_SEED) -> Dict[str, torch.Tensor]:
    """Every site's scaled mask for one training step of TwoTowerEngine with its dropout counter
    ``engine.seed_dev`` holding ``counter`` (see counter_after), as float32 tensors under the keys of the
    oracle's ``drop=``:

      "emb"                  (B, L, D)     after the embedding LayerNorm; row = token b*L + l
      "layers.{l}.attn"      (B, H, L, L)  attention probabilities; index ((b*H + h)*L + q)*L + k
      "layers.{l}.out_proj"  (B, L, D)     out_proj output (GEMM epilogue; chain_bwd drop2 in the backward)
      "layers.{l}.ffn"       (B, L, 4D)    after the FFN ReLU (GEMM epilogue; the gated dgrad in the backward)
      "layers.{l}.linear2"   (B, L, D)     linear2 output (GEMM epilogue; chain_bwd drop2 in the backward)
      "item"                 (B, 512)      after the item BatchNorm-ReLU, rate 0.1 whenever cfg.dropout > 0

    GEMM sites index row*N + col. With ``prune_last_layer`` the last layer's out_proj / linear1 /
    linear2 run on the compact [B, .] rows, so at the one row of each sequence that is read
    (b, last_b) their masks are those of compact row b; the single-query attention keeps the
    full-sequence index (b*H + h)*L + last_b. Rows the step never reads keep the token-row masks."""
    B, L = batch["history_ids"].shape
    D, FF, H, NL = cfg.embedding_dim, cfg.ff_dim, cfg.num_heads, cfg.num_layers
    p = float(cfg.dropout)
    seed = (base_seed + int(counter)) % (1 << 64)
    last = last_index(batch)
    out = {"emb": scaled_mask(seed, SITE_EMB, (B, L, D), p)}
    for l in range(NL):
        out[f"layers.{l}.attn"] = scaled_mask(seed, _site(l, 0), (B, H, L, L), p)
        for which, name, width in ((1, "out_proj", D), (2, "ffn", FF), (3, "linear2", D)):
            m = scaled_mask(seed, _site(l, which), (B, L, width), p)
            if prune_last_layer and l == NL - 1:
                m[np.arange(B), last] = scaled_mask(seed, _site(l, which), (B, width), p)
            out[f"layers.{l}.{name}"] = m
    out["item"] = scaled_mask(seed, SITE_ITEM, (B, cfg.fusion_hidden), ITEM_P if p > 0 else 0.0)
    return {k: torch.from_numpy(v) for k, v in out.items()}


def redraw(masks: Dict[str, torch.Tensor], key: str, seed: int = 0xBAD5EED) -> Dict[str, torch.Tensor]:
    """``masks`` with the one at ``key`` replaced by an independent draw of the same rate and scale."""
    m = masks[key]
    scale = float(m.max())
    p = 1.0 - 1.0 / scale if scale > 1.0 else 0.0
    out = dict(masks)
    out[key] = torch.from_numpy(scaled_mask(seed, 999, tuple(m.shape), p))
    return out
