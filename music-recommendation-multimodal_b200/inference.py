"""Single-user recommendation path (reference: src/inference.py:213-323, `recommend_for_user`).

In scope is the arithmetic of that function — user tower on the (truncated) history, re-normalisation, scores
against the item index, exclusion of the padding id and of the history items, top-k with scores. The CSV /
metadata / printing around it stays with the caller. Everything runs on the CUDA kernels of the catalog
retrieval path: the exclusion is applied AFTER an exact top-(k + |history|) selection, which contains the
top-k of the non-excluded items whatever the history is.

`recommend_batch` is the batched form for serving: histories of any model window, exclusion lists of up to 4096
ids per user, sharded catalogs; the exclusion happens inside the selection kernels (`retrieval.Exclusions`).
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from . import retrieval


def recommend_topk(user_emb: torch.Tensor, index: retrieval.CatalogIndex, exclude_ids: Optional[torch.Tensor] = None,
                   k: int = 10) -> Tuple[torch.Tensor, torch.Tensor]:
    """Top-k (item ids int64 (U, k), scores fp32 (U, k)) per user, canonical order (score descending, item id
    ascending), with item 0 and the ids in ``exclude_ids`` (U, m) int64 (0 = no entry) removed — the masking of
    src/inference.py:296-302 for a batch of users."""
    assert user_emb.is_cuda and user_emb.dim() == 2
    U = user_emb.shape[0]
    u = F.normalize(user_emb.float(), p=2, dim=1, eps=1e-8)            # src/inference.py:286
    m = 0 if exclude_ids is None else exclude_ids.shape[1]
    K = k + m
    if K > 256:
        raise ValueError(f"recommend_topk: k + history length = {K} > 256 candidates per user is not supported")
    K = min(K, index.vocab_size - 1)
    idx, score, _ = retrieval.retrieve_topk(u, index, K, mask_item0=True)
    if m == 0:
        return idx[:, :k].long(), score[:, :k]
    ex = exclude_ids.to(user_emb.device).long()
    banned = (idx.long().unsqueeze(2) == ex.unsqueeze(1)).any(dim=2)   # (U, K); id 0 never appears in idx
    # stable partition: kept entries first, in their canonical order
    order = torch.argsort(banned.to(torch.int8), dim=1, stable=True)[:, :k]
    out_s = torch.gather(score, 1, order)
    # fewer than k admissible items (tiny catalogs): the tail is masked like the reference's -inf scores
    out_s = torch.where(torch.gather(banned, 1, order), torch.full_like(out_s, float("-inf")), out_s)
    return torch.gather(idx.long(), 1, order), out_s


def recommend_for_user(model, index: retrieval.CatalogIndex, history_ids: Sequence[int], user_gender: int = 0,
                       user_country: int = 0, k: int = 10, max_len: int = 50) -> Tuple[torch.Tensor, torch.Tensor]:
    """The compute of `recommend_for_user` for one user: ``history_ids`` are the mapped integer item ids in
    time order (src/inference.py:251); the last ``max_len`` are used (:254-258). Returns (item ids (k,) int64,
    scores (k,) fp32), best first."""
    hist = [int(h) for h in history_ids][-max_len:]
    if not hist:
        raise ValueError("recommend_for_user: empty history (the reference returns without recommending)")
    dev = model.engine.device
    L = model.engine.cfg.max_seq_len
    if len(hist) > L:
        raise ValueError(f"history of {len(hist)} items exceeds the model's max_seq_len {L}")
    ids = torch.zeros(1, L, dtype=torch.long)
    ids[0, :len(hist)] = torch.tensor(hist, dtype=torch.long)          # right-padded prefix, mask = ids != 0
    was_training = model.training
    model.eval()
    with torch.no_grad():
        u = model.get_user_embedding(ids.to(dev), history_mask=(ids != 0).long().to(dev),
                                     user_gender=torch.tensor([user_gender], device=dev),
                                     user_country=torch.tensor([user_country], device=dev))
    model.train(was_training)
    ex = torch.zeros(1, max_len, dtype=torch.long)
    ex[0, :len(hist)] = torch.tensor(hist, dtype=torch.long)
    idx, score = recommend_topk(u, index, ex.to(dev), k)
    return idx[0], score[0]


#: users per user-tower call in `recommend_batch`: bounds the tower's workspace (B = 10 k at L = 512 would otherwise
#: size every activation buffer for all users at once)
_TOWER_CHUNK = 1024


def recommend_batch(model, index: retrieval.CatalogIndex, history_ids: torch.Tensor,
                    history_mask: Optional[torch.Tensor] = None, user_gender: Optional[torch.Tensor] = None,
                    user_country: Optional[torch.Tensor] = None, k: int = 10, exclude_ids: Optional[torch.Tensor] = None,
                    group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """`recommend_for_user` (src/inference.py:283-306) for a batch of B users.

    ``history_ids`` (B, L) int64, L <= the model's max_seq_len, right-padded with 0; ``history_mask`` (B, L), default
    ``history_ids != 0``; ``user_gender`` / ``user_country`` (B,), default 0. The eval-mode user tower runs in chunks of
    1024 users, its output is re-normalised (eps 1e-8, :286), and the padding id 0 and every excluded item are
    masked (:296-302) inside the selection kernels. The excluded items are ``exclude_ids`` (B, m) int64 (0 = empty
    slot, m <= 4096: e.g. a full listening history longer than the tower's window) if given, otherwise the valid
    history positions. On a sharded ``index`` the top k is taken over the whole catalog across ``group``
    (collective: every rank passes its copy of the same users).

    Returns (item ids int64 (B, k), scores fp32 (B, k)), best first in the canonical order (score descending, item id
    ascending). When a user has fewer than k admissible items, the tail is id -1 with score -inf."""
    chunk = _TOWER_CHUNK
    if not 1 <= k <= 256:
        raise ValueError(f"recommend_batch: k = {k} outside [1, 256]")
    dev = model.engine.device
    ids = history_ids.to(dev).long()
    B, L = ids.shape
    if L > model.engine.cfg.max_seq_len:
        raise ValueError(f"history window {L} exceeds the model's max_seq_len {model.engine.cfg.max_seq_len}")
    mask = (ids != 0).long() if history_mask is None else history_mask.to(dev).long()
    gender = torch.zeros(B, dtype=torch.long, device=dev) if user_gender is None else user_gender.to(dev).long()
    country = torch.zeros(B, dtype=torch.long, device=dev) if user_country is None else user_country.to(dev).long()
    was_training = model.training
    model.eval()
    with torch.no_grad():
        u = torch.cat([model.get_user_embedding(ids[s:s + chunk], mask[s:s + chunk], gender[s:s + chunk],
                                                country[s:s + chunk]) for s in range(0, B, chunk)])
    model.train(was_training)
    u = F.normalize(u.float(), p=2, dim=1, eps=1e-8)                     # src/inference.py:286
    ex = ids * (mask != 0) if exclude_ids is None else exclude_ids.to(dev).long()
    if ex.shape[0] != B:
        raise ValueError(f"exclude_ids has {ex.shape[0]} rows for {B} users")
    exclude = retrieval.Exclusions(ex, index.vocab_size)
    if index.is_sharded:
        idx, score = retrieval.sharded_topk(u, index, k, group=group, exclude=exclude)
    else:
        idx, score, _ = retrieval.retrieve_topk(u, index, k, exclude=exclude)
    return idx.long(), score
