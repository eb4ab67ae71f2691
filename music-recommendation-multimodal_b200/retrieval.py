"""Catalog retrieval on the B200: fused scoring + streaming top-K, exact re-score, canonical
order, Recall@K / NDCG@K — the device side of the reference's ``calculate_metrics_global``
(src/evaluate_metrics.py:106-192) and of its item-embedding cache (:92-104, 323-326).
"""
from __future__ import annotations

import ctypes
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import ops
from ._lib import TopkPlan, check, lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class CatalogIndex:
    """Device-resident item table in the reference's cache layout: fp32 (V, 256), row i = embedding
    of item id i, row 0 = padding. ``shard`` = (first_row, num_rows) keeps only a contiguous slice
    on this GPU (catalog sharding); indices returned by retrieval are always global.

    A built index takes live catalog updates: `upsert` adds or re-embeds songs, `retire` removes them. No retrieval
    call on the index (`retrieve_topk` and its exact fallback, `retrieve_candidates`, `sharded_topk`, and everything
    built on them: recommendations with or without diversity, sessions, metrics) ever returns a retired song; that
    combines with per-user `Exclusions` and ``mask_item0``, and a user with fewer than K live admissible songs gets
    an id -1 / score -inf tail. The mask is a bitmap of one bit per row that the scoring kernel reads; it exists
    from the first `retire` on (before that the index launches exactly the kernels of an index without updates).
    Updates are ordered on the current stream like every other call on the index; updates concurrent with queries
    on other streams are not supported. The index never grows: to leave room for new songs, build it with
    ``vocab_size`` = the wanted capacity and retire the ids not yet in use."""

    def __init__(self, item_embeddings: torch.Tensor, device=None, shard: Optional[Tuple[int, int]] = None):
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        V = item_embeddings.shape[0]
        first, rows = (0, V) if shard is None else shard
        self.vocab_size = V
        self.item_base = first
        #: True = this object holds ONE contiguous slice of the catalog and its peers hold the rest: retrieval
        #: must merge across the process group. Never inferred from torch.distributed's global state.
        self.is_sharded = shard is not None
        self._group_checked = set()
        self.table = item_embeddings[first:first + rows].to(device=dev, dtype=torch.float32).contiguous()
        assert self.table.shape[1] == 256
        self.table_bf16 = torch.empty(self.table.shape, device=dev, dtype=torch.bfloat16)
        ops.cast_bf16(self.table.view(-1), self.table_bf16.view(-1))
        self._error_terms()
        self._scratch: Dict[Tuple[int, int], Dict[str, torch.Tensor]] = {}
        self._plans: Dict[Tuple[int, int], TopkPlan] = {}
        #: int32 bitmap, bit r = row r of this index is retired (tt_score_topk_live layout); None until `retire`
        self.retired_bits: Optional[torch.Tensor] = None

    @classmethod
    def from_shard(cls, shard_rows: torch.Tensor, first_row: int, vocab_size: int, device=None) -> "CatalogIndex":
        """Index over rows [first_row, first_row + len(shard_rows)) of a catalog of ``vocab_size`` rows whose other
        rows live on the other ranks (the slice is already cut: no full table on this rank)."""
        self = cls(shard_rows, device=device)
        self.item_base, self.vocab_size, self.is_sharded = first_row, vocab_size, True
        return self

    @classmethod
    def from_device_tables(cls, table: torch.Tensor, table_bf16: torch.Tensor) -> "CatalogIndex":
        """Adopt device tables produced by catalog indexing (fp32 cache + the bf16 copy, same shape): no copy."""
        assert table.is_cuda and table.dtype == torch.float32 and table.is_contiguous() and table.shape[1] == 256
        assert table_bf16.dtype == torch.bfloat16 and table_bf16.shape == table.shape and table_bf16.is_contiguous()
        self = cls.__new__(cls)
        self.vocab_size, self.item_base, self.is_sharded, self._group_checked = table.shape[0], 0, False, set()
        self.table, self.table_bf16 = table, table_bf16
        self._error_terms()
        self._scratch, self._plans = {}, {}
        self.retired_bits = None
        return self

    def _error_terms(self) -> None:
        """terms of the bound |bf16-path score - exact score| that depend on the items only (chunked: the
        fp32 copy of a 10 M-row bf16 table would be 10 GB)"""
        de, ne = 0.0, 0.0
        for s0 in range(0, self.table.shape[0], 1 << 20):
            t16 = self.table_bf16[s0:s0 + (1 << 20)].float()
            de = max(de, (t16 - self.table[s0:s0 + (1 << 20)]).norm(dim=1).max().item())
            ne = max(ne, t16.norm(dim=1).max().item())
        self.de_max, self.ne_max = de, ne

    @property
    def num_rows(self) -> int:
        return self.table.shape[0]

    def _check_update_ids(self, item_ids, what: str) -> torch.Tensor:
        """the ids of an update as a host int64 vector; ValueError (before any launch) for id 0, ids outside
        [1, vocab_size) and ids that appear twice"""
        if not torch.is_tensor(item_ids) or item_ids.dim() != 1 or item_ids.dtype.is_floating_point \
                or item_ids.is_complex() or item_ids.dtype == torch.bool:
            raise ValueError(f"{what}: item_ids must be a 1-D integer tensor")
        ids = item_ids.to("cpu", torch.int64)
        if ids.numel() and (int(ids.min()) < 1 or int(ids.max()) >= self.vocab_size):
            raise ValueError(f"{what}: item ids must lie in [1, {self.vocab_size}) (id 0 is the padding row)")
        s = np.sort(ids.numpy())                 # cheaper on the host than torch.unique
        if (s[1:] == s[:-1]).any():
            raise ValueError(f"{what}: duplicate item ids")
        return ids

    def _owned(self, ids: torch.Tensor) -> np.ndarray:
        a = ids.numpy()
        return (a >= self.item_base) & (a < self.item_base + self.num_rows)

    def retire(self, item_ids: torch.Tensor) -> None:
        """Remove songs from retrieval: their fp32 and bf16 rows become zero (so `table` stays the reference's cache
        of the live catalog, a retired row indistinguishable from an unlisted one) and their retired bits are set.
        ``item_ids``: integer tensor on any device; ids outside this index's rows are skipped (every shard may be
        handed the same batch), retiring a retired id does nothing. The certificate terms ``de_max`` / ``ne_max`` are
        never lowered: the bound stays valid, only conservative. The first call that retires a row of this index
        allocates the bitmap (ceil(rows / 256) * 32 bytes)."""
        ids = self._check_update_ids(item_ids, "retire")
        own = torch.from_numpy(ids.numpy()[self._owned(ids)])
        if own.numel() == 0:
            return
        dev = self.table.device
        if self.retired_bits is None:
            self.retired_bits = torch.zeros((self.num_rows + 255) // 256 * 8, device=dev, dtype=torch.int32)
        ops.catalog_retire(own.to(dev), self.vocab_size, self.item_base, self.table, self.table_bf16,
                           self.retired_bits)

    def retired_ids(self) -> torch.Tensor:
        """Global ids of this index's retired rows, int64, ascending, on the index's device (with `retire` the round
        trip that persists the retired set)."""
        dev = self.table.device
        if self.retired_bits is None:
            return torch.empty(0, device=dev, dtype=torch.int64)
        bits = (self.retired_bits[:, None] >> torch.arange(32, device=dev, dtype=torch.int32)) & 1
        return torch.nonzero(bits.flatten()[:self.num_rows]).flatten() + self.item_base

    def upsert(self, model, item_features: Dict[str, torch.Tensor], item_ids: torch.Tensor,
               batch_size: int = 131072) -> None:
        """Add new songs or re-embed existing ones: the item tower runs in eval mode with the model's CURRENT weights
        over ``item_features`` (the four (n, modality_dim) feature tensors of catalog indexing, any device) and row
        ``item_ids[i]`` gets song i's embedding; the song is live afterwards, also when it had been retired. The
        arithmetic is `TwoTowerEngine.index_items`' (folded BatchNorm, GEMM, GEMM, the index-rows tail), so a row is
        bit-identical to the one a from-scratch `index_catalog_device` writes for the same song and weights. Ids
        outside this index's rows are skipped; id 0, ids outside [1, vocab_size), duplicates and malformed features
        raise ValueError before any launch. Ids at or above the MODEL's vocab_size can be upserted and recommended,
        but the user tower cannot take them in a history (`UserSessions` rejects them).

        The certificate terms ``de_max`` / ``ne_max`` are raised on the device and read back once: one host
        synchronisation per call."""
        ids = self._check_update_ids(item_ids, "upsert")
        n = ids.numel()
        keys = ("target_audio", "target_image", "target_input_ids", "target_tabular")
        m = model.engine.cfg.modality_dim
        if not isinstance(item_features, dict) or any(k not in item_features for k in keys):
            raise ValueError(f"upsert: item_features must hold {keys}")
        for k in keys:
            f = item_features[k]
            if not torch.is_tensor(f) or not f.dtype.is_floating_point or tuple(f.shape) != (n, m):
                raise ValueError(f"upsert: item_features[{k!r}] must be a floating tensor of shape ({n}, {m})")
        own = self._owned(ids)
        if not bool(own.any()):
            return
        dev = self.table.device
        if bool(own.all()):
            feats = {k: item_features[k].to(dev, dtype=torch.float32).contiguous() for k in keys}
        else:
            sel = torch.from_numpy(np.nonzero(own)[0])
            feats = {k: item_features[k][sel.to(item_features[k].device)].to(dev, dtype=torch.float32).contiguous()
                     for k in keys}
            ids = ids[sel]
        eng = model.engine
        model.eval()
        if hasattr(model, "_sync_shadow"):
            model._sync_shadow()
        stats = torch.zeros(2, device=dev)
        eng.index_items(feats, ids.to(dev), self.table, self.table_bf16, batch_size=batch_size,
                        live=(self.vocab_size, self.item_base, self.retired_bits, stats))
        de, ne = stats.tolist()
        self.de_max, self.ne_max = max(self.de_max, de), max(self.ne_max, ne)

    def check_group(self, U: int, group=None) -> None:
        """Once per (group, U): the shards of the group's ranks must tile [0, vocab_size) without gaps or overlaps
        and every rank must bring the same number of users (the merge pairs row u of every rank). One small
        host-synchronising all-gather; raises on every rank alike."""
        import torch.distributed as dist
        key = (id(group), U)
        if key in self._group_checked:
            return
        ws = dist.get_world_size(group)
        mine = torch.tensor([self.item_base, self.num_rows, U, self.vocab_size], dtype=torch.int64,
                            device=self.table.device if dist.get_backend(group) == "nccl" else "cpu")
        allv = torch.empty(ws * 4, dtype=torch.int64, device=mine.device)
        dist.all_gather_into_tensor(allv, mine, group=group)
        rows = sorted(tuple(r) for r in allv.view(ws, 4).tolist())
        nxt = 0
        for first, n, u, v in rows:
            if u != U or v != self.vocab_size:
                raise ValueError(f"sharded retrieval: ranks disagree on users / vocab size: {rows}")
            if first != nxt:
                raise ValueError(f"sharded retrieval: shards do not tile the catalog (gap or overlap at row {nxt}): {rows}")
            nxt = first + n
        if nxt != self.vocab_size:
            raise ValueError(f"sharded retrieval: shards cover {nxt} of {self.vocab_size} rows: {rows}")
        self._group_checked.add(key)

    def plan(self, U: int, kprime: int) -> TopkPlan:
        key = (U, kprime)
        if key not in self._plans:
            p = TopkPlan()
            check(lib().tt_topk_plan_make(U, self.num_rows, kprime, ctypes.byref(p)), "tt_topk_plan_make")
            self._plans[key] = p
            dev = self.table.device
            self._scratch[key] = {
                "cand": torch.empty(p.cand_bytes // 8, device=dev, dtype=torch.int64),
                "cnt": torch.empty(p.cnt_bytes // 4, device=dev, dtype=torch.int32),
                "thr": torch.empty(p.thr_bytes // 8, device=dev, dtype=torch.int64),
                "smax": (torch.empty(p.smax_bytes // 4, device=dev, dtype=torch.float32) if p.smax_bytes else None),
                "users_bf16": torch.empty(U, 256, device=dev, dtype=torch.bfloat16),
                "eps_stats": torch.zeros(2, device=dev),
                "keys": None,
            }
        return self._plans[key]


class Exclusions:
    """Per-user sets of item ids that retrieval must never return (a user's listening history: the masking of
    src/inference.py:296-302), in the device form the selection kernels probe (tt_exclusions_build): a sorted,
    de-duplicated int32 list per user, its length and a 4096-bit hashed bitmap. Build it once per batch.

    ``ids`` (U, m) integer tensor, m <= 4096; 0 marks an empty slot and ids <= 0 or >= ``vocab_size`` are dropped.
    The selection kernel drops excluded items from the candidate lists before it prunes or hands them over, so the
    result is the exact top K of the admissible items; rows of a sharded catalog may name items of any shard."""

    def __init__(self, ids: torch.Tensor, vocab_size: int):
        assert ids.dim() == 2 and ids.is_cuda
        U, m = ids.shape
        if m > 4096:
            raise ValueError(f"Exclusions: {m} ids per user exceed 4096")
        ids = ids.long().contiguous()
        dev = ids.device
        self.ld = max(m, 1)
        self.ids = torch.empty(U, self.ld, device=dev, dtype=torch.int32)
        self.cnt = torch.empty(U, device=dev, dtype=torch.int32)
        self.bits = torch.empty(U, 128, device=dev, dtype=torch.int32)
        check(lib().tt_exclusions_build(ids.data_ptr(), U, m, max(m, 1), vocab_size, self.ids.data_ptr(), self.ld,
                                        self.cnt.data_ptr(), self.bits.data_ptr(), _stream()), "tt_exclusions_build")

    @property
    def num_users(self) -> int:
        return self.cnt.shape[0]

    def rows(self, sel: torch.Tensor) -> "Exclusions":
        """The exclusions of users ``sel`` (index tensor), in that order: no rebuild."""
        out = Exclusions.__new__(Exclusions)
        out.ld = self.ld
        out.ids, out.cnt, out.bits = self.ids[sel].contiguous(), self.cnt[sel].contiguous(), self.bits[sel].contiguous()
        return out


def _check_exclude(exclude: Optional[Exclusions], U: int) -> None:
    if exclude is not None and exclude.num_users != U:
        raise ValueError(f"exclusions for {exclude.num_users} users, {U} user embeddings")


def _exclude_kw(exclude: Optional[Exclusions]) -> dict:
    """keyword arguments that pass ``exclude`` on only when it is set: without exclusions the sharded protocol makes
    exactly the calls it always made"""
    return {} if exclude is None else {"exclude": exclude}


def exchange_buffers(index, U: int, ld: int, world: int, group=None) -> Dict[str, torch.Tensor]:
    """Reused buffers of the sharded protocol: this shard's packed rows [U, ld] int32, the gathered ones
    [world * U, ld], the certificate flags. On an NCCL group of one NVLink domain the gathered buffer lives in a
    symmetric arena and `exchange` moves the rows with this repo's all-gather kernel (peer / multicast stores + an
    in-kernel barrier); otherwise (gloo tests, no peer access) with the library collective. Collective on first use."""
    key = ("xchg", U, ld, world)
    if key not in index._scratch:
        dev = index.table.device
        buf = {"pack": torch.empty(U, ld, device=dev, dtype=torch.int32),
               "bad": torch.zeros(U, device=dev, dtype=torch.int32), "arena": None}
        if dev.type == "cuda" and os.environ.get("TT_COMM", "") != "nccl":
            from . import symm
            if symm.available(group):
                try:
                    buf["arena"] = symm.SymmArena({"all": world * U * ld * 4}, group, dev)
                    buf["all"] = buf["arena"].view("all", torch.int32, (world * U, ld))
                except Exception:          # same outcome on every rank: fall back to the library collective
                    buf["arena"] = None
        if buf["arena"] is None:
            buf["all"] = torch.empty(world * U, ld, device=dev, dtype=torch.int32)
        index._scratch[key] = buf
    return index._scratch[key]


def _pitch(k: int) -> int:
    """Row pitch (int32 words) of the exchange layout [k scores | k ids | bound | flag], padded to 16 bytes."""
    return (2 * k + 2 + 3) // 4 * 4


def exchange(buf: Dict[str, torch.Tensor], group=None) -> None:
    """buf['all'][r * U:(r + 1) * U] = rank r's buf['pack'] on every rank."""
    if buf["arena"] is not None:
        # leading barrier: a peer may still be merging the previous pass out of its gathered buffer
        buf["arena"].allgather([(buf["pack"], "all")], pre_barrier=True)
    else:
        import torch.distributed as dist
        dist.all_gather_into_tensor(buf["all"], buf["pack"], group=group)


def retrieve_topk(user_emb: torch.Tensor, index: CatalogIndex, K: int, kprime: int = 256,
                  mask_item0: bool = True, exact_fallback: bool = True, flags_out: Optional[torch.Tensor] = None,
                  exclude: Optional[Exclusions] = None):
    """Top-K items of this shard for every user, canonical order; ``exclude``: per-user item ids never returned
    (a user with fewer than K admissible items gets id -1 / score -inf in the tail).

    Returns (idx int32 (U, K) global item ids, score fp32 (U, K), n_fallback). Scores are the
    exact fp32 dot products (fp64-accumulated, rounded once). Users whose exactness certificate
    fails are recomputed by brute force (``n_fallback`` of them; needs one host sync).
    ``exact_fallback=False`` skips that read-back: the result is only certified for users whose entry of
    ``flags_out`` (int32 (U,), filled by the pass) is 0 — the caller must look at it."""
    assert user_emb.is_cuda and user_emb.dtype == torch.float32 and user_emb.shape[1] == 256
    user_emb = user_emb.contiguous()
    U = user_emb.shape[0]
    kprime = max(kprime, K)
    _check_exclude(exclude, U)
    plan, sc = _score_pass(user_emb, index, kprime, mask_item0, exclude)
    dev = user_emb.device
    out_idx = torch.empty(U, K, device=dev, dtype=torch.int32)
    out_score = torch.empty(U, K, device=dev, dtype=torch.float32)
    flags = torch.empty(U, device=dev, dtype=torch.int32) if flags_out is None else flags_out
    assert flags.dtype == torch.int32 and flags.numel() == U and flags.is_cuda
    check(lib().tt_topk_finalize(ctypes.byref(plan), sc["cand"].data_ptr(), sc["cnt"].data_ptr(),
                                 sc["thr"].data_ptr(), user_emb.data_ptr(),
                                 index.table.data_ptr(), index.item_base, K, 0.0, sc["eps_stats"].data_ptr(),
                                 index.ne_max, index.de_max, out_idx.data_ptr(),
                                 out_score.data_ptr(), flags.data_ptr(), _stream()), "tt_topk_finalize")
    n_fallback = 0
    if exact_fallback:
        bad = torch.nonzero(flags).flatten().tolist()
        n_fallback = len(bad)
        if bad:
            if sc["keys"] is None:
                sc["keys"] = torch.empty(index.num_rows, device=dev, dtype=torch.int64)
            for u in bad:
                ex_ids, ex_cnt = (None, None) if exclude is None else (exclude.ids[u].data_ptr(),
                                                                       exclude.cnt[u:].data_ptr())
                if index.retired_bits is None:
                    check(lib().tt_exact_topk_excl(user_emb[u].data_ptr(), index.table.data_ptr(), index.num_rows,
                                                   index.item_base, int(mask_item0), K, ex_ids, ex_cnt,
                                                   sc["keys"].data_ptr(), out_score[u].data_ptr(),
                                                   out_idx[u].data_ptr(), _stream()), "tt_exact_topk_excl")
                else:
                    check(lib().tt_exact_topk_live(user_emb[u].data_ptr(), index.table.data_ptr(), index.num_rows,
                                                   index.item_base, int(mask_item0), K, ex_ids, ex_cnt,
                                                   index.retired_bits.data_ptr(), sc["keys"].data_ptr(),
                                                   out_score[u].data_ptr(), out_idx[u].data_ptr(), _stream()),
                          "tt_exact_topk_live")
    return out_idx, out_score, n_fallback


def _score_pass(user_emb: torch.Tensor, index: "CatalogIndex", kprime: int, mask_item0: bool,
                exclude: Optional[Exclusions] = None):
    """bf16 scoring + streaming candidate selection of this shard (tt_score_topk); returns (plan, scratch).
    The user-side terms of the certificate's error bound (max ||bf16(u) - u||, max ||u||) are reduced on the device by
    the cast kernel into scratch['eps_stats'] and combined with the index's item-side terms inside the finalize kernel
    (rigorous bound on |u^.e^ - u.e|: Cauchy-Schwarz on the bf16 rounding errors + fp32 accumulation slack) — nothing
    is read back to the host before or between the launches."""
    U = user_emb.shape[0]
    plan = index.plan(U, kprime)
    sc = index._scratch[(U, kprime)]
    check(lib().tt_users_prepare(user_emb.data_ptr(), sc["users_bf16"].data_ptr(), U, sc["eps_stats"].data_ptr(),
                                 _stream()), "tt_users_prepare")
    ex = (None, None, None, 0) if exclude is None else (exclude.ids.data_ptr(), exclude.cnt.data_ptr(),
                                                         exclude.bits.data_ptr(), exclude.ld)
    smax = None if sc["smax"] is None else sc["smax"].data_ptr()
    if index.retired_bits is None:
        check(lib().tt_score_topk_excl(sc["users_bf16"].data_ptr(), index.table_bf16.data_ptr(), index.item_base,
                                       ctypes.byref(plan), sc["cand"].data_ptr(), sc["cnt"].data_ptr(),
                                       sc["thr"].data_ptr(), smax, int(mask_item0), *ex, _stream()),
              "tt_score_topk_excl")
    else:
        check(lib().tt_score_topk_live(sc["users_bf16"].data_ptr(), index.table_bf16.data_ptr(), index.item_base,
                                       ctypes.byref(plan), sc["cand"].data_ptr(), sc["cnt"].data_ptr(),
                                       sc["thr"].data_ptr(), smax, int(mask_item0), *ex,
                                       index.retired_bits.data_ptr(), _stream()), "tt_score_topk_live")
    return plan, sc


def retrieve_candidates(user_emb: torch.Tensor, index: "CatalogIndex", kprime: int, mask_item0: bool = True,
                        pack: Optional[torch.Tensor] = None, exclude: Optional[Exclusions] = None):
    """Sharded catalogs: ALL ``kprime`` candidates of this shard per user, re-scored exactly.

    Returns (idx int32 (U, kprime) global ids, -1 padded; score fp32 (U, kprime); bound fp32 (U,): every item of
    the shard that is not in the list has exact score <= bound; overflow int32 (U,): 1 = tie flood, use the exact
    path). With G shards a shard needs about 1/G of the single-GPU candidate budget (`shard_kprime`).
    ``pack`` int32 (U, >= 2 * kprime + 2): the kernel writes the exchange layout [scores | ids | bound | flag] of
    `sharded_topk` directly and the four results are views of it. ``exclude``: as in `retrieve_topk`; the lists and
    bounds then cover the admissible items only."""
    assert user_emb.is_cuda and user_emb.dtype == torch.float32 and user_emb.shape[1] == 256
    user_emb = user_emb.contiguous()
    U = user_emb.shape[0]
    _check_exclude(exclude, U)
    plan, sc = _score_pass(user_emb, index, kprime, mask_item0, exclude)
    dev = user_emb.device
    if pack is None:
        pack = torch.empty(U, 2 * kprime + 2, device=dev, dtype=torch.int32)
    ld = pack.shape[1]           # row pitch in words: >= 2 * kprime + 2 (padded so rows stay 16-byte multiples)
    assert pack.dtype == torch.int32 and pack.shape[0] == U and ld >= 2 * kprime + 2 and pack.is_contiguous()
    base = pack.data_ptr()
    check(lib().tt_topk_finalize_bounded(ctypes.byref(plan), sc["cand"].data_ptr(), sc["cnt"].data_ptr(),
                                         sc["thr"].data_ptr(), user_emb.data_ptr(), index.table.data_ptr(),
                                         index.item_base, 0.0, sc["eps_stats"].data_ptr(), index.ne_max, index.de_max,
                                         base + 4 * kprime, base, ld, base + 8 * kprime, base + 8 * kprime + 4, ld,
                                         _stream()), "tt_topk_finalize_bounded")
    return (pack[:, kprime:2 * kprime], pack[:, :kprime].view(torch.float32), pack[:, 2 * kprime].view(torch.float32),
            pack[:, 2 * kprime + 1])


#: users of the most recent `sharded_topk` call that needed the per-shard exact fallback (bench bookkeeping)
last_fallback_users = 0


def shard_kprime(kprime: int, shards: int) -> int:
    """Candidates per user and shard: 1.5x the even share of the single-GPU budget plus 16 (the number of a
    user's global top-K' items that fall into one shard is binomial), a multiple of 8 in [48, kprime]."""
    if shards <= 1:
        return kprime
    k = int(1.5 * kprime / shards + 16 + 7) // 8 * 8
    return max(48, min(kprime, k))


def merge_bounded(scores: torch.Tensor, idx: torch.Tensor, bounds: torch.Tensor, K: int):
    """Merge per-shard candidate lists [G, U, K'] (exact scores) into the global top K and certify it:
    the result for user u is exact when its K-th score beats every shard's bound (an item missing from
    shard s's list scores at most bounds[s, u]). Returns (idx (U, K), score (U, K), uncertified bool (U,))."""
    G, U, Kin = scores.shape
    scores, idx = scores.contiguous(), idx.contiguous()
    out_s = torch.empty(U, K, device=scores.device, dtype=torch.float32)
    out_i = torch.empty(U, K, device=scores.device, dtype=torch.int32)
    check(lib().tt_topk_merge_lists(scores.data_ptr(), idx.data_ptr(), G, U, Kin, K, out_s.data_ptr(),
                                    out_i.data_ptr(), _stream()), "tt_topk_merge_lists")
    bmax = bounds.max(dim=0).values
    # fewer than K items in the union is fine when every shard listed ALL its items (bound = -inf)
    ok = torch.where(out_i[:, K - 1] >= 0, out_s[:, K - 1] > bmax, torch.isneginf(bmax))
    return out_i, out_s, ~ok


def sharded_topk(user_emb: torch.Tensor, index: "CatalogIndex", K: int, kprime: int = 256, group=None,
                 bounded: Optional[bool] = None, defer_check: bool = False, exclude: Optional[Exclusions] = None):
    """Exact global top K over a catalog sharded across the ranks of ``group`` (every rank gets the result).

    bounded protocol (default from 4 shards): per-shard candidate lists of `shard_kprime` entries +
    completeness bounds, one all-gather, merge + certificate; users whose certificate fails (and only those) go
    through the per-shard exact top-K protocol. ``bounded=False`` (default below 4 shards) always uses the latter.
    ``defer_check=True`` (bounded protocol only) returns (idx, score, bad) without reading the certificate back:
    the caller checks ``bad`` together with its own read-back and calls `finish_sharded_topk` if any flag is set.
    ``exclude`` (`Exclusions` of these users, built against the global vocabulary): never return those items."""
    import torch.distributed as dist
    ws = dist.get_world_size(group)
    index.check_group(user_emb.shape[0], group)
    if bounded is None:
        # Measured (tools/dist_retrieval_check.py, 2 GPUs over NCCL, 10 k users x 1 M items): with 2 shards the
        # lists are nearly as long as the single-GPU budget (208 of 256) and the bounded pass is the slower one
        # (3.27 vs 3.06 ms); a 1/8 shard takes 1.14 ms with 64-entry lists against 1.76 ms with K' = 256.
        bounded = ws >= 4

    def per_shard_exact(users):
        i, s, _ = retrieve_topk(users, index, K, kprime, **_exclude_kw(exclude))
        n = s.shape[0]
        # one exchange of [scores | ids | bound = -inf | flag = 0] rows, merged in place like the bounded protocol
        # (every shard's list IS its exact top K, so the certificate is trivially satisfied)
        xb = exchange_buffers(index, n, _pitch(K), ws, group)
        pk = xb["pack"]
        pk[:, :K] = s.view(torch.int32)
        pk[:, K:2 * K] = i
        pk[:, 2 * K] = -8388608        # fp32 -inf as int32 (0xFF800000)
        pk[:, 2 * K + 1] = 0
        exchange(xb, group)
        return merge_packed(xb["all"], ws, n, K, K, xb["bad"])

    global last_fallback_users
    last_fallback_users = 0
    if not bounded or K > ws * shard_kprime(kprime, ws):
        out = per_shard_exact(user_emb)
        return (out[0], out[1], torch.zeros(user_emb.shape[0], device=user_emb.device, dtype=torch.int32)) \
            if defer_check else out
    kps = shard_kprime(kprime, ws)
    U = user_emb.shape[0]
    buf = exchange_buffers(index, U, _pitch(kps), ws, group)
    # the finalize kernel writes this shard's lists, bounds and flags in the exchange layout; ONE all-gather; the merge
    # kernel reads the gathered buffer in place and emits the certificate
    retrieve_candidates(user_emb, index, kps, pack=buf["pack"], **_exclude_kw(exclude))
    exchange(buf, group)
    bad = buf["bad"]
    out_i, out_s = merge_packed(buf["all"], ws, U, kps, K, bad)
    if defer_check:
        return out_i, out_s, bad
    finish_sharded_topk(user_emb, index, K, out_i, out_s, bad, kprime, group, exclude)
    return out_i, out_s


def merge_packed(allp: torch.Tensor, G: int, U: int, kps: int, K: int, bad: torch.Tensor):
    """Merge the all-gathered exchange buffer [G * U, ld >= 2 * kps + 2] (rows [scores | ids | bound | flag]) into the global
    top K per user, in place of any unpacking; ``bad`` (int32 (U,)) receives the certificate (1 = not certified)."""
    out_s = torch.empty(U, K, device=allp.device, dtype=torch.float32)
    out_i = torch.empty(U, K, device=allp.device, dtype=torch.int32)
    check(lib().tt_topk_merge_packed(allp.data_ptr(), allp.shape[1], G, U, kps, K, out_s.data_ptr(), out_i.data_ptr(),
                                     bad.data_ptr(), _stream()), "tt_topk_merge_packed")
    return out_i, out_s


def finish_sharded_topk(user_emb, index, K, out_i, out_s, bad, kprime: int = 256, group=None,
                        exclude: Optional[Exclusions] = None) -> int:
    """Second half of the bounded protocol: users whose merged list is not certified (`bad`, identical on every rank
    because it was computed from all-gathered data) go through the per-shard exact top-K + merge, in place. One host
    read of the flags; returns the number of such users. Collective."""
    import torch.distributed as dist
    global last_fallback_users
    ws = dist.get_world_size(group)
    sel = torch.nonzero(bad).flatten()        # host sync: the (rare) fallback is a different launch sequence
    n = sel.numel()
    last_fallback_users = n
    if n == 0:
        return 0
    # scratch buffers are cached per user count: pad to a multiple of 256 (repeating the first user) so that
    # a long evaluation with a few uncertified users per batch does not accumulate one scratch set per count
    padded = torch.cat([sel, sel[:1].expand((-n) % 256)])
    users = user_emb[padded].contiguous()
    i, s, _ = retrieve_topk(users, index, K, kprime, **_exclude_kw(None if exclude is None else exclude.rows(padded)))
    m = s.shape[0]
    all_s = torch.empty(ws * m, K, device=s.device, dtype=s.dtype)
    all_i = torch.empty(ws * m, K, device=i.device, dtype=i.dtype)
    dist.all_gather_into_tensor(all_s, s.contiguous(), group=group)
    dist.all_gather_into_tensor(all_i, i.contiguous(), group=group)
    fi, fs = merge_topk(all_s.view(ws, m, K), all_i.view(ws, m, K))
    out_i[sel], out_s[sel] = fi[:n], fs[:n]
    return n


def merge_topk(scores: torch.Tensor, idx: torch.Tensor):
    """Merge per-shard lists [G, U, K] (each canonical) into the global top-K per user."""
    G, U, K = scores.shape
    scores, idx = scores.contiguous(), idx.contiguous()
    out_s = torch.empty(U, K, device=scores.device, dtype=torch.float32)
    out_i = torch.empty(U, K, device=scores.device, dtype=torch.int32)
    check(lib().tt_topk_merge(scores.data_ptr(), idx.data_ptr(), G, U, K, out_s.data_ptr(), out_i.data_ptr(),
                              _stream()), "tt_topk_merge")
    return out_i, out_s


#: bytes of gathered pool rows per `diversify` chunk on a sharded index
_DIVERSIFY_CHUNK_BYTES = 256 << 20


def check_diversity(diversity: float) -> None:
    if not 0.0 <= diversity <= 1.0:            # also rejects NaN
        raise ValueError(f"diversity = {diversity} outside [0, 1]")


def diversify(idx: torch.Tensor, score: torch.Tensor, index: CatalogIndex, k: int, diversity: float, group=None):
    """k maximal-marginal-relevance picks from each user's candidate pool: ``idx`` / ``score`` (U, P), P <= 256, the
    exact top P of `retrieve_topk` / `sharded_topk` in canonical order (-1 / -inf tail).

    With lambda = 1 - diversity and mu = 1 - lambda, each step picks the unpicked candidate with the largest
    lambda * score - mu * (its largest similarity to the items picked so far), ties to the earlier pool position;
    similarity is the dot product of the index's fp32 rows (fp64 accumulate, rounded to fp32). diversity = 0 returns
    the pool's first k; diversity = 1 starts with the best item and then takes the one least similar to the picks.

    Returns (idx int32 (U, k), score fp32 (U, k)): the picks in pick order with their exact scores — NOT sorted by
    score when diversity > 0 — and -1 / -inf where fewer than k candidates are admissible. On a sharded index this is
    collective over ``group`` (every rank brings the same users, as in `sharded_topk`): each rank writes the pool rows
    it owns into a zeroed buffer, one all-reduce (sum) assembles them, and the result is bit-identical to the
    single-GPU one."""
    check_diversity(diversity)
    U, P = idx.shape
    if not 1 <= k <= P <= 256:
        raise ValueError(f"diversify: need 1 <= k = {k} <= pool = {P} <= 256")
    lam = 1.0 - float(diversity)
    mu = 1.0 - lam
    idx = idx.to(torch.int32).contiguous()
    score = score.contiguous()
    if not index.is_sharded:
        return ops.mmr_select(idx, score, k, lam, mu, ops.MMR_ROWS_TABLE, index.table, index.item_base,
                              index.num_rows)
    import torch.distributed as dist
    chunk = max(1, _DIVERSIFY_CHUNK_BYTES // (P * 1024))
    rows = torch.empty(min(U, chunk), P, 256, device=idx.device, dtype=torch.float32)
    out_i = torch.empty(U, k, device=idx.device, dtype=torch.int32)
    out_s = torch.empty(U, k, device=idx.device, dtype=torch.float32)
    for s0 in range(0, U, chunk):
        n = min(chunk, U - s0)
        buf = rows[:n]
        ops.mmr_gather_rows(idx[s0:s0 + n], index.table, index.item_base, buf)
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)     # one non-zero contributor per element: exact
        out_i[s0:s0 + n], out_s[s0:s0 + n] = ops.mmr_select(idx[s0:s0 + n], score[s0:s0 + n], k, lam, mu,
                                                            ops.MMR_ROWS_GATHERED, buf)
    return out_i, out_s


def gain_table(K: int) -> torch.Tensor:
    """1/log2(rank+2) exactly as the reference computes it (fp32 torch ops, evaluate_metrics.py:180)."""
    return 1.0 / torch.log2(torch.arange(K).float() + 2.0)


_METRIC_CONSTANTS: dict = {}


def _metric_constants(k_list: tuple, K: int, dev: torch.device):
    """The cut-off list and the gain table on the device, built once per (k_list, K, device): creating them per call
    costs two pageable host->device copies, each of which stalls the host until the stream has drained (measured
    6.2 ms per call behind the sharded exchange, gpurun r3_b2a)."""
    key = (k_list, K, dev.type, dev.index)
    hit = _METRIC_CONSTANTS.get(key)
    if hit is None:
        hit = (torch.tensor(list(k_list), dtype=torch.int32, device=dev), gain_table(K).to(dev))
        _METRIC_CONSTANTS[key] = hit
    return hit


def rank_metrics(topk_idx: torch.Tensor, targets: torch.Tensor, k_list: Sequence[int]):
    """Per-row Recall@k / NDCG@k on the device -> (recall [nk, U], ndcg [nk, U]) fp32."""
    U, K = topk_idx.shape
    dev = topk_idx.device
    kl, gt = _metric_constants(tuple(int(k) for k in k_list), K, dev)
    recall = torch.empty(len(k_list), U, device=dev)
    ndcg = torch.empty(len(k_list), U, device=dev)
    check(lib().tt_rank_metrics(topk_idx.data_ptr(), targets.contiguous().data_ptr(), U, K, kl.data_ptr(),
                                len(k_list), gt.data_ptr(), recall.data_ptr(), ndcg.data_ptr(), _stream()),
          "tt_rank_metrics")
    return recall, ndcg


def metrics_from_embeddings(user_emb: torch.Tensor, targets: torch.Tensor, index: CatalogIndex,
                            k_list: Sequence[int] = (10, 20), kprime: int = 256,
                            group=None) -> Dict[str, float]:
    """Recall@k / NDCG@k of precomputed user embeddings against the (possibly sharded) catalog.
    With an index built over one shard (``CatalogIndex(shard=...)`` / ``from_shard``) every rank of ``group``
    (default: the world group) scores its shard and the per-shard lists are all-gathered and merged — the result
    does not depend on the number of shards. An unsharded index never communicates, whatever process group
    happens to be initialised (every rank then evaluates its own users against the whole catalog)."""
    K = max(k_list)
    targets = targets.to(user_emb.device)
    if index.is_sharded:
        # the certificate flags travel to the host WITH the metrics: one synchronisation per call; only if a flag is
        # set (rare) the exact per-shard protocol repairs those users and the metrics are taken again
        idx, score, bad = sharded_topk(user_emb, index, K, kprime, group, defer_check=True)
        recall, ndcg = rank_metrics(idx, targets, k_list)
        packed = torch.cat([recall.flatten(), ndcg.flatten(), bad.max().float().view(1)]).cpu()
        if packed[-1].item() != 0:
            finish_sharded_topk(user_emb, index, K, idx, score, bad, kprime, group)
            recall, ndcg = rank_metrics(idx, targets, k_list)
            packed = torch.cat([recall.flatten(), ndcg.flatten()]).cpu()
        r = packed[:recall.numel()].view(recall.shape)
        n = packed[recall.numel():2 * recall.numel()].view(ndcg.shape)
    else:
        idx, score, _ = retrieve_topk(user_emb, index, K, kprime)
        recall, ndcg = rank_metrics(idx, targets, k_list)
        packed = torch.cat([recall.flatten(), ndcg.flatten()]).cpu()    # one read-back; the mean is taken on the host
        r = packed[:recall.numel()].view(recall.shape)                  # exactly like the reference (:188-190)
        n = packed[recall.numel():].view(ndcg.shape)
    out = {}
    for j, k in enumerate(k_list):
        out[f"Recall@{k}"] = r[j].mean().item()
    for j, k in enumerate(k_list):
        out[f"NDCG@{k}"] = n[j].mean().item()
    return out
