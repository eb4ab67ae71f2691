"""Listening sessions: a user's embedding updated after each new listen from cached attention keys and values.

A streaming service refreshes a user's recommendations after every listen. Re-running the user tower on the whole
window costs the full padded window per update. The encoder is causal and a history is a right-padded prefix, so
appending item p to a history of length p < L leaves every earlier position unchanged in every layer: per layer only
the new row's Q/K/V, one query over the cached K/V of positions 0..p (tt_session_attn), out_proj and the FFN remain,
then the fusion head (TwoTowerEngine.session_append).

`UserSessions` owns, on the device, the K/V planes of every layer (bf16 [capacity, 4, L, 64] each: 2 KB per token at
two layers), the window ids [capacity, L] and gender / country per slot, plus a host copy of every slot's length, so
choosing the incremental path needs no device synchronisation. The caller owns the slot numbers (no eviction policy).

A full window (length L) follows the reference's window semantics, the last L items (src/inference.py:254-258): the
oldest item drops out and every position shifts, so such rows are re-run through the whole tower on the shifted window
(one batched call) and their caches refilled. That is exact, and the only path for full windows.

Caches derive from the weights. Every slot records `engine.weights_epoch` and the model's parameter version when it is
filled; `append` and `recommend` raise RuntimeError for a slot filled under other weights.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import inference, retrieval

IntsLike = Union[Sequence[int], torch.Tensor, np.ndarray]


class UserSessions:
    def __init__(self, model, capacity: int):
        eng = model.engine
        if eng.table_rows is not None or eng.peer_table is not None:
            raise NotImplementedError("user sessions need a local ID table (no row-sharded or peer table)")
        if capacity < 1:
            raise ValueError(f"capacity = {capacity}: at least one slot")
        cfg, dev = eng.cfg, eng.device
        self.model, self.engine, self.capacity = model, eng, capacity
        self.L, H = cfg.max_seq_len, cfg.num_heads
        bf = dict(device=dev, dtype=torch.bfloat16)
        self.k_cache = [torch.zeros(capacity, H, self.L, 64, **bf) for _ in range(cfg.num_layers)]
        self.v_cache = [torch.zeros(capacity, H, self.L, 64, **bf) for _ in range(cfg.num_layers)]
        self.window = torch.zeros(capacity, self.L, device=dev, dtype=torch.long)
        self.gender = torch.zeros(capacity, device=dev, dtype=torch.long)
        self.country = torch.zeros(capacity, device=dev, dtype=torch.long)
        self.emb = torch.zeros(capacity, cfg.embedding_dim, device=dev)
        #: host copy of each slot's history length (0 = empty)
        self.lengths = np.zeros(capacity, dtype=np.int64)
        self._epoch = np.full(capacity, -1, dtype=np.int64)
        self._version = np.full(capacity, -1, dtype=np.int64)
        self._ws: Dict[int, Dict[str, torch.Tensor]] = {}

    # ------------------------------------------------------------------ checks
    def _slots(self, slots: IntsLike) -> np.ndarray:
        s = np.asarray(torch.as_tensor(slots).cpu(), dtype=np.int64).reshape(-1)
        if s.size == 0:
            raise ValueError("no slots given")
        if s.min() < 0 or s.max() >= self.capacity:
            raise ValueError(f"slot outside [0, {self.capacity})")
        if np.unique(s).size != s.size:
            raise ValueError("a slot appears more than once in one call")
        return s

    def _check_fresh(self, s: np.ndarray) -> int:
        """RuntimeError if a non-empty slot of ``s`` was filled under other weights; returns the parameter version."""
        version = self.model._param_version()
        filled = self.lengths[s] > 0
        stale = filled & ((self._epoch[s] != self.engine.weights_epoch) | (self._version[s] != version))
        if stale.any():
            raise RuntimeError(f"slots {s[stale].tolist()[:8]} were filled under other weights: open them again")
        return version

    def _ids_of(self, s: np.ndarray) -> torch.Tensor:
        return torch.from_numpy(s).to(self.engine.device)

    # ------------------------------------------------------------------ full tower
    def _fill(self, s: np.ndarray, win: torch.Tensor, lengths: np.ndarray, gender: torch.Tensor,
              country: torch.Tensor) -> torch.Tensor:
        """Eval-mode tower on the windows ``win`` (n, L) int64 (right-padded) of slots ``s``; K/V of every layer and
        position go to the caches. Returns the normalised embeddings (n, 256)."""
        model, eng, L = self.model, self.engine, self.L
        H = eng.cfg.num_heads
        chunk = min(inference._TOWER_CHUNK, inference._TOWER_TOKENS // L)
        was_training = model.training
        model.eval()
        outs = []
        with torch.no_grad():
            for c0 in range(0, s.size, chunk):
                sl = self._ids_of(s[c0:c0 + chunk])
                w = win[c0:c0 + chunk]
                b = w.shape[0]
                outs.append(model.get_user_embedding(w, (w != 0).long(), gender[c0:c0 + chunk],
                                                     country[c0:c0 + chunk]))
                ws = eng.workspace(b, L)
                for l in range(eng.cfg.num_layers):
                    kv = ws[f"qkv_{l}"].view(b, L, 3, H, 64)
                    self.k_cache[l][sl] = kv[:, :, 1].transpose(1, 2)
                    self.v_cache[l][sl] = kv[:, :, 2].transpose(1, 2)
        model.train(was_training)
        u = torch.cat(outs)
        sl = self._ids_of(s)
        self.window[sl] = win
        self.gender[sl] = gender
        self.country[sl] = country
        self.emb[sl] = u
        self.lengths[s] = lengths
        self._epoch[s] = eng.weights_epoch
        self._version[s] = model._param_version()
        return u

    # ------------------------------------------------------------------ public interface
    def open(self, slots: IntsLike, history_ids: torch.Tensor, history_mask: Optional[torch.Tensor] = None,
             user_gender: Optional[torch.Tensor] = None, user_country: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Start (or restart) the sessions of ``slots`` from ``history_ids`` (n, Lh) int64, Lh <= max_seq_len: non-empty
        right-padded prefixes (``history_mask`` (n, Lh), default ids != 0). Returns the normalised user embeddings
        (n, 256) fp32, those of `TwoTowerModel.get_user_embedding` on the same histories."""
        s = self._slots(slots)
        cfg, dev = self.engine.cfg, self.engine.device
        ids = torch.as_tensor(history_ids).cpu().long()
        if ids.dim() != 2 or ids.shape[0] != s.size:
            raise ValueError(f"history_ids {tuple(ids.shape)} for {s.size} slots")
        n, Lh = ids.shape
        if Lh > self.L:
            raise ValueError(f"history window {Lh} exceeds the model's max_seq_len {self.L}")
        mask = (ids != 0) if history_mask is None else (torch.as_tensor(history_mask).cpu() != 0)
        if mask.shape != ids.shape:
            raise ValueError("history_mask and history_ids differ in shape")
        lengths = mask.sum(dim=1)
        if (lengths == 0).any():
            raise ValueError("empty history")
        if not torch.equal(mask, torch.arange(Lh)[None, :] < lengths[:, None]):
            raise ValueError("histories must be right-padded prefixes")
        valid = ids[mask]
        if (valid < 1).any() or (valid >= cfg.vocab_size).any():
            raise ValueError(f"history item id outside [1, {cfg.vocab_size})")
        win = torch.zeros(n, self.L, dtype=torch.long)
        win[:, :Lh] = ids * mask
        gender = self._demographic(user_gender, n, cfg.num_genders, "user_gender")
        country = self._demographic(user_country, n, cfg.num_countries, "user_country")
        return self._fill(s, win.to(dev), lengths.numpy(), gender.to(dev), country.to(dev)).clone()

    @staticmethod
    def _demographic(t, n: int, bound: int, what: str) -> torch.Tensor:
        if t is None:
            return torch.zeros(n, dtype=torch.long)
        t = torch.as_tensor(t).cpu().long().reshape(-1)
        if t.numel() != n or (t < 0).any() or (t >= bound).any():
            raise ValueError(f"{what}: {n} values in [0, {bound}) expected")
        return t

    def _append_ws(self, n: int) -> Dict[str, torch.Tensor]:
        """Row views of a session workspace sized to the next power of two (few distinct allocations)."""
        if n not in self._ws:
            full = self.engine.session_workspace(1 << (n - 1).bit_length())
            self._ws[n] = {k: v[:n] for k, v in full.items()}
        return self._ws[n]

    def append(self, slots: IntsLike, item_ids: IntsLike) -> torch.Tensor:
        """One new listen per slot: item ``item_ids[r]`` is appended to the history of ``slots[r]``. Returns the
        normalised embeddings (n, 256) fp32 of the extended windows. An empty slot starts at position 0; a full
        window drops its oldest item (those rows are re-run through the whole tower)."""
        s = self._slots(slots)
        items = np.asarray(torch.as_tensor(item_ids).cpu(), dtype=np.int64).reshape(-1)
        V = self.engine.cfg.vocab_size
        if items.size != s.size:
            raise ValueError(f"{items.size} item ids for {s.size} slots")
        if items.min() < 1 or items.max() >= V:
            raise ValueError(f"item id outside [1, {V})")
        version = self._check_fresh(s)
        self.model._sync_shadow()
        dev = self.engine.device
        full = self.lengths[s] >= self.L
        inc = np.flatnonzero(~full)
        out = None if inc.size == s.size else torch.empty(s.size, self.engine.cfg.embedding_dim, device=dev)
        if inc.size:
            si, pi, n = s[inc], self.lengths[s[inc]], inc.size
            packed = np.empty(4 * n, dtype=np.int32)          # slots | positions | item ids as int64: one copy
            packed[:n], packed[n:2 * n] = si, pi
            packed[2 * n:].view(np.int64)[:] = items[inc]
            d = torch.from_numpy(packed).to(dev, non_blocking=True)
            d_slot, d_pos, d_item = d[:n], d[n:2 * n], d[2 * n:].view(torch.int64)
            ws = self._append_ws(n)
            u = self.engine.session_append(ws, d_item, d_slot, d_pos, self.k_cache, self.v_cache,
                                           self.gender[d_slot.long()], self.country[d_slot.long()])
            d_slot = d_slot.long()
            self.window[d_slot, d_pos.long()] = d_item
            self.emb[d_slot] = u
            if out is None:
                out = u.clone()
            else:
                out[torch.from_numpy(inc).to(dev)] = u
            self.lengths[si] += 1
            self._epoch[si] = self.engine.weights_epoch      # slots that started empty take the current weights
            self._version[si] = version
        fi = np.flatnonzero(full)
        if fi.size:
            sf = s[fi]
            sl = self._ids_of(sf)
            win = torch.cat([self.window[sl, 1:], torch.from_numpy(items[fi]).to(dev)[:, None]], dim=1)
            u = self._fill(sf, win, np.full(fi.size, self.L), self.gender[sl], self.country[sl])
            out[torch.from_numpy(fi).to(dev)] = u
        return out

    def recommend(self, slots: IntsLike, index: retrieval.CatalogIndex, k: int = 10,
                  exclude_ids: Optional[torch.Tensor] = None, group=None, diversity: float = 0.0,
                  pool: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """`inference.recommend_batch`'s selection on the sessions' current embeddings: top k of plain or sharded
        ``index``, excluding ``exclude_ids`` (n, m) int64 or, by default, each slot's window ids. Returns (item ids int64
        (n, k), scores fp32 (n, k)); id -1 / score -inf where fewer than k items are admissible. ``diversity`` /
        ``pool``: as in `inference.recommend_embeddings` (diversity > 0: pick order, not sorted by score)."""
        if not 1 <= k <= 256:
            raise ValueError(f"recommend: k = {k} outside [1, 256]")
        s = self._slots(slots)
        if (self.lengths[s] == 0).any():
            raise ValueError("recommend on an empty slot")
        self._check_fresh(s)
        sl = self._ids_of(s)
        ex = self.window[sl] if exclude_ids is None else exclude_ids.to(self.engine.device).long()
        return inference.recommend_embeddings(self.emb[sl], index, ex, k, group, diversity, pool)

    def reset(self, slots: IntsLike) -> None:
        """Empty the slots: the next `append` starts a history at position 0 (gender / country 0)."""
        s = self._slots(slots)
        sl = self._ids_of(s)
        self.window[sl] = 0
        self.gender[sl] = 0
        self.country[sl] = 0
        self.lengths[s] = 0
        self._epoch[s] = -1
        self._version[s] = -1
