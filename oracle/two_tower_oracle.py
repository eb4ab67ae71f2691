"""CPU ORACLE — test infrastructure only, never a product path.

A plain-PyTorch, CPU, dtype-generic restatement of the reference's two-tower hot path
(DiegoPaniagua23/music-recommendation-multimodal). Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` leg may
import this module; the product package must never import it.

Pinning: the reference ships no tests, golden vectors or fixtures for this path
(SURVEY.md §4), so this oracle is pinned against outputs of the *reference's own modules*
run in the dev container — ``tests/golden/make_golden.py`` imports ``/root/reference``
(with the three harness-side stubs of SURVEY.md §8c), feeds it the seeded synthetic
parameters/batches of ``synthetic.py`` and stores outputs under ``tests/golden/``;
``tests/test_oracle_golden.py`` checks this file against them.

Each function cites the reference lines it restates (paths relative to the reference root).
The arithmetic the reference delegates to torch (nn.TransformerEncoderLayer,
F.cross_entropy, nn.BatchNorm1d ...) is written out explicitly here from its published
definition (torch 2.9.1 pinned by the reference's uv.lock; 2.11 in this image).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Params = Dict[str, torch.Tensor]


# ----------------------------------------------------------------------------------
# building blocks
# ----------------------------------------------------------------------------------
def layer_norm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """nn.LayerNorm over the last dim, biased variance (user_tower.py:47,54; item_tower.py:128)."""
    mu = x.mean(dim=-1, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w + b


def l2_normalize(x: torch.Tensor, eps: float = 1e-12) -> torch.Tensor:
    """F.normalize(p=2, dim=1) (two_tower.py:100-101,157,168)."""
    n = torch.sqrt((x * x).sum(dim=1, keepdim=True))
    return x / n.clamp_min(eps)


def encoder_layer(x: torch.Tensor, p: Params, prefix: str, num_heads: int,
                  key_is_pad: torch.Tensor, drop: Optional[Params] = None) -> torch.Tensor:
    """One pre-LN nn.TransformerEncoderLayer(d, nhead, 4d, batch_first, norm_first=True)
    (user_tower.py:37-45, called at :111-116 with a causal mask and a key-padding mask).
    torch semantics: x += OutProj(Attn(LN1(x))); x += W2 ReLU(W1 LN2(x)).
    Dropout is off unless ``drop`` gives this layer's scaled masks (keep / (1 - p)), applied where
    nn.TransformerEncoderLayer applies its dropouts: "attn" (B,H,L,L) on the softmax probabilities,
    "out_proj" (B,L,D) and "linear2" (B,L,D) before the residual adds, "ffn" (B,L,4D) after the ReLU."""
    B, L, D = x.shape
    dh = D // num_heads
    h = layer_norm(x, p[prefix + "norm1.weight"], p[prefix + "norm1.bias"])
    qkv = h @ p[prefix + "self_attn.in_proj_weight"].t() + p[prefix + "self_attn.in_proj_bias"]
    q, k, v = qkv.split(D, dim=-1)                      # in_proj rows are [Q; K; V]
    q = q.view(B, L, num_heads, dh).transpose(1, 2)
    k = k.view(B, L, num_heads, dh).transpose(1, 2)
    v = v.view(B, L, num_heads, dh).transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) / math.sqrt(dh)       # (B,H,L,L)
    causal = torch.triu(torch.ones(L, L, dtype=torch.bool), diagonal=1)
    neg = torch.finfo(s.dtype).min if False else float("-inf")
    s = s.masked_fill(causal, neg)
    s = s.masked_fill(key_is_pad[:, None, None, :], neg)
    a = torch.softmax(s, dim=-1)
    if drop is not None:
        a = a * drop["attn"]
    ctx = (a @ v).transpose(1, 2).reshape(B, L, D)
    if drop is None:
        x = x + ctx @ p[prefix + "self_attn.out_proj.weight"].t() + p[prefix + "self_attn.out_proj.bias"]
    else:
        x = x + (ctx @ p[prefix + "self_attn.out_proj.weight"].t() + p[prefix + "self_attn.out_proj.bias"]) * drop["out_proj"]
    h2 = layer_norm(x, p[prefix + "norm2.weight"], p[prefix + "norm2.bias"])
    f = torch.relu(h2 @ p[prefix + "linear1.weight"].t() + p[prefix + "linear1.bias"])
    if drop is None:
        x = x + f @ p[prefix + "linear2.weight"].t() + p[prefix + "linear2.bias"]
    else:
        f = f * drop["ffn"]
        x = x + (f @ p[prefix + "linear2.weight"].t() + p[prefix + "linear2.bias"]) * drop["linear2"]
    return x


def user_tower(p: Params, history_ids: torch.Tensor, user_gender: torch.Tensor,
               user_country: torch.Tensor, history_mask: Optional[torch.Tensor] = None,
               num_heads: int = 4, prefix: str = "user_tower.", drop: Optional[Params] = None) -> torch.Tensor:
    """SequentialUserEncoder.forward (user_tower.py:73-144). Dropout is off unless ``drop`` holds the
    scaled masks "emb" (B,L,D), after the embedding LayerNorm, and "layers.{l}.<site>" of encoder_layer.
    Returns the un-normalised (B, D) user embedding."""
    B, L = history_ids.shape
    E = p[prefix + "item_embedding.weight"]
    x = E[history_ids] + p[prefix + "position_embedding.weight"][:L].unsqueeze(0)     # :86-92
    x = layer_norm(x, p[prefix + "layer_norm.weight"], p[prefix + "layer_norm.bias"])  # :93
    if drop is not None:
        x = x * drop["emb"]
    if history_mask is not None:                                                        # :100-103
        key_is_pad = history_mask == 0
        lengths = history_mask.sum(dim=1).long() - 1                                    # :122-125
    else:
        key_is_pad = history_ids == 0
        lengths = (history_ids != 0).sum(dim=1).long() - 1
    num_layers = 0
    while f"{prefix}transformer_encoder.layers.{num_layers}.norm1.weight" in p:
        num_layers += 1
    for l in range(num_layers):                                                         # :111-116
        ld = None if drop is None else {k: drop[f"layers.{l}.{k}"] for k in ("attn", "out_proj", "ffn", "linear2")}
        x = encoder_layer(x, p, f"{prefix}transformer_encoder.layers.{l}.", num_heads, key_is_pad, ld)
    lengths = lengths.clamp(min=0)                                                      # :128
    seq = x[torch.arange(B), lengths]                                                   # :132
    g = p[prefix + "gender_embedding.weight"][user_gender]                              # :135-136
    c = p[prefix + "country_embedding.weight"][user_country]
    z = torch.cat([seq, g, c], dim=1)                                                   # :139
    z = z @ p[prefix + "fusion_layer.0.weight"].t() + p[prefix + "fusion_layer.0.bias"]  # :52-57
    z = layer_norm(z, p[prefix + "fusion_layer.1.weight"], p[prefix + "fusion_layer.1.bias"])
    z = torch.relu(z)
    return z @ p[prefix + "fusion_layer.3.weight"].t() + p[prefix + "fusion_layer.3.bias"]


def item_fusion(p: Params, audio: torch.Tensor, visual: torch.Tensor, text: torch.Tensor,
                tabular: torch.Tensor, training: bool, bn_eps: float = 1e-5,
                prefix: str = "item_tower.fusion_layer.", drop: Optional[torch.Tensor] = None,
                ) -> Tuple[torch.Tensor, Optional[Tuple[torch.Tensor, torch.Tensor]]]:
    """MultimodalItemEncoder.forward from the concat on (item_tower.py:147-150) with
    fusion_layer = Linear(512,512) -> BatchNorm1d -> ReLU -> Dropout -> Linear(512,256)
    -> LayerNorm (item_tower.py:121-129). Concat order: audio, visual, text, tabular.
    The Dropout is off unless ``drop`` gives its scaled (B, 512) mask.
    Returns (un-normalised item embedding, (batch_mean, batch_var_biased) in training mode)."""
    x = torch.cat([audio, visual, text, tabular], dim=1)
    y = x @ p[prefix + "0.weight"].t() + p[prefix + "0.bias"]
    stats = None
    if training:
        mu = y.mean(dim=0)
        var = ((y - mu) ** 2).mean(dim=0)          # biased: what BN normalises with
        stats = (mu, var)
    else:
        mu, var = p[prefix + "1.running_mean"].to(y.dtype), p[prefix + "1.running_var"].to(y.dtype)
    y = (y - mu) / torch.sqrt(var + bn_eps) * p[prefix + "1.weight"] + p[prefix + "1.bias"]
    y = torch.relu(y)
    if drop is not None:
        y = y * drop
    y = y @ p[prefix + "4.weight"].t() + p[prefix + "4.bias"]
    return layer_norm(y, p[prefix + "5.weight"], p[prefix + "5.bias"]), stats


def bn_running_update(running_mean, running_var, batch_mean, batch_var_biased, n: int, momentum: float = 0.1):
    """nn.BatchNorm1d buffer update in training mode: running stats take the UNBIASED variance."""
    unbiased = batch_var_biased * (n / max(n - 1, 1))
    return ((1 - momentum) * running_mean + momentum * batch_mean,
            (1 - momentum) * running_var + momentum * unbiased)


def infonce(user_emb: torch.Tensor, item_emb: torch.Tensor, temperature: float,
            user_idx: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Symmetric InfoNCE on already-normalised embeddings (two_tower.py:106-140).
    Same-user off-diagonal logits are overwritten with -1e4. Returns (loss, logits)."""
    logits = user_emb @ item_emb.t() / temperature
    if user_idx is not None:
        coll = user_idx.unsqueeze(1) == user_idx.unsqueeze(0)
        coll = coll & ~torch.eye(coll.shape[0], dtype=torch.bool)
        logits = logits.masked_fill(coll, -1e4)
    B = logits.shape[0]
    lse_r = torch.logsumexp(logits, dim=1)
    lse_c = torch.logsumexp(logits, dim=0)
    diag = logits.diagonal()
    loss = 0.5 * ((lse_r - diag).mean() + (lse_c - diag).mean())
    return loss, logits


def two_tower_forward(p: Params, batch: Dict[str, torch.Tensor], temperature: float = 0.07,
                      num_heads: int = 4, training: bool = True, drop: Optional[Params] = None):
    """TwoTowerModel.forward (two_tower.py:68-142) with the four modality encoders replaced
    by identity (north_star): batch['target_audio'|'target_image'|'target_input_ids'|
    'target_tabular'] carry precomputed (B,128) embeddings. ``drop``: every dropout site's
    scaled mask (user_tower's keys and "item"); None runs without dropout.
    Returns (loss, logits, user_emb, item_emb, bn_stats)."""
    u = user_tower(p, batch["history_ids"], batch["user_gender"], batch["user_country"],
                   batch.get("history_mask"), num_heads, drop=drop)
    dt = u.dtype
    i, stats = item_fusion(p, batch["target_audio"].to(dt), batch["target_image"].to(dt),
                           batch["target_input_ids"].to(dt), batch["target_tabular"].to(dt), training,
                           drop=None if drop is None else drop["item"])
    u = l2_normalize(u)
    i = l2_normalize(i)
    loss, logits = infonce(u, i, temperature, batch.get("user_idx"))
    return loss, logits, u, i, stats


TRAINABLE_SKIP = ("running_mean", "running_var", "num_batches_tracked")


def loss_and_grads(p: Params, batch, temperature: float = 0.07, num_heads: int = 4,
                   dtype: torch.dtype = torch.float32, drop: Optional[Params] = None):
    """Forward + autograd backward of the restated path (train.py:57-63 without AMP:
    on a CPU host autocast/GradScaler disable themselves, SURVEY.md App. A). ``drop``: the
    scaled dropout masks of two_tower_forward (None: dropout off)."""
    q = {}
    for k, v in p.items():
        if k.endswith(TRAINABLE_SKIP):
            q[k] = v.clone()
        else:
            q[k] = v.detach().to(dtype).clone().requires_grad_(True)
    loss, logits, u, i, stats = two_tower_forward(q, batch, temperature, num_heads, training=True, drop=drop)
    loss.backward()
    grads = {k: v.grad for k, v in q.items() if isinstance(v, torch.Tensor) and v.requires_grad}
    for k, g in list(grads.items()):
        if g is None:
            grads[k] = torch.zeros_like(q[k])
    # padding_idx=0: the reference's nn.Embedding never accumulates into row 0 (user_tower.py:26)
    grads["user_tower.item_embedding.weight"][0] = 0
    return loss.detach(), logits.detach(), u.detach(), i.detach(), grads, stats


def adamw_step(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, step: int,
               lr: float = 1e-4, beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-8,
               weight_decay: float = 0.01):
    """torch.optim.AdamW defaults as used at train.py:302 (lr=1e-4), dense, decoupled decay."""
    p = p * (1 - lr * weight_decay)
    m = beta1 * m + (1 - beta1) * g
    v = beta2 * v + (1 - beta2) * g * g
    bc1 = 1 - beta1 ** step
    bc2 = 1 - beta2 ** step
    denom = v.sqrt() / math.sqrt(bc2) + eps
    p = p - (lr / bc1) * m / denom
    return p, m, v


# ----------------------------------------------------------------------------------
# retrieval (evaluate_metrics.py:106-192)
# ----------------------------------------------------------------------------------
def canonical_topk(scores: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Top-k under the canonical order (score descending, item index ascending).
    torch.topk (evaluate_metrics.py:156) leaves tie order unspecified; a stable descending
    sort returns the lowest index first among equal scores."""
    vals, idx = torch.sort(scores, dim=1, descending=True, stable=True)
    return vals[:, :k], idx[:, :k]


def retrieval_scores(user_emb: torch.Tensor, item_embeddings: torch.Tensor) -> torch.Tensor:
    """scores = U @ E^T in fp32 with column 0 (padding id) masked (evaluate_metrics.py:148-152)."""
    s = user_emb @ item_embeddings.t()
    s[:, 0] = float("-inf")
    return s


def recommend(user_emb: torch.Tensor, item_embeddings: torch.Tensor, history_ids: Sequence[int],
              k: int = 10) -> Tuple[torch.Tensor, torch.Tensor]:
    """The scoring part of recommend_for_user (src/inference.py:283-303) for ONE user: re-normalise with
    eps 1e-8 (:286), scores = u @ E^T (:291), padding id 0 and every history item masked to -inf (:296-302),
    top-k (:306) under the canonical order. Returns (scores (k,), item ids (k,))."""
    u = F.normalize(user_emb.view(1, -1), p=2, dim=1, eps=1e-8)
    s = (u @ item_embeddings.t()).squeeze(0)
    s[0] = float("-inf")
    for h in history_ids:
        if h < s.numel():
            s[h] = float("-inf")
    vals, idx = canonical_topk(s.view(1, -1), k)
    return vals[0], idx[0]


def rank_metrics(topk_idx: torch.Tensor, targets: torch.Tensor, k_list: Sequence[int]) -> Dict[str, torch.Tensor]:
    """Per-row Recall@k / NDCG@k (evaluate_metrics.py:159-185): hit if target in the first k;
    gain 1/log2(rank+2) with the 0-based rank, single relevant item => IDCG = 1."""
    out = {}
    t = targets.view(-1, 1)
    for k in k_list:
        eq = topk_idx[:, :k] == t
        hit = eq.any(dim=1)
        rank = eq.float().argmax(dim=1)
        gain = 1.0 / torch.log2(rank.float() + 2.0)
        out[f"Recall@{k}"] = hit.float()
        out[f"NDCG@{k}"] = torch.where(hit, gain, torch.zeros_like(gain))
    return out


def calculate_metrics_global(user_emb: torch.Tensor, item_embeddings: torch.Tensor, targets: torch.Tensor,
                             k_list: Sequence[int] = (10, 20), batch_size: int = 64) -> Dict[str, float]:
    """The scoring / top-K / metric part of calculate_metrics_global (evaluate_metrics.py:106-192)
    on precomputed user embeddings, batched like the reference (val batch 64, :203)."""
    per = {f"Recall@{k}": [] for k in k_list}
    per.update({f"NDCG@{k}": [] for k in k_list})
    kmax = max(k_list)
    for s in range(0, user_emb.shape[0], batch_size):
        sc = retrieval_scores(user_emb[s:s + batch_size], item_embeddings)
        _, idx = canonical_topk(sc, kmax)
        m = rank_metrics(idx, targets[s:s + batch_size], k_list)
        for k, v in m.items():
            per[k].append(v)
    return {k: torch.cat(v).mean().item() for k, v in per.items()}


# ----------------------------------------------------------------------------------
# in-batch validation (train.py:78-111)
# ----------------------------------------------------------------------------------
def inbatch_hits(logits: torch.Tensor, k: int = 10) -> torch.Tensor:
    """Per-row hit flags of the in-batch Recall@k of ``evaluate`` (train.py:100-103): row i hits when
    column i is among the k best logits of row i. torch.topk leaves the order of equal logits
    unspecified; here ties are resolved by the canonical order (logit descending, column ascending),
    i.e. hit <=> #{j : l_ij > l_ii or (l_ij == l_ii and j < i)} < k. With k >= B every row hits
    (the reference's topk would raise for k > B: callers keep k <= B)."""
    B = logits.shape[0]
    diag = logits.diagonal().unsqueeze(1)
    col = torch.arange(logits.shape[1]).unsqueeze(0)
    row = torch.arange(B).unsqueeze(1)
    better = (logits > diag) | ((logits == diag) & (col < row))
    return better.sum(dim=1) < k


def evaluate_inbatch(logit_batches: Sequence[torch.Tensor], k: int = 10) -> float:
    """``evaluate`` (train.py:78-111) given the per-batch logits of model(batch): hits / total over all
    batches (the all_reduce(SUM) of :106-109 adds the per-rank hits and totals before the division)."""
    hits, total = 0.0, 0.0
    for lg in logit_batches:
        hits += float(inbatch_hits(lg, k).sum().item())
        total += lg.shape[0]
    return hits / total if total > 0 else 0.0


# ----------------------------------------------------------------------------------
# catalog indexing (evaluate_metrics.py:24-104)
# ----------------------------------------------------------------------------------
def index_catalog(p: Params, features: Dict[str, torch.Tensor], item_ids: torch.Tensor, vocab_size: int,
                  batch_size: int = 64) -> torch.Tensor:
    """``compute_all_item_embeddings`` on precomputed modality embeddings: per batch (evaluate_metrics.py:63-87)
    emb = get_item_embedding(...) = F.normalize(item tower in eval mode) (two_tower.py:159-168, eps 1e-12);
    if the batch holds a NaN, nan_to_num(nan=0) (:79-81); F.normalize(eps=1e-8) again (:85). Then the dense
    scatter (:98-102): table[item_id] = embedding, row 0 and every id not listed stay zero.
    Returns the (vocab_size, D) table in the dtype of the parameters."""
    dt = p["item_tower.fusion_layer.0.weight"].dtype
    rows = []
    for s in range(0, item_ids.shape[0], batch_size):
        sl = slice(s, s + batch_size)
        e, _ = item_fusion(p, features["target_audio"][sl].to(dt), features["target_image"][sl].to(dt),
                           features["target_input_ids"][sl].to(dt), features["target_tabular"][sl].to(dt),
                           training=False)
        e = l2_normalize(e)
        if torch.isnan(e).any():
            e = torch.nan_to_num(e, nan=0.0)
        rows.append(F.normalize(e, p=2, dim=1, eps=1e-8))
    emb = torch.cat(rows, dim=0)
    dense = torch.zeros(vocab_size, emb.shape[1], dtype=emb.dtype)
    dense[item_ids.long()] = emb
    return dense


# ----------------------------------------------------------------------------------
# data-parallel step with all-gathered negatives (BASELINE.json configs[3]; SURVEY.md §8e)
# ----------------------------------------------------------------------------------
def dp_loss_and_grads(p: Params, batches: Sequence[Dict[str, torch.Tensor]], temperature: float = 0.07,
                      num_heads: int = 4, dtype: torch.dtype = torch.float64, tower_grads: bool = True):
    """G data-parallel ranks, rank r holding ``batches[r]``: the towers run per rank (BatchNorm batch statistics
    per rank: the reference wraps the model in plain DDP, no SyncBatchNorm, train.py:300), the normalised
    embeddings and user ids of all ranks are concatenated and ONE symmetric InfoNCE (two_tower.py:106-140) is
    taken over the global batch. Returns (loss, {param: d loss / d param}, user_emb_all, item_emb_all,
    d loss / d user_emb_all, d loss / d item_emb_all); ``tower_grads=False`` stops at the embedding gradients
    (parameter gradients None). The averaged per-rank gradient the DP step applies equals this gradient. Memory stays that of one rank:
    embeddings first without autograd, then one autograd pass per rank seeded with d loss / d embedding."""
    q = {k: (v.clone() if k.endswith(TRAINABLE_SKIP) else v.detach().to(dtype)) for k, v in p.items()}

    def towers(params, b):
        u = user_tower(params, b["history_ids"], b["user_gender"], b["user_country"], b.get("history_mask"), num_heads)
        i, _ = item_fusion(params, b["target_audio"].to(dtype), b["target_image"].to(dtype),
                           b["target_input_ids"].to(dtype), b["target_tabular"].to(dtype), True)
        return l2_normalize(u), l2_normalize(i)

    with torch.no_grad():
        embs = [towers(q, b) for b in batches]
    U = torch.cat([e[0] for e in embs]).requires_grad_(True)
    I = torch.cat([e[1] for e in embs]).requires_grad_(True)
    uid = torch.cat([b["user_idx"] for b in batches]) if "user_idx" in batches[0] else None
    loss, _ = infonce(U, I, temperature, uid)
    loss.backward()
    if not tower_grads:
        return loss.detach(), None, U.detach(), I.detach(), U.grad, I.grad
    grads = None
    off = 0
    for b in batches:
        n = b["history_ids"].shape[0]
        qr = {k: (v if k.endswith(TRAINABLE_SKIP) else v.clone().requires_grad_(True)) for k, v in q.items()}
        u, i = towers(qr, b)
        torch.autograd.backward([u, i], [U.grad[off:off + n], I.grad[off:off + n]])
        gr = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in qr.items()
              if isinstance(v, torch.Tensor) and v.requires_grad}
        grads = gr if grads is None else {k: grads[k] + gr[k] for k in gr}
        off += n
    grads["user_tower.item_embedding.weight"][0] = 0
    return loss.detach(), grads, U.detach(), I.detach(), U.grad, I.grad
