"""Kernel sequencing for the two-tower hot path: forward, backward and the fused AdamW step.

The engine owns
  * one flat fp32 parameter buffer (reference state-dict tensors are views into it), a flat
    fp32 gradient buffer of the same layout, AdamW moments, and a bf16 shadow of the dense
    region (tensor-core operands);
  * per-(batch, seq_len) activation workspaces, allocated once and reused (CUDA-graph safe);
and launches the C-ABI kernels of libtt_b200.so in order on the current stream. There is no
autograd here: the backward pass is written out by hand, mirroring the forward.

Reference call sites: SequentialUserEncoder.forward (src/models/user_tower.py:73-144),
MultimodalItemEncoder.fusion_layer (src/models/item_tower.py:121-129,147-150),
TwoTowerModel.forward (src/models/two_tower.py:68-142), the step body of train_one_epoch
(src/train.py:48-67).
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import os

import torch

from . import ops
from .synthetic import TwoTowerConfig

_ALIGN = 64  # elements; keeps every bf16 view 128-byte aligned (TMA needs 16)

# dropout sites (hash domain separation)
SITE_EMB = 1
SITE_ITEM = 60


def _site(layer: int, which: int) -> int:
    """which: 0 attention probabilities, 1 after out_proj, 2 inside FFN, 3 after linear2."""
    return 10 + 4 * layer + which


def param_shapes(cfg: TwoTowerConfig) -> List[Tuple[str, Tuple[int, ...]]]:
    """(name, shape) of every trainable tensor, reference key names (SURVEY.md §8b).
    Order = flat-buffer order: ID table, small embeddings, then the dense region."""
    D, FF, H = cfg.embedding_dim, cfg.ff_dim, cfg.fusion_hidden
    ut = "user_tower."
    out = [
        (ut + "item_embedding.weight", (cfg.vocab_size, D)),
        (ut + "position_embedding.weight", (cfg.max_seq_len, D)),
        (ut + "gender_embedding.weight", (cfg.num_genders, 16)),
        (ut + "country_embedding.weight", (cfg.num_countries, 32)),
    ]
    for l in range(cfg.num_layers):
        p = f"{ut}transformer_encoder.layers.{l}."
        out += [
            (p + "self_attn.in_proj_weight", (3 * D, D)), (p + "self_attn.in_proj_bias", (3 * D,)),
            (p + "self_attn.out_proj.weight", (D, D)), (p + "self_attn.out_proj.bias", (D,)),
            (p + "linear1.weight", (FF, D)), (p + "linear1.bias", (FF,)),
            (p + "linear2.weight", (D, FF)), (p + "linear2.bias", (D,)),
            (p + "norm1.weight", (D,)), (p + "norm1.bias", (D,)),
            (p + "norm2.weight", (D,)), (p + "norm2.bias", (D,)),
        ]
    out += [
        (ut + "layer_norm.weight", (D,)), (ut + "layer_norm.bias", (D,)),
        (ut + "fusion_layer.0.weight", (D, D + 48)), (ut + "fusion_layer.0.bias", (D,)),
        (ut + "fusion_layer.1.weight", (D,)), (ut + "fusion_layer.1.bias", (D,)),
        (ut + "fusion_layer.3.weight", (D, D)), (ut + "fusion_layer.3.bias", (D,)),
    ]
    it = "item_tower.fusion_layer."
    out += [
        (it + "0.weight", (H, 4 * cfg.modality_dim)), (it + "0.bias", (H,)),
        (it + "1.weight", (H,)), (it + "1.bias", (H,)),
        (it + "4.weight", (D, H)), (it + "4.bias", (D,)),
        (it + "5.weight", (D,)), (it + "5.bias", (D,)),
    ]
    return out


_NUM_SPARSE = 4  # table, positions, gender, country come before the dense region
#: longest history window the attention kernels take (tt_attn_causal_*, tt_attn_lastq_*)
MAX_SEQ_LEN = 4096
#: most tokens (B * L) one user-tower call may hold: the bound the kernels' 32-bit indices were checked against
#: (T * 4D = 2^30; the GEMM epilogues' 32-bit dropout index row * N + col wraps from 2^22 tokens)
MAX_TOKENS = 1 << 20


class TwoTowerEngine:
    def __init__(self, cfg: TwoTowerConfig, device: Optional[torch.device] = None):
        assert cfg.embedding_dim == 256 and cfg.num_heads == 4, \
            "the sm_100a kernels are specialised for d_model=256, 4 heads of 64 (the reference's configuration)"
        assert cfg.fusion_hidden == 512 and 4 * cfg.modality_dim == 512
        if not 1 <= cfg.max_seq_len <= MAX_SEQ_LEN:
            raise ValueError(f"max_seq_len = {cfg.max_seq_len} outside [1, {MAX_SEQ_LEN}]")
        self.cfg = cfg
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        shapes = param_shapes(cfg)
        self.layout: Dict[str, Tuple[int, Tuple[int, ...]]] = {}
        off = 0
        for i, (name, shape) in enumerate(shapes):
            if i == _NUM_SPARSE:
                self.dense_begin = off
            n = 1
            for s in shape:
                n *= s
            self.layout[name] = (off, shape)
            off += (n + _ALIGN - 1) // _ALIGN * _ALIGN
        off += _ALIGN  # tail padding: ragged MN-major chunks may read up to 63 elements past a tensor
        off = (off + 2047) // 2048 * 2048   # divisible into 1/2/4/8 equal, 16-byte aligned optimizer shards
        self.numel = off
        dev = self.device
        self.flat = torch.zeros(off, device=dev)
        self.grad = torch.zeros(off, device=dev)
        self.exp_avg: Optional[torch.Tensor] = None
        self.exp_avg_sq: Optional[torch.Tensor] = None
        self.shadow = torch.zeros(off - self.dense_begin, device=dev, dtype=torch.bfloat16)
        self.p: Dict[str, torch.Tensor] = {}
        self.g: Dict[str, torch.Tensor] = {}
        self.w: Dict[str, torch.Tensor] = {}   # bf16 shadows (dense region only)
        self.rebind_hooks = []
        self._bind_views()
        H = cfg.fusion_hidden
        self.bn_running_mean = torch.zeros(H, device=dev)
        self.bn_running_var = torch.ones(H, device=dev)
        self.bn_num_batches = torch.zeros((), device=dev, dtype=torch.long)
        self.step_dev = torch.zeros((), device=dev, dtype=torch.long)     # AdamW step count
        self.seed_dev = torch.zeros((), device=dev, dtype=torch.long)     # dropout seed offset
        self.base_seed = 0x5EED
        self._ws: Dict[Tuple[int, int], Dict[str, torch.Tensor]] = {}
        self.shadow_valid = False
        #: compute the last encoder layer's query / out_proj / FFN only for the row that is read
        #: (exact; SURVEY.md §8 a5). False runs every layer on every position like the reference.
        self.prune_last_layer = True
        #: run weight-gradient GEMMs / bias column sums on a second stream (see _wg)
        #: measurement aid: issue everything on the current stream (per-kernel event timing without overlap)
        self.serialize = False
        #: row-sharded ID table (sharding.RowShardedTable, config 5): when set, `table_rows` [1 + B*L, 256] holds
        #: the rows the exchange fetched for this step's tokens (row 0 unused) and the embedding kernels index
        #: it with the token number instead of the item id; `table_rows_grad` receives the per-token gradient
        #: rows, which the owner ranks then scatter-add. The flat buffer's own table region is a 2-row dummy.
        self.table_rows: Optional[torch.Tensor] = None
        self.table_rows_grad: Optional[torch.Tensor] = None
        self._virt_ids: Dict[Tuple[int, int], torch.Tensor] = {}
        #: sharding.SymmShardedTable: the ID table lives row-sharded in a symmetric NVLink arena; the embedding
        #: kernels read rows from / add gradient rows into the OWNER's memory directly (no exchange step). The flat
        #: buffer's own table region is a 2-row dummy.
        self.peer_table = None
        self._sparse: Dict[int, Dict[str, torch.Tensor]] = {}
        #: deterministic table gradient (TT_DETERMINISTIC=1): the per-token gradient rows of duplicate ids are summed
        #: in 64-bit fixed point per distinct id (tt_embed_ln_bwd_det), so the result does not depend on the order the
        #: atomics land in. Local (replicated / single-GPU) table only; costs the id de-duplication (3 small kernels)
        #: and 2 KB of accumulator per distinct id and step.
        self.deterministic_table_grad = os.environ.get("TT_DETERMINISTIC", "0") == "1"
        self._det: Dict[int, Dict[str, torch.Tensor]] = {}
        #: host-side count of parameter updates (load_state_dict, the AdamW steps, TrainStepRunner steps): state derived
        #: from the weights, such as the K/V caches of sessions.UserSessions, records it and is refused once it moved
        self.weights_epoch = 0

    # ------------------------------------------------------------------ parameters
    def use_external_table(self, B: int, L: int) -> None:
        """Switch the ID-embedding lookups to the per-step row buffer of a row-sharded table."""
        D = self.cfg.embedding_dim
        self.table_rows = torch.zeros(1 + B * L, D, device=self.device)
        self.table_rows_grad = torch.zeros(1 + B * L, D, device=self.device)

    def _embed_operands(self, ids: torch.Tensor):
        """(ids, table, table_grad) the embedding kernels see: the real ones, or token numbers 1..B*L into the
        fetched-rows buffer when the table is row-sharded."""
        ut = "user_tower."
        if self.table_rows is None:
            return ids.view(-1), self.p[ut + "item_embedding.weight"], self.g[ut + "item_embedding.weight"]
        B, L = ids.shape
        assert self.table_rows.shape[0] == 1 + B * L, "use_external_table was sized for another (B, L)"
        if (B, L) not in self._virt_ids:
            self._virt_ids[(B, L)] = torch.arange(1, 1 + B * L, device=self.device, dtype=torch.long)
        return self._virt_ids[(B, L)], self.table_rows, self.table_rows_grad

    def _bind_views(self) -> None:
        self.p, self.g, self.w = {}, {}, {}
        for name, (o, shape) in self.layout.items():
            n = 1
            for s in shape:
                n *= s
            self.p[name] = self.flat[o:o + n].view(shape)
            self.g[name] = self.grad[o:o + n].view(shape)
            if o >= self.dense_begin:
                so = o - self.dense_begin
                self.w[name] = self.shadow[so:so + n].view(shape)

    def rebind_storage(self, flat: torch.Tensor, grad: torch.Tensor, shadow: torch.Tensor) -> None:
        """Move the parameters, gradients and the bf16 operand shadow into caller-provided buffers of the same
        sizes (blocks of a symmetric arena, symm.SymmArena) and re-point every view at them. CUDA graphs and
        workspaces that captured the old buffers must be rebuilt by their owners; `rebind_hooks` lets the
        nn.Module wrappers re-point their Parameters."""
        assert flat.numel() == self.numel and grad.numel() == self.numel and shadow.numel() == self.shadow.numel()
        assert flat.dtype == torch.float32 and grad.dtype == torch.float32 and shadow.dtype == torch.bfloat16
        flat.copy_(self.flat)
        grad.copy_(self.grad)
        shadow.copy_(self.shadow)
        self.flat, self.grad, self.shadow = flat, grad, shadow
        self._bind_views()
        for hook in getattr(self, "rebind_hooks", []):
            hook()

    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        """Copy a reference-format state dict (src/train.py:327-330; optional 'module.' prefix,
        encoder keys ignored) into the flat buffer. With a row-sharded table the ID table entry is skipped
        (RowShardedTable.load_full takes it)."""
        sd = {(k[7:] if k.startswith("module.") else k): v for k, v in sd.items()}
        for name, t in self.p.items():
            if name == "user_tower.item_embedding.weight" and self.peer_table is not None:
                self.peer_table.load_full(sd[name])       # every rank keeps the rows it owns
                continue
            if self.table_rows is not None and name == "user_tower.item_embedding.weight":
                continue
            t.copy_(sd[name].to(device=self.device, dtype=torch.float32))
        it = "item_tower.fusion_layer.1."
        if it + "running_mean" in sd:
            self.bn_running_mean.copy_(sd[it + "running_mean"])
            self.bn_running_var.copy_(sd[it + "running_var"])
            self.bn_num_batches.copy_(sd[it + "num_batches_tracked"])
        self.shadow_valid = False
        self.weights_epoch += 1

    def state_dict(self) -> Dict[str, torch.Tensor]:
        out = {k: v.detach().clone() for k, v in self.p.items()}
        if self.peer_table is not None:      # collective: the owners' shards are all-gathered
            out["user_tower.item_embedding.weight"] = self.peer_table.gather_full()
        it = "item_tower.fusion_layer.1."
        out[it + "running_mean"] = self.bn_running_mean.clone()
        out[it + "running_var"] = self.bn_running_var.clone()
        out[it + "num_batches_tracked"] = self.bn_num_batches.clone()
        return out

    def refresh_shadow(self) -> None:
        ops.cast_bf16(self.flat[self.dense_begin:], self.shadow)
        self.shadow_valid = True

    # ------------------------------------------------------------------ workspaces
    def workspace(self, B: int, L: int) -> Dict[str, torch.Tensor]:
        """Activation buffers of a (B, L) user-tower call; B * L <= MAX_TOKENS, else ValueError."""
        key = (B, L)
        if key in self._ws:
            return self._ws[key]
        cfg, dev = self.cfg, self.device
        D, FF, NL, Hh = cfg.embedding_dim, cfg.ff_dim, cfg.num_layers, cfg.num_heads
        T = B * L
        if T > MAX_TOKENS:
            raise ValueError(f"{B} sequences x {L} positions = {T} tokens in one call; at most {MAX_TOKENS}")
        f32 = dict(device=dev, dtype=torch.float32)
        bf = dict(device=dev, dtype=torch.bfloat16)
        ws: Dict[str, torch.Tensor] = {}
        ws["last_idx"] = torch.zeros(B, device=dev, dtype=torch.int32)
        ws["x_in0"] = torch.empty(T, D, **f32)
        for l in range(NL):
            ws[f"h1_{l}"] = torch.empty(T, D, **bf)
            ws[f"qkv_{l}"] = torch.empty(T, 3 * D, **bf)
            ws[f"ctx_{l}"] = torch.empty(T, D, **bf)
            ws[f"lse_{l}"] = torch.empty(B, Hh, L, **f32)
            ws[f"xmid_{l}"] = torch.empty(T, D, **f32)
            ws[f"h2_{l}"] = torch.empty(T, D, **bf)
            ws[f"f_{l}"] = torch.empty(T, FF, **bf)
            ws[f"xout_{l}"] = torch.empty(T, D, **f32)
        # last-layer single-row path (B rows instead of B*L)
        ws["zero_idx"] = torch.zeros(B, device=dev, dtype=torch.int32)
        ws["hq"] = torch.empty(B, D, **bf)
        ws["xq_in"] = torch.empty(B, D, **f32)
        ws["qq"] = torch.empty(B, D, **bf)
        ws["ctxq"] = torch.empty(B, D, **bf)
        ws["lseq"] = torch.empty(B, Hh, **f32)
        ws["xmid_q"] = torch.empty(B, D, **f32)
        ws["h2q"] = torch.empty(B, D, **bf)
        ws["fq"] = torch.empty(B, FF, **bf)
        ws["xout_q"] = torch.empty(B, D, **f32)
        ws["dxq"] = torch.empty(B, D, **f32)
        ws["dy_q"] = torch.empty(B, D, **bf)
        ws["dy_q1"] = torch.empty(B, D, **bf)
        ws["dpre_q"] = torch.empty(B, FF, **bf)
        ws["dh_q"] = torch.empty(B, D, **f32)
        ws["dxmid_q"] = torch.empty(B, D, **f32)
        ws["dctx_q"] = torch.empty(B, D, **bf)
        ws["dq_q"] = torch.empty(B, D, **bf)
        ws["dhq"] = torch.empty(B, D, **f32)
        ws["cat"] = torch.zeros(B + 1, D + 48, **bf)[:B]          # +1 row: ragged MN-major reads
        ws["z1"] = torch.empty(B, D, **f32)
        ws["a1"] = torch.empty(B, D, **bf)
        ws["u"] = torch.empty(B, D, **f32)
        ws["un"] = torch.empty(B, D, **f32)
        ws["un_bf"] = torch.empty(B, D, **bf)
        ws["xi"] = torch.empty(B, 4 * cfg.modality_dim, **bf)
        ws["y1"] = torch.empty(B, cfg.fusion_hidden, **f32)
        ws["bn_mean"] = torch.empty(cfg.fusion_hidden, **f32)
        ws["bn_rstd"] = torch.empty(cfg.fusion_hidden, **f32)
        ws["a"] = torch.empty(B, cfg.fusion_hidden, **bf)
        ws["y2"] = torch.empty(B, D, **f32)
        ws["in"] = torch.empty(B, D, **f32)
        ws["in_bf"] = torch.empty(B, D, **bf)
        # loss
        Bp = (B + 7) // 8 * 8                      # leading dimensions padded for 16-byte rows
        ws["S"] = torch.empty(B, Bp, **f32)[:, :B]
        ws["S2"] = torch.empty(B, Bp, **f32)[:, :B]
        for k in ("lse_r", "pos_r", "lse_c", "pos_c"):
            ws[k] = torch.empty(B, **f32)
        ws["loss"] = torch.zeros((), **f32)
        # backward
        ws["dS"] = torch.zeros(B, Bp, **bf)[:, :B]
        ws["dS2"] = torch.zeros(B, Bp, **bf)[:, :B]
        ws["dun"] = torch.empty(B, D, **f32)
        ws["din"] = torch.empty(B, D, **f32)
        ws["du_bf"] = torch.empty(B, D, **bf)
        ws["da1"] = torch.empty(B, D, **f32)
        ws["dz1_bf"] = torch.empty(B, D, **bf)
        ws["dcat"] = torch.empty(B, D + 48, **f32)
        ws["dy2i_bf"] = torch.empty(B, D, **bf)
        ws["da"] = torch.empty(B, cfg.fusion_hidden, **f32)
        ws["dy1i_bf"] = torch.empty(B, cfg.fusion_hidden, **bf)
        ws["dx_a"] = torch.empty(T, D, **f32)      # gradient of the residual stream (ping)
        ws["dx_b"] = torch.empty(T, D, **f32)      # (pong)
        # bf16 gradients fed to the dgrad/wgrad GEMMs: one buffer per use (the wgrad stream reads them
        # while the main stream moves on, so nothing is recycled inside one backward pass)
        for l in range(NL):
            ws[f"dy2_{l}"] = torch.empty(T, D, **bf)      # grad of linear2's output (dropout-masked)
            ws[f"dy1_{l}"] = torch.empty(T, D, **bf)      # grad of out_proj's output
            ws[f"dqkv_{l}"] = torch.empty(T, 3 * D, **bf)
            if l < NL - 1 or not self.prune_last_layer:
                ws[f"dpre_{l}"] = torch.empty(T, FF, **bf)
        ws["dh"] = torch.empty(T, D, **f32)        # grad w.r.t. a LayerNorm output
        ws["dh_bf"] = torch.empty(T, D, **bf)      # the same in bf16 (what a Linear's backward returns under autocast)
        ws["dctx"] = torch.empty(T, D, **bf)
        self._ws[key] = ws
        return ws

    def session_workspace(self, n: int) -> Dict[str, torch.Tensor]:
        """Buffers of a session append (`session_append`): n rows per layer, no (B, L) token buffers."""
        key = ("session", n)
        if key in self._ws:
            return self._ws[key]
        cfg, dev = self.cfg, self.device
        D, FF = cfg.embedding_dim, cfg.ff_dim
        f32 = dict(device=dev, dtype=torch.float32)
        bf = dict(device=dev, dtype=torch.bfloat16)
        ws: Dict[str, torch.Tensor] = {"x_in0": torch.empty(n, D, **f32), "zero_idx": torch.zeros(n, device=dev,
                                                                                                  dtype=torch.int32)}
        for l in range(cfg.num_layers):
            ws[f"h1_{l}"] = torch.empty(n, D, **bf)
            ws[f"qkv_{l}"] = torch.empty(n, 3 * D, **bf)
            ws[f"ctx_{l}"] = torch.empty(n, D, **bf)
            ws[f"xmid_{l}"] = torch.empty(n, D, **f32)
            ws[f"h2_{l}"] = torch.empty(n, D, **bf)
            ws[f"f_{l}"] = torch.empty(n, FF, **bf)
            ws[f"xout_{l}"] = torch.empty(n, D, **f32)
        ws["cat"] = torch.zeros(n + 1, D + 48, **bf)[:n]          # +1 row: ragged MN-major reads
        ws["z1"] = torch.empty(n, D, **f32)
        ws["a1"] = torch.empty(n, D, **bf)
        ws["u"] = torch.empty(n, D, **f32)
        ws["un"] = torch.empty(n, D, **f32)
        ws["un_bf"] = torch.empty(n, D, **bf)
        self._ws[key] = ws
        return ws

    def session_append(self, ws, item_ids, slots, pos, k_caches, v_caches, gender, country) -> torch.Tensor:
        """User tower for ONE new history item per row, from the K/V of the earlier positions (eval, no dropout).

        Row r appends ``item_ids[r]`` (int64) at position ``pos[r]`` (int32) of cache slot ``slots[r]`` (int32, distinct);
        ``k_caches[l]`` / ``v_caches[l]`` are layer l's planes, bf16 [capacity, 4, L, 64], holding that slot's K/V for
        positions < pos[r]. The new row's K/V are written into them. Returns ws['un'] fp32 [n, 256]: the normalised user
        embedding of the extended history (user_forward on the whole window gives the same)."""
        if self.table_rows is not None or self.peer_table is not None:
            raise NotImplementedError("user sessions need a local ID table (no row-sharded or peer table)")
        cfg, p, w = self.cfg, self.p, self.w
        ut = "user_tower."
        if not self.shadow_valid:
            self.refresh_shadow()
        ops.embed_ln_fwd_pos(item_ids, pos, p[ut + "item_embedding.weight"], p[ut + "position_embedding.weight"],
                             p[ut + "layer_norm.weight"], p[ut + "layer_norm.bias"], p[self._lp(0, "norm1.weight")],
                             p[self._lp(0, "norm1.bias")], ws["x_in0"], ws["h1_0"])
        x_in = ws["x_in0"]
        for l in range(cfg.num_layers):
            self._gemm(ws[f"h1_{l}"], w[self._lp(l, "self_attn.in_proj_weight")],
                       bias=p[self._lp(l, "self_attn.in_proj_bias")], out_bf16=ws[f"qkv_{l}"])
            ops.session_attn(ws[f"qkv_{l}"], k_caches[l], v_caches[l], slots, pos, ws[f"ctx_{l}"])
            self._layer_tail(l, ws[f"ctx_{l}"], x_in, ws[f"xmid_{l}"], ws[f"h2_{l}"], ws[f"f_{l}"], ws[f"xout_{l}"],
                             0.0, self.base_seed, None)
            x_in = ws[f"xout_{l}"]
            if l + 1 < cfg.num_layers:
                ops.chain_fwd(x_in, ln=(p[self._lp(l + 1, "norm1.weight")], p[self._lp(l + 1, "norm1.bias")]),
                              out_bf16=ws[f"h1_{l + 1}"])
        n = item_ids.shape[0]
        ops.gather_cat_fwd(x_in, ws["zero_idx"], gender, country, p[ut + "gender_embedding.weight"],
                           p[ut + "country_embedding.weight"], n, 1, ws["cat"])
        return self._user_head(ws)

    def _sparse_ws(self, T: int) -> Dict[str, torch.Tensor]:
        """Scratch of the id de-duplication for T tokens per step (direct-address flag / slot tables over the
        vocabulary, distinct-id list, per-token slots, compact row cache and gradient accumulator)."""
        if T not in self._sparse:
            dev, V, D = self.device, self.peer_table.vocab_size, self.cfg.embedding_dim
            self._sparse[T] = {
                "flag": torch.zeros(V, device=dev, dtype=torch.int32), "slot": torch.zeros(V, device=dev, dtype=torch.int32),
                "uniq": torch.zeros(T + 1, device=dev, dtype=torch.int64), "state": torch.zeros(2, device=dev, dtype=torch.int32),
                "inverse": torch.zeros(T, device=dev, dtype=torch.int64),
                "cache": torch.zeros(T + 1, D, device=dev), "gacc": torch.zeros(T + 1, D, device=dev)}
        return self._sparse[T]

    def _det_ws(self, T: int) -> Dict[str, torch.Tensor]:
        if T not in self._det:
            dev, V, D = self.device, self.cfg.vocab_size, self.cfg.embedding_dim
            self._det[T] = {
                "flag": torch.zeros(V, device=dev, dtype=torch.int32), "slot": torch.zeros(V, device=dev, dtype=torch.int32),
                "uniq": torch.zeros(T + 1, device=dev, dtype=torch.int64), "state": torch.zeros(2, device=dev, dtype=torch.int32),
                "inverse": torch.zeros(T, device=dev, dtype=torch.int64),
                "acc64": torch.zeros(T + 1, D, device=dev, dtype=torch.int64)}
        return self._det[T]

    def release_workspaces(self) -> None:
        """Drop every activation workspace (they are rebuilt on demand; CUDA graphs that captured them must be
        dropped by their owner first)."""
        self._ws.clear()

    def item_workspace(self, B: int) -> Dict[str, torch.Tensor]:
        """Buffers of the item tower alone (catalog indexing / get_item_embedding: no (B, L) user-tower workspace)."""
        key = ("item", B)
        if key in self._ws:
            return self._ws[key]
        cfg, dev = self.cfg, self.device
        D, H = cfg.embedding_dim, cfg.fusion_hidden
        f32 = dict(device=dev, dtype=torch.float32)
        bf = dict(device=dev, dtype=torch.bfloat16)
        ws = {"xi": torch.empty(B, 4 * cfg.modality_dim, **bf), "y1": torch.empty(B, H, **f32),
              "bn_mean": torch.empty(H, **f32), "bn_rstd": torch.empty(H, **f32), "a": torch.empty(B, H, **bf),
              "y2": torch.empty(B, D, **f32), "in": torch.empty(B, D, **f32), "in_bf": torch.empty(B, D, **bf)}
        self._ws[key] = ws
        return ws

    # ------------------------------------------------------------------ helpers
    def _gemm(self, A, B, **kw):
        """tt_gemm_bf16; with ``self.gemm_log`` set (a list), every launch is bracketed by CUDA events
        and logged as (event0, event1, algorithmic flops, algorithmic bytes) — bench.py's roofline measurement."""
        log = getattr(self, "gemm_log", None)
        if log is None:
            ops.gemm(A, B, **kw)
            return
        a_mn, b_mn = kw.get("a_mn", False), kw.get("b_mn", False)
        M = A.shape[1] if a_mn else A.shape[0]
        K = A.shape[0] if a_mn else A.shape[1]
        N = B.shape[1] if b_mn else B.shape[0]
        nbytes = 2.0 * (M * K + N * K)                      # bf16 operands
        if kw.get("out_bf16") is not None:
            nbytes += 2.0 * M * N
        if kw.get("out_f32") is not None:
            nbytes += (8.0 if kw.get("accumulate") else 4.0) * M * N
        if kw.get("residual") is not None:
            nbytes += 4.0 * M * N
        if kw.get("gate") is not None:
            nbytes += 2.0 * M * N
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.gemm(A, B, **kw)
        e1.record()
        log.append((e0, e1, 2.0 * M * N * K, nbytes, (M, N, K)))

    def _side_stream(self) -> torch.cuda.Stream:
        if self.serialize:
            return torch.cuda.current_stream()
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(device=self.device)
        return self._side

    def _wgrad_stream(self) -> torch.cuda.Stream:
        if self.serialize:
            return torch.cuda.current_stream()
        if getattr(self, "_wside", None) is None:
            self._wside = torch.cuda.Stream(device=self.device)
        return self._wside

    def _wg(self, fn, *a, **kw) -> None:
        """Issue a weight-gradient kernel (wgrad GEMM, bias column sum) on the wgrad stream, ordered after
        everything issued so far on the current stream. Nothing on the critical dgrad chain depends on
        these results before the optimizer, so they become parallel branches of the captured graph; the
        ~25 tiny B-row wgrads then overlap the dgrad chain instead of extending it. Every buffer they read
        is written once per backward (no reuse), so the only cross-stream hazard is the read-after-write
        edge this helper orders."""
        main = torch.cuda.current_stream()
        wst = self._wgrad_stream()
        wst.wait_stream(main)
        with torch.cuda.stream(wst):
            fn(*a, **kw)

    def _dgrad_bias(self, dy, W, gbias, **kw) -> None:
        """dX = dY W on the main chain together with the bias gradient sum(dY, dim=0) -> gbias (accumulated).
        The GEMM's two idle warps take the column sums from the dY tiles it stages anyway (``a_colsum``)."""
        self._gemm(dy, W, b_mn=True, a_colsum=gbias, **kw)

    def _lp(self, l: int, name: str) -> str:
        return f"user_tower.transformer_encoder.layers.{l}.{name}"

    def _drop(self, training: bool) -> float:
        return self.cfg.dropout if training else 0.0

    # ------------------------------------------------------------------ forward pieces
    def user_forward(self, ws, ids, mask, gender, country, training: bool) -> torch.Tensor:
        """SASRec user tower -> L2-normalised user embedding (fp32 [B,256])."""
        cfg, p, w = self.cfg, self.p, self.w
        B, L = ids.shape
        dp = self._drop(training)
        seed, sdev = self.base_seed, self.seed_dev
        ut = "user_tower."
        ops.last_index(ids, mask, ws["last_idx"])
        if self.peer_table is not None:
            # distinct ids of the step -> each distinct row crosses NVLink once into a compact (L2-resident) cache;
            # the embedding kernel then runs on the cache with the slot numbers as ids
            t, sp = self.peer_table, self._sparse_ws(B * L)
            ops.ids_dedup(ids.view(-1), t.vocab_size, sp["flag"], sp["slot"], sp["uniq"], sp["state"], sp["inverse"])
            ops.rows_gather(sp["uniq"], sp["state"], sp["cache"], team=t.arena.team, weight_offset=t.arena.offset("weight"))
            ops.embed_ln_fwd(sp["inverse"], sp["cache"], p[ut + "position_embedding.weight"],
                             p[ut + "layer_norm.weight"], p[ut + "layer_norm.bias"],
                             p[self._lp(0, "norm1.weight")], p[self._lp(0, "norm1.bias")], B, L,
                             ws["x_in0"], ws["h1_0"], drop_p=dp, seed=seed, seed_dev=sdev, site=SITE_EMB)
        else:
            e_ids, e_table, _ = self._embed_operands(ids)
            ops.embed_ln_fwd(e_ids, e_table, p[ut + "position_embedding.weight"],
                             p[ut + "layer_norm.weight"], p[ut + "layer_norm.bias"],
                             p[self._lp(0, "norm1.weight")], p[self._lp(0, "norm1.bias")], B, L,
                             ws["x_in0"], ws["h1_0"], drop_p=dp, seed=seed, seed_dev=sdev, site=SITE_EMB)
        x_in = ws["x_in0"]
        for l in range(cfg.num_layers):
            if self.prune_last_layer and l == cfg.num_layers - 1:
                self._last_layer_forward(ws, l, x_in, B, L, dp, seed, sdev)
                x_in = None
                break
            self._gemm(ws[f"h1_{l}"], w[self._lp(l, "self_attn.in_proj_weight")],
                       bias=p[self._lp(l, "self_attn.in_proj_bias")], out_bf16=ws[f"qkv_{l}"])
            ops.attn_fwd(ws[f"qkv_{l}"], ws[f"ctx_{l}"], ws[f"lse_{l}"], B, L, cfg.num_heads, drop_p=dp,
                         drop_seed=seed, drop_seed_dev=sdev, drop_site=_site(l, 0))
            self._layer_tail(l, ws[f"ctx_{l}"], x_in, ws[f"xmid_{l}"], ws[f"h2_{l}"], ws[f"f_{l}"], ws[f"xout_{l}"],
                             dp, seed, sdev)
            x_in = ws[f"xout_{l}"]
            if l + 1 < cfg.num_layers:
                ops.chain_fwd(x_in, ln=(p[self._lp(l + 1, "norm1.weight")], p[self._lp(l + 1, "norm1.bias")]),
                              out_bf16=ws[f"h1_{l + 1}"])
        if x_in is None:   # pruned last layer: its output exists for the gathered rows only
            ops.gather_cat_fwd(ws["xout_q"], ws["zero_idx"], gender, country, p[ut + "gender_embedding.weight"],
                               p[ut + "country_embedding.weight"], B, 1, ws["cat"])
        else:
            ops.gather_cat_fwd(x_in, ws["last_idx"], gender, country, p[ut + "gender_embedding.weight"],
                               p[ut + "country_embedding.weight"], B, L, ws["cat"])
        return self._user_head(ws)

    def _user_head(self, ws) -> torch.Tensor:
        """Fusion MLP on ws['cat'] (last encoder row | gender | country) -> L2-normalised user embedding ws['un']."""
        p, w = self.p, self.w
        ut = "user_tower."
        self._gemm(ws["cat"], w[ut + "fusion_layer.0.weight"], bias=p[ut + "fusion_layer.0.bias"], out_f32=ws["z1"])
        ops.chain_fwd(ws["z1"], ln=(p[ut + "fusion_layer.1.weight"], p[ut + "fusion_layer.1.bias"]), relu=True,
                      out_bf16=ws["a1"])
        self._gemm(ws["a1"], w[ut + "fusion_layer.3.weight"], bias=p[ut + "fusion_layer.3.bias"], out_f32=ws["u"])
        ops.chain_fwd(ws["u"], l2norm=True, out_f32=ws["un"], out_bf16=ws["un_bf"])
        return ws["un"]

    def _layer_tail(self, l, ctx, x_in, xmid, h2, f, xout, dp, seed, sdev) -> None:
        """Encoder layer l after the attention, on whichever rows ``ctx`` holds: out_proj + residual x_in -> xmid,
        norm2 -> h2, linear1 + ReLU -> f, linear2 + residual -> xout."""
        p, w = self.p, self.w
        self._gemm(ctx, w[self._lp(l, "self_attn.out_proj.weight")], bias=p[self._lp(l, "self_attn.out_proj.bias")],
                   drop_p=dp, drop_seed=seed, drop_seed_dev=sdev, drop_site=_site(l, 1), residual=x_in, out_f32=xmid)
        ops.chain_fwd(xmid, ln=(p[self._lp(l, "norm2.weight")], p[self._lp(l, "norm2.bias")]), out_bf16=h2)
        self._gemm(h2, w[self._lp(l, "linear1.weight")], bias=p[self._lp(l, "linear1.bias")], relu=True,
                   drop_p=dp, drop_seed=seed, drop_seed_dev=sdev, drop_site=_site(l, 2), out_bf16=f)
        self._gemm(f, w[self._lp(l, "linear2.weight")], bias=p[self._lp(l, "linear2.bias")], drop_p=dp,
                   drop_seed=seed, drop_seed_dev=sdev, drop_site=_site(l, 3), residual=xmid, out_f32=xout)

    def _last_layer_forward(self, ws, l, x_in, B, L, dp, seed, sdev) -> None:
        """Last encoder layer, exact single-row form: K/V for every position, everything downstream of
        the attention for the row len-1 of each sequence only."""
        cfg, p, w = self.cfg, self.p, self.w
        D = cfg.embedding_dim
        Wqkv, bqkv = w[self._lp(l, "self_attn.in_proj_weight")], p[self._lp(l, "self_attn.in_proj_bias")]
        self._gemm(ws[f"h1_{l}"], Wqkv[D:], bias=bqkv[D:], out_bf16=ws[f"qkv_{l}"][:, D:])          # K | V
        ops.gather_rows(ws["last_idx"], B, L, x_f32=x_in, out_f32=ws["xq_in"], x_bf16=ws[f"h1_{l}"], out_bf16=ws["hq"])
        self._gemm(ws["hq"], Wqkv[:D], bias=bqkv[:D], out_bf16=ws["qq"])                          # Q, B rows
        ops.attn_lastq_fwd(ws["qq"], ws[f"qkv_{l}"], ws["last_idx"], ws["ctxq"], ws["lseq"], B, L, cfg.num_heads,
                           drop_p=dp, seed=seed, seed_dev=sdev, site=_site(l, 0))
        self._layer_tail(l, ws["ctxq"], ws["xq_in"], ws["xmid_q"], ws["h2q"], ws["fq"], ws["xout_q"], dp, seed, sdev)

    def _last_layer_backward(self, ws, l, x_in, B, L, dp, seed, sdev, dx, dx_other):
        """Backward of _last_layer_forward. ws['dxq'] holds d(loss)/d(xout_q) (B rows). Returns the
        (dx, dx_other) ping-pong with dx = gradient w.r.t. the layer input (all positions)."""
        cfg, p, w, g = self.cfg, self.p, self.w, self.g
        D = cfg.embedding_dim
        gemm = self._gemm
        ffn_scale = 1.0 / (1.0 - dp) if dp > 0 else 1.0
        Wqkv = w[self._lp(l, "self_attn.in_proj_weight")]
        gW, gb = g[self._lp(l, "self_attn.in_proj_weight")], g[self._lp(l, "self_attn.in_proj_bias")]
        # --- FFN and out_proj on the B gathered rows (weight gradients go to the wgrad stream)
        wg = self._wg
        ops.chain_bwd(ws["dxq"], dout=ws["dxq"], dx_bf16=ws["dy_q"], drop2_p=dp, drop2_site=_site(l, 3), seed=seed,
                      seed_dev=sdev, dx_colsum=g[self._lp(l, "linear2.bias")])
        wg(gemm, ws["dy_q"], ws["fq"], a_mn=True, b_mn=True, out_f32=g[self._lp(l, "linear2.weight")], accumulate=True)
        gemm(ws["dy_q"], w[self._lp(l, "linear2.weight")], b_mn=True, gate=ws["fq"], gate_scale=ffn_scale,
             out_bf16=ws["dpre_q"])
        wg(gemm, ws["dpre_q"], ws["h2q"], a_mn=True, b_mn=True, out_f32=g[self._lp(l, "linear1.weight")], accumulate=True)
        self._dgrad_bias(ws["dpre_q"], w[self._lp(l, "linear1.weight")], g[self._lp(l, "linear1.bias")], out_f32=ws["dh_q"])
        ops.chain_bwd(ws["xmid_q"], ln=(p[self._lp(l, "norm2.weight")], p[self._lp(l, "norm2.bias")]), dout=ws["dh_q"],
                      resid=ws["dxq"], dx_f32=ws["dxmid_q"], dx_bf16=ws["dy_q1"], drop2_p=dp, drop2_site=_site(l, 1),
                      seed=seed, seed_dev=sdev, dgamma=g[self._lp(l, "norm2.weight")],
                      dbeta=g[self._lp(l, "norm2.bias")], dx_colsum=g[self._lp(l, "self_attn.out_proj.bias")])
        wg(gemm, ws["dy_q1"], ws["ctxq"], a_mn=True, b_mn=True, out_f32=g[self._lp(l, "self_attn.out_proj.weight")],
           accumulate=True)
        gemm(ws["dy_q1"], w[self._lp(l, "self_attn.out_proj.weight")], b_mn=True, out_bf16=ws["dctx_q"])
        # --- single-query attention backward: dq (B rows), dK/dV for every position
        dqkv = ws[f"dqkv_{l}"]
        ops.attn_lastq_bwd(ws["qq"], ws[f"qkv_{l}"], ws["last_idx"], ws["ctxq"], ws["dctx_q"], ws["lseq"], ws["dq_q"],
                           dqkv, B, L, cfg.num_heads, drop_p=dp, seed=seed, seed_dev=sdev, site=_site(l, 0))
        wg(gemm, ws["dq_q"], ws["hq"], a_mn=True, b_mn=True, out_f32=gW[:D], accumulate=True)
        self._dgrad_bias(ws["dq_q"], Wqkv[:D], gb[:D], out_f32=ws["dhq"])
        dkv = dqkv[:, D:]
        wg(gemm, dkv, ws[f"h1_{l}"], a_mn=True, b_mn=True, out_f32=gW[D:], accumulate=True)
        self._dgrad_bias(dkv, Wqkv[D:], gb[D:], out_f32=ws["dh"])
        ops.scatter_rows_add(ws["dhq"], ws["last_idx"], B, L, ws["dh"], accumulate=True)
        # --- residual gradient of the layer input: only the gathered rows carry one
        # the residual-stream gradient into this layer's input is non-zero for ONE row per sequence
        # (dxmid_q): chain_bwd adds it to that row instead of reading a zero-filled [T, 256] tensor
        extra = {}
        if l > 0:
            extra = dict(dx_bf16=ws[f"dy2_{l - 1}"], drop2_p=dp, drop2_site=_site(l - 1, 3),
                         dx_colsum=g[self._lp(l - 1, "linear2.bias")])
        ops.chain_bwd(x_in, ln=(p[self._lp(l, "norm1.weight")], p[self._lp(l, "norm1.bias")]), dout=ws["dh"],
                      resid_rows=ws["dxmid_q"], resid_last_idx=ws["last_idx"], resid_seq_len=L, dx_f32=dx_other,
                      seed=seed, seed_dev=sdev, dgamma=g[self._lp(l, "norm1.weight")],
                      dbeta=g[self._lp(l, "norm1.bias")], **extra)
        return dx_other, dx

    def item_forward(self, ws, audio, visual, text, tabular, training: bool) -> torch.Tensor:
        """Late-fusion item tower on precomputed modality embeddings -> normalised item embedding."""
        p, w = self.p, self.w
        it = "item_tower.fusion_layer."
        ops.concat4_bf16(audio, visual, text, tabular, ws["xi"])
        self._gemm(ws["xi"], w[it + "0.weight"], bias=p[it + "0.bias"], out_f32=ws["y1"])
        ops.bn_relu_fwd(ws["y1"], p[it + "1.weight"], p[it + "1.bias"], self.bn_running_mean, self.bn_running_var,
                        self.bn_num_batches, training=training, drop_p=(0.1 if training and self.cfg.dropout > 0 else 0.0),
                        seed=self.base_seed, seed_dev=self.seed_dev, site=SITE_ITEM, save_mean=ws["bn_mean"],
                        save_rstd=ws["bn_rstd"], out_bf16=ws["a"])
        self._gemm(ws["a"], w[it + "4.weight"], bias=p[it + "4.bias"], out_f32=ws["y2"])
        ops.chain_fwd(ws["y2"], ln=(p[it + "5.weight"], p[it + "5.bias"]), l2norm=True, out_f32=ws["in"],
                      out_bf16=ws["in_bf"])
        return ws["in"]

    def index_items(self, features: Dict[str, torch.Tensor], item_ids: torch.Tensor, table: torch.Tensor,
                    table_bf16: Optional[torch.Tensor] = None, batch_size: int = 131072) -> None:
        """Catalog indexing (src/evaluate_metrics.py:24-104) on device tensors: item tower in eval mode over
        ``features`` (four (n, 128) fp32 device tensors), NaN -> 0, re-normalise (eps 1e-8), rows scattered by
        ``item_ids`` into ``table`` fp32 (V, 256) (+ its bf16 copy). Eval-mode BatchNorm is an affine map per
        column, so it is folded into the first Linear once per call (W' = diag(gamma * rstd) W, b' = (b - mean)
        * gamma * rstd + beta): GEMM -> bias+ReLU epilogue -> bf16 replaces GEMM -> fp32 -> BatchNorm kernel, and
        an item costs 9.5 KB of HBM traffic against the 3 KB (2 KB of features in, 1 KB of embedding out) it must."""
        p = self.p
        it = "item_tower.fusion_layer."
        n = item_ids.shape[0]
        scale = p[it + "1.weight"] * torch.rsqrt(self.bn_running_var + 1e-5)
        w_fold = (p[it + "0.weight"] * scale[:, None]).to(torch.bfloat16).contiguous()
        b_fold = ((p[it + "0.bias"] - self.bn_running_mean) * scale + p[it + "1.bias"]).contiguous()
        if not self.shadow_valid:
            self.refresh_shadow()
        ws = self.item_workspace(min(batch_size, n))
        f = [features[k] for k in ("target_audio", "target_image", "target_input_ids", "target_tabular")]
        for s0 in range(0, n, batch_size):
            r = min(batch_size, n - s0)
            ops.concat4_bf16(f[0][s0:s0 + r], f[1][s0:s0 + r], f[2][s0:s0 + r], f[3][s0:s0 + r], ws["xi"][:r])
            self._gemm(ws["xi"][:r], w_fold, bias=b_fold, relu=True, out_bf16=ws["a"][:r])
            self._gemm(ws["a"][:r], self.w[it + "4.weight"], bias=p[it + "4.bias"], out_f32=ws["y2"][:r])
            ops.index_rows(ws["y2"][:r], p[it + "5.weight"], p[it + "5.bias"], item_ids[s0:s0 + r], table, table_bf16)

    # -- InfoNCE, written for data parallelism with all-gathered negatives --------------------
    # Rank r holds B local users/items and the G*B gathered ones; its positives sit at column
    # r*B + i. S = U_loc I_all^T / tau and S2 = I_loc U_all^T / tau are ROW problems; the column
    # log-sum-exps needed by the gradient are the other matrix's row log-sum-exps on the owning
    # ranks (two small all-gathers, no reduce-scatter). With one rank everything is local.
    def gathered_workspace(self, ws, G: int) -> Dict[str, torch.Tensor]:
        B, D = ws["un"].shape
        key = f"_gath{G}"
        if key not in ws:
            dev = self.device
            ws[key] = {
                "U_all": torch.empty(G * B, D, device=dev, dtype=torch.bfloat16),
                "I_all": torch.empty(G * B, D, device=dev, dtype=torch.bfloat16),
                "uid_all": torch.zeros(G * B, device=dev, dtype=torch.long),
                "S": torch.empty(B, (G * B + 7) // 8 * 8, device=dev)[:, :G * B],
                "S2": torch.empty(B, (G * B + 7) // 8 * 8, device=dev)[:, :G * B],
                "dS": torch.zeros(B, (G * B + 7) // 8 * 8, device=dev, dtype=torch.bfloat16)[:, :G * B],
                "dS2": torch.zeros(B, (G * B + 7) // 8 * 8, device=dev, dtype=torch.bfloat16)[:, :G * B],
                "lse_r_all": torch.empty(G * B, device=dev), "lse_c_all": torch.empty(G * B, device=dev),
            }
        return ws[key]

    def loss_forward(self, ws, user_idx: Optional[torch.Tensor], gathered: Optional[Dict[str, torch.Tensor]] = None,
                     rank: int = 0, offsets: Optional[Tuple[torch.Tensor, torch.Tensor]] = None) -> torch.Tensor:
        """Logits + masked row log-sum-exps (+ the local loss when not gathered). With `gathered`
        (U_all, I_all, uid_all filled by the caller's all-gather) the caller must all-gather
        ws['lse_r'] / ws['lse_c'] into gathered['lse_r_all' / 'lse_c_all'] and then call loss_value().
        ``offsets`` = (oi, ou), fp32 over the (global) batch rows: log q of each row's item / user (logQ correction,
        train.LogQCorrection). The row log-sum-exps, positives and backward() then use x_ij - oi[j] (user rows) and
        x_ij - ou[j] (item rows); the logits in ws / gathered stay the uncorrected masked ones."""
        B = ws["un"].shape[0]
        inv_t = 1.0 / self.cfg.temperature
        self._gathered = None if gathered is None else (gathered, rank)
        self._offsets = offsets
        if gathered is None:
            S, S2, U_all, I_all, uid_all, pos0 = ws["S"], ws["S2"], ws["un_bf"], ws["in_bf"], user_idx, 0
        else:
            S, S2, U_all, I_all, pos0 = gathered["S"], gathered["S2"], gathered["U_all"], gathered["I_all"], rank * B
            uid_all = gathered["uid_all"] if user_idx is not None else None
        self._gemm(ws["un_bf"], I_all, alpha=inv_t, out_f32=S)
        self._gemm(ws["in_bf"], U_all, alpha=inv_t, out_f32=S2)
        if offsets is None:
            ops.infonce_rows(S, user_idx, uid_all, pos0, ws["lse_r"], ws["pos_r"])
            ops.infonce_rows(S2, user_idx, uid_all, pos0, ws["lse_c"], ws["pos_c"])
        else:
            ops.infonce_rows_off(S, user_idx, uid_all, pos0, offsets[0], ws["lse_r"], ws["pos_r"])
            ops.infonce_rows_off(S2, user_idx, uid_all, pos0, offsets[1], ws["lse_c"], ws["pos_c"])
        if gathered is None:
            self.loss_value(ws, B)
        return ws["loss"]

    def loss_value(self, ws, global_batch: int) -> torch.Tensor:
        """loss contribution of the local rows: 0.5/global_batch * sum_i (lse - positive) over both directions
        (sum over ranks = the global symmetric InfoNCE)."""
        ops.infonce_loss(ws["lse_r"], ws["pos_r"], ws["lse_c"], ws["pos_c"], 0.5 / global_batch, ws["loss"])
        return ws["loss"]

    def forward_towers(self, batch: Dict[str, torch.Tensor], training: bool = True):
        ids = batch["history_ids"]
        B, L = ids.shape
        if B % 4 != 0:
            raise ValueError(f"batch size {B}: the InfoNCE logit tiles need a multiple of 4 (16-byte fp32 rows)")
        ws = self.workspace(B, L)
        if not self.shadow_valid:
            self.refresh_shadow()
        # The item tower (a handful of tiny kernels) is independent of the user tower: it runs on a
        # side stream (a parallel branch of the captured graph) and fills the tails of the big kernels.
        main = torch.cuda.current_stream()
        side = self._side_stream()
        side.wait_stream(main)
        with torch.cuda.stream(side):
            self.item_forward(ws, batch["target_audio"], batch["target_image"], batch["target_input_ids"],
                              batch["target_tabular"], training)
        self.user_forward(ws, ids, batch.get("history_mask"), batch["user_gender"], batch["user_country"], training)
        main.wait_stream(side)
        self._last = (ws, batch, training)
        self._gathered = None
        self._offsets = None
        return ws

    def forward(self, batch: Dict[str, torch.Tensor], training: bool = True):
        """TwoTowerModel.forward (src/models/two_tower.py:68-142) ->
        (loss, logits, user_emb, item_emb); tensors are workspace views valid until the next call."""
        ws = self.forward_towers(batch, training)
        self.loss_forward(ws, batch.get("user_idx"))
        return ws["loss"], ws["S"], ws["un"], ws["in"]

    # ------------------------------------------------------------------ backward
    def _item_backward(self, ws, training, seed, sdev) -> None:
        cfg, p, w, g = self.cfg, self.p, self.w, self.g
        it = "item_tower.fusion_layer."
        gemm = self._gemm
        ops.chain_bwd(ws["y2"], ln=(p[it + "5.weight"], p[it + "5.bias"]), l2norm=True, dout=ws["din"],
                      dx_bf16=ws["dy2i_bf"], dgamma=g[it + "5.weight"], dbeta=g[it + "5.bias"],
                      dx_colsum=g[it + "4.bias"])
        gemm(ws["dy2i_bf"], ws["a"], a_mn=True, b_mn=True, out_f32=g[it + "4.weight"], accumulate=True)
        gemm(ws["dy2i_bf"], w[it + "4.weight"], b_mn=True, out_f32=ws["da"])
        ops.bn_relu_bwd(ws["y1"], p[it + "1.weight"], p[it + "1.bias"], self.bn_running_mean, self.bn_running_var,
                        None, training=training, drop_p=(0.1 if training and cfg.dropout > 0 else 0.0),
                        seed=seed, seed_dev=sdev, site=SITE_ITEM, save_mean=ws["bn_mean"], save_rstd=ws["bn_rstd"],
                        dout=ws["da"], dy_bf16=ws["dy1i_bf"], dgamma=g[it + "1.weight"], dbeta=g[it + "1.bias"],
                        dy_colsum=g[it + "0.bias"])
        gemm(ws["dy1i_bf"], ws["xi"], a_mn=True, b_mn=True, out_f32=g[it + "0.weight"], accumulate=True)


    def backward(self, loss_scale: float = 1.0) -> None:
        """Accumulates d(loss_scale * loss)/d(param) into self.grad (self.g views)."""
        ws, batch, training = self._last
        cfg, p, w, g = self.cfg, self.p, self.w, self.g
        ids = batch["history_ids"]
        B, L = ids.shape
        T, D = B * L, cfg.embedding_dim
        dp = self._drop(training)
        seed, sdev = self.base_seed, self.seed_dev
        inv_t = 1.0 / cfg.temperature
        ut, it = "user_tower.", "item_tower.fusion_layer."
        gemm = self._gemm

        # ---- InfoNCE -> d(normalised embeddings)
        gath = getattr(self, "_gathered", None)
        off = getattr(self, "_offsets", None)
        if gath is None:
            coef = 0.5 / B * loss_scale
            if off is None:
                ops.infonce_grad(ws["S"], ws["lse_r"], ws["lse_c"], 0, coef, ws["dS"])
                ops.infonce_grad(ws["S2"], ws["lse_c"], ws["lse_r"], 0, coef, ws["dS2"])
            else:
                ops.infonce_grad_off(ws["S"], ws["lse_r"], ws["lse_c"], 0, coef, off[0], off[1], ws["dS"])
                ops.infonce_grad_off(ws["S2"], ws["lse_c"], ws["lse_r"], 0, coef, off[1], off[0], ws["dS2"])
            gemm(ws["dS"], ws["in_bf"], b_mn=True, alpha=inv_t, out_f32=ws["dun"])
            gemm(ws["dS2"], ws["un_bf"], b_mn=True, alpha=inv_t, out_f32=ws["din"])
        else:
            g_, rank = gath
            coef = 0.5 / B * loss_scale     # per-rank normalisation; the gradient all-reduce AVERAGES
            if off is None:
                ops.infonce_grad(g_["S"], ws["lse_r"], g_["lse_c_all"], rank * B, coef, g_["dS"])
                ops.infonce_grad(g_["S2"], ws["lse_c"], g_["lse_r_all"], rank * B, coef, g_["dS2"])
            else:
                ops.infonce_grad_off(g_["S"], ws["lse_r"], g_["lse_c_all"], rank * B, coef, off[0], off[1], g_["dS"])
                ops.infonce_grad_off(g_["S2"], ws["lse_c"], g_["lse_r_all"], rank * B, coef, off[1], off[0],
                                     g_["dS2"])
            gemm(g_["dS"], g_["I_all"], b_mn=True, alpha=inv_t, out_f32=ws["dun"])
            gemm(g_["dS2"], g_["U_all"], b_mn=True, alpha=inv_t, out_f32=ws["din"])

        # ---- item tower (side stream: independent of the user tower's backward)
        main = torch.cuda.current_stream()
        side = self._side_stream()
        side.wait_stream(main)
        with torch.cuda.stream(side):
            self._item_backward(ws, training, seed, sdev)

        # ---- user head
        ops.chain_bwd(ws["u"], l2norm=True, dout=ws["dun"], dx_bf16=ws["du_bf"],
                      dx_colsum=g[ut + "fusion_layer.3.bias"])
        wg = self._wg
        wg(gemm, ws["du_bf"], ws["a1"], a_mn=True, b_mn=True, out_f32=g[ut + "fusion_layer.3.weight"], accumulate=True)
        gemm(ws["du_bf"], w[ut + "fusion_layer.3.weight"], b_mn=True, out_f32=ws["da1"])
        ops.chain_bwd(ws["z1"], ln=(p[ut + "fusion_layer.1.weight"], p[ut + "fusion_layer.1.bias"]), relu=True,
                      dout=ws["da1"], dx_bf16=ws["dz1_bf"], dgamma=g[ut + "fusion_layer.1.weight"],
                      dbeta=g[ut + "fusion_layer.1.bias"], dx_colsum=g[ut + "fusion_layer.0.bias"])
        wg(gemm, ws["dz1_bf"], ws["cat"], a_mn=True, b_mn=True, out_f32=g[ut + "fusion_layer.0.weight"], accumulate=True)
        gemm(ws["dz1_bf"], w[ut + "fusion_layer.0.weight"], b_mn=True, out_f32=ws["dcat"])
        dx, dx_other = ws["dx_a"], ws["dx_b"]
        top = cfg.num_layers - 1
        if self.prune_last_layer:
            # d(loss)/d(xout_q): one row per sequence; the pruned last layer takes it from there
            ops.gather_cat_bwd(ws["dcat"], ws["zero_idx"], batch["user_gender"], batch["user_country"], B, 1, ws["dxq"],
                               None, g[ut + "gender_embedding.weight"], g[ut + "country_embedding.weight"])
        else:
            dx.zero_()
            ops.gather_cat_bwd(ws["dcat"], ws["last_idx"], batch["user_gender"], batch["user_country"], B, L, dx, None,
                               g[ut + "gender_embedding.weight"], g[ut + "country_embedding.weight"])
            # dy = dropout-mask(dx) as bf16 for the top layer's linear2, with its column sums (bias grad)
            ops.chain_bwd(dx, dout=dx, dx_bf16=ws[f"dy2_{top}"], drop2_p=dp, drop2_site=_site(top, 3), seed=seed,
                          seed_dev=sdev, dx_colsum=g[self._lp(top, "linear2.bias")])

        # ---- encoder layers, last to first
        for l in range(cfg.num_layers - 1, -1, -1):
            x_in = ws[f"xout_{l - 1}"] if l > 0 else ws["x_in0"]
            if self.prune_last_layer and l == top:
                dx, dx_other = self._last_layer_backward(ws, l, x_in, B, L, dp, seed, sdev, dx, dx_other)
                continue
            ffn_scale = 1.0 / (1.0 - dp) if dp > 0 else 1.0
            # linear2: dW2 = dy^T f ; dpre = (dy W2) gated by f (ReLU and FFN dropout in one test)
            if f"dpre_{l}" not in ws:      # prune_last_layer toggled after the workspace was built
                ws[f"dpre_{l}"] = torch.empty(B * L, cfg.ff_dim, dtype=torch.bfloat16, device=self.device)
            dy2, dy1, dpre, dqkv = ws[f"dy2_{l}"], ws[f"dy1_{l}"], ws[f"dpre_{l}"], ws[f"dqkv_{l}"]
            wg(gemm, dy2, ws[f"f_{l}"], a_mn=True, b_mn=True, out_f32=g[self._lp(l, "linear2.weight")], accumulate=True)
            gemm(dy2, w[self._lp(l, "linear2.weight")], b_mn=True, gate=ws[f"f_{l}"], gate_scale=ffn_scale,
                 out_bf16=dpre)
            wg(gemm, dpre, ws[f"h2_{l}"], a_mn=True, b_mn=True, out_f32=g[self._lp(l, "linear1.weight")],
               accumulate=True)
            # the gradient a Linear hands back to the LayerNorm in front of it is bf16 like the reference's autocast
            # backward (half the bytes between the dgrad GEMM and the LayerNorm backward)
            self._dgrad_bias(dpre, w[self._lp(l, "linear1.weight")], g[self._lp(l, "linear1.bias")],
                             out_bf16=ws["dh_bf"])
            # norm2 backward (+ residual); emits dy for out_proj (dropout-1 mask) and its bias grad
            ops.chain_bwd(ws[f"xmid_{l}"], ln=(p[self._lp(l, "norm2.weight")], p[self._lp(l, "norm2.bias")]),
                          resid=dx, dx_f32=dx_other, dx_bf16=dy1, drop2_p=dp, dout_bf16=ws["dh_bf"],
                          drop2_site=_site(l, 1), seed=seed, seed_dev=sdev,
                          dgamma=g[self._lp(l, "norm2.weight")], dbeta=g[self._lp(l, "norm2.bias")],
                          dx_colsum=g[self._lp(l, "self_attn.out_proj.bias")])
            dx, dx_other = dx_other, dx
            wg(gemm, dy1, ws[f"ctx_{l}"], a_mn=True, b_mn=True, out_f32=g[self._lp(l, "self_attn.out_proj.weight")],
               accumulate=True)
            gemm(dy1, w[self._lp(l, "self_attn.out_proj.weight")], b_mn=True, out_bf16=ws["dctx"])
            ops.attn_bwd(ws[f"qkv_{l}"], ws[f"ctx_{l}"], ws["dctx"], ws[f"lse_{l}"], dqkv, B, L, cfg.num_heads,
                         drop_p=dp, drop_seed=seed, drop_seed_dev=sdev, drop_site=_site(l, 0))
            wg(gemm, dqkv, ws[f"h1_{l}"], a_mn=True, b_mn=True, out_f32=g[self._lp(l, "self_attn.in_proj_weight")],
               accumulate=True)
            self._dgrad_bias(dqkv, w[self._lp(l, "self_attn.in_proj_weight")], g[self._lp(l, "self_attn.in_proj_bias")],
                             out_bf16=ws["dh_bf"])
            # norm1 backward (+ residual); for l > 0 also dy for the previous layer's linear2
            extra = {}
            if l > 0:
                extra = dict(dx_bf16=ws[f"dy2_{l - 1}"], drop2_p=dp, drop2_site=_site(l - 1, 3),
                             dx_colsum=g[self._lp(l - 1, "linear2.bias")])
            ops.chain_bwd(x_in, ln=(p[self._lp(l, "norm1.weight")], p[self._lp(l, "norm1.bias")]),
                          dout_bf16=ws["dh_bf"], resid=dx, dx_f32=dx_other, seed=seed, seed_dev=sdev,
                          dgamma=g[self._lp(l, "norm1.weight")], dbeta=g[self._lp(l, "norm1.bias")], **extra)
            dx, dx_other = dx_other, dx

        # ---- embedding LayerNorm + lookup
        if self.peer_table is not None:
            # per-token gradient rows are combined in the compact local buffer (atomics on L2-resident memory), then
            # ONE remote reduction per distinct row goes to its owner
            t, sp = self.peer_table, self._sparse_ws(B * L)
            ops.embed_ln_bwd(sp["inverse"], sp["cache"], p[ut + "position_embedding.weight"],
                             p[ut + "layer_norm.weight"], p[ut + "layer_norm.bias"], dx, B, L,
                             sp["gacc"], g[ut + "position_embedding.weight"],
                             g[ut + "layer_norm.weight"], g[ut + "layer_norm.bias"], drop_p=dp, seed=seed,
                             seed_dev=sdev, site=SITE_EMB)
            ops.rows_scatter_add(sp["uniq"], sp["state"], sp["gacc"], team=t.arena.team, grad_offset=t.arena.offset("grad"))
        elif self.deterministic_table_grad and self.table_rows is None:
            dw = self._det_ws(T)
            ops.ids_dedup(ids.view(-1), cfg.vocab_size, dw["flag"], dw["slot"], dw["uniq"], dw["state"], dw["inverse"])
            ops.embed_ln_bwd_det(ids.view(-1), p[ut + "item_embedding.weight"], p[ut + "position_embedding.weight"],
                                 p[ut + "layer_norm.weight"], p[ut + "layer_norm.bias"], dx, B, L, dw["inverse"],
                                 dw["acc64"], g[ut + "position_embedding.weight"], g[ut + "layer_norm.weight"],
                                 g[ut + "layer_norm.bias"], drop_p=dp, seed=seed, seed_dev=sdev, site=SITE_EMB)
            ops.rows_scatter_add_i64(dw["uniq"], dw["state"], dw["acc64"], g[ut + "item_embedding.weight"])
        else:
            e_ids, e_table, e_grad = self._embed_operands(ids)
            ops.embed_ln_bwd(e_ids, e_table, p[ut + "position_embedding.weight"],
                             p[ut + "layer_norm.weight"], p[ut + "layer_norm.bias"], dx, B, L,
                             e_grad, g[ut + "position_embedding.weight"],
                             g[ut + "layer_norm.weight"], g[ut + "layer_norm.bias"], drop_p=dp, seed=seed,
                             seed_dev=sdev, site=SITE_EMB)
        main.wait_stream(side)
        main.wait_stream(self._wgrad_stream())

    # ------------------------------------------------------------------ optimizer
    def adamw_step(self, lr: float = 1e-4, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01,
                   zero_grad: bool = True) -> None:
        """torch.optim.AdamW semantics over the whole flat buffer (src/train.py:302, 64-65), dense
        on the ID table like the reference; refreshes the bf16 shadow of the dense region and
        zeroes the gradient buffer in the same pass; advances the step / dropout-seed counters."""
        if self.exp_avg is None or self.exp_avg.numel() != self.numel:
            self.exp_avg = torch.zeros_like(self.flat)
            self.exp_avg_sq = torch.zeros_like(self.flat)
        ops.step_counters_advance(self.step_dev, self.seed_dev)
        ops.adamw_step(self.flat, self.grad, self.exp_avg, self.exp_avg_sq, self.step_dev, lr, betas[0], betas[1],
                       eps, weight_decay, shadow=self.shadow, shadow_begin=self.dense_begin, shadow_end=self.numel,
                       zero_grad=zero_grad)
        self.shadow_valid = True
        self.weights_epoch += 1

    def adamw_step_sharded(self, rank: int, world: int, grad_shard: torch.Tensor, lr: float = 1e-4,
                           betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01) -> torch.Tensor:
        """Optimizer-state sharding for data parallelism: this rank owns elements
        [rank*n/world, (rank+1)*n/world) of the flat buffer, holds AdamW moments for them only and
        updates them from the reduce-scattered, averaged gradient `grad_shard`. The caller all-gathers
        the parameter shards afterwards and refreshes the bf16 shadow. Returns the parameter shard view."""
        assert self.numel % world == 0, \
            f"flat buffer of {self.numel} elements does not split into {world} equal optimizer shards"
        n = self.numel // world
        lo = rank * n
        if self.exp_avg is None or self.exp_avg.numel() != n:
            self.exp_avg = torch.zeros(n, device=self.device)
            self.exp_avg_sq = torch.zeros(n, device=self.device)
        ops.step_counters_advance(self.step_dev, self.seed_dev)
        p_shard = self.flat[lo:lo + n]
        ops.adamw_step(p_shard, grad_shard, self.exp_avg, self.exp_avg_sq, self.step_dev, lr, betas[0], betas[1],
                       eps, weight_decay, shadow=None, zero_grad=False)
        self.shadow_valid = False
        self.weights_epoch += 1
        return p_shard

    def train_step(self, batch: Dict[str, torch.Tensor], lr: float = 1e-4) -> torch.Tensor:
        """One step of the train_one_epoch body (src/train.py:54-65): forward, backward, AdamW."""
        loss, _, _, _ = self.forward(batch, training=True)
        self.backward()
        self.adamw_step(lr=lr)
        return loss
