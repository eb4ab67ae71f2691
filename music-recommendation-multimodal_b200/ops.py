"""Thin tensor-level wrappers over the C ABI (pointer + size marshalling only)."""
from __future__ import annotations

import ctypes
from typing import Optional

import torch

from ._lib import GemmArgs, check, lib


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise ValueError("tt ops take CUDA tensors only (no CPU fallback)")


def gemm(A: torch.Tensor, B: torch.Tensor, *, a_mn: bool = False, b_mn: bool = False,
         alpha: float = 1.0, bias: Optional[torch.Tensor] = None, relu: bool = False,
         drop_p: float = 0.0, drop_seed: int = 0, drop_site: int = 0,
         drop_seed_dev: Optional[torch.Tensor] = None, gate: Optional[torch.Tensor] = None, gate_scale: float = 1.0,
         residual: Optional[torch.Tensor] = None,
         out_f32: Optional[torch.Tensor] = None, out_bf16: Optional[torch.Tensor] = None,
         accumulate: bool = False, k_splits: int = 0, block_n: int = 0, a_colsum: Optional[torch.Tensor] = None,
         M: Optional[int] = None, N: Optional[int] = None, K: Optional[int] = None) -> None:
    """C[M,N] = epi(alpha * A @ B^T). See ``tt_gemm_bf16`` in include/tt_b200.h.

    a_mn=False: A is [M,K]; a_mn=True: A is stored [K,M]. Same for B with N.
    """
    _require_cuda(A, B, bias, gate, residual, out_f32, out_bf16, a_colsum)
    assert A.dtype == torch.bfloat16 and B.dtype == torch.bfloat16
    assert A.dim() == 2 and B.dim() == 2 and A.stride(1) == 1 and B.stride(1) == 1
    if a_mn:
        k_a, m_a = A.shape
    else:
        m_a, k_a = A.shape
    if b_mn:
        k_b, n_b = B.shape
    else:
        n_b, k_b = B.shape
    M = m_a if M is None else M
    N = n_b if N is None else N
    K = min(k_a, k_b) if K is None else K
    args = GemmArgs()
    args.A, args.B = A.data_ptr(), B.data_ptr()
    args.lda, args.ldb = A.stride(0), B.stride(0)
    args.a_mn, args.b_mn = int(a_mn), int(b_mn)
    args.M, args.N, args.K = M, N, K
    args.alpha = alpha
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.is_contiguous() and bias.numel() >= N
    args.bias = _ptr(bias)
    args.relu = int(relu)
    args.drop_p, args.drop_seed, args.drop_site = drop_p, drop_seed, drop_site
    args.drop_seed_dev = _ptr(drop_seed_dev)
    if gate is not None:
        assert gate.dtype == torch.bfloat16 and gate.stride(1) == 1
        args.ld_gate = gate.stride(0)
    args.gate = _ptr(gate)
    args.gate_scale = gate_scale
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.stride(1) == 1
        args.ld_res = residual.stride(0)
    args.residual = _ptr(residual)
    if out_f32 is not None:
        assert out_f32.dtype == torch.float32 and out_f32.stride(1) == 1
        args.ld_f32 = out_f32.stride(0)
    args.out_f32 = _ptr(out_f32)
    if out_bf16 is not None:
        assert out_bf16.dtype == torch.bfloat16 and out_bf16.stride(1) == 1
        args.ld_bf16 = out_bf16.stride(0)
    args.out_bf16 = _ptr(out_bf16)
    args.accumulate = int(accumulate)
    args.k_splits = k_splits
    args.block_n = block_n
    if a_colsum is not None:      # a_colsum[k] += sum_m A[m, k]: the bias gradient next to a dgrad GEMM
        assert a_colsum.dtype == torch.float32 and a_colsum.is_contiguous() and a_colsum.numel() >= K and not a_mn
    args.a_colsum = _ptr(a_colsum)
    check(lib().tt_gemm_bf16(ctypes.byref(args), _stream()), "tt_gemm_bf16")


def attn_fwd(qkv: torch.Tensor, ctx: torch.Tensor, lse: Optional[torch.Tensor], B: int, L: int, H: int,
             drop_p: float = 0.0, drop_seed: int = 0, drop_site: int = 0,
             drop_seed_dev: Optional[torch.Tensor] = None) -> None:
    """Causal self-attention forward (tt_attn_causal_fwd). qkv bf16 [B*L, 3*H*64] -> ctx bf16 [B*L, H*64]."""
    _require_cuda(qkv, ctx, lse)
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous() and qkv.shape == (B * L, 3 * H * 64)
    assert ctx.dtype == torch.bfloat16 and ctx.is_contiguous() and ctx.shape == (B * L, H * 64)
    if lse is not None:
        assert lse.dtype == torch.float32 and lse.is_contiguous() and lse.numel() == B * H * L
    check(lib().tt_attn_causal_fwd(qkv.data_ptr(), ctx.data_ptr(), _ptr(lse), B, L, H, drop_p,
                                   drop_seed, _ptr(drop_seed_dev), drop_site, _stream()), "tt_attn_causal_fwd")


def attn_bwd(qkv: torch.Tensor, ctx: torch.Tensor, dctx: torch.Tensor, lse: torch.Tensor,
             dqkv: torch.Tensor, B: int, L: int, H: int, drop_p: float = 0.0, drop_seed: int = 0,
             drop_site: int = 0, drop_seed_dev: Optional[torch.Tensor] = None) -> None:
    """Causal self-attention backward (tt_attn_causal_bwd): dqkv bf16 [B*L, 3*H*64]."""
    _require_cuda(qkv, ctx, dctx, lse, dqkv)
    for t in (qkv, ctx, dctx, dqkv):
        assert t.dtype == torch.bfloat16 and t.is_contiguous()
    assert lse.dtype == torch.float32 and lse.is_contiguous()
    check(lib().tt_attn_causal_bwd(qkv.data_ptr(), ctx.data_ptr(), dctx.data_ptr(), lse.data_ptr(),
                                   dqkv.data_ptr(), B, L, H, drop_p, drop_seed, _ptr(drop_seed_dev), drop_site, _stream()),
          "tt_attn_causal_bwd")


# --------------------------------------------------------------------------------------
# row-wise kernels
# --------------------------------------------------------------------------------------
from ._lib import BnArgs, ChainArgs  # noqa: E402


def cast_bf16(src: torch.Tensor, dst: torch.Tensor) -> None:
    _require_cuda(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == torch.bfloat16 and src.numel() == dst.numel()
    assert src.is_contiguous() and dst.is_contiguous()
    check(lib().tt_cast_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()), "tt_cast_bf16")


def last_index(ids: torch.Tensor, mask: Optional[torch.Tensor], out: torch.Tensor) -> None:
    _require_cuda(ids, mask, out)
    B, L = ids.shape
    assert ids.dtype == torch.int64 and ids.is_contiguous() and out.dtype == torch.int32
    if mask is not None:
        assert mask.dtype == torch.int64 and mask.is_contiguous() and mask.shape == ids.shape
    check(lib().tt_last_index(ids.data_ptr(), _ptr(mask), B, L, out.data_ptr(), _stream()), "tt_last_index")


def embed_ln_fwd(ids, E, P, ln_w, ln_b, next_w, next_b, B, L, x0, h, drop_p=0.0, seed=0, seed_dev=None, site=0):
    _require_cuda(ids, E, P, x0, h)
    assert ids.dtype == torch.int64 and E.dtype == torch.float32 and E.shape[1] == 256 and P.shape[0] >= L
    check(lib().tt_embed_ln_fwd(ids.data_ptr(), E.data_ptr(), P.data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(),
                                next_w.data_ptr(), next_b.data_ptr(), B, L, drop_p, seed, _ptr(seed_dev), site,
                                x0.data_ptr(), h.data_ptr(), _stream()), "tt_embed_ln_fwd")


def embed_ln_fwd_pos(ids, pos, E, P, ln_w, ln_b, next_w, next_b, x0, h) -> None:
    """tt_embed_ln_fwd_pos: embed_ln_fwd's rows for item ids[r] at position pos[r] (eval, local table)."""
    _require_cuda(ids, pos, E, P, x0, h)
    n = ids.numel()
    assert ids.dtype == torch.int64 and ids.is_contiguous() and pos.dtype == torch.int32 and pos.is_contiguous()
    assert pos.numel() == n and E.dtype == torch.float32 and E.shape[1] == 256
    assert x0.dtype == torch.float32 and x0.is_contiguous() and x0.shape == (n, 256)
    assert h.dtype == torch.bfloat16 and h.is_contiguous() and h.shape == (n, 256)
    check(lib().tt_embed_ln_fwd_pos(ids.data_ptr(), pos.data_ptr(), E.data_ptr(), P.data_ptr(), ln_w.data_ptr(),
                                    ln_b.data_ptr(), next_w.data_ptr(), next_b.data_ptr(), n, x0.data_ptr(),
                                    h.data_ptr(), _stream()), "tt_embed_ln_fwd_pos")


def session_attn(qkv, k_cache, v_cache, slots, pos, ctx) -> None:
    """tt_session_attn: each new row's K/V into cache[slot, :, pos], ctx = its attention over positions 0..pos.
    qkv bf16 [n, 3*H*64], caches bf16 [capacity, H, L, 64], slots / pos int32 [n] -> ctx bf16 [n, H*64]."""
    _require_cuda(qkv, k_cache, v_cache, slots, pos, ctx)
    n = slots.numel()
    cap, H, L, dh = k_cache.shape
    assert dh == 64 and v_cache.shape == k_cache.shape
    for t in (qkv, k_cache, v_cache, ctx):
        assert t.dtype == torch.bfloat16 and t.is_contiguous()
    assert qkv.shape == (n, 3 * H * 64) and ctx.shape == (n, H * 64)
    assert slots.dtype == torch.int32 and pos.dtype == torch.int32 and pos.numel() == n
    assert slots.is_contiguous() and pos.is_contiguous()
    check(lib().tt_session_attn(qkv.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), slots.data_ptr(),
                                pos.data_ptr(), n, H, L, cap, ctx.data_ptr(), _stream()), "tt_session_attn")


#: row sources of tt_mmr_select (include/tt_b200.h)
MMR_ROWS_TABLE, MMR_ROWS_GATHERED = 0, 1


def mmr_select(pool_idx, pool_score, k: int, lam: float, mu: float, source: int, rows, item_base: int = 0,
               num_rows: int = 0):
    """tt_mmr_select: k maximal-marginal-relevance picks per user from its pool (int32 / fp32 [U, P], canonical order).
    ``rows``: the shard's fp32 table [num_rows, 256] (MMR_ROWS_TABLE) or the gathered pool rows [U, P, 256]
    (MMR_ROWS_GATHERED). Returns (ids int32 [U, k], relevances fp32 [U, k]) in pick order."""
    _require_cuda(pool_idx, pool_score, rows)
    U, P = pool_idx.shape
    assert pool_idx.dtype == torch.int32 and pool_score.dtype == torch.float32 and pool_score.shape == (U, P)
    assert pool_idx.is_contiguous() and pool_score.is_contiguous()
    assert rows.dtype == torch.float32 and rows.is_contiguous() and rows.shape[-1] == 256
    out_idx = torch.empty(U, k, device=pool_idx.device, dtype=torch.int32)
    out_score = torch.empty(U, k, device=pool_idx.device, dtype=torch.float32)
    check(lib().tt_mmr_select(pool_idx.data_ptr(), pool_score.data_ptr(), U, P, k, lam, mu, source, rows.data_ptr(),
                              item_base, num_rows, out_idx.data_ptr(), out_score.data_ptr(), _stream()),
          "tt_mmr_select")
    return out_idx, out_score


def mmr_gather_rows(pool_idx, table, item_base: int, out) -> None:
    """tt_mmr_gather_rows: out [.., 256] row r = table row of pool_idx.flatten()[r] when this shard (rows
    [item_base, item_base + len(table))) owns it, zeros otherwise."""
    _require_cuda(pool_idx, table, out)
    n = pool_idx.numel()
    assert pool_idx.dtype == torch.int32 and pool_idx.is_contiguous()
    assert table.dtype == torch.float32 and table.is_contiguous() and table.shape[1] == 256
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == n * 256
    check(lib().tt_mmr_gather_rows(pool_idx.data_ptr(), n, table.data_ptr(), item_base, table.shape[0], out.data_ptr(),
                                   _stream()), "tt_mmr_gather_rows")


def embed_ln_bwd(ids, E, P, ln_w, ln_b, dx0, B, L, dE, dP, dgamma, dbeta, drop_p=0.0, seed=0, seed_dev=None, site=0):
    _require_cuda(ids, E, P, dx0, dE, dP, dgamma, dbeta)
    check(lib().tt_embed_ln_bwd(ids.data_ptr(), E.data_ptr(), P.data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(),
                                dx0.data_ptr(), B, L, drop_p, seed, _ptr(seed_dev), site, dE.data_ptr(),
                                dP.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), _stream()), "tt_embed_ln_bwd")


def embed_ln_bwd_det(ids, E, P, ln_w, ln_b, dx0, B, L, slot_of_token, acc64, dP, dgamma, dbeta, drop_p=0.0, seed=0,
                     seed_dev=None, site=0):
    """tt_embed_ln_bwd_det: the table gradient is accumulated per distinct id in 64-bit fixed point (order-independent,
    bit-identical from run to run); rows_scatter_add_i64 rounds the sums into the table's gradient."""
    _require_cuda(ids, E, P, dx0, slot_of_token, acc64, dP, dgamma, dbeta)
    assert acc64.dtype == torch.int64 and acc64.is_contiguous() and acc64.shape[1] == 256
    assert slot_of_token.dtype == torch.int64 and slot_of_token.numel() == B * L
    check(lib().tt_embed_ln_bwd_det(ids.data_ptr(), E.data_ptr(), P.data_ptr(), ln_w.data_ptr(), ln_b.data_ptr(),
                                    dx0.data_ptr(), B, L, drop_p, seed, _ptr(seed_dev), site, slot_of_token.data_ptr(),
                                    acc64.data_ptr(), dP.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), _stream()),
          "tt_embed_ln_bwd_det")


def rows_scatter_add_i64(uniq, state, acc64, grad_local) -> None:
    _require_cuda(uniq, state, acc64, grad_local)
    assert acc64.dtype == torch.int64 and acc64.is_contiguous() and acc64.shape[1] == 256
    assert grad_local.dtype == torch.float32 and grad_local.is_contiguous()
    check(lib().tt_rows_scatter_add_i64(grad_local.data_ptr(), uniq.data_ptr(), state.data_ptr() + 4, acc64.shape[0],
                                        acc64.data_ptr(), _stream()), "tt_rows_scatter_add_i64")


def ids_dedup(ids, V, flag, slot, uniq, state, inverse) -> None:
    """tt_ids_dedup: distinct ids of a step (uniq, state[1] = count) and every token's slot (inverse)."""
    _require_cuda(ids, flag, slot, uniq, state, inverse)
    T = ids.numel()
    assert ids.dtype == torch.int64 and ids.is_contiguous() and inverse.dtype == torch.int64 and inverse.numel() == T
    assert flag.dtype == torch.int32 and slot.dtype == torch.int32 and flag.numel() >= V and slot.numel() >= V
    assert uniq.dtype == torch.int64 and uniq.numel() >= T + 1 and state.dtype == torch.int32 and state.numel() >= 2
    check(lib().tt_ids_dedup(ids.data_ptr(), T, V, flag.data_ptr(), slot.data_ptr(), uniq.data_ptr(), state.data_ptr(),
                             inverse.data_ptr(), _stream()), "tt_ids_dedup")


def rows_gather(uniq, state, cache, team=None, weight_offset=0, table_local=None) -> None:
    _require_cuda(uniq, state, cache, table_local)
    assert cache.dtype == torch.float32 and cache.is_contiguous() and cache.shape[1] == 256
    check(lib().tt_rows_gather(None if team is None else ctypes.byref(team), weight_offset, _ptr(table_local),
                               uniq.data_ptr(), state.data_ptr() + 4, cache.shape[0], cache.data_ptr(), _stream()),
          "tt_rows_gather")


def rows_scatter_add(uniq, state, gacc, team=None, grad_offset=0, grad_local=None) -> None:
    _require_cuda(uniq, state, gacc, grad_local)
    assert gacc.dtype == torch.float32 and gacc.is_contiguous() and gacc.shape[1] == 256
    check(lib().tt_rows_scatter_add(None if team is None else ctypes.byref(team), grad_offset, _ptr(grad_local),
                                    uniq.data_ptr(), state.data_ptr() + 4, gacc.shape[0], gacc.data_ptr(), _stream()),
          "tt_rows_scatter_add")


def _chain_args(x, *, ln=None, relu=False, drop_p=0.0, seed=0, seed_dev=None, site=0, l2norm=False,
                l2_eps=1e-12, out_f32=None, out_bf16=None, dout=None, resid=None, dx_f32=None, dx_bf16=None,
                drop2_p=0.0, drop2_site=0, dgamma=None, dbeta=None, dx_colsum=None, resid_rows=None,
                resid_last_idx=None, resid_seq_len=0, dout_bf16=None) -> ChainArgs:
    _require_cuda(x, out_f32, out_bf16, dout, dout_bf16, resid, dx_f32, dx_bf16, dgamma, dbeta, dx_colsum, resid_rows,
                  resid_last_idx)
    assert x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous()
    a = ChainArgs()
    a.x, a.rows, a.width = x.data_ptr(), x.shape[0], x.shape[1]
    if ln is not None:
        a.ln_w, a.ln_b = ln[0].data_ptr(), ln[1].data_ptr()
    a.ln_eps = 1e-5
    a.relu = int(relu)
    a.drop_p, a.drop_seed, a.drop_seed_dev, a.drop_site = drop_p, seed, _ptr(seed_dev), site
    a.l2norm, a.l2_eps = int(l2norm), l2_eps
    a.out_f32, a.out_bf16 = _ptr(out_f32), _ptr(out_bf16)
    a.dout, a.resid, a.dx_f32, a.dx_bf16 = _ptr(dout), _ptr(resid), _ptr(dx_f32), _ptr(dx_bf16)
    a.drop2_p, a.drop2_site = drop2_p, drop2_site
    a.dgamma, a.dbeta, a.dx_colsum = _ptr(dgamma), _ptr(dbeta), _ptr(dx_colsum)
    if resid_rows is not None:
        assert resid is None and resid_last_idx is not None and resid_seq_len > 0
        assert resid_rows.dtype == torch.float32 and resid_rows.is_contiguous() and resid_rows.shape[1] == x.shape[1]
        assert resid_last_idx.dtype == torch.int32 and x.shape[0] == resid_rows.shape[0] * resid_seq_len
    a.resid_rows, a.resid_last_idx, a.resid_seq_len = _ptr(resid_rows), _ptr(resid_last_idx), resid_seq_len
    if dout_bf16 is not None:
        assert dout is None and dout_bf16.dtype == torch.bfloat16 and dout_bf16.is_contiguous() and dout_bf16.shape == x.shape
    a.dout_bf16 = _ptr(dout_bf16)
    return a


def chain_fwd(x, **kw) -> None:
    """[LayerNorm] -> [ReLU] -> [dropout] -> [L2 normalise] (tt_chain_fwd)."""
    a = _chain_args(x, **kw)
    check(lib().tt_chain_fwd(ctypes.byref(a), _stream()), "tt_chain_fwd")


def chain_bwd(x, **kw) -> None:
    a = _chain_args(x, **kw)
    check(lib().tt_chain_bwd(ctypes.byref(a), _stream()), "tt_chain_bwd")


def gather_cat_fwd(x, last_idx, gender, country, G, C, B, L, cat) -> None:
    _require_cuda(x, last_idx, gender, country, G, C, cat)
    check(lib().tt_gather_cat_fwd(x.data_ptr(), last_idx.data_ptr(), _ptr(gender), _ptr(country), G.data_ptr(),
                                  C.data_ptr(), B, L, cat.data_ptr(), _stream()), "tt_gather_cat_fwd")


def gather_cat_bwd(dcat, last_idx, gender, country, B, L, dx, dx_bf16, dG, dC) -> None:
    _require_cuda(dcat, last_idx, gender, country, dx, dx_bf16, dG, dC)
    check(lib().tt_gather_cat_bwd(dcat.data_ptr(), last_idx.data_ptr(), _ptr(gender), _ptr(country), B, L,
                                  _ptr(dx), _ptr(dx_bf16), dG.data_ptr(), dC.data_ptr(), _stream()),
          "tt_gather_cat_bwd")


def concat4_bf16(a, b, c, d, out) -> None:
    _require_cuda(a, b, c, d, out)
    B, m = a.shape
    for t in (a, b, c, d):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.shape == (B, m)
    check(lib().tt_concat4_bf16(a.data_ptr(), b.data_ptr(), c.data_ptr(), d.data_ptr(), B, m, out.data_ptr(),
                                _stream()), "tt_concat4_bf16")


def _bn_args(y, w, b, running_mean, running_var, num_batches, *, training, momentum=0.1, eps=1e-5, drop_p=0.0,
             seed=0, seed_dev=None, site=0, save_mean=None, save_rstd=None, out_bf16=None, dout=None,
             dy_bf16=None, dgamma=None, dbeta=None, dy_colsum=None) -> BnArgs:
    _require_cuda(y, w, b, running_mean, running_var, num_batches, save_mean, save_rstd, out_bf16, dout, dy_bf16)
    a = BnArgs()
    a.y, a.B, a.C = y.data_ptr(), y.shape[0], y.shape[1]
    a.w, a.b = w.data_ptr(), b.data_ptr()
    a.running_mean, a.running_var, a.num_batches_tracked = _ptr(running_mean), _ptr(running_var), _ptr(num_batches)
    a.training, a.momentum, a.eps = int(training), momentum, eps
    a.drop_p, a.drop_seed, a.drop_seed_dev, a.drop_site = drop_p, seed, _ptr(seed_dev), site
    a.save_mean, a.save_rstd, a.out_bf16 = _ptr(save_mean), _ptr(save_rstd), _ptr(out_bf16)
    a.dout, a.dy_bf16, a.dgamma, a.dbeta, a.dy_colsum = _ptr(dout), _ptr(dy_bf16), _ptr(dgamma), _ptr(dbeta), _ptr(dy_colsum)
    return a


def bn_relu_fwd(y, w, b, running_mean, running_var, num_batches, **kw) -> None:
    a = _bn_args(y, w, b, running_mean, running_var, num_batches, **kw)
    check(lib().tt_bn_relu_fwd(ctypes.byref(a), _stream()), "tt_bn_relu_fwd")


def bn_relu_bwd(y, w, b, running_mean, running_var, num_batches, **kw) -> None:
    a = _bn_args(y, w, b, running_mean, running_var, num_batches, **kw)
    check(lib().tt_bn_relu_bwd(ctypes.byref(a), _stream()), "tt_bn_relu_bwd")


def adamw_step(p, g, m, v, step_dev, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.01,
               shadow=None, shadow_begin=0, shadow_end=0, zero_grad=True, grad_scale=1.0) -> None:
    _require_cuda(p, g, m, v, step_dev, shadow)
    for t in (p, g, m, v):
        assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == p.numel()
    assert step_dev.dtype == torch.int64
    check(lib().tt_adamw_step(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, beta1, beta2,
                              eps, weight_decay, grad_scale, step_dev.data_ptr(), _ptr(shadow), shadow_begin, shadow_end,
                              int(zero_grad), _stream()), "tt_adamw_step")


def step_counters_advance(step_dev, seed_dev) -> None:
    check(lib().tt_step_counters_advance(_ptr(step_dev), _ptr(seed_dev), _stream()), "tt_step_counters_advance")


def infonce_rows(S, uid_rows, uid_cols, pos0, row_lse, pos_logit) -> None:
    _require_cuda(S, uid_rows, uid_cols, row_lse, pos_logit)
    assert S.dtype == torch.float32 and S.stride(1) == 1
    check(lib().tt_infonce_rows(S.data_ptr(), S.shape[0], S.shape[1], S.stride(0), _ptr(uid_rows), _ptr(uid_cols),
                                pos0, row_lse.data_ptr(), pos_logit.data_ptr(), _stream()), "tt_infonce_rows")


def infonce_grad(S, row_lse, col_lse, pos0, coef, dS) -> None:
    _require_cuda(S, row_lse, col_lse, dS)
    assert dS.dtype == torch.bfloat16 and dS.stride(1) == 1
    check(lib().tt_infonce_grad(S.data_ptr(), S.shape[0], S.shape[1], S.stride(0), row_lse.data_ptr(),
                                col_lse.data_ptr(), pos0, coef, dS.data_ptr(), dS.stride(0), _stream()),
          "tt_infonce_grad")


def _offsets(off, n: int, what: str) -> None:
    if off.dtype != torch.float32 or not off.is_contiguous() or off.numel() != n:
        raise ValueError(f"{what}: offsets must be contiguous fp32 with {n} values, got {off.dtype} {tuple(off.shape)}")


def infonce_rows_off(S, uid_rows, uid_cols, pos0, col_off, row_lse, pos_logit) -> None:
    """tt_infonce_rows over S[i, j] - col_off[j] (logQ correction); S keeps the uncorrected masked logits."""
    _require_cuda(S, uid_rows, uid_cols, col_off, row_lse, pos_logit)
    assert S.dtype == torch.float32 and S.stride(1) == 1
    _offsets(col_off, S.shape[1], "infonce_rows_off")
    check(lib().tt_infonce_rows_off(S.data_ptr(), S.shape[0], S.shape[1], S.stride(0), _ptr(uid_rows), _ptr(uid_cols),
                                    pos0, col_off.data_ptr(), row_lse.data_ptr(), pos_logit.data_ptr(), _stream()),
          "tt_infonce_rows_off")


def infonce_grad_off(S, row_lse, col_lse, pos0, coef, col_off, row_off, dS) -> None:
    """tt_infonce_grad with the logQ offsets of the columns (col_off) and of the other side's rows (row_off)."""
    _require_cuda(S, row_lse, col_lse, col_off, row_off, dS)
    assert dS.dtype == torch.bfloat16 and dS.stride(1) == 1
    _offsets(col_off, S.shape[1], "infonce_grad_off")
    _offsets(row_off, S.shape[1], "infonce_grad_off")
    check(lib().tt_infonce_grad_off(S.data_ptr(), S.shape[0], S.shape[1], S.stride(0), row_lse.data_ptr(),
                                    col_lse.data_ptr(), pos0, coef, col_off.data_ptr(), row_off.data_ptr(),
                                    dS.data_ptr(), dS.stride(0), _stream()), "tt_infonce_grad_off")


def logq_table_gather(ids, table, floor: float, out) -> None:
    """out[i] = table[ids[i]] for ids in [0, len(table)), ``floor`` otherwise (tt_logq_table_gather)."""
    _require_cuda(ids, table, out)
    assert ids.dtype == torch.int64 and ids.is_contiguous() and table.dtype == torch.float32 and table.is_contiguous()
    _offsets(out, ids.numel(), "logq_table_gather")
    check(lib().tt_logq_table_gather(ids.data_ptr(), ids.numel(), table.data_ptr(), table.numel(), floor,
                                     out.data_ptr(), _stream()), "tt_logq_table_gather")


def logq_stream_update(ids, A, Bv, step_dev, alpha: float, one_minus_alpha: float, out) -> None:
    """One step of the streaming frequency estimator (tt_logq_stream_update): A int64 / Bv fp32 [h, 2^b], step_dev
    int64 [1]; out[i] = log q of ids[i] after the update."""
    _require_cuda(ids, A, Bv, step_dev, out)
    h, H = A.shape
    assert ids.dtype == torch.int64 and ids.is_contiguous() and A.dtype == torch.int64 and A.is_contiguous()
    assert Bv.dtype == torch.float32 and Bv.is_contiguous() and Bv.shape == A.shape and H & (H - 1) == 0
    assert step_dev.dtype == torch.int64
    _offsets(out, ids.numel(), "logq_stream_update")
    check(lib().tt_logq_stream_update(ids.data_ptr(), ids.numel(), A.data_ptr(), Bv.data_ptr(), h, H.bit_length() - 1,
                                      step_dev.data_ptr(), alpha, one_minus_alpha, out.data_ptr(), _stream()),
          "tt_logq_stream_update")


def infonce_loss(lse_a, pos_a, lse_b, pos_b, coef, loss) -> None:
    _require_cuda(lse_a, pos_a, lse_b, pos_b, loss)
    check(lib().tt_infonce_loss(lse_a.data_ptr(), pos_a.data_ptr(), lse_b.data_ptr(), pos_b.data_ptr(),
                                lse_a.numel(), coef, loss.data_ptr(), _stream()), "tt_infonce_loss")


def inbatch_recall(S, pos0: int, k: int, acc) -> None:
    """acc[0] += hits, acc[1] += rows of the in-batch Recall@k on logits S (tt_inbatch_recall)."""
    _require_cuda(S, acc)
    assert S.dtype == torch.float32 and S.stride(1) == 1 and acc.dtype == torch.float32 and acc.numel() == 2
    check(lib().tt_inbatch_recall(S.data_ptr(), S.shape[0], S.shape[1], S.stride(0), pos0, k, acc.data_ptr(),
                                  _stream()), "tt_inbatch_recall")


def index_rows(y, ln_w, ln_b, ids, table, table_bf16=None) -> None:
    """LayerNorm -> normalise -> NaN->0 -> normalise(eps 1e-8) -> table[ids] (tt_index_rows)."""
    _require_cuda(y, ln_w, ln_b, ids, table, table_bf16)
    assert y.dtype == torch.float32 and y.is_contiguous() and y.shape[1] == 256
    assert ids.dtype == torch.int64 and ids.is_contiguous() and ids.numel() == y.shape[0]
    assert table.dtype == torch.float32 and table.is_contiguous() and table.shape[1] == 256
    if table_bf16 is not None:
        assert table_bf16.dtype == torch.bfloat16 and table_bf16.is_contiguous() and table_bf16.shape == table.shape
    check(lib().tt_index_rows(y.data_ptr(), y.shape[0], ln_w.data_ptr(), ln_b.data_ptr(), ids.data_ptr(),
                              table.shape[0], table.data_ptr(), _ptr(table_bf16), _stream()), "tt_index_rows")


# --------------------------------------------------------------------------------------
# last-layer specialisation (one query row per sequence)
# --------------------------------------------------------------------------------------
def gather_rows(last_idx, B, L, x_f32=None, out_f32=None, x_bf16=None, out_bf16=None) -> None:
    _require_cuda(last_idx, x_f32, out_f32, x_bf16, out_bf16)
    W = (x_f32 if x_f32 is not None else x_bf16).shape[1]
    check(lib().tt_gather_rows(_ptr(x_f32), _ptr(x_bf16), last_idx.data_ptr(), B, L, W, _ptr(out_f32), _ptr(out_bf16),
                               _stream()), "tt_gather_rows")


def scatter_rows_add(rows, last_idx, B, L, x, accumulate: bool) -> None:
    _require_cuda(rows, last_idx, x)
    assert rows.dtype == torch.float32 and x.dtype == torch.float32 and rows.is_contiguous() and x.is_contiguous()
    check(lib().tt_scatter_rows_add(rows.data_ptr(), last_idx.data_ptr(), B, L, rows.shape[1], x.data_ptr(),
                                    int(accumulate), _stream()), "tt_scatter_rows_add")


def attn_lastq_fwd(q, qkv, last_idx, ctx, lse, B, L, H, drop_p=0.0, seed=0, seed_dev=None, site=0) -> None:
    _require_cuda(q, qkv, last_idx, ctx, lse)
    assert q.is_contiguous() and qkv.is_contiguous() and ctx.is_contiguous()
    check(lib().tt_attn_lastq_fwd(q.data_ptr(), qkv.data_ptr(), last_idx.data_ptr(), ctx.data_ptr(), _ptr(lse), B, L, H,
                                  drop_p, seed, _ptr(seed_dev), site, _stream()), "tt_attn_lastq_fwd")


def attn_lastq_bwd(q, qkv, last_idx, ctx, dctx, lse, dq, dqkv, B, L, H, drop_p=0.0, seed=0, seed_dev=None, site=0) -> None:
    _require_cuda(q, qkv, last_idx, ctx, dctx, lse, dq, dqkv)
    check(lib().tt_attn_lastq_bwd(q.data_ptr(), qkv.data_ptr(), last_idx.data_ptr(), ctx.data_ptr(), dctx.data_ptr(),
                                  lse.data_ptr(), dq.data_ptr(), dqkv.data_ptr(), B, L, H, drop_p, seed, _ptr(seed_dev),
                                  site, _stream()), "tt_attn_lastq_bwd")
