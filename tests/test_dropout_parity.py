"""Dropout parity: every kernel's mask against the numpy restatement of the hash (tests/_dropout_ref.py), the
dropout backward passes against fp32 autograd given that mask, and the engine's dropout training step against the
fp64 oracle given the masks the engine's conventions produce.

A mask is stored nowhere: each kernel recomputes its keep bits from (seed + step counter, site, element index), and
a backward often rebuilds a mask in another kernel than the forward that applied it (GEMM epilogue -> chain_bwd
drop2, attn_fwd -> attn_bwd, embed_ln_fwd -> embed_ln_bwd, bn_relu_fwd -> bn_relu_bwd). A pair that disagrees on the
seed, counter, site, row numbering or index width gives ~18 % of a site's elements a wrong gradient while training
still converges, so the pins below compare keep bits exactly and the end-to-end tests use the parity tolerance,
which test_the_end_to_end_tolerance_sees_a_wrong_mask_at_every_site shows is tight enough to see any one wrong site.

Measured values are appended to the parity report that test_engine.py writes (its ``_report``).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import _dropout_ref as R
from test_engine import _report

gpu = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

# (seed, device counter or None, site): the engine's base seed with no counter at site 0, and a seed with a non-zero
# high word plus a non-zero counter at a non-zero site (both halves of drop_key and the seed + *seed_dev read)
CASES = [(R.BASE_SEED, None, 0), (0x1_2345_6789, 7, 37)]
CASE_IDS = ["seed", "seed+counter"]


def _counter(ctr):
    return None if ctr is None else torch.tensor(ctr, dtype=torch.long, device="cuda")


def _keep(case, shape, p):
    seed, ctr, site = case
    n = int(np.prod(shape))
    return torch.from_numpy(R.keep_bits(seed + (ctr or 0), site, n, p).reshape(shape)).cuda()


def _randn(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).cuda()


def _close(a, ref, rel):
    err = (a.float() - ref).abs().max().item()
    assert err <= rel * max(1.0, ref.abs().max().item()), (err, ref.abs().max().item())


# ----------------------------------------------------------------------------------------------------------------
# the numpy restatement itself (CPU)
# ----------------------------------------------------------------------------------------------------------------
def test_mask_reference_rates_and_threshold():
    """Keep fraction 1 - p, the host threshold and scale as the .cu files compute them, and the uint64 arithmetic
    agreeing with plain Python integers on a sample of indices (including both words of a 64-bit seed)."""
    assert R.drop_threshold(0.0) == 0 and R.drop_threshold(1e-12) == 1
    assert R.drop_threshold(0.1) == int(float(np.float32(0.1)) * 2.0 ** 32)
    assert R.drop_scale(0.1) == np.float32(1.0) / np.float32(0.9)
    for p in (0.1, 0.25):
        frac = R.keep_bits(0x1_2345_6789, 37, 1 << 20, p).mean()
        assert abs(frac - (1 - p)) < 2e-3, (p, frac)

    def mix(x):
        x ^= x >> 16; x = (x * 0x7FEB352D) & 0xFFFFFFFF
        x ^= x >> 15; x = (x * 0x846CA68B) & 0xFFFFFFFF
        return x ^ (x >> 16)

    seed, site, thresh = 0x1_2345_6789 + 7, 37, R.drop_threshold(0.1)
    key = mix((seed & 0xFFFFFFFF) ^ mix(((seed >> 32) + site * 0x9E3779B9) & 0xFFFFFFFF))
    assert R.drop_key(seed, site) == key
    idx = [0, 1, 2, 3, 4, 5, 6, 7, 1023, 40_960_001, (1 << 32) - 1]
    muls = [1, 0x9E3779B1, 0x85EBCA6B, 0xC2B2AE35]
    want = [((mix((i >> 2) ^ key) * muls[i & 3]) & 0xFFFFFFFF) >= thresh for i in idx]
    assert R.drop_keep_k(key, np.array(idx, dtype=np.uint64), thresh).tolist() == want


# ----------------------------------------------------------------------------------------------------------------
# kernel masks, bit for bit
# ----------------------------------------------------------------------------------------------------------------
def _embed_operands(B, L, V=1001, seed=0):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(0, V, (B, L), generator=g).cuda()
    E, P = _randn(V, 256, seed=seed + 1, scale=0.1), _randn(L, 256, seed=seed + 2, scale=0.1)
    w, b = 1 + _randn(256, seed=seed + 3, scale=0.1), _randn(256, seed=seed + 4, scale=0.1)
    w1, b1 = 1 + _randn(256, seed=seed + 5, scale=0.1), _randn(256, seed=seed + 6, scale=0.1)
    return ids, E, P, w, b, w1, b1


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("B,L", [(3, 50), (64, 50)])
def test_embed_ln_fwd_mask(B, L, case):
    """The zeros of x0 are the embedding dropout's mask; the kept elements are the p = 0 output times 1/(1-p)."""
    from mrm_b200 import ops
    seed, ctr, site = case
    ids, E, P, w, b, w1, b1 = _embed_operands(B, L)
    out = []
    for p in (0.0, 0.1):
        x0 = torch.empty(B * L, 256, device="cuda")
        h = torch.empty(B * L, 256, device="cuda", dtype=torch.bfloat16)
        ops.embed_ln_fwd(ids.view(-1), E, P, w, b, w1, b1, B, L, x0, h, drop_p=p, seed=seed,
                         seed_dev=_counter(ctr), site=site)
        out.append(x0)
    torch.cuda.synchronize()
    keep = _keep(case, (B * L, 256), 0.1)
    assert torch.equal(out[1] != 0, keep)
    assert torch.allclose(out[1], torch.where(keep, out[0] * float(R.drop_scale(0.1)), 0.0), rtol=1e-6, atol=0)


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("M,N,epi", [(200, 256, "plain"), (333, 256, "residual"), (37, 1024, "relu"),
                                     (25_000, 1024, "relu"), (25_001, 256, "residual")])
def test_gemm_epilogue_mask(M, N, epi, case):
    """A = 0 and bias = 1 make the epilogue's output keep * 1/(1-p) (+ residual): the mask of the out_proj / linear1 /
    linear2 launches, ragged M, and M large enough for CTA pairs (25,000 rows: 196 row blocks)."""
    from mrm_b200 import ops
    seed, ctr, site = case
    K = 256
    A = torch.zeros(M, K, device="cuda", dtype=torch.bfloat16)
    W = _randn(N, K, seed=M + N).bfloat16()
    bias = torch.ones(N, device="cuda")
    kw = dict(bias=bias, drop_p=0.1, drop_seed=seed, drop_seed_dev=_counter(ctr), drop_site=site)
    keep = _keep(case, (M, N), 0.1)
    scaled = torch.where(keep, float(R.drop_scale(0.1)), 0.0)
    if epi == "relu":
        out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
        ops.gemm(A, W, relu=True, out_bf16=out, **kw)
        want = scaled.bfloat16()
    elif epi == "residual":
        res = _randn(M, N, seed=5)
        out = torch.empty(M, N, device="cuda")
        ops.gemm(A, W, residual=res, out_f32=out, **kw)
        want = scaled + res
    else:
        out = torch.empty(M, N, device="cuda")
        ops.gemm(A, W, out_f32=out, **kw)
        want = scaled
    torch.cuda.synchronize()
    assert torch.equal(out, want)


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("R_", [600, 777])
def test_chain_fwd_and_bwd_drop2_masks(R_, case):
    """chain_fwd's dropout on x = 1 and chain_bwd's drop2 (the dy of out_proj / linear2 in the backward) on dout = 1,
    no LayerNorm: both outputs are keep * 1/(1-p), with row * 256 + col as the GEMM epilogue numbers it."""
    from mrm_b200 import ops
    seed, ctr, site = case
    ones = torch.ones(R_, 256, device="cuda")
    fwd = torch.empty(R_, 256, device="cuda")
    ops.chain_fwd(ones, drop_p=0.1, seed=seed, seed_dev=_counter(ctr), site=site, out_f32=fwd)
    bwd = torch.empty(R_, 256, device="cuda", dtype=torch.bfloat16)
    ops.chain_bwd(ones, dout=ones, dx_bf16=bwd, drop2_p=0.1, drop2_site=site, seed=seed, seed_dev=_counter(ctr))
    torch.cuda.synchronize()
    scaled = torch.where(_keep(case, (R_, 256), 0.1), float(R.drop_scale(0.1)), 0.0)
    assert torch.equal(fwd, scaled)
    assert torch.equal(bwd, scaled.bfloat16())


def _bn_operands(B, C=512, big_bias=False):
    y = _randn(B, C, seed=B)
    w = 1 + _randn(C, seed=B + 1, scale=0.1)
    b = torch.full((C,), 100.0, device="cuda") if big_bias else _randn(C, seed=B + 2, scale=0.1)
    stats = dict(save_mean=torch.empty(C, device="cuda"), save_rstd=torch.empty(C, device="cuda"))
    return y, w, b, stats


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("B", [37, 256])
def test_bn_relu_fwd_mask(B, case):
    """A large BatchNorm bias lets the ReLU pass everything: the zeros of the output are the item dropout's mask."""
    from mrm_b200 import ops
    seed, ctr, site = case
    y, w, b, stats = _bn_operands(B, big_bias=True)
    out = torch.empty(B, 512, device="cuda", dtype=torch.bfloat16)
    ops.bn_relu_fwd(y, w, b, torch.zeros(512, device="cuda"), torch.ones(512, device="cuda"), None, training=True,
                    drop_p=0.1, seed=seed, seed_dev=_counter(ctr), site=site, out_bf16=out, **stats)
    torch.cuda.synchronize()
    keep = _keep(case, (B, 512), 0.1)
    assert torch.equal(out != 0, keep)
    ref = (F.batch_norm(y, None, None, w, b, training=True) * float(R.drop_scale(0.1)))
    _close(out.float()[keep], ref[keep], 1e-2)


def _probs_readout(qkv, B, L, H, **drop):
    """[B, H, L, L] probabilities as attn_fwd forms them (dropout applied), read out through one-hot V blocks."""
    from mrm_b200 import ops
    D = H * 64
    out = torch.zeros(B, H, L, L, device="cuda")
    x = qkv.clone().view(B, L, 3, H, 64)
    ctx = torch.empty(B * L, D, device="cuda", dtype=torch.bfloat16)
    for k0 in range(0, L, 64):
        x[:, :, 2] = 0
        n = min(64, L - k0)
        x[:, k0:k0 + n, 2, :, :n] = torch.eye(n, device="cuda", dtype=torch.bfloat16)[None, :, None, :]
        ops.attn_fwd(x.view(B * L, 3 * D), ctx, None, B, L, H, **drop)
        out[:, :, :, k0:k0 + n] = ctx.float().view(B, L, H, 64)[..., :n].permute(0, 2, 1, 3)
    torch.cuda.synchronize()
    return out


def _attn_ref(qkv, B, L, H, mask, dctx):
    """fp32 causal attention with the probabilities multiplied by ``mask`` (B, H, L, L); returns (o, dqkv)."""
    x = qkv.float().view(B, L, 3, H, 64).requires_grad_(True)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) / 8.0
    s = s.masked_fill(torch.triu(torch.ones(L, L, dtype=torch.bool, device="cuda"), 1), float("-inf"))
    o = ((torch.softmax(s, dim=-1) * mask) @ v).transpose(1, 2).reshape(B * L, H * 64)
    o.backward(dctx.float())
    return o.detach(), x.grad.reshape(B * L, 3 * H * 64)


# odd B*H (and L = 50, 129, 300: every alignment of the index, so the quad, pair and single hash forms all run);
# the persistent kernels for L <= 256, the tiled forward and the four-tile per-item backward for 256 < L <= 512
ATTN_SHAPES = [(3, 50, 1), (1, 129, 3), (3, 200, 1), (2, 200, 4), (1, 256, 3), (3, 300, 1), (1, 512, 3)]


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("B,L,H", ATTN_SHAPES)
def test_attention_masks_forward_and_backward(B, L, H, case):
    """The forward's keep bits, read out through one-hot V, equal the numpy mask wherever the probability is
    resolvable (P > 1e-5); the backward equals fp32 autograd with the numpy mask."""
    from mrm_b200 import ops
    seed, ctr, site = case
    p = 0.1
    D = H * 64
    g = torch.Generator().manual_seed(7 * L + B + H)
    qkv = torch.randn(B * L, 3 * D, generator=g).cuda().bfloat16()
    dctx = torch.randn(B * L, D, generator=g).cuda().bfloat16()
    drop = dict(drop_p=p, drop_seed=seed, drop_seed_dev=_counter(ctr), drop_site=site)
    keep = _keep(case, (B, H, L, L), p)
    P0 = _probs_readout(qkv, B, L, H)
    Pd = _probs_readout(qkv, B, L, H, **drop)
    known = P0 > 1e-5
    assert known.sum().item() > 0.5 * B * H * L * (L + 1) / 2    # most of the causal triangle is resolvable
    assert torch.equal((Pd > 0.5 * P0)[known], keep[known])
    mask = torch.where(keep, float(R.drop_scale(p)), 0.0)
    o_ref, d_ref = _attn_ref(qkv, B, L, H, mask, dctx)
    ctx = torch.empty(B * L, D, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H, **drop)
    dqkv = torch.full((B * L, 3 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attn_bwd(qkv, ctx, dctx, lse, dqkv, B, L, H, **drop)
    torch.cuda.synchronize()
    assert (ctx.float() - o_ref).abs().max().item() <= 4e-2
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        err = (dqkv[:, sl].float() - d_ref[:, sl]).abs().max().item()
        assert err <= 4e-2 * max(d_ref[:, sl].abs().max().item(), 1.0), (name, err)


def _lastq_operands(B, L, H, last, seed):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B * L, 3 * H * 64, generator=g).cuda().bfloat16()
    q = torch.stack([qkv.view(B, L, -1)[b, int(last[b]), :H * 64] for b in range(B)]).contiguous()
    return qkv, q


def _lastq_last(B, L):
    return torch.tensor([0, L - 1, L // 2, 5, L - 2][:B], dtype=torch.int32).cuda()


@gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
@pytest.mark.parametrize("L", [77, 200, 512])
def test_attn_lastq_fwd_mask_equals_the_full_kernel_row(L, case):
    """attn_lastq_fwd (the pruned last layer's attention) draws its mask at the full-sequence index
    ((b*H + h)*L + last)*L + k: its probabilities, read out through one-hot V, keep the numpy mask's bits and equal
    row `last` of the full kernel's."""
    from mrm_b200 import ops
    seed, ctr, site = case
    B, H, p = 5, 4, 0.1
    D = H * 64
    last = _lastq_last(B, L)
    qkv, q = _lastq_operands(B, L, H, last, seed=L)
    drop = dict(drop_p=p, seed=seed, seed_dev=_counter(ctr), site=site)

    def rows(**kw):
        out = torch.zeros(B, H, L, device="cuda")
        x = qkv.clone().view(B, L, 3, H, 64)
        ctx = torch.empty(B, D, device="cuda", dtype=torch.bfloat16)
        for k0 in range(0, L, 64):
            x[:, :, 2] = 0
            n = min(64, L - k0)
            x[:, k0:k0 + n, 2, :, :n] = torch.eye(n, device="cuda", dtype=torch.bfloat16)[None, :, None, :]
            ops.attn_lastq_fwd(q, x.view(B * L, 3 * D), last, ctx, None, B, L, H, **kw)
            out[:, :, k0:k0 + n] = ctx.float().view(B, H, 64)[..., :n]
        torch.cuda.synchronize()
        return out

    P0, Pd = rows(), rows(**drop)
    keep = _keep(case, (B, H, L, L), p)
    bi = torch.arange(B, device="cuda")
    keep_rows = keep[bi, :, last.long()]                              # (B, H, L)
    known = P0 > 1e-5
    assert torch.equal((Pd > 0.5 * P0)[known], keep_rows[known])
    full = _probs_readout(qkv, B, L, H, drop_p=p, drop_seed=seed, drop_seed_dev=_counter(ctr),
                          drop_site=site)[bi, :, last.long()]
    assert torch.equal((full > 0)[known], (Pd > 0)[known])
    assert torch.allclose(full, Pd, rtol=1e-2, atol=1e-4)


@gpu
@pytest.mark.parametrize("L", [77, 200, 512])
def test_attn_lastq_bwd_with_dropout_matches_autograd(L):
    from mrm_b200 import ops
    seed, ctr, site = CASES[1]
    B, H, p = 5, 4, 0.1
    D = H * 64
    last = _lastq_last(B, L)
    qkv, q = _lastq_operands(B, L, H, last, seed=100 + L)
    drop = dict(drop_p=p, seed=seed, seed_dev=_counter(ctr), site=site)
    ctx = torch.empty(B, D, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, device="cuda")
    ops.attn_lastq_fwd(q, qkv, last, ctx, lse, B, L, H, **drop)
    dctx = _randn(B, D, seed=L).bfloat16()
    dq = torch.empty_like(q)
    dqkv = torch.full_like(qkv, float("nan"))
    ops.attn_lastq_bwd(q, qkv, last, ctx, dctx, lse, dq, dqkv, B, L, H, **drop)
    torch.cuda.synchronize()
    mask = torch.where(_keep(CASES[1], (B, H, L, L), p), float(R.drop_scale(p)), 0.0)
    x = qkv.float().view(B, L, 3, H, 64)
    for b in range(B):
        n = int(last[b]) + 1
        qq = q[b].float().view(H, 64).clone().requires_grad_(True)
        k = x[b, :n, 1].clone().requires_grad_(True)
        v = x[b, :n, 2].clone().requires_grad_(True)
        s = torch.einsum("hd,nhd->hn", qq, k) / 8.0
        o = torch.einsum("hn,nhd->hd", torch.softmax(s, dim=-1) * mask[b, :, n - 1, :n], v)
        assert (ctx[b].float().view(H, 64) - o).abs().max().item() < 2e-2
        o.backward(dctx[b].float().view(H, 64))
        _close(dq[b].float().view(H, 64), qq.grad, 3e-2)
        dk = dqkv.view(B, L, 3, H, 64)[b, :, 1].float()
        dv = dqkv.view(B, L, 3, H, 64)[b, :, 2].float()
        _close(dk[:n], k.grad, 3e-2)
        _close(dv[:n], v.grad, 3e-2)
        if n < L:
            assert dk[n:].abs().max().item() == 0.0 and dv[n:].abs().max().item() == 0.0


# ----------------------------------------------------------------------------------------------------------------
# dropout backward passes against fp32 autograd with the numpy mask
# ----------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("p", [0.1, 0.25])
def test_embed_ln_bwd_dropout_matches_autograd(p):
    """B = 64, L = 50: several row splits per position (the c2 step runs four)."""
    from mrm_b200 import ops
    case = CASES[1]
    seed, ctr, site = case
    B, L = 64, 50
    ids, E, P, w, b, _, _ = _embed_operands(B, L, seed=30)
    kw = dict(drop_p=p, seed=seed, seed_dev=_counter(ctr), site=site)
    mask = torch.where(_keep(case, (B * L, 256), p), float(R.drop_scale(p)), 0.0)
    dx0 = _randn(B * L, 256, seed=40)
    dE, dP, dg, db = (torch.zeros_like(E), torch.zeros_like(P), torch.zeros(256, device="cuda"),
                      torch.zeros(256, device="cuda"))
    ops.embed_ln_bwd(ids.view(-1), E, P, w, b, dx0, B, L, dE, dP, dg, db, **kw)
    torch.cuda.synchronize()
    Er, Pr, wr, br = (t.clone().requires_grad_(True) for t in (E, P, w, b))
    x = F.layer_norm(Er[ids] + Pr[:L].unsqueeze(0), (256,), wr, br).view(B * L, 256) * mask
    x.backward(dx0)
    dE_ref = Er.grad.clone()
    dE_ref[0] = 0                     # padding_idx
    for a, r in zip((dE, dP, dg, db), (dE_ref, Pr.grad, wr.grad, br.grad)):
        _close(a, r, 1e-4)


@gpu
@pytest.mark.parametrize("B", [37, 256])
def test_bn_relu_bwd_with_dropout_matches_autograd(B):
    from mrm_b200 import ops
    case = CASES[1]
    seed, ctr, site = case
    y, w, b, stats = _bn_operands(B)
    kw = dict(training=True, drop_p=0.1, seed=seed, seed_dev=_counter(ctr), site=site, **stats)
    rm, rv = torch.zeros(512, device="cuda"), torch.ones(512, device="cuda")
    out = torch.empty(B, 512, device="cuda", dtype=torch.bfloat16)
    ops.bn_relu_fwd(y, w, b, rm, rv, None, out_bf16=out, **kw)
    dout = _randn(B, 512, seed=B + 9)
    dy = torch.empty(B, 512, device="cuda", dtype=torch.bfloat16)
    dg, db = torch.zeros(512, device="cuda"), torch.zeros(512, device="cuda")
    ops.bn_relu_bwd(y, w, b, rm, rv, None, dout=dout, dy_bf16=dy, dgamma=dg, dbeta=db, **kw)
    torch.cuda.synchronize()
    mask = torch.where(_keep(case, (B, 512), 0.1), float(R.drop_scale(0.1)), 0.0)
    yr, wr, br = (t.clone().requires_grad_(True) for t in (y, w, b))
    a = torch.relu(F.batch_norm(yr, None, None, wr, br, training=True)) * mask
    _close(out.float(), a.detach(), 1e-2)
    a.backward(dout)
    _close(dy.float(), yr.grad, 1e-2)
    _close(dg, wr.grad, 1e-4)
    _close(db, br.grad, 1e-4)


# ----------------------------------------------------------------------------------------------------------------
# end to end: the engine's dropout step against the fp64 oracle given the engine's masks
# ----------------------------------------------------------------------------------------------------------------
def _fixture(name, dropout):
    from mrm_b200 import synthetic
    gold = torch.load(os.path.join(GOLDEN, name), weights_only=False)
    cfg = synthetic.TwoTowerConfig(**gold["config"])
    cfg.dropout = dropout
    sd = synthetic.make_state_dict(cfg, seed=gold["seed_w"])
    batch = synthetic.make_batch(cfg, gold["batch_size"], seed=gold["seed_b"], full_length=gold["full_length"])
    return gold["bf16_autocast_err"], cfg, sd, batch


def _oracle(cfg, sd, batch, masks):
    from oracle import two_tower_oracle as oracle
    b64 = {k: (v.double() if v.is_floating_point() else v) for k, v in batch.items()}
    loss, logits, u, i, grads, _ = oracle.loss_and_grads(sd, b64, cfg.temperature, cfg.num_heads, dtype=torch.float64,
                                                         drop=masks)
    return dict(loss=loss, logits=logits, user_emb=u, item_emb=i, grads=grads)


def _engine_step(cfg, sd, batch, counter, prune):
    from mrm_b200.engine import TwoTowerEngine
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(sd)
    eng.prune_last_layer = prune
    eng.seed_dev.fill_(counter - (1 << 64) if counter >= 1 << 63 else counter)     # int64 view of the uint64 counter
    loss, logits, u, i = eng.forward({k: v.cuda() for k, v in batch.items()}, training=True)
    eng.backward()
    torch.cuda.synchronize()
    return dict(loss=loss.cpu().double(), logits=logits.cpu().double(), user_emb=u.cpu().double(),
                item_emb=i.cpu().double(), grads={k: v.cpu().double() for k, v in eng.g.items()})


# The autocast anchors were measured at dropout 0. With dropout 0.1 the user-head gradients (country / gender
# embeddings, fusion_layer.0/1) carry up to 1.17x the dropout-0 bound of bf16 noise (B200, 1000 W: train_l200,
# full schedule), so the gradient bounds get this factor; a wrong mask at any one site still moves some compared
# quantity by >= 4.3x the bound (test_the_end_to_end_tolerance_sees_a_wrong_mask_at_every_site keeps >= 2x).
DROPOUT_GRAD_FACTOR = 1.5


def _bounds(auto, ref):
    """The parity rule of test_engine.test_backward_matches_oracle: err(ours, fp64) <= max(2 * err(the reference
    under bf16 autocast, fp64), floor), the autocast errors measured at dropout 0 on the same batch (gradient bounds
    times DROPOUT_GRAD_FACTOR). Where the batch has same-user collisions the reference's bf16 -1e4 logit mask alone
    is off by 16; the logits keep the floor."""
    b = {"loss": max(2 * auto["loss_abs"], 5e-3), "user_emb": max(2 * auto["user_emb_abs"], 5e-3),
         "item_emb": max(2 * auto["item_emb_abs"], 5e-3),
         "logits": 8e-2 if auto["logits_abs"] >= 1.0 else max(2 * auto["logits_abs"], 8e-2)}
    for k, g in ref["grads"].items():
        b[k] = DROPOUT_GRAD_FACTOR * max(2 * auto["grad_abs"].get(k, 0.0), 3e-2 * g.norm().item() + 1e-5 * g.numel() ** 0.5)
    return b


def _errors(got, ref):
    e = {k: (got[k] - ref[k]).abs().max().item() for k in ("loss", "user_emb", "item_emb", "logits")}
    for k, g in ref["grads"].items():
        e[k] = (got["grads"][k] - g).norm().item()
    return e


def _check(test, got, ref, bounds, **info):
    err = _errors(got, ref)
    rows = sorted(((err[k] / bounds[k], k, err[k], bounds[k]) for k in err), reverse=True)
    _report(test=test, **info, worst=[(k, e, b) for _, k, e, b in rows[:6]],
            forward={k: (err[k], bounds[k]) for k in ("loss", "user_emb", "item_emb", "logits")})
    bad = [(k, e, b) for r, k, e, b in rows if r > 1.0]
    assert not bad, bad[:6]
    return rows


E2E = [("train_c1.pt", 0.1, True), ("train_c1.pt", 0.1, False), ("train_l200.pt", 0.1, True),
       ("train_l200.pt", 0.1, False),
       ("train_c1.pt", 0.25, True)]      # user sites follow cfg.dropout, the item site stays at 0.1


@gpu
@pytest.mark.parametrize("name,dropout,prune", E2E)
def test_dropout_step_matches_oracle_with_engine_masks(name, dropout, prune):
    """Forward + backward of one dropout training step (the counter of the fourth step) against the fp64 oracle given the masks the
    engine's kernels draw: loss, embeddings, logits and every parameter gradient. The pruned last layer draws its
    out_proj / linear1 / linear2 masks at the compact rows, the full schedule at the token rows: each path is
    checked with its own masks."""
    auto, cfg, sd, batch = _fixture(name, dropout)
    ctr = R.counter_after(3)
    got = _engine_step(cfg, sd, batch, ctr, prune=prune)
    ref = _oracle(cfg, sd, batch, R.engine_masks(cfg, batch, ctr, prune_last_layer=prune))
    _check("dropout_step", got, ref, _bounds(auto, ref), fixture=name, dropout=dropout, prune=prune)
    assert got["grads"]["user_tower.item_embedding.weight"][0].abs().max().item() == 0.0


@gpu
def test_dropout_step_seq512_matches_oracle():
    """L = 512 (four attention tiles, the per-item backward) at B = 8, bounds of
    test_engine.test_seq512_training_step_matches_oracle: 8 sequences give the bf16 noise no averaging."""
    from mrm_b200 import synthetic
    cfg = synthetic.TwoTowerConfig(vocab_size=3001, max_seq_len=512, dropout=0.1)
    sd = synthetic.make_state_dict(cfg, seed=12)
    batch = synthetic.make_batch(cfg, 8, seed=13)
    batch["history_ids"][0, :] = torch.randint(1, 3001, (512,), generator=torch.Generator().manual_seed(14))
    batch["history_mask"][0, :] = 1
    ctr = R.counter_after(5)
    got = _engine_step(cfg, sd, batch, ctr, prune=True)
    ref = _oracle(cfg, sd, batch, R.engine_masks(cfg, batch, ctr))
    bounds = {"loss": 2e-2, "user_emb": 1e-2, "item_emb": 1e-2, "logits": 1e-2 / cfg.temperature}
    for k, g in ref["grads"].items():
        bounds[k] = 0.15 * g.norm().item() + 5e-5 * g.numel() ** 0.5
    _check("dropout_step_seq512", got, ref, bounds)


@gpu
def test_c2_dropout_step_matches_fp64_oracle():
    """The benchmarked c2 step (B = 256, L = 200, V = 100,001, dropout 0.1) from the seeded start, one step, against
    the fp64 oracle with the engine's masks; tolerance anchors of tests/golden/anchor_c2.pt (measured at dropout 0)."""
    from mrm_b200 import synthetic
    cfg = synthetic.TwoTowerConfig(vocab_size=100_001, max_seq_len=200, dropout=0.1)
    sd = synthetic.make_state_dict(cfg, seed=0)
    batch = synthetic.make_c2_parity_batch(cfg, 256)
    auto = torch.load(os.path.join(GOLDEN, "anchor_c2.pt"), weights_only=False)["bf16_autocast_err"]
    got = _engine_step(cfg, sd, batch, counter=0, prune=True)
    torch.set_num_threads(os.cpu_count() or 1)
    ref = _oracle(cfg, sd, batch, R.engine_masks(cfg, batch, 0))
    bounds = _bounds(auto, ref)
    err = _errors(got, ref)
    _report(test="c2_dropout_step_all_grads", grads={k: (err[k], bounds[k]) for k in ref["grads"]})
    _check("c2_dropout_step", got, ref, bounds)


@gpu
def test_cuda_graph_replay_reads_the_dropout_counter():
    """TrainStepRunner: step 1 eager, step 2 captured and replayed, step 3 replayed. Each step's loss and embeddings
    equal the oracle's at the counter of that step (0, then advanced by every optimizer step) on the
    oracle-AdamW-updated parameters: the graph reads the counter from the device, not a value fixed at capture."""
    from oracle import two_tower_oracle as oracle
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import TrainStepRunner
    auto, cfg, sd, batch = _fixture("train_c1.pt", 0.1)
    B, L = batch["history_ids"].shape
    lr = 1e-4
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(sd)
    runner = TrainStepRunner(eng, B, L, lr=lr, use_graph=True)
    runner.load_batch({k: v.cuda() for k, v in batch.items()})
    p = {k: (v.double() if v.is_floating_point() else v.clone()) for k, v in sd.items()}
    m = {k: torch.zeros_like(v) for k, v in p.items() if v.is_floating_point()}
    v2 = {k: torch.zeros_like(v) for k, v in p.items() if v.is_floating_point()}
    for t in range(3):
        ctr = int(eng.seed_dev.item()) % (1 << 64)
        assert ctr == R.counter_after(t)
        loss = runner.step_resident().item()
        ws = eng.workspace(B, L)
        got = dict(loss=torch.tensor(loss, dtype=torch.float64), user_emb=ws["un"].cpu().double(),
                   item_emb=ws["in"].cpu().double())
        ref = _oracle(cfg, p, batch, R.engine_masks(cfg, batch, ctr))
        bounds = _bounds(auto, ref)
        err = {k: (got[k] - ref[k]).abs().max().item() for k in ("loss", "user_emb", "item_emb")}
        _report(test="graph_replay_counter", step=t, err=err)
        assert all(err[k] <= bounds[k] for k in err), (t, err)
        for k, g in ref["grads"].items():
            p[k], m[k], v2[k] = oracle.adamw_step(p[k], g, m[k], v2[k], t + 1, lr=lr)
    assert int(eng.seed_dev.item()) % (1 << 64) == R.counter_after(3)


# ----------------------------------------------------------------------------------------------------------------
# the end-to-end tolerance sees a wrong mask at every site (CPU)
# ----------------------------------------------------------------------------------------------------------------
def test_the_end_to_end_tolerance_sees_a_wrong_mask_at_every_site():
    """For each dropout site in turn the mask is replaced by an independent draw, and for two plausible bookkeeping
    mistakes (the pruned layer's GEMM masks at token rows instead of compact rows; the previous step's counter) the
    masks are built the wrong way: the oracle's result must then move at least twice the bound on some quantity the
    end-to-end test compares. The counter mistake is also checked on the loss and embeddings alone, the quantities
    the CUDA-graph test compares."""
    torch.set_num_threads(os.cpu_count() or 1)
    auto, cfg, sd, batch = _fixture("train_c1.pt", 0.1)
    masks = R.engine_masks(cfg, batch, R.counter_after(3))
    ref = _oracle(cfg, sd, batch, masks)
    bounds = _bounds(auto, ref)
    mutations = {k: R.redraw(masks, k) for k in masks}
    mutations["pruned layer at token rows"] = R.engine_masks(cfg, batch, R.counter_after(3), prune_last_layer=False)
    mutations["previous counter"] = R.engine_masks(cfg, batch, R.counter_after(2))
    weak = {}
    for name, mm in mutations.items():
        err = _errors(_oracle(cfg, sd, batch, mm), ref)
        score = {k: err[k] / bounds[k] for k in err}
        top = max(score, key=score.get)
        if score[top] < 2.0:
            weak[name] = (top, score[top])
        if name == "previous counter":
            assert max(score[k] for k in ("loss", "user_emb", "item_emb")) >= 2.0, score
    assert len(mutations) == 1 + 4 * cfg.num_layers + 1 + 2
    assert not weak, weak
