"""tcgen05 causal attention against an fp32 torch restatement on the same bf16 inputs.

Tolerances: P is rounded to bf16 before P@V (relative 2^-9 per term) and the output is bf16,
so abs error <= 2e-2 on O(1) outputs; dq/dk/dv likewise (bf16 dS, bf16 outputs).
"""
import math

import pytest
import torch

import _dropout_ref as R

pytestmark = pytest.mark.gpu


def _ref_attention(qkv, B, L, H, dctx=None, drop_mask=None):
    """fp32 causal attention; ``drop_mask`` (B, H, L, L), if given, multiplies the probabilities."""
    D = H * 64
    x = qkv.float().view(B, L, 3, H, 64).requires_grad_(dctx is not None)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) / 8.0
    mask = torch.triu(torch.ones(L, L, dtype=torch.bool, device=qkv.device), 1)
    s = s.masked_fill(mask, float("-inf"))
    lse = torch.logsumexp(s, dim=-1)                         # (B,H,L)
    prob = torch.softmax(s, dim=-1)
    if drop_mask is not None:
        prob = prob * drop_mask
    o = (prob @ v).transpose(1, 2).reshape(B * L, D)
    if dctx is None:
        return o, lse, None
    o.backward(dctx.float())
    return o.detach(), lse.detach(), x.grad.reshape(B * L, 3 * D)


@pytest.mark.parametrize("B,L,H", [(2, 128, 4), (3, 200, 4), (2, 50, 4), (1, 256, 2), (2, 384, 4), (1, 512, 4)])
def test_attn_fwd(B, L, H):
    from mrm_b200 import ops
    g = torch.Generator().manual_seed(L)
    qkv = (torch.randn(B * L, 3 * H * 64, generator=g) * 1.5).cuda().bfloat16()
    ctx = torch.full((B * L, H * 64), float("nan"), device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H)
    torch.cuda.synchronize()
    o, lse_ref, _ = _ref_attention(qkv, B, L, H)
    err = (ctx.float() - o).abs().max().item()
    lerr = (lse - lse_ref).abs().max().item()
    assert err <= 3e-2, f"ctx err {err}"
    assert lerr <= 2e-3, f"lse err {lerr}"


@pytest.mark.parametrize("B,L,H", [(2, 128, 4), (3, 200, 4), (2, 50, 4), (2, 256, 4), (2, 300, 4), (1, 512, 4)])
def test_attn_bwd(B, L, H):
    from mrm_b200 import ops
    g = torch.Generator().manual_seed(100 + L)
    qkv = (torch.randn(B * L, 3 * H * 64, generator=g) * 1.2).cuda().bfloat16()
    dctx = torch.randn(B * L, H * 64, generator=g).cuda().bfloat16()
    ctx = torch.empty((B * L, H * 64), device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H)
    dqkv = torch.full((B * L, 3 * H * 64), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attn_bwd(qkv, ctx, dctx, lse, dqkv, B, L, H)
    torch.cuda.synchronize()
    _, _, dref = _ref_attention(qkv, B, L, H, dctx)
    D = H * 64
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        a, r = dqkv[:, sl].float(), dref[:, sl]
        err = (a - r).abs().max().item()
        scale = r.abs().max().item()
        assert err <= 3e-2 * max(scale, 1.0), f"{name}: err {err} scale {scale}"


def test_attn_dropout_statistics():
    """Dropout on the probabilities: deterministic per seed, unbiased on average."""
    from mrm_b200 import ops
    B, L, H = 4, 128, 4
    g = torch.Generator().manual_seed(7)
    qkv = (torch.randn(B * L, 3 * H * 64, generator=g) * 0.3).cuda().bfloat16()
    base = torch.empty((B * L, H * 64), device="cuda", dtype=torch.bfloat16)
    ops.attn_fwd(qkv, base, None, B, L, H)
    acc = torch.zeros((B * L, H * 64), device="cuda")
    n = 24
    outs = []
    for s in range(n):
        o = torch.empty_like(base)
        ops.attn_fwd(qkv, o, None, B, L, H, drop_p=0.2, drop_seed=1000 + s, drop_site=3)
        acc += o.float()
        outs.append(o)
    o2 = torch.empty_like(base)
    ops.attn_fwd(qkv, o2, None, B, L, H, drop_p=0.2, drop_seed=1000, drop_site=3)
    torch.cuda.synchronize()
    assert torch.equal(o2, outs[0])
    assert not torch.equal(outs[0], outs[1])
    # rows deep in the sequence average many keys: the mean over seeds approaches the no-dropout output
    deep = slice(L // 2, L)
    diff = (acc / n - base.float()).view(B, L, -1)[:, deep].abs().mean().item()
    ref = base.float().view(B, L, -1)[:, deep].abs().mean().item()
    assert diff <= 0.25 * ref, (diff, ref)


# More (sequence, head) items than SMs (a persistent CTA walks several items) and fewer; with and without dropout.
REPEAT_SHAPES = [(160, 200, 4, 0.1), (150, 50, 4, 0.1), (40, 256, 2, 0.2), (37, 129, 4, 0.1), (3, 200, 4, 0.0),
                 (2, 128, 4, 0.0), (64, 384, 4, 0.1), (40, 512, 4, 0.1), (48, 300, 4, 0.0)]


def _drop_mask(B, L, H, drop, seed, site):
    """The kernels' dropout mask of the probabilities (index ((b*H + h)*L + q)*L + k), scaled, or None."""
    if drop == 0.0:
        return None
    return torch.from_numpy(R.scaled_mask(seed, site, (B, H, L, L), drop)).cuda()


@pytest.mark.parametrize("B,L,H,drop", REPEAT_SHAPES)
def test_attn_fwd_repeated_launches_match_reference(B, L, H, drop):
    """Two forward launches give the very same bits (the second must not depend on state the first left behind),
    finite, and equal to fp32 attention with the kernels' dropout mask."""
    from mrm_b200 import ops
    g = torch.Generator().manual_seed(11 * L + B)
    qkv = (torch.randn(B * L, 3 * H * 64, generator=g) * 1.2).cuda().bfloat16()
    out = []
    for _ in range(2):
        ctx = torch.full((B * L, H * 64), float("nan"), device="cuda", dtype=torch.bfloat16)
        lse = torch.full((B, H, L), float("nan"), device="cuda")
        ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=drop, drop_seed=11, drop_site=2)
        out.append((ctx, lse))
    torch.cuda.synchronize()
    (ctx, lse), (ctx2, lse2) = out
    assert torch.isfinite(ctx.float()).all() and torch.isfinite(lse).all()
    assert torch.equal(ctx, ctx2) and torch.equal(lse, lse2)
    o, lse_ref, _ = _ref_attention(qkv, B, L, H, drop_mask=_drop_mask(B, L, H, drop, 11, 2))
    tol = 4e-2 if drop > 0 else 3e-2
    err = (ctx.float() - o).abs().max().item()
    lerr = (lse - lse_ref).abs().max().item()
    assert err <= tol, f"ctx err {err}"
    assert lerr <= 2e-3, f"lse err {lerr}"


@pytest.mark.parametrize("B,L,H,drop", REPEAT_SHAPES)
def test_attn_bwd_repeated_launches_match_reference(B, L, H, drop):
    """Two backward launches give the very same bits (the second must not depend on state the first left behind),
    finite, and equal to fp32 autograd with the kernels' dropout mask."""
    from mrm_b200 import ops
    g = torch.Generator().manual_seed(7 * L + B)
    qkv = (torch.randn(B * L, 3 * H * 64, generator=g) * 1.2).cuda().bfloat16()
    dctx = torch.randn(B * L, H * 64, generator=g).cuda().bfloat16()
    ctx = torch.empty((B * L, H * 64), device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=drop, drop_seed=11, drop_site=2)
    out = []
    for _ in range(2):
        d = torch.full((B * L, 3 * H * 64), float("nan"), device="cuda", dtype=torch.bfloat16)
        ops.attn_bwd(qkv, ctx, dctx, lse, d, B, L, H, drop_p=drop, drop_seed=11, drop_site=2)
        out.append(d)
    torch.cuda.synchronize()
    dqkv, dqkv2 = out
    assert torch.isfinite(dqkv.float()).all()
    assert torch.equal(dqkv, dqkv2)
    _, _, dref = _ref_attention(qkv, B, L, H, dctx, drop_mask=_drop_mask(B, L, H, drop, 11, 2))
    tol = 4e-2 if drop > 0 else 3e-2
    D = H * 64
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        a, r = dqkv[:, sl].float(), dref[:, sl]
        err = (a - r).abs().max().item()
        scale = r.abs().max().item()
        assert err <= tol * max(scale, 1.0), f"{name}: err {err} scale {scale}"


@pytest.mark.parametrize("B,L,H", [(2, 200, 2), (2, 384, 2), (1, 512, 2), (2, 300, 4)])
def test_attn_bwd_uses_the_forward_dropout_mask(B, L, H):
    """The backward re-creates the forward's dropout mask from the hash. Here the mask is READ OUT of the forward kernel
    (one-hot V blocks turn ctx into the dropped probabilities themselves) and a torch backward with exactly that mask
    is the reference — for the persistent kernels (L <= 256) and for the tiled forward with the four-tile backward
    (256 < L <= 512), whose hash evaluations differ (one word per 4 / 2 / 1 keys depending on alignment)."""
    from mrm_b200 import ops
    p_drop, seed, site = 0.3, 4242, 5
    D = H * 64
    g = torch.Generator().manual_seed(7 * L + B)
    qkv = (torch.randn(B * L, 3 * D, generator=g) * 1.0).cuda().bfloat16()

    def probs(drop):
        """[B, H, L, L] probabilities as the kernel forms them (dropout applied when drop > 0), via one-hot V."""
        out = torch.zeros(B, H, L, L, device="cuda")
        x = qkv.clone().view(B, L, 3, H, 64)
        ctx = torch.empty(B * L, D, device="cuda", dtype=torch.bfloat16)
        for k0 in range(0, L, 64):
            x[:, :, 2] = 0
            n = min(64, L - k0)
            x[:, k0:k0 + n, 2, :, :n] = torch.eye(n, device="cuda", dtype=torch.bfloat16)[None, :, None, :]
            ops.attn_fwd(x.view(B * L, 3 * D), ctx, None, B, L, H, drop_p=drop, drop_seed=seed, drop_site=site)
            out[:, :, :, k0:k0 + n] = ctx.float().view(B, L, H, 64)[..., :n].permute(0, 2, 1, 3)
        return out

    P, Pd = probs(0.0), probs(p_drop)
    known = P > 1e-5          # bf16 keeps the relative precision of small probabilities; below this they do not matter
    keep = torch.where(known, Pd > 0.5 * P, torch.ones_like(known))
    frac = keep[known].float().mean().item()
    assert abs(frac - (1 - p_drop)) < 0.03, frac
    # the backward on the real V with the hash-made mask against torch with the read-out mask
    dctx = torch.randn(B * L, D, generator=g).cuda().bfloat16()
    ctx = torch.empty(B * L, D, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=p_drop, drop_seed=seed, drop_site=site)
    dqkv = torch.empty(B * L, 3 * D, device="cuda", dtype=torch.bfloat16)
    ops.attn_bwd(qkv, ctx, dctx, lse, dqkv, B, L, H, drop_p=p_drop, drop_seed=seed, drop_site=site)
    torch.cuda.synchronize()
    x = qkv.float().view(B, L, 3, H, 64).requires_grad_(True)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) / 8.0
    s = s.masked_fill(torch.triu(torch.ones(L, L, dtype=torch.bool, device="cuda"), 1), float("-inf"))
    o = ((torch.softmax(s, dim=-1) * keep / (1 - p_drop)) @ v).transpose(1, 2).reshape(B * L, D)
    assert (ctx.float() - o.detach()).abs().max().item() <= 4e-2
    o.backward(dctx.float())
    dref = x.grad.reshape(B * L, 3 * D)
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        a, r = dqkv[:, sl].float(), dref[:, sl]
        err = (a - r).abs().max().item()
        assert err <= 4e-2 * max(r.abs().max().item(), 1.0), f"{name}: err {err}"
