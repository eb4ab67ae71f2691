"""fp64 reference of the attention kernels, with a per-element error bound and an RMS error model.

The reference takes the kernels' own bf16 inputs. A product of two bf16 values is exact in fp64 and a
64-term sum of them loses nothing a bf16 result could show, so the reference is exact up to fp64
rounding. It runs on batched (item, row, 64) tensors, one item per (sequence, head) or per single
query, on whatever device the inputs live on; query row r of item n sees keys j <= qpos[n, r]
(the causal predicate for full sequences, ``last`` for the single-query kernels, ``pos`` for the
session kernel). An optional scaled dropout mask multiplies the probabilities (tests/_dropout_ref).

Notation: s = scale Q K^T (scale = 1/8), p = softmax(s), P~ = p * mask, O = P~ V, lse = log sum exp s;
backward G = dO V^T, Delta_i = dO_i . ctx_i on the bf16 ctx the forward STORED (as the kernels form it),
dS = p (mask G - Delta) scale, dQ = dS K, dK = dS^T Q, dV = P~^T dO. u = 2^-8 is the bf16 unit
roundoff, e = 2^-24 the fp32 one.

What the kernels round (tt_attention.cu; tt_lastrow.cu and tt_session.cu keep P and dS in fp32):
  * S is an fp32 sum of 64 exact products: |error| <= 64 e scale sum_d |Q_id K_jd|. With the fp32
    exponent arithmetic (S c1 - m c1, ex2.approx) every probability carries a relative error
        eps_ij = e (64 scale sum_d |Q_id K_jd| + 4 (|s_ij| + max_j |s_ij|)) + 2^-21.
    A common factor of a row cancels in the normalisation, so O moves by sum_j P~_ij d_ij (V_jd - O_id)
    for relative errors d_ij of the probabilities, which is at most (P~ eps) |V| + |O| (p eps) 1.
  * P~ (the unnormalised P, dropout applied) is rounded to bf16 before the PV product: u sum_j P~_ij |V_jd|.
  * The fp32 PV accumulation and the row sum l over L terms: (L e) sum_j P~_ij |V_jd| and (L e) |O_id|.
  * ctx = O / l is rounded to bf16: u |O_id|.
  Forward bound per (i, d):
        (u + L e) sum_j P~_ij |V_jd| + (u + L e) |O_id| + (P~ eps |V|)_id + |O_id| (p eps 1)_i
  (the first u only where P is rounded). lse = m scale + log l: (p eps 1)_i + L e + 2^-22 (ex2 in l)
  + 2^-20 (the MUFU log) + 2^-23 |lse_i|.
  Backward: the recomputed probability carries eta_ij = eps_ij + (lse bound)_i (the kernel subtracts its
  own fp32 lse). G and Delta are fp32 sums of 64 exact products (g = 64 e). Per element of dS
        |d dS_ij| <= |dS_ij| (u + eta_ij) + p_ij scale (mask_ij g sum_d|dO_id V_jd| + g sum_d |dO_id ctx_id|)
  with u for the bf16 rounding of dS, and |d P~_ij| <= P~_ij (u + eta_ij) for the bf16 Pd. Then
        dQ: (|d dS| |K|) + (L e)(|dS| |K|) + u |dQ|,   dK: (|d dS|^T |Q|) + (L e)(|dS|^T |Q|) + u |dK|,
        dV: (|d P~|^T |dO|) + (L e)(P~^T |dO|) + u |dV|.
  attn_bwd_kernel (256 < L <= 512) rounds P to bf16 before forming dS from it: 2u on dS there.
  Underflow: a probability below 2^-126 of the row maximum may flush to 0 (ex2.approx.ftz) and a result
  below 2^-126 may lose its bits in fp32 / bf16 subnormals, so each probability and dS carries an absolute
  TINY = 2^-126 (times the factor it multiplies) and each output TINY more: nothing above ~1e-37 moves.
  Every bound is a product of absolute values in fp64. It is NOT compared with |reference|: prefix
  means cancel, and for q = 0 at L = 4096 a correct bound is about a fifth of the median |ctx|.

RMS model: each rounding above is an independent error of variance at most u^2 / 3 times the square of
the rounded value (a bf16 value in [2^k, 2^k+1) has a spacing of 2u 2^k, so a uniform rounding error
has variance (2u 2^k)^2 / 12 <= u^2 x^2 / 3). Per output element
        var(O_id)  = (u^2/3) (sum_j (P~_ij V_jd)^2 + O_id^2),
        var(dQ_id) = (u^2/3) (sum_j (dS_ij K_jd)^2 + dQ_id^2), likewise dK (dS^T, Q) and dV (P~^T, dO),
without the sum where P / dS stay fp32, with it twice for dQ / dK where dS is rounded twice. dQ / dK also
carry the fp32 roundings of G and Delta, var(dS_ij) = (p_ij scale)^2 (64 e^2 / 3) ((mask G~)^2 + Delta~^2)
with G~, Delta~ the sums of absolute products: they matter only where G - Delta cancels. Elements whose
modelled deviation is below 2^-100 (exact results, the underflow range) are left out of the RMS sums and
held to the worst-case bound alone. The score and accumulation errors are orders smaller and left
out. ``rms_ratio`` is sqrt(sum err^2 / sum var) per block of ``BLOCK`` rows of one item; correct
rounding lands near 0.6 (the mantissa spread makes the average variance u^2 x^2 / 6), a 2^-6 error in
Delta near 2 and one in the row sum near 5.

Every test uses the same constants: the error may reach KAPPA times the worst-case bound, and the
largest block RMS ratio must lie in [RMS_MIN, RMS_MAX]. RMS_MIN catches a model that overstates the
rounding tenfold as surely as RMS_MAX catches a wrong kernel.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

U = 2.0 ** -8
E32 = 2.0 ** -24
SCALE = 0.125
KAPPA = 2.0
RMS_MAX = 1.5
RMS_MIN = 0.1
BLOCK = 128
_G = 64 * E32
TINY = 2.0 ** -126    # fp32 underflow (ex2.approx.ftz flushes below it) and the bf16 subnormal range
_CHUNK = 1 << 25      # fp64 elements of one (item, query, key) tensor processed at a time


def causal_qpos(n: int, L: int, device=None) -> torch.Tensor:
    """qpos of full causal sequences: row i sees keys 0..i."""
    return torch.arange(L, device=device).expand(n, L)


def _chunks(n: int, lq: int, lk: int):
    step = max(1, _CHUNK // max(1, lq * lk))
    for a in range(0, n, step):
        yield slice(a, min(n, a + step))


def forward(q, k, v, qpos, drop: Optional[torch.Tensor] = None, rounded: bool = True) -> Dict[str, torch.Tensor]:
    """q (N, Lq, 64), k / v (N, Lk, 64), qpos (N, Lq), drop (N, Lq, Lk) scaled mask or None.
    Returns ctx, lse, their worst-case bounds ctx_bound / lse_bound and the model variance ctx_var."""
    out = {n: [] for n in ("ctx", "lse", "ctx_bound", "lse_bound", "ctx_var", "p")}
    for sl in _chunks(q.shape[0], q.shape[1], k.shape[1]):
        r = _forward(q[sl].double(), k[sl].double(), v[sl].double(), qpos[sl],
                     None if drop is None else drop[sl].double(), rounded)
        for n in out:
            out[n].append(r[n])
    return {n: torch.cat(t) for n, t in out.items()}


def _scores(q, k, qpos):
    Lk = k.shape[1]
    vis = torch.arange(Lk, device=q.device)[None, None, :] <= qpos[..., None]
    s = (q @ k.transpose(1, 2)) * SCALE
    s = s.masked_fill(~vis, -math.inf)
    mabs = s.abs().masked_fill(~vis, 0).amax(-1, keepdim=True)
    eps = E32 * (64 * SCALE * (q.abs() @ k.abs().transpose(1, 2)) + 4 * (s.abs().masked_fill(~vis, 0) + mabs)) + 2.0 ** -21
    return s, vis, eps


def _forward(q, k, v, qpos, drop, rounded):
    Lk = k.shape[1]
    s, vis, eps = _scores(q, k, qpos)
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse[..., None]).masked_fill(~vis, 0)
    pt = p if drop is None else p * drop
    o = pt @ v
    acc = Lk * E32
    pe = pt * eps
    ctx_bound = ((U if rounded else 0.0) + acc) * (pt @ v.abs()) + (U + acc) * o.abs() + pe @ v.abs() \
        + o.abs() * (p * eps).sum(-1, keepdim=True) + TINY * ((vis.double() if drop is None else vis * drop) @ v.abs() + 1)
    lse_bound = (p * eps).sum(-1) + acc + 2.0 ** -22 + 2.0 ** -20 + 2.0 ** -23 * lse.abs()
    ctx_var = (U * U / 3) * (((pt * pt) @ (v * v) if rounded else 0.0) + o * o)
    return {"ctx": o, "lse": lse, "ctx_bound": ctx_bound, "lse_bound": lse_bound, "ctx_var": ctx_var, "p": p}


def backward(q, k, v, qpos, do, ctx, drop: Optional[torch.Tensor] = None, rounded: bool = True,
             parked_p: bool = False) -> Dict[str, torch.Tensor]:
    """Gradients of the forward above for the output gradient ``do`` (N, Lq, 64), with Delta formed on
    ``ctx`` (the bf16 ctx the kernel stored). ``parked_p``: P itself is rounded to bf16 before dS is formed
    from it (attn_bwd_kernel, 256 < L <= 512, keeps P in the dS tile while dP takes the TMEM of S), a second
    rounding of every dS. Returns dq, dk, dv, their bounds *_bound and variances *_var."""
    names = ("dq", "dk", "dv", "dq_bound", "dk_bound", "dv_bound", "dq_var", "dk_var", "dv_var")
    out = {n: [] for n in names}
    for sl in _chunks(q.shape[0], q.shape[1], k.shape[1]):
        r = _backward(q[sl].double(), k[sl].double(), v[sl].double(), qpos[sl], do[sl].double(), ctx[sl].double(),
                      None if drop is None else drop[sl].double(), rounded, parked_p)
        for n in out:
            out[n].append(r[n])
    return {n: torch.cat(t) for n, t in out.items()}


def _backward(q, k, v, qpos, do, ctx, drop, rounded, parked_p):
    Lk = k.shape[1]
    s, vis, eps = _scores(q, k, qpos)
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse[..., None]).masked_fill(~vis, 0)
    lse_bound = (p * eps).sum(-1) + Lk * E32 + 2.0 ** -22 + 2.0 ** -20 + 2.0 ** -23 * lse.abs()
    m = torch.ones_like(p) if drop is None else drop
    pt = p * m
    g = do @ v.transpose(1, 2)
    delta = (do * ctx).sum(-1, keepdim=True)
    ds = p * (m * g - delta) * SCALE
    dq, dk, dv = ds @ k, ds.transpose(1, 2) @ q, pt.transpose(1, 2) @ do
    r = U if rounded else 0.0
    acc = Lk * E32
    eta = eps + lse_bound[..., None]
    nds = 2 if parked_p else 1                      # bf16 roundings every dS carries
    dds = ds.abs() * (nds * r + eta) + p * SCALE * _G * (m * (do.abs() @ v.abs().transpose(1, 2))
                                                         + (do.abs() * ctx.abs()).sum(-1, keepdim=True)) \
        + TINY * vis * (1 + SCALE * (m * g.abs() + delta.abs()))
    dpt = pt * (r + eta) + TINY * vis * m
    out = {"dq": dq, "dk": dk, "dv": dv}
    out["dq_bound"] = dds @ k.abs() + acc * (ds.abs() @ k.abs()) + U * dq.abs() + TINY
    out["dk_bound"] = dds.transpose(1, 2) @ q.abs() + acc * (ds.abs().transpose(1, 2) @ q.abs()) + U * dk.abs() + TINY
    out["dv_bound"] = dpt.transpose(1, 2) @ do.abs() + acc * (pt.transpose(1, 2) @ do.abs()) + U * dv.abs() + TINY
    c = U * U / 3
    ds2 = nds * ds * ds
    # fp32 G and Delta: 64 roundings each, which matter where G - Delta cancels (a nearly one-hot row)
    vds = (p * SCALE) ** 2 * (64 * E32 * E32 / 3) * ((m * (do.abs() @ v.abs().transpose(1, 2))) ** 2
                                                     + (do.abs() * ctx.abs()).sum(-1, keepdim=True) ** 2)
    out["dq_var"] = c * ((ds2 @ (k * k) if rounded else 0.0) + dq * dq) + vds @ (k * k)
    out["dk_var"] = c * ((ds2.transpose(1, 2) @ (q * q) if rounded else 0.0) + dk * dk) + vds.transpose(1, 2) @ (q * q)
    out["dv_var"] = c * (((pt * pt).transpose(1, 2) @ (do * do) if rounded else 0.0) + dv * dv)
    return out


def worst_ratio(got, ref, bound) -> float:
    """max |got - ref| / bound (0 where both the error and the bound are 0; inf where only the bound is)."""
    err = (got.double() - ref).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return r.max().item()


def rms_ratio(got, ref, var, rows=None) -> float:
    """Largest sqrt(sum err^2 / sum var) over blocks of BLOCK rows of each item (all items together when an item
    has fewer rows); got / ref / var (N, R, 64).
    ``rows`` (N, R) bool restricts the sums to the rows it marks."""
    err2 = (got.double() - ref) ** 2
    var = var.clone()
    tiny = var < 2.0 ** -200
    err2[tiny], var[tiny] = 0.0, 0.0
    if rows is not None:
        err2 = err2 * rows[..., None]
        var = var * rows[..., None]
    R = err2.shape[1]
    e, w = err2.sum(-1), var.sum(-1)
    if R < BLOCK:
        # the roundings of one row are shared by its 64 columns: pool short items so that a block has many rows
        e, w = e.sum().view(1), w.sum().view(1)
    else:
        # blocks of BLOCK rows, the last one taking the remainder
        blk = (torch.arange(R, device=e.device) // BLOCK).clamp(max=R // BLOCK - 1)
        e = torch.zeros(e.shape[0], R // BLOCK, dtype=e.dtype, device=e.device).index_add_(1, blk, e)
        w = torch.zeros(w.shape[0], R // BLOCK, dtype=w.dtype, device=w.device).index_add_(1, blk, w)
    live = w > 0
    return torch.sqrt(e[live] / w[live]).max().item() if live.any() else 0.0


class Ratios:
    """Collects the worst-case and RMS ratios of one test, prints them, and asserts the file's limits."""

    def __init__(self, name: str):
        self.name, self.worst, self.rms = name, {}, {}

    def add(self, what: str, got, ref, bound, var=None, rows=None):
        self.worst[what] = max(self.worst.get(what, 0.0), worst_ratio(got, ref, bound))
        if var is not None:
            self.rms[what] = max(self.rms.get(what, 0.0), rms_ratio(got, ref, var, rows))

    def check(self, floor: bool = True):
        w = max(self.worst.values())
        r = max(self.rms.values()) if self.rms else 0.0
        detail = " ".join(f"{k}={self.worst[k]:.3f}/{self.rms.get(k, float('nan')):.3f}" for k in self.worst)
        print(f"[{self.name}] worst-case ratio {w:.3f} (limit {KAPPA}), RMS ratio {r:.3f} "
              f"(limits {RMS_MIN}..{RMS_MAX}); {detail}")
        bad = {k: v for k, v in self.worst.items() if not v <= KAPPA}
        assert not bad, f"{self.name}: error beyond {KAPPA} x the worst-case bound: {bad}"
        bad = {k: v for k, v in self.rms.items() if not v <= RMS_MAX}
        assert not bad, f"{self.name}: RMS error beyond {RMS_MAX} x the rounding model: {bad}"
        if floor:
            assert r >= RMS_MIN, f"{self.name}: RMS ratio {r} below {RMS_MIN}: the model overstates the rounding"


# ---------------------------------------------------------------------------------------------------------------------
# Input families. Every generator returns float tensors holding bf16 values (CPU, seeded): qkv (B*L, 3*H*64) and
# dctx (B*L, H*64); the tests call check_family on the reference probabilities for the property a family exists for.
# ---------------------------------------------------------------------------------------------------------------------
FAMILIES = ("random", "peaked", "rising", "falling", "uniform", "poisoned")
TILE = 128
POISON_K = 160.0      # added to dim 0 of a poisoned key; every query has Q[0] = POISON_Q: score + 40
POISON_Q = 2.0
POISON_V = 1024.0
POISON_DO = 32.0


def poisoned_items(B: int, H: int) -> torch.Tensor:
    """(B, H) bool: alternate sequences and alternate heads (a checkerboard), so every clean (sequence, head)
    has poisoned neighbours in both directions."""
    return (torch.arange(B)[:, None] + torch.arange(H)[None, :]) % 2 == 1


def poison_rows_(x, g):
    """Poison the rows of a (..., 3, 64) Q | K | V tensor in place: K[0] += POISON_K, V = +-POISON_V."""
    x[..., 1, 0] += POISON_K
    sign = torch.randint(0, 2, x[..., 2, :].shape, generator=g).float() * 2 - 1
    x[..., 2, :] = sign * POISON_V


def make_inputs(family: str, B: int, L: int, H: int, seed: int):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, L, 3, H, 64, generator=g)
    do = torch.randn(B, L, H, 64, generator=g)
    if family == "random":
        x *= 1.2
    elif family == "peaked":                       # scores of standard deviation 25: most rows nearly one-hot
        x[:, :, :2] *= 5.0
    elif family in ("rising", "falling"):
        # small noise, a shared direction in Q (dim 1) and a per-tile offset in K: 4 score units per 128-key tile
        x *= 0.25
        x[:, :, 0, :, 1] = 4.0
        t = (torch.arange(L) // TILE).float()
        x[:, :, 1, :, 1] = (8.0 if family == "rising" else -8.0) * t[None, :, None]
    elif family == "uniform":
        x[:, :, 0] = 0.0
    elif family == "poisoned":
        x *= 1.2
        x[:, :, 0, :, 0] = POISON_Q
        bad = poisoned_items(B, H)
        xp = x.permute(0, 3, 1, 2, 4)                  # (B, H, L, 3, 64) view
        xb = xp[bad]
        poison_rows_(xb, g)
        xp[bad] = xb
        dp = do.permute(0, 2, 1, 3)
        dp[bad] = dp[bad] * POISON_DO
    else:
        raise ValueError(family)
    qkv = x.reshape(B * L, 3 * H * 64).bfloat16().float()
    return qkv, do.reshape(B * L, H * 64).bfloat16().float()


def split_heads(qkv, B: int, L: int, H: int):
    """qkv (B*L, 3*H*64) -> q, k, v as (B*H, L, 64), item = b*H + h."""
    x = qkv.view(B, L, 3, H, 64).permute(2, 0, 3, 1, 4).reshape(3, B * H, L, 64)
    return x[0], x[1], x[2]


def heads(t, B: int, L: int, H: int):
    """(B*L, H*64) -> (B*H, L, 64)."""
    return t.view(B, L, H, 64).permute(0, 2, 1, 3).reshape(B * H, L, 64)


def check_family(family: str, q, k, v, qpos, p, ctx, B: int, H: int):
    """Assert the property ``family`` exists for, on the reference probabilities p (N, Lq, Lk)."""
    L = k.shape[1]
    vis = torch.arange(L, device=p.device)[None, None, :] <= qpos[..., None]
    if family == "peaked":
        top = p.amax(-1)[qpos >= 1]
        if top.numel() == 0:
            return
        frac = (top > 0.9).double().mean().item()
        assert frac >= 0.4, f"peaked: only {frac:.2f} of rows have a top weight above 0.9"
    elif family in ("rising", "falling"):
        if L <= TILE:
            return
        s = (q.double() @ k.double().transpose(1, 2)).masked_fill(~vis, math.nan)
        nt = (L + TILE - 1) // TILE
        s = torch.nn.functional.pad(s, (0, nt * TILE - L), value=math.nan).view(*s.shape[:2], nt, TILE)
        tmax = torch.where(torch.isnan(s), torch.full_like(s, -math.inf), s).amax(-1)   # (N, Lq, nt)
        d = tmax[..., 1:] - tmax[..., :-1]
        seen = torch.isfinite(tmax[..., 1:])
        if family == "rising":
            assert (d[seen] > 0).all(), "rising: a per-tile row maximum does not increase"
        else:
            assert (d[seen] < 0).all(), "falling: a per-tile row maximum does not decrease"
    elif family == "uniform":
        n = qpos.double() + 1
        pref = torch.cumsum(v.double(), 1)[:, : qpos.shape[1]] / n[..., None]
        assert torch.allclose(ctx, pref, rtol=0, atol=1e-9), "uniform: ctx is not the prefix mean of V"
    elif family == "poisoned":
        bad = poisoned_items(B, H).reshape(-1).to(p.device)
        good = (~bad).nonzero().flatten()
        if not bad.any() or good.numel() == 0:
            return
        # a clean item's queries against its poisoned neighbour's keys score far above its own row maximum
        step = H if B > 1 else 1
        nb = torch.where(good + step < B * H, good + step, good - step)
        own = (q[good].double() @ k[good].double().transpose(1, 2)).masked_fill(~vis[good], -math.inf).amax(-1)
        cross = (q[good].double() @ k[nb].double().transpose(1, 2)).amin(-1)
        assert bad[nb].all() and ((cross - own) * SCALE > 10).all(), "poisoned: a neighbour's keys would not stand out"
