"""Every attention kernel against the fp64 oracle of tests/_attn_oracle.py, element by element.

Each GPU test checks the kernel's outputs against the oracle's worst-case bound (times KAPPA) and its RMS
rounding model, prints both ratios, and covers one dispatch edge or one input family meant to break a
kernel: nearly one-hot softmax rows, row maxima that climb or fall by 4 score units every 128-key tile,
q = 0, and neighbouring sequences / heads / stale keys poisoned so that any read across a boundary dominates
its softmax. The CPU tests at the top check the oracle itself.
"""
import numpy as np
import pytest
import torch

import _attn_oracle as A
import _dropout_ref as R

SEED, SITE = 0x5EED, 9


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the oracle against autograd, and against an emulation of the kernels' roundings
# ---------------------------------------------------------------------------------------------------------------------
def _emulate(q, k, v, do, drop=None, delta_scale=1.0, l_scale=1.0):
    """The tcgen05 kernels' arithmetic on (N, L, 64) bf16-valued fp32 tensors: fp32 scores and sums, the
    unnormalised P rounded to bf16, bf16 ctx, P recomputed from the fp32 lse, bf16 Pd and dS, bf16 outputs."""
    bf = lambda t: t.bfloat16().float()
    L = q.shape[1]
    c1 = float(np.float32(0.125 * 1.4426950408889634))
    mask = torch.triu(torch.ones(L, L, dtype=torch.bool), 1)
    s = (q @ k.transpose(1, 2)).masked_fill(mask, -float("inf"))
    m = s.amax(-1, keepdim=True)
    p = torch.exp2(s * c1 - m * c1)
    l = p.sum(-1, keepdim=True) * l_scale
    dm = torch.ones_like(p) if drop is None else drop.float()
    ctx = bf((bf(p * dm) @ v) / l)
    lse = (m * 0.125 + torch.log(l)).squeeze(-1)
    p2 = torch.exp2(s * c1 - lse[..., None] * float(np.float32(1.4426950408889634)))
    g = do @ v.transpose(1, 2)
    delta = (do * ctx).sum(-1, keepdim=True) * delta_scale
    ds = bf(p2 * (dm * g - delta) * 0.125)
    pd = bf(p2 * dm)
    return ctx, lse, bf(ds @ k), bf(ds.transpose(1, 2) @ q), bf(pd.transpose(1, 2) @ do)


def _cpu_inputs(N, L, seed, drop):
    g = torch.Generator().manual_seed(seed)
    q, k, v, do = (torch.randn(N, L, 64, generator=g).mul(1.2).bfloat16().float() for _ in range(4))
    dm = None
    if drop:
        dm = torch.from_numpy(R.scaled_mask(seed, SITE, (N, L, L), drop))
    return q, k, v, do, dm


def _emulated_ratios(L, drop, **mutation):
    q, k, v, do, dm = _cpu_inputs(2, L, 7 * L, drop)
    ctx, lse, dq, dk, dv = _emulate(q, k, v, do, dm, **mutation)
    qpos = A.causal_qpos(2, L)
    f = A.forward(q, k, v, qpos, dm)
    b = A.backward(q, k, v, qpos, do, ctx, dm)
    r = A.Ratios(f"emulated L={L} drop={drop} {mutation}")
    r.add("ctx", ctx, f["ctx"], f["ctx_bound"], f["ctx_var"])
    r.add("lse", lse, f["lse"], f["lse_bound"])
    for n, t in (("dq", dq), ("dk", dk), ("dv", dv)):
        r.add(n, t, b[n], b[n + "_bound"], b[n + "_var"])
    return r


@pytest.mark.parametrize("L,drop", [(1, 0.0), (5, 0.0), (37, 0.2), (130, 0.1)])
def test_oracle_gradients_equal_fp64_autograd(L, drop):
    q, k, v, do, dm = _cpu_inputs(3, L, L, drop)
    x = [t.double().requires_grad_(True) for t in (q, k, v)]
    s = (x[0] @ x[1].transpose(1, 2)) * A.SCALE
    s = s.masked_fill(torch.triu(torch.ones(L, L, dtype=torch.bool), 1), -float("inf"))
    p = torch.softmax(s, -1)
    o = (p if dm is None else p * dm.double()) @ x[2]
    lse = torch.logsumexp(s, -1)
    o.backward(do.double())
    qpos = A.causal_qpos(3, L)
    f = A.forward(q, k, v, qpos, dm)
    b = A.backward(q, k, v, qpos, do, o.detach(), dm)
    torch.testing.assert_close(f["ctx"], o.detach(), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(f["lse"], lse.detach(), rtol=1e-12, atol=1e-12)
    for n, t in zip(("dq", "dk", "dv"), x):
        torch.testing.assert_close(b[n], t.grad, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("L,drop", [(65, 0.0), (257, 0.1), (513, 0.0), (1024, 0.0)])
def test_emulated_kernel_rounding_stays_inside_both_tolerances(L, drop):
    r = _emulated_ratios(L, drop)
    r.check()


@pytest.mark.parametrize("L", [65, 300, 1024])
@pytest.mark.parametrize("mutation", [{"delta_scale": 1 + 2.0 ** -6}, {"l_scale": 1 + 2.0 ** -6}])
def test_emulated_error_of_2_to_the_minus_6_fails_the_rms_check(L, mutation):
    r = _emulated_ratios(L, 0.0, **mutation)
    with pytest.raises(AssertionError):
        r.check()
    assert max(r.rms.values()) > A.RMS_MAX


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _ops():
    from mrm_b200 import ops
    return ops


def _drop_mask(B, L, H, drop, first_item=0, n_items=None):
    """Scaled dropout mask (items, L, L) of the causal kernels for items first_item.. (index (item*L + i)*L + j)."""
    n = B * H - first_item if n_items is None else n_items
    if drop == 0.0:
        return None
    bits = R.keep_bits(SEED, SITE, n * L * L, drop, start=first_item * L * L)
    return torch.from_numpy(np.where(bits, R.drop_scale(drop), np.float32(0)).astype(np.float32).reshape(n, L, L)).cuda()


def _run_causal(qkv, do, B, L, H, drop):
    """Forward then backward of the causal kernels on bf16 copies; ctx / lse / dqkv start as NaN."""
    ops = _ops()
    D = H * 64
    x = qkv.cuda().bfloat16()
    ctx = torch.full((B * L, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    lse = torch.full((B, H, L), float("nan"), device="cuda")
    ops.attn_fwd(x, ctx, lse, B, L, H, drop_p=drop, drop_seed=SEED, drop_site=SITE)
    dqkv = torch.full((B * L, 3 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attn_bwd(x, ctx, do.cuda().bfloat16(), lse, dqkv, B, L, H, drop_p=drop, drop_seed=SEED, drop_site=SITE)
    torch.cuda.synchronize()
    return ctx.float(), lse, dqkv.float()


def _check_causal(name, family, qkv, do, B, L, H, drop, ctx, lse, dqkv, items=None, dm=None):
    """Oracle comparison of a causal forward + backward for the given items (default: all)."""
    N = B * H
    q, k, v = (t.cuda().double() for t in A.split_heads(qkv, B, L, H))
    dO = A.heads(do, B, L, H).cuda().double()
    ck = A.heads(ctx, B, L, H).double()
    lk = lse.view(N, L).double()
    dq, dk, dv = (A.heads(dqkv[:, i * H * 64:(i + 1) * H * 64], B, L, H).double() for i in range(3))
    if items is not None:
        q, k, v, dO, ck, lk, dq, dk, dv = (t[items] for t in (q, k, v, dO, ck, lk, dq, dk, dv))
    if dm is None and drop > 0:
        dm = _drop_mask(B, L, H, drop)
    qpos = A.causal_qpos(q.shape[0], L, "cuda")
    f = A.forward(q, k, v, qpos, dm)
    if family is not None:
        A.check_family(family, q, k, v, qpos, f["p"], f["ctx"], B, H)
    r = A.Ratios(name)
    r.add("ctx", ck, f["ctx"], f["ctx_bound"], f["ctx_var"])
    r.add("lse", lk, f["lse"], f["lse_bound"])
    b = A.backward(q, k, v, qpos, dO, ck, dm, parked_p=256 < L <= 512)
    for n, t in (("dq", dq), ("dk", dk), ("dv", dv)):
        r.add(n, t, b[n], b[n + "_bound"], b[n + "_var"])
    if L == 1:
        # a one-key softmax is exactly 1: ctx is V itself and the floor on the RMS ratio does not apply
        assert torch.equal(ck, v) or drop > 0
    r.check(floor=L > 1)
    return r


L_ALL = [1, 2, 3, 31, 64, 65, 127, 128, 129, 255, 256, 257, 300, 511, 512, 513, 1025, 2048, 4096]
CAUSAL_CASES = []
for _i, _L in enumerate(L_ALL):
    _H = (1, 3, 4)[_i % 3]
    for _f in (A.FAMILIES if _L < 4096 else ("random", "rising")):
        CAUSAL_CASES.append((_L, _H, _f, 0.0))
    if _L > 1:
        CAUSAL_CASES.append((_L, _H, "random", 0.1))
CAUSAL_CASES.append((300, 3, "rising", 0.1))
CAUSAL_CASES.append((1025, 1, "poisoned", 0.1))


@pytest.mark.gpu
@pytest.mark.parametrize("L,H,family,drop", CAUSAL_CASES)
def test_causal_attention_inside_the_fp64_bounds(L, H, family, drop):
    """Causal forward (ctx, lse) and backward (dq, dk, dv) at every dispatch edge of L, three sequences (ragged
    tail tiles between them whenever L % 128 != 0), against both tolerances."""
    B = 3
    qkv, do = A.make_inputs(family, B, L, H, seed=L * 31 + H)
    ctx, lse, dqkv = _run_causal(qkv, do, B, L, H, drop)
    _check_causal(f"causal L={L} H={H} {family} drop={drop}", family, qkv, do, B, L, H, drop, ctx, lse, dqkv)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [100, 256])
@pytest.mark.parametrize("extra", [None, -1, 0, 1, "2n+1"])
def test_persistent_kernels_over_every_grid_shape(L, extra):
    """The persistent kernels walk B*H items over min(B*H, SMs) CTAs: one item, one short of a full wave, a full wave,
    one item more (a CTA takes a second item) and two waves plus one. Dropout on, and checked for every item."""
    from mrm_b200._lib import lib
    sms = int(lib().tt_num_sms())
    n = 1 if extra is None else (2 * sms + 1 if extra == "2n+1" else sms + extra)
    B, H = n, 1
    qkv, do = A.make_inputs("random", B, L, H, seed=n + L)
    ctx, lse, dqkv = _run_causal(qkv, do, B, L, H, 0.1)
    _check_causal(f"persistent L={L} B*H={n} (SMs {sms})", "random", qkv, do, B, L, H, 0.1, ctx, lse, dqkv)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 65, 257, 513, 1000])
@pytest.mark.parametrize("family", ["random", "peaked"])
def test_forward_probabilities_are_exactly_causal(L, family):
    """The probabilities read out of the forward through one-hot V blocks (ctx column d = P[:, k0 + d]): exactly 0
    above the diagonal, inside the bound below it, and (random inputs) positive on and below the diagonal."""
    ops = _ops()
    B, H = 2, 3
    D = H * 64
    qkv, _ = A.make_inputs(family, B, L, H, seed=L + 5)
    q, k, v = (t.cuda().double() for t in A.split_heads(qkv, B, L, H))
    qpos = A.causal_qpos(B * H, L, "cuda")
    x = qkv.clone().view(B, L, 3, H, 64)
    ctx = torch.empty(B * L, D, device="cuda", dtype=torch.bfloat16)
    got = torch.zeros(B * H, L, L, device="cuda", dtype=torch.float64)
    r = A.Ratios(f"causal P read-out L={L} {family}")
    for k0 in range(0, L, 64):
        n = min(64, L - k0)
        x[:, :, 2] = 0
        x[:, k0:k0 + n, 2, :, :n] = torch.eye(n)[None, :, None, :]
        xv = x.view(B * L, 3 * D)
        ops.attn_fwd(xv.cuda().bfloat16(), ctx, None, B, L, H)
        torch.cuda.synchronize()
        ck = A.heads(ctx.float(), B, L, H).double()
        vb = A.split_heads(xv, B, L, H)[2].cuda().double()
        f = A.forward(q, k, vb, qpos)
        r.add("P", ck, f["ctx"], f["ctx_bound"], f["ctx_var"])
        got[:, :, k0:k0 + n] = ck[..., :n]
    above = torch.triu(torch.ones(L, L, dtype=torch.bool, device="cuda"), 1)
    assert (got[:, above] == 0).all(), "probability above the diagonal"
    if family == "random":
        assert (got[:, ~above] > 0).all(), "a visible key got probability 0"
    r.check(floor=L > 1)


def _lastq_inputs(family, L, lasts, H, seed):
    """B = len(lasts) sequences; every key after a sequence's ``last`` is poisoned, and q is the Q row ``last``."""
    B = len(lasts)
    qkv, do = A.make_inputs(family, B, L, H, seed)
    g = torch.Generator().manual_seed(seed + 1)
    x = qkv.view(B, L, 3, H, 64)
    x[:, :, 0, :, 0] = A.POISON_Q
    for b, last in enumerate(lasts):
        if last + 1 < L:
            A.poison_rows_(x[b, last + 1:].transpose(1, 2), g)      # (L', H, 3, 64)
    last_t = torch.tensor(lasts, dtype=torch.int32)
    qrow = x[torch.arange(B), last_t.long(), 0].reshape(B, H * 64)
    return qkv, qrow, do.view(B, L, H * 64)[:, 0].contiguous(), last_t


def _lastq_oracle(qkv, qrow, last_t, B, L, H, dm=None):
    _, k, v = (t.cuda().double() for t in A.split_heads(qkv, B, L, H))
    q1 = qrow.view(B * H, 1, 64).cuda().double()
    qpos = last_t.long().repeat_interleave(H).view(B * H, 1).cuda()
    return q1, k, v, qpos, A.forward(q1, k, v, qpos, dm, rounded=False)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [77, 512, 513, 1000, 2048, 4096])
@pytest.mark.parametrize("family", ["random", "peaked", "rising"])
def test_single_query_attention_inside_the_fp64_bounds(L, family):
    """attn_lastq_fwd / _bwd at both instantiations (L <= 512, L <= 4096) and the switch between them, for last on
    the warp and tile edges, with every key after last poisoned: dK / dV rows after last are exactly 0."""
    ops = _ops()
    H, D = 4, 256
    lasts = sorted({x for x in (0, 31, 32, 511, 512, L - 2, L - 1) if 0 <= x < L})
    B = len(lasts)
    qkv, qrow, dctx, last_t = _lastq_inputs(family, L, lasts, H, seed=L + 3)
    xq, xkv, li = qrow.cuda().bfloat16(), qkv.cuda().bfloat16(), last_t.cuda()
    ctx = torch.full((B, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    lse = torch.full((B, H), float("nan"), device="cuda")
    ops.attn_lastq_fwd(xq, xkv, li, ctx, lse, B, L, H)
    dq = torch.full((B, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    dqkv = torch.full((B * L, 3 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attn_lastq_bwd(xq, xkv, li, ctx, dctx.cuda().bfloat16(), lse, dq, dqkv, B, L, H)
    torch.cuda.synchronize()
    q1, k, v, qpos, f = _lastq_oracle(qkv, qrow, last_t, B, L, H)
    A.check_family(family, q1, k, v, qpos, f["p"], f["ctx"], B, H)
    r = A.Ratios(f"single query L={L} {family} last={lasts}")
    ck = ctx.float().view(B * H, 1, 64).double()
    r.add("ctx", ck, f["ctx"], f["ctx_bound"], f["ctx_var"])
    r.add("lse", lse.view(B * H, 1).double(), f["lse"], f["lse_bound"])
    dO = dctx.view(B * H, 1, 64).cuda().double()
    b = A.backward(q1, k, v, qpos, dO, ck, rounded=False)
    r.add("dq", dq.float().view(B * H, 1, 64).double(), b["dq"], b["dq_bound"], b["dq_var"])
    after = torch.arange(L, device="cuda")[None, :] > qpos
    for i, n in ((1, "dk"), (2, "dv")):
        t = A.heads(dqkv[:, i * D:(i + 1) * D].float(), B, L, H).double()
        assert (t[after] == 0).all(), f"{n}: rows after last are not 0"
        r.add(n, t, b[n], b[n + "_bound"], b[n + "_var"])
    r.check()


@pytest.mark.gpu
def test_single_query_dropout_above_2_to_the_32_matches_the_tiled_forward():
    """At L = 4096, B = 65, H = 4 the last sequence's element indices pass 2^32. Its dropout pattern read out of the
    single-query kernel (L <= 4096 instantiation) equals row ``last`` of the tiled forward and the 64-bit numpy
    mask, and the read-out probabilities are inside the bound."""
    ops = _ops()
    B, L, H, D, p = 65, 4096, 4, 256, 0.1
    g = torch.Generator().manual_seed(65)
    qkv = torch.randn(B * L, 3 * D, generator=g).bfloat16().float()
    last = L - 1
    last_t = torch.randint(0, L, (B,), generator=g, dtype=torch.int32)
    last_t[-1] = last
    b0 = B - 1
    assert (b0 * H) * L * L >= 1 << 32
    x = qkv.cuda().bfloat16().view(B, L, 3, H, 64)
    qrow = x[torch.arange(B), last_t.long(), 0].reshape(B, D).contiguous()
    ctx1 = torch.empty(B, D, device="cuda", dtype=torch.bfloat16)
    ctxf = torch.empty(B * L, D, device="cuda", dtype=torch.bfloat16)
    lq = torch.zeros(H, L, dtype=torch.float64)
    tf = torch.zeros(H, L, dtype=torch.float64)
    li = last_t.cuda()
    for k0 in range(0, L, 64):
        x[:, :, 2] = 0
        x[:, k0:k0 + 64, 2, :, :] = torch.eye(64, device="cuda")[None, :, None, :]
        xv = x.view(B * L, 3 * D)
        ops.attn_lastq_fwd(qrow, xv, li, ctx1, None, B, L, H, drop_p=p, seed=SEED, site=SITE)
        ops.attn_fwd(xv, ctxf, None, B, L, H, drop_p=p, drop_seed=SEED, drop_site=SITE)
        torch.cuda.synchronize()
        lq[:, k0:k0 + 64] = ctx1[b0].float().view(H, 64).double().cpu()
        tf[:, k0:k0 + 64] = ctxf[b0 * L + last].float().view(H, 64).double().cpu()
    keep = torch.from_numpy(R.keep_bits(SEED, SITE, H * L * L, p, start=b0 * H * L * L).reshape(H, L, L)[:, last])
    assert 0.85 < keep.double().mean().item() < 0.95
    assert torch.equal(lq > 0, keep), "single-query dropout differs from the 64-bit mask"
    assert torch.equal(tf > 0, keep), "tiled forward dropout differs from the 64-bit mask"
    _, k, v = (t[b0 * H:(b0 + 1) * H] for t in A.split_heads(qkv, B, L, H))
    q1 = qrow[b0].float().view(H, 1, 64).double().cuda()
    qpos = torch.full((H, 1), last, device="cuda")
    dm = (keep.double() * float(R.drop_scale(p))).view(H, 1, L).cuda()
    r = A.Ratios("single query read-out above 2^32")
    eye = torch.eye(L, dtype=torch.float64, device="cuda").expand(H, L, L)
    f = A.forward(q1, k.cuda().double(), eye, qpos, dm, rounded=False)
    r.add("P", lq.view(H, 1, L).cuda(), f["ctx"], f["ctx_bound"], f["ctx_var"])
    r.check()


@pytest.mark.gpu
@pytest.mark.parametrize("L,positions", [(200, (0, 1, 100, 198, 199)), (512, (0, 255, 256, 257, 511)),
                                         (4096, (0, 511, 512, 513, 1023, 2048, 4095))])
@pytest.mark.parametrize("family", ["random", "peaked", "rising"])
def test_session_attention_ignores_stale_cache_entries(L, positions, family):
    """tt_session_attn with pos on the edges of its split chunks (chunk 224 / 256 / 512 at L = 200 / 512 / 4096) and
    every cache entry at or after pos poisoned, as in a reused slot: ctx against both tolerances, and the new K / V
    row lands in the cache."""
    ops = _ops()
    H, D = 4, 256
    n = len(positions)
    cap = n + 2
    g = torch.Generator().manual_seed(L + len(family))
    hist, _ = A.make_inputs(family, cap, L, H, seed=L + 11)          # (cap*L, 3D): K | V rows of each slot
    x = hist.view(cap, L, 3, H, 64)
    x[:, :, 0, :, 0] = A.POISON_Q
    slots = torch.randperm(cap, generator=g)[:n].int()
    pos = torch.tensor(positions, dtype=torch.int32)
    new = torch.empty(n, 3, H, 64)
    for r_, (s, p_) in enumerate(zip(slots.tolist(), positions)):
        new[r_] = x[s, p_]
        A.poison_rows_(x[s, p_:].transpose(1, 2), g)                  # stale entries from an earlier user
    kc = x[:, :, 1].permute(0, 2, 1, 3).contiguous()                  # (cap, H, L, 64)
    vc = x[:, :, 2].permute(0, 2, 1, 3).contiguous()
    qkv = new.view(n, 3 * D)
    kc_d, vc_d = kc.cuda().bfloat16(), vc.cuda().bfloat16()
    ctx = torch.full((n, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.session_attn(qkv.cuda().bfloat16(), kc_d, vc_d, slots.cuda(), pos.cuda(), ctx)
    torch.cuda.synchronize()
    k = kc[slots.long()].clone()
    v = vc[slots.long()].clone()
    for r_, p_ in enumerate(positions):
        k[r_, :, p_] = new[r_, 1]
        v[r_, :, p_] = new[r_, 2]
        assert torch.equal(kc_d[slots[r_], :, p_].float().cpu(), new[r_, 1]), "new key not in the cache"
        assert torch.equal(vc_d[slots[r_], :, p_].float().cpu(), new[r_, 2]), "new value not in the cache"
    q1 = new[:, 0].reshape(n * H, 1, 64).cuda().double()
    k, v = k.view(n * H, L, 64).cuda().double(), v.view(n * H, L, 64).cuda().double()
    qpos = pos.long().repeat_interleave(H).view(n * H, 1).cuda()
    f = A.forward(q1, k, v, qpos, rounded=False)
    A.check_family(family, q1, k, v, qpos, f["p"], f["ctx"], n, H)
    r = A.Ratios(f"session L={L} {family} pos={positions}")
    r.add("ctx", ctx.float().view(n * H, 1, 64).double(), f["ctx"], f["ctx_bound"], f["ctx_var"])
    r.check()


# ---------------------------------------------------------------------------------------------------------------------
# Element-index limit of the 32-bit dropout hash (buffers of 3-9 GB, every launch in bounds)
# ---------------------------------------------------------------------------------------------------------------------
def _big_inputs(B, L, H):
    g = torch.Generator(device="cuda").manual_seed(B + L)
    qkv = torch.empty(B * L, 3 * H * 64, device="cuda", dtype=torch.bfloat16).normal_(generator=g)
    do = torch.empty(B * L, H * 64, device="cuda", dtype=torch.bfloat16).normal_(generator=g)
    return qkv, do


def _last_item(t, B, L, H, width):
    """(B*L, width*H*64) -> the last (sequence, head) of each third as (1, L, 64) fp64 tensors."""
    rows = t[(B - 1) * L:].float().view(L, width, H, 64)[:, :, H - 1]
    return [rows[:, i].double()[None] for i in range(width)]


@pytest.mark.gpu
@pytest.mark.parametrize("L,B", [(512, 4096), (256, 16384)])
def test_dropout_at_the_last_32_bit_element_index(L, B):
    """B*H*L*L = 2^32 at H = 4: the last index a 32-bit hash can form. The last (sequence, head) matches the oracle
    with the 64-bit numpy mask in the forward and in the backward."""
    ops = _ops()
    H, p = 4, 0.1
    assert B * H * L * L == 1 << 32
    qkv, do = _big_inputs(B, L, H)
    ctx = torch.empty(B * L, H * 64, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=p, drop_seed=SEED, drop_site=SITE)
    dqkv = torch.empty(B * L, 3 * H * 64, device="cuda", dtype=torch.bfloat16)
    ops.attn_bwd(qkv, ctx, do, lse, dqkv, B, L, H, drop_p=p, drop_seed=SEED, drop_site=SITE)
    torch.cuda.synchronize()
    q, k, v = _last_item(qkv, B, L, H, 3)
    (dO,), (ck,) = _last_item(do, B, L, H, 1), _last_item(ctx, B, L, H, 1)
    dq, dk, dv = _last_item(dqkv, B, L, H, 3)
    lk = lse[B - 1, H - 1].double()[None]
    dm = _drop_mask(B, L, H, p, first_item=B * H - 1)
    del qkv, do, ctx, dqkv
    qpos = A.causal_qpos(1, L, "cuda")
    f = A.forward(q, k, v, qpos, dm)
    b = A.backward(q, k, v, qpos, dO, ck, dm, parked_p=256 < L <= 512)
    r = A.Ratios(f"last 32-bit index L={L} B={B}")
    r.add("ctx", ck, f["ctx"], f["ctx_bound"], f["ctx_var"])
    r.add("lse", lk, f["lse"], f["lse_bound"])
    for n, t in (("dq", dq), ("dk", dk), ("dv", dv)):
        r.add(n, t, b[n], b[n + "_bound"], b[n + "_var"])
    r.check()
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_backward_refuses_dropout_past_the_32_bit_index():
    """B = 4097, L = 512, H = 4: the tiled forward (64-bit index) still matches the oracle on the last (sequence, head),
    and the per-item backward, whose hash index is 32-bit, refuses the dropout instead of applying another mask."""
    from mrm_b200._lib import TTError
    ops = _ops()
    B, L, H, p = 4097, 512, 4, 0.1
    qkv, do = _big_inputs(B, L, H)
    ctx = torch.empty(B * L, H * 64, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, H, L, device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=p, drop_seed=SEED, drop_site=SITE)
    torch.cuda.synchronize()
    q, k, v = _last_item(qkv, B, L, H, 3)
    (ck,) = _last_item(ctx, B, L, H, 1)
    dm = _drop_mask(B, L, H, p, first_item=B * H - 1)
    f = A.forward(q, k, v, A.causal_qpos(1, L, "cuda"), dm)
    r = A.Ratios(f"tiled forward past 2^32 L={L} B={B}")
    r.add("ctx", ck, f["ctx"], f["ctx_bound"], f["ctx_var"])
    r.add("lse", lse[B - 1, H - 1].double()[None], f["lse"], f["lse_bound"])
    r.check()
    dqkv = torch.empty(B * L, 3 * H * 64, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(TTError, match="2\\^32"):
        ops.attn_bwd(qkv, ctx, do, lse, dqkv, B, L, H, drop_p=p, drop_seed=SEED, drop_site=SITE)
    torch.cuda.synchronize()
    del qkv, do, ctx, dqkv
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_persistent_forward_refuses_dropout_past_the_32_bit_index():
    """B = 16385, L = 256, H = 4: B*H*L*L passes 2^32 and the persistent forward refuses the dropout."""
    from mrm_b200._lib import TTError
    ops = _ops()
    B, L, H = 16385, 256, 4
    qkv = torch.zeros(B * L, 3 * H * 64, device="cuda", dtype=torch.bfloat16)
    ctx = torch.empty(B * L, H * 64, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(TTError, match="2\\^32"):
        ops.attn_fwd(qkv, ctx, None, B, L, H, drop_p=0.1, drop_seed=SEED, drop_site=SITE)
    torch.cuda.synchronize()
    del qkv, ctx
    torch.cuda.empty_cache()
