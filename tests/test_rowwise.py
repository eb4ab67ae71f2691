"""Row-wise CUDA kernels against plain PyTorch fp32 (autograd for the backward passes)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _randn(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).cuda()


def test_cast_and_last_index():
    from mrm_b200 import ops
    x = _randn(4096, seed=1)
    y = torch.empty(4096, device="cuda", dtype=torch.bfloat16)
    ops.cast_bf16(x, y)
    assert torch.equal(y, x.bfloat16())
    ids = torch.tensor([[5, 3, 0, 0], [1, 2, 3, 4], [7, 0, 0, 0], [0, 0, 0, 0]], device="cuda")
    out = torch.empty(4, device="cuda", dtype=torch.int32)
    ops.last_index(ids, None, out)
    assert out.tolist() == [1, 3, 0, 0]
    ops.last_index(ids, (ids != 0).long(), out)
    assert out.tolist() == [1, 3, 0, 0]


def test_embed_ln_fwd_bwd():
    from mrm_b200 import ops
    B, L, V = 6, 37, 101
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(0, V, (B, L), generator=g).cuda()
    E, P = _randn(V, 256, seed=4, scale=0.1), _randn(64, 256, seed=5, scale=0.1)
    w, b = 1 + _randn(256, seed=6, scale=0.1), _randn(256, seed=7, scale=0.1)
    nw, nb = 1 + _randn(256, seed=8, scale=0.1), _randn(256, seed=9, scale=0.1)
    x0 = torch.empty(B * L, 256, device="cuda")
    h = torch.empty(B * L, 256, device="cuda", dtype=torch.bfloat16)
    ops.embed_ln_fwd(ids.view(-1), E, P, w, b, nw, nb, B, L, x0, h)
    Er, Pr, wr, br = (t.clone().requires_grad_(True) for t in (E, P, w, b))
    e = Er[ids] + Pr[:L].unsqueeze(0)
    x_ref = F.layer_norm(e, (256,), wr, br).view(B * L, 256)
    assert (x0 - x_ref).abs().max().item() < 2e-5
    h_ref = F.layer_norm(x_ref, (256,), nw, nb)
    assert (h.float() - h_ref).abs().max().item() < 3e-2
    dx0 = _randn(B * L, 256, seed=10)
    dE, dP = torch.zeros_like(E), torch.zeros_like(P)
    dg, db = torch.zeros(256, device="cuda"), torch.zeros(256, device="cuda")
    ops.embed_ln_bwd(ids.view(-1), E, P, w, b, dx0, B, L, dE, dP, dg, db)
    x_ref.backward(dx0)
    dE_ref = Er.grad.clone()
    dE_ref[0] = 0  # padding_idx
    assert (dE - dE_ref).abs().max().item() < 1e-4
    assert (dP - Pr.grad).abs().max().item() < 1e-4
    assert (dg - wr.grad).abs().max().item() < 1e-3
    assert (db - br.grad).abs().max().item() < 1e-3


@pytest.mark.parametrize("ln,relu,l2", [(True, False, False), (True, True, False), (False, False, True),
                                        (True, False, True)])
def test_chain_fwd_bwd(ln, relu, l2):
    from mrm_b200 import ops
    R, W = 300, 256
    x = _randn(R, W, seed=11)
    w, b = 1 + _randn(W, seed=12, scale=0.1), _randn(W, seed=13, scale=0.1)
    out = torch.empty(R, W, device="cuda")
    out16 = torch.empty(R, W, device="cuda", dtype=torch.bfloat16)
    ops.chain_fwd(x, ln=(w, b) if ln else None, relu=relu, l2norm=l2, out_f32=out, out_bf16=out16)
    xr, wr, br = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = F.layer_norm(xr, (W,), wr, br) if ln else xr
    if relu:
        y = torch.relu(y)
    if l2:
        y = F.normalize(y, dim=1)
    assert (out - y).abs().max().item() < 2e-5
    assert (out16.float() - y).abs().max().item() < 2e-2
    dout, resid = _randn(R, W, seed=14), _randn(R, W, seed=15)
    dx = torch.empty(R, W, device="cuda")
    dx16 = torch.empty(R, W, device="cuda", dtype=torch.bfloat16)
    dg, db, cs = (torch.zeros(W, device="cuda") for _ in range(3))
    ops.chain_bwd(x, ln=(w, b) if ln else None, relu=relu, l2norm=l2, dout=dout, resid=resid, dx_f32=dx,
                  dx_bf16=dx16, dgamma=dg if ln else None, dbeta=db if ln else None, dx_colsum=cs)
    y.backward(dout)
    ref = xr.grad + resid
    assert (dx - ref).abs().max().item() < 1e-4 * max(1.0, ref.abs().max().item())
    assert (cs - dx16.float().sum(0)).abs().max().item() < 1e-2
    if ln:
        assert (dg - wr.grad).abs().max().item() < 2e-3
        assert (db - br.grad).abs().max().item() < 2e-3


def test_chain_bwd_sparse_residual_equals_dense():
    """resid_rows (one row per sequence, selected by last_idx) == a dense residual that is zero elsewhere."""
    from mrm_b200 import ops
    Bq, L, W = 12, 25, 256
    R = Bq * L
    x, dout = _randn(R, W, seed=31), _randn(R, W, seed=32)
    w, b = 1 + _randn(W, seed=33, scale=0.1), _randn(W, seed=34, scale=0.1)
    rows = _randn(Bq, W, seed=35)
    last = torch.randint(0, L, (Bq,), device="cuda", dtype=torch.int32)
    dense = torch.zeros(R, W, device="cuda")
    dense[torch.arange(Bq, device="cuda") * L + last.long()] = rows
    outs = []
    for kw in (dict(resid=dense), dict(resid_rows=rows, resid_last_idx=last, resid_seq_len=L)):
        dx = torch.empty(R, W, device="cuda")
        dg, db = torch.zeros(W, device="cuda"), torch.zeros(W, device="cuda")
        ops.chain_bwd(x, ln=(w, b), dout=dout, dx_f32=dx, dgamma=dg, dbeta=db, **kw)
        outs.append((dx, dg, db))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0])
    assert torch.allclose(outs[0][1], outs[1][1], atol=1e-4) and torch.allclose(outs[0][2], outs[1][2], atol=1e-4)


def test_chain_bwd_bf16_incoming_gradient():
    """dout_bf16 == dout holding the same (bf16-representable) values: the incoming gradient of a LayerNorm whose
    consumer is a Linear arrives in bf16 under autocast; only the load differs."""
    from mrm_b200 import ops
    from mrm_b200._lib import TTError
    R, W = 777, 256
    x, resid = _randn(R, W, seed=41), _randn(R, W, seed=43)
    d16 = _randn(R, W, seed=42).to(torch.bfloat16)
    w, b = 1 + _randn(W, seed=44, scale=0.1), _randn(W, seed=45, scale=0.1)
    outs = []
    for kw in (dict(dout=d16.float()), dict(dout_bf16=d16)):
        dx, dxb = torch.empty(R, W, device="cuda"), torch.empty(R, W, device="cuda", dtype=torch.bfloat16)
        dg, db, cs = (torch.zeros(W, device="cuda") for _ in range(3))
        ops.chain_bwd(x, ln=(w, b), resid=resid, dx_f32=dx, dx_bf16=dxb, dgamma=dg, dbeta=db, dx_colsum=cs, **kw)
        outs.append((dx, dxb, dg, db, cs))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    for a, c in zip(outs[0][2:], outs[1][2:]):
        assert torch.allclose(a, c, atol=1e-3, rtol=1e-5)
    with pytest.raises(TTError):       # exactly one of the two
        ops.chain_bwd(x, ln=(w, b), dx_f32=outs[0][0], dgamma=outs[0][2], dbeta=outs[0][3])


def test_chain_dropout_fwd_bwd_consistent():
    """Same (seed, site) in forward and backward: d/dx of sum(dropout(LN(x)) * c) matches a finite mask."""
    from mrm_b200 import ops
    R, W = 64, 256
    x = _randn(R, W, seed=21)
    w, b = torch.ones(W, device="cuda"), torch.zeros(W, device="cuda")
    out = torch.empty(R, W, device="cuda")
    ops.chain_fwd(x, ln=(w, b), drop_p=0.3, seed=77, site=5, out_f32=out)
    mask = (out != 0).float()
    assert 0.65 < mask.mean().item() < 0.75
    xr = x.clone().requires_grad_(True)
    y = F.layer_norm(xr, (W,), w, b) * mask / 0.7
    assert (out - y).abs().max().item() < 1e-4
    dout = _randn(R, W, seed=22)
    y.backward(dout)
    dx = torch.empty(R, W, device="cuda")
    dg, db = torch.zeros(W, device="cuda"), torch.zeros(W, device="cuda")
    ops.chain_bwd(x, ln=(w, b), drop_p=0.3, seed=77, site=5, dout=dout, dx_f32=dx, dgamma=dg, dbeta=db)
    assert (dx - xr.grad).abs().max().item() < 1e-4


def test_gather_cat_and_concat4():
    from mrm_b200 import ops
    B, L = 5, 9
    x = _randn(B * L, 256, seed=31)
    last = torch.tensor([0, 8, 3, 5, 1], device="cuda", dtype=torch.int32)
    gender = torch.tensor([0, 2, 1, 1, 0], device="cuda")
    country = torch.tensor([3, 0, 6, 6, 2], device="cuda")
    G, C = _randn(3, 16, seed=32), _randn(7, 32, seed=33)
    cat = torch.zeros(B, 304, device="cuda", dtype=torch.bfloat16)
    ops.gather_cat_fwd(x, last, gender, country, G, C, B, L, cat)
    rows = x.view(B, L, 256)[torch.arange(B), last.long()]
    ref = torch.cat([rows, G[gender], C[country]], dim=1)
    assert torch.equal(cat, ref.bfloat16())
    dcat = _randn(B, 304, seed=34)
    dx = torch.zeros(B * L, 256, device="cuda")
    dG, dC = torch.zeros_like(G), torch.zeros_like(C)
    ops.gather_cat_bwd(dcat, last, gender, country, B, L, dx, None, dG, dC)
    dx_ref = torch.zeros(B, L, 256, device="cuda")
    dx_ref[torch.arange(B), last.long()] = dcat[:, :256]
    assert torch.equal(dx, dx_ref.view(B * L, 256))
    dG_ref = torch.zeros_like(G).index_add_(0, gender, dcat[:, 256:272])
    dC_ref = torch.zeros_like(C).index_add_(0, country, dcat[:, 272:])
    assert (dG - dG_ref).abs().max().item() < 1e-5 and (dC - dC_ref).abs().max().item() < 1e-5
    parts = [_randn(B, 128, seed=40 + i) for i in range(4)]
    out = torch.empty(B, 512, device="cuda", dtype=torch.bfloat16)
    ops.concat4_bf16(*parts, out)
    assert torch.equal(out, torch.cat(parts, dim=1).bfloat16())


@pytest.mark.parametrize("training", [True, False])
def test_bn_relu_fwd_bwd(training):
    from mrm_b200 import ops
    B, C = 96, 512
    y = _randn(B, C, seed=51)
    w, b = 1 + _randn(C, seed=52, scale=0.1), _randn(C, seed=53, scale=0.1)
    bn = torch.nn.BatchNorm1d(C).cuda()
    with torch.no_grad():
        bn.weight.copy_(w)
        bn.bias.copy_(b)
        bn.running_mean.copy_(_randn(C, seed=54, scale=0.1))
        bn.running_var.copy_(1 + _randn(C, seed=55, scale=0.1).abs())
    rm, rv, nb = bn.running_mean.clone(), bn.running_var.clone(), bn.num_batches_tracked.clone()
    bn.train(training)
    yr = y.clone().requires_grad_(True)
    ref = torch.relu(bn(yr))
    out = torch.empty(B, C, device="cuda", dtype=torch.bfloat16)
    sm, sr = torch.empty(C, device="cuda"), torch.empty(C, device="cuda")
    ops.bn_relu_fwd(y, w, b, rm, rv, nb, training=training, save_mean=sm, save_rstd=sr, out_bf16=out)
    assert (out.float() - ref).abs().max().item() < 3e-2
    assert (rm - bn.running_mean).abs().max().item() < 1e-5
    assert (rv - bn.running_var).abs().max().item() < 1e-5
    assert nb.item() == bn.num_batches_tracked.item()
    if training:
        dout = _randn(B, C, seed=56)
        ref.backward(dout)
        dy = torch.empty(B, C, device="cuda", dtype=torch.bfloat16)
        dg, db, cs = (torch.zeros(C, device="cuda") for _ in range(3))
        ops.bn_relu_bwd(y, w, b, rm, rv, None, training=True, save_mean=sm, save_rstd=sr, dout=dout, dy_bf16=dy,
                        dgamma=dg, dbeta=db, dy_colsum=cs)
        assert (dy.float() - yr.grad).abs().max().item() < 2e-2 * max(1.0, yr.grad.abs().max().item())
        assert (dg - bn.weight.grad).abs().max().item() < 2e-3
        assert (db - bn.bias.grad).abs().max().item() < 2e-3
        assert (cs - dy.float().sum(0)).abs().max().item() < 1e-2


def test_adamw():
    from mrm_b200 import ops
    from oracle import two_tower_oracle as oracle
    n = 4096 + 64
    p, g = _randn(n, seed=62), _randn(n, seed=63, scale=0.01)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    shadow = torch.zeros(1024, device="cuda", dtype=torch.bfloat16)
    step = torch.zeros((), device="cuda", dtype=torch.long)
    pr, mr, vr = p.cpu().double(), torch.zeros(n).double(), torch.zeros(n).double()
    for t in range(1, 4):
        gt = g * t
        gcpu = gt.cpu().double()
        ops.step_counters_advance(step, None)
        ops.adamw_step(p, gt, m, v, step, shadow=shadow, shadow_begin=64, shadow_end=64 + 1024, zero_grad=True)
        pr, mr, vr = oracle.adamw_step(pr, gcpu, mr, vr, t)
        assert gt.abs().max().item() == 0.0
    assert (p.cpu().double() - pr).abs().max().item() < 1e-6
    assert torch.equal(shadow, p[64:64 + 1024].bfloat16())


def test_infonce_rows_grad_loss():
    from mrm_b200 import ops
    B = 70
    S = _randn(B, B, seed=71, scale=4.0)
    uid = torch.randint(0, 20, (B,), generator=torch.Generator().manual_seed(72)).cuda()
    Sr = S.clone().requires_grad_(True)
    coll = (uid[:, None] == uid[None, :]) & ~torch.eye(B, dtype=torch.bool, device="cuda")
    Sm = Sr.masked_fill(coll, -1e4)
    labels = torch.arange(B, device="cuda")
    loss_ref = 0.5 * (F.cross_entropy(Sm, labels) + F.cross_entropy(Sm.t(), labels))
    loss_ref.backward()
    S1, S2 = S.clone(), S.t().contiguous()
    lr, pr_, lc, pc = (torch.empty(B, device="cuda") for _ in range(4))
    ops.infonce_rows(S1, uid, uid, 0, lr, pr_)
    ops.infonce_rows(S2, uid, uid, 0, lc, pc)
    assert torch.equal(S1, Sm.detach())
    loss = torch.zeros((), device="cuda")
    ops.infonce_loss(lr, pr_, lc, pc, 0.5 / B, loss)
    assert abs(loss.item() - loss_ref.item()) < 1e-4
    dS = torch.empty(B, B, device="cuda", dtype=torch.bfloat16)
    ops.infonce_grad(S1, lr, lc, 0, 0.5 / B, dS)
    assert (dS.float() - Sr.grad).abs().max().item() < 1e-4
