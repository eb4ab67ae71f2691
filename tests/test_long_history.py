"""Long listening histories: 512 < L <= 4096 through the tiled attention kernels, the single-query last layer, the
training step, CUDA-graph replay and recommend_batch.

Attention references are the fp32 torch restatement of tests/test_attention.py on the same bf16 inputs, with its
tolerances; dropout references apply the numpy mask of tests/_dropout_ref.drop_keep_k (64-bit element index
((b*H + h)*L + q)*L + k)."""
import numpy as np
import pytest
import torch

import _dropout_ref as R

gpu = pytest.mark.gpu


def _ref_attention(qkv, B, L, H, dctx=None, mask=None):
    """ctx, lse, dqkv of causal attention in fp32 autograd; ``mask`` (B, H, L, L) scaled dropout mask or None."""
    D = H * 64
    x = qkv.float().view(B, L, 3, H, 64).requires_grad_(dctx is not None)
    q, k, v = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2), x[:, :, 2].transpose(1, 2)
    s = (q @ k.transpose(-1, -2)) / 8.0
    causal = torch.triu(torch.ones(L, L, dtype=torch.bool, device=qkv.device), 1)
    s = s.masked_fill(causal, float("-inf"))
    lse = torch.logsumexp(s, dim=-1)
    p = torch.softmax(s, dim=-1)
    if mask is not None:
        p = p * mask
    o = (p @ v).transpose(1, 2).reshape(B * L, D)
    if dctx is None:
        return o.detach(), lse.detach(), None
    o.backward(dctx.float())
    return o.detach(), lse.detach(), x.grad.reshape(B * L, 3 * D)


def _attn_mask(L, H, bh, seed, site, p):
    """Scaled dropout mask (L, L) of (sequence, head) item bh = b*H + h, from the 64-bit element index."""
    idx = (np.uint64(bh) * np.uint64(L) + np.arange(L, dtype=np.uint64)[:, None]) * np.uint64(L) \
        + np.arange(L, dtype=np.uint64)[None, :]
    keep = R.drop_keep_k(R.drop_key(seed, site), idx, R.drop_threshold(p))
    return torch.from_numpy(np.where(keep, R.drop_scale(p), np.float32(0.0)).astype(np.float32))


def _run(qkv, dctx, B, L, H, drop=0.0, seed=0, site=0):
    from mrm_b200 import ops
    D = H * 64
    ctx = torch.full((B * L, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    lse = torch.full((B, H, L), float("nan"), device="cuda")
    ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=drop, drop_seed=seed, drop_site=site)
    dqkv = torch.full((B * L, 3 * D), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.attn_bwd(qkv, ctx, dctx, lse, dqkv, B, L, H, drop_p=drop, drop_seed=seed, drop_site=site)
    torch.cuda.synchronize()
    return ctx, lse, dqkv


def _check_grads(dqkv, dref, D):
    for name, sl in (("dq", slice(0, D)), ("dk", slice(D, 2 * D)), ("dv", slice(2 * D, 3 * D))):
        a, r = dqkv[:, sl].float(), dref[:, sl]
        err = (a - r).abs().max().item()
        scale = r.abs().max().item()
        assert err <= 3e-2 * max(scale, 1.0), f"{name}: err {err} scale {scale}"


@gpu
@pytest.mark.parametrize("B,L,H", [(2, 513, 4), (2, 640, 4), (1, 1000, 4), (2, 1024, 4), (1, 2048, 4), (1, 4096, 2)])
def test_long_attention_matches_torch(B, L, H):
    """Forward ctx / lse and backward dq / dk / dv, tail tiles and L not a multiple of 4 included."""
    g = torch.Generator().manual_seed(L + B)
    D = H * 64
    qkv = (torch.randn(B * L, 3 * D, generator=g) * 1.2).cuda().bfloat16()
    dctx = torch.randn(B * L, D, generator=g).cuda().bfloat16()
    ctx, lse, dqkv = _run(qkv, dctx, B, L, H)
    o, lse_ref, dref = _ref_attention(qkv, B, L, H, dctx)
    assert (ctx.float() - o).abs().max().item() <= 3e-2
    assert (lse - lse_ref).abs().max().item() <= 2e-3
    _check_grads(dqkv, dref, D)


@gpu
def test_long_attention_backward_is_deterministic():
    B, L, H = 2, 2048, 4
    g = torch.Generator().manual_seed(5)
    qkv = (torch.randn(B * L, 3 * H * 64, generator=g) * 1.2).cuda().bfloat16()
    dctx = torch.randn(B * L, H * 64, generator=g).cuda().bfloat16()
    _, _, a = _run(qkv, dctx, B, L, H, drop=0.1, seed=77, site=3)
    _, _, b = _run(qkv, dctx, B, L, H, drop=0.1, seed=77, site=3)
    assert torch.isfinite(a.float()).all()
    assert torch.equal(a, b)


@gpu
@pytest.mark.parametrize("B,L,H", [(2, 1001, 4), (1, 2048, 4)])
def test_long_attention_dropout_uses_the_hash_mask(B, L, H):
    """Forward and backward with dropout 0.1 against torch autograd applying the numpy mask of every (sequence, head)."""
    p, seed, site = 0.1, 4242, 5
    D = H * 64
    g = torch.Generator().manual_seed(3 * L)
    qkv = (torch.randn(B * L, 3 * D, generator=g) * 1.2).cuda().bfloat16()
    dctx = torch.randn(B * L, D, generator=g).cuda().bfloat16()
    ctx, lse, dqkv = _run(qkv, dctx, B, L, H, drop=p, seed=seed, site=site)
    mask = torch.stack([_attn_mask(L, H, bh, seed, site, p) for bh in range(B * H)]).view(B, H, L, L).cuda()
    o, lse_ref, dref = _ref_attention(qkv, B, L, H, dctx, mask)
    assert (ctx.float() - o).abs().max().item() <= 3e-2
    assert (lse - lse_ref).abs().max().item() <= 2e-3
    _check_grads(dqkv, dref, D)


@gpu
def test_long_attention_dropout_index_above_2_32():
    """B = 65, L = 4096, H = 4: the last (sequence, head) draws from element indices >= 2^32 only. Its ctx and its
    head's dq / dk / dv match torch with the numpy mask of the 64-bit index."""
    B, L, H, p, seed, site = 65, 4096, 4, 0.1, 99, 2
    D = H * 64
    bh = B * H - 1
    assert bh * L * L >= 1 << 32
    g = torch.Generator().manual_seed(65)
    qkv = (torch.randn(B * L, 3 * D, generator=g) * 1.2).cuda().bfloat16()
    dctx = torch.randn(B * L, D, generator=g).cuda().bfloat16()
    ctx, lse, dqkv = _run(qkv, dctx, B, L, H, drop=p, seed=seed, site=site)
    b, h = divmod(bh, H)
    rows = slice(b * L, (b + 1) * L)
    heads = [slice(t * D + h * 64, t * D + h * 64 + 64) for t in range(3)]
    one = torch.cat([qkv[rows, s] for s in heads], dim=1).contiguous()         # (L, 3*64): one head
    mask = _attn_mask(L, H, bh, seed, site, p).view(1, 1, L, L).cuda()
    o, lse_ref, dref = _ref_attention(one, 1, L, 1, dctx[rows, h * 64:h * 64 + 64], mask)
    assert (ctx[rows, h * 64:h * 64 + 64].float() - o).abs().max().item() <= 3e-2
    assert (lse[b, h] - lse_ref[0, 0]).abs().max().item() <= 2e-3
    got = torch.cat([dqkv[rows, s] for s in heads], dim=1)
    _check_grads(got, dref, 64)


def _long_batch(cfg, seed):
    """B = 4 at max_seq_len 2048: two full-length histories, one of length 1, one of length 1000."""
    from mrm_b200 import synthetic
    L = cfg.max_seq_len
    batch = synthetic.make_batch(cfg, 4, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    ids = torch.randint(1, cfg.vocab_size, (4, L), generator=g)
    lens = torch.tensor([L, L, 1, 1000])
    valid = torch.arange(L)[None, :] < lens[:, None]
    batch["history_ids"] = ids * valid
    batch["history_mask"] = valid.long()
    return batch


GRAD_KEYS = ("user_tower.transformer_encoder.layers.0.self_attn.in_proj_weight",
             "user_tower.transformer_encoder.layers.0.linear1.weight",
             "user_tower.transformer_encoder.layers.1.self_attn.in_proj_weight",
             "user_tower.position_embedding.weight", "user_tower.item_embedding.weight")


@gpu
@pytest.mark.parametrize("dropout", [0.0, 0.1])
def test_long_training_step_matches_oracle(dropout):
    """One engine training step at max_seq_len 2048 against the fp64 oracle (with the engine's own dropout masks when
    dropout > 0), with the bounds of test_engine.test_seq512_training_step_matches_oracle."""
    import os
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    from oracle import two_tower_oracle as oracle
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = synthetic.TwoTowerConfig(vocab_size=3001, max_seq_len=2048, dropout=dropout)
    sd = synthetic.make_state_dict(cfg, seed=21)
    batch = _long_batch(cfg, seed=22)
    ctr = R.counter_after(2)
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(sd)
    eng.seed_dev.fill_(ctr)
    loss, _, u, _ = eng.forward({k: v.cuda() for k, v in batch.items()}, training=True)
    eng.backward()
    torch.cuda.synchronize()
    drop = R.engine_masks(cfg, batch, ctr) if dropout > 0 else None
    b64 = {k: (v.double() if v.is_floating_point() else v) for k, v in batch.items()}
    ref_loss, _, ref_u, _, grads, _ = oracle.loss_and_grads(sd, b64, cfg.temperature, cfg.num_heads,
                                                            dtype=torch.float64, drop=drop)
    errs = {"loss": abs(loss.item() - ref_loss.item()), "user_emb": (u.cpu().double() - ref_u).abs().max().item()}
    for k in GRAD_KEYS:
        ref = grads[k]
        errs[k] = ((eng.g[k].cpu().double() - ref).norm().item(), ref.norm().item())
    print("long_training_step", dropout, errs)
    assert errs["loss"] <= 2e-2, errs
    assert errs["user_emb"] <= 1e-2, errs
    for k in GRAD_KEYS:
        err, n = errs[k]
        assert err <= 0.15 * n + 5e-5 * grads[k].numel() ** 0.5, (k, err, n)


@gpu
def test_long_pruned_last_layer_equals_full_computation():
    """At dropout 0 the single-row last layer gives the loss, embeddings and user-tower gradients of the full
    computation. (With B = 4 the item tower's gradients are small enough that bf16 noise of the two paths' different
    user embeddings dominates them; test_engine.test_pruned_last_layer_equals_full_computation covers all of them.)"""
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    cfg = synthetic.TwoTowerConfig(vocab_size=3001, max_seq_len=2048, dropout=0.0)
    sd = synthetic.make_state_dict(cfg, seed=31)
    dbatch = {k: v.cuda() for k, v in _long_batch(cfg, seed=32).items()}
    out = {}
    for prune in (True, False):
        e = TwoTowerEngine(cfg)
        e.load_state_dict(sd)
        e.prune_last_layer = prune
        loss, _, u, _ = e.forward(dbatch, training=True)
        e.backward()
        torch.cuda.synchronize()
        out[prune] = (loss.item(), u.clone(), {k: v.clone() for k, v in e.g.items()})
    assert abs(out[True][0] - out[False][0]) <= 5e-3
    assert (out[True][1] - out[False][1]).abs().max().item() <= 3e-3
    for k in GRAD_KEYS:
        gp, gf = out[True][2][k], out[False][2][k]
        err = (gp - gf).norm().item()
        assert err <= 0.12 * gf.norm().item() + 5e-5 * gf.numel() ** 0.5, (k, err, gf.norm().item())


@gpu
def test_long_graph_replay_matches_eager_steps():
    """TrainStepRunner at L = 1024, dropout 0.1: a graph runner (step 1 eager, step 2 captured and replayed, steps 3-4
    replayed) against an eager runner, in lockstep from the same state. Each step's loss and every parameter's gradient
    agree. The gradient is read from AdamW's first moment, m_t = b1 m_{t-1} + (1 - b1) g_t, before the update can
    amplify it. After each step the graph runner's parameters, moments and bf16 shadow are set to the eager runner's
    (in place, the graph keeps its pointers), so every step starts from one state: the two gradients then differ only
    by fp32 atomic summation order, and the replays must read the advancing dropout counter."""
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import TrainStepRunner
    cfg = synthetic.TwoTowerConfig(vocab_size=3001, max_seq_len=1024, dropout=0.1)
    sd = synthetic.make_state_dict(cfg, seed=41)
    batch = {k: v.cuda() for k, v in synthetic.make_batch(cfg, 8, seed=42).items()}
    batch["history_ids"][0] = torch.randint(1, 3001, (1024,), device="cuda")
    batch["history_mask"][0] = 1
    b1 = 0.9
    engs, runners = [], []
    for graph in (False, True):
        eng = TwoTowerEngine(cfg)
        eng.load_state_dict(sd)
        runner = TrainStepRunner(eng, 8, 1024, lr=1e-3, betas=(b1, 0.999), use_graph=graph)
        runner.load_batch(batch)
        engs.append(eng)
        runners.append(runner)
    ea, eg = engs
    worst = 0.0
    for step in range(4):
        m_prev = ea.exp_avg.clone() if ea.exp_avg is not None else torch.zeros_like(ea.flat)
        la = runners[0].step_resident().item()
        lg = runners[1].step_resident().item()
        torch.cuda.synchronize()
        assert abs(la - lg) <= 1e-4 * abs(la), (step, la, lg)
        assert int(ea.seed_dev.item()) == int(eg.seed_dev.item()) and int(ea.step_dev.item()) == int(eg.step_dev.item())
        ga = (ea.exp_avg - b1 * m_prev) / (1 - b1)
        gg = (eg.exp_avg - b1 * m_prev) / (1 - b1)
        for name, (off, shape) in ea.layout.items():
            n = int(np.prod(shape))
            a, g = ga[off:off + n], gg[off:off + n]
            err, ref = (a - g).norm().item(), a.norm().item()
            bound = 1e-2 * ref + 1e-6 * n ** 0.5
            worst = max(worst, err / bound)
            assert err <= bound, (step, name, err, ref)
        eg.flat.copy_(ea.flat)
        eg.exp_avg.copy_(ea.exp_avg)
        eg.exp_avg_sq.copy_(ea.exp_avg_sq)
        eg.shadow.copy_(ea.shadow)
    print("graph_replay worst gradient error / bound", worst)


@gpu
def test_long_recommend_batch_matches_oracle():
    """recommend_batch at max_seq_len 2048 (towers in chunks of 256 users) against get_user_embedding +
    oracle.recommend per user, histories longer than 512 included."""
    from mrm_b200 import inference, retrieval, synthetic
    from mrm_b200.models import TwoTowerModel
    from oracle import two_tower_oracle as oracle
    from test_recommend_exclusion import _assert_no_excluded, _assert_same_ranking
    V, B, L = 2001, 300, 2048
    model = TwoTowerModel(vocab_size=V, tabular_input_dim=17, num_genders=3, num_countries=50, max_seq_len=L,
                          user_embedding_dim=256, item_embedding_dim=256, use_lora=True, seed=6)
    table = synthetic.make_catalog(V - 1, 256, seed=8)
    index = retrieval.CatalogIndex(table)
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(1, V, (B, L), generator=g)
    lengths = torch.randint(1, L + 1, (B,), generator=g)
    lengths[:5] = L
    lengths[5:10] = torch.tensor([513, 700, 1000, 1500, 2047])
    ids[torch.arange(L)[None, :] >= lengths[:, None]] = 0
    gender = torch.randint(0, 3, (B,), generator=g)
    country = torch.randint(0, 50, (B,), generator=g)
    model.eval()
    with torch.no_grad():
        u = model.get_user_embedding(ids.cuda(), (ids != 0).long().cuda(), gender.cuda(), country.cuda()).cpu()
    model.train()
    idx, score = inference.recommend_batch(model, index, ids, user_gender=gender, user_country=country, k=10)
    for b in range(B):
        want_s, want_i = oracle.recommend(u[b], table, [h for h in ids[b].tolist() if h], 10)
        _assert_same_ranking(idx[b], score[b], want_i, want_s)
    _assert_no_excluded(idx.cpu(), ids)


@gpu
def test_more_tokens_per_call_than_the_bound_are_rejected():
    from mrm_b200 import synthetic
    from mrm_b200.engine import MAX_TOKENS, TwoTowerEngine
    eng = TwoTowerEngine(synthetic.TwoTowerConfig(vocab_size=11, max_seq_len=4096))
    assert MAX_TOKENS == 256 * 4096
    with pytest.raises(ValueError):
        eng.workspace(257, 4096)


def test_max_seq_len_above_4096_is_rejected():
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    with pytest.raises(ValueError):
        TwoTowerEngine(synthetic.TwoTowerConfig(vocab_size=11, max_seq_len=4097))
