"""User sessions (sessions.UserSessions): the incremental user tower over cached keys / values.

Kernels: tt_session_attn against fp32 torch attention over the same cache, with the cache checked for stray writes;
tt_embed_ln_fwd_pos against tt_embed_ln_fwd's rows. Sessions: every append against the full tower
(get_user_embedding on the same window) and the fp64 oracle, through the window boundary; recommendations against the
oracle; every guard.
"""
import pytest
import torch
import torch.nn.functional as F

gpu = pytest.mark.gpu
POSITIONS = (0, 1, 31, 32, 33, 511, 512, 513, 2047, 4095)


def _ref_session_attn(qkv, kc, vc, slots, pos):
    """fp32: each row's query over cache[slot, h, :pos] plus its own key / value at pos."""
    n = qkv.shape[0]
    H = kc.shape[1]
    out = torch.empty(n, H * 64)
    for r in range(n):
        s, p = int(slots[r]), int(pos[r])
        for h in range(H):
            q = qkv[r, h * 64:(h + 1) * 64].float()
            k = torch.cat([kc[s, h, :p].float(), qkv[r, 256 + h * 64:256 + (h + 1) * 64].float()[None]])
            v = torch.cat([vc[s, h, :p].float(), qkv[r, 512 + h * 64:512 + (h + 1) * 64].float()[None]])
            out[r, h * 64:(h + 1) * 64] = torch.softmax(k @ q / 8.0, dim=0) @ v
    return out


@gpu
@pytest.mark.parametrize("L", [200, 512, 4096])
@pytest.mark.parametrize("n", [1, 300])
def test_session_attn_matches_torch(L, n):
    """Random caches, positions 0 ... 4095 (those below L), permuted slots of a larger cache: ctx within 3e-2 of fp32
    torch; the cache changes only in each row's (slot, pos) entry, which holds the K / V thirds of qkv; a second
    identical call gives a bit-identical ctx."""
    from mrm_b200 import ops
    g = torch.Generator().manual_seed(L + n)
    cap, H = n + 7, 4
    kc = (torch.randn(cap, H, L, 64, generator=g)).bfloat16().cuda()
    vc = (torch.randn(cap, H, L, 64, generator=g)).bfloat16().cuda()
    qkv = (torch.randn(n, 768, generator=g) * 1.5).bfloat16().cuda()
    slots = torch.randperm(cap, generator=g)[:n].int()
    ps = [p for p in POSITIONS if p < L] + [L - 1]
    pos = torch.tensor([ps[i % len(ps)] for i in range(n)], dtype=torch.int32)
    if n == 1:
        pos[0] = L - 1
    k0, v0 = kc.cpu(), vc.cpu()
    ctx = torch.empty(n, 256, dtype=torch.bfloat16, device="cuda")
    ops.session_attn(qkv, kc, vc, slots.cuda(), pos.cuda(), ctx)
    torch.cuda.synchronize()
    ref = _ref_session_attn(qkv.cpu(), k0, v0, slots, pos)
    assert (ctx.cpu().float() - ref).abs().max().item() <= 3e-2
    k1, v1 = kc.cpu(), vc.cpu()
    want_k, want_v = k0.clone(), v0.clone()
    q = qkv.cpu()
    for r in range(n):
        want_k[slots[r], :, pos[r]] = q[r, 256:512].view(H, 64)
        want_v[slots[r], :, pos[r]] = q[r, 512:].view(H, 64)
    assert torch.equal(k1, want_k) and torch.equal(v1, want_v)
    ctx2 = torch.empty_like(ctx)
    ops.session_attn(qkv, kc, vc, slots.cuda(), pos.cuda(), ctx2)
    torch.cuda.synchronize()
    assert torch.equal(ctx, ctx2)


@gpu
def test_embed_ln_fwd_pos_equals_embed_ln_fwd_rows():
    from mrm_b200 import ops, synthetic
    from mrm_b200.engine import TwoTowerEngine
    cfg = synthetic.TwoTowerConfig(vocab_size=3001, max_seq_len=512)
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(synthetic.make_state_dict(cfg, seed=3))
    p, ut = eng.p, "user_tower."
    B, L = 6, 512
    g = torch.Generator().manual_seed(5)
    ids = torch.randint(0, cfg.vocab_size, (B, L), generator=g).cuda()
    args = (p[ut + "position_embedding.weight"], p[ut + "layer_norm.weight"], p[ut + "layer_norm.bias"],
            p[eng._lp(0, "norm1.weight")], p[eng._lp(0, "norm1.bias")])
    x0 = torch.empty(B * L, 256, device="cuda")
    h = torch.empty(B * L, 256, device="cuda", dtype=torch.bfloat16)
    ops.embed_ln_fwd(ids.view(-1), p[ut + "item_embedding.weight"], *args[:3], *args[3:], B, L, x0, h)
    rows = torch.randperm(B * L, generator=g)[:333].cuda()
    pos = (rows % L).int()
    x0p = torch.empty(333, 256, device="cuda")
    hp = torch.empty(333, 256, device="cuda", dtype=torch.bfloat16)
    ops.embed_ln_fwd_pos(ids.view(-1)[rows].contiguous(), pos, p[ut + "item_embedding.weight"], *args, x0p, hp)
    torch.cuda.synchronize()
    assert torch.equal(x0p, x0[rows]) and torch.equal(hp, h[rows])


def _model(L, seed, prune=True, V=3001):
    from mrm_b200.models import TwoTowerModel
    m = TwoTowerModel(vocab_size=V, tabular_input_dim=17, num_genders=3, num_countries=50, max_seq_len=L,
                      user_embedding_dim=256, item_embedding_dim=256, use_lora=True, seed=seed)
    m.engine.prune_last_layer = prune
    return m


def _tower(model, windows, gender, country):
    model.eval()
    with torch.no_grad():
        ids = windows.cuda()
        return model.get_user_embedding(ids, (ids != 0).long(), gender.cuda(), country.cuda())


def _oracle(model, windows, gender, country):
    from oracle import two_tower_oracle as oracle
    sd = {k: v.detach().cpu().double() for k, v in model.engine.p.items()}
    u = oracle.user_tower(sd, windows, gender, country, (windows != 0).long())
    return F.normalize(u, p=2, dim=1)


def _bf16_ulps(a, b):
    """Largest distance in bf16 units in the last place between two bf16 tensors of equal signs (0 when equal)."""
    ia, ib = a.view(torch.int16).int(), b.view(torch.int16).int()
    same_sign = (ia < 0) == (ib < 0)
    d = torch.where(same_sign, (ia - ib).abs(), torch.full_like(ia, 1 << 20))
    d = torch.where(a.float() == b.float(), torch.zeros_like(d), d)
    return int(d.max().item())


@gpu
@pytest.mark.parametrize("L,prune", [(200, True), (512, True), (2048, True), (200, False), (2048, False)])
def test_sessions_follow_the_full_tower(L, prune):
    """Users opened at lengths 1, L/2, L - 3 and L - 3, plus one never-opened slot, append one item at a time for 5
    steps (through the full window and past it, where the window shifts). After every append the embedding is within
    3e-3 of get_user_embedding on the same window; at the first and last step within 1e-2 of the fp64 oracle. Layer 0's
    cached K / V of the appended positions equal the full tower's within one bf16 ulp."""
    model = _model(L, seed=7 + L, prune=prune)
    V = model.engine.cfg.vocab_size
    from mrm_b200.sessions import UserSessions
    sess = UserSessions(model, capacity=9)
    g = torch.Generator().manual_seed(L)
    slots = [6, 2, 8, 0]
    lens = [1, L // 2, L - 3, L - 3]
    hist = [torch.randint(1, V, (n,), generator=g).tolist() for n in lens]
    ids = torch.zeros(4, L, dtype=torch.long)
    for i, h in enumerate(hist):
        ids[i, :len(h)] = torch.tensor(h)
    gender = torch.tensor([0, 1, 2, 1])
    country = torch.tensor([3, 49, 0, 7])
    u0 = sess.open(slots, ids[:, :max(lens)], user_gender=gender, user_country=country)
    assert (u0 - _tower(model, ids, gender, country)).abs().max().item() == 0.0
    fresh = 4
    all_slots = slots + [fresh]
    hist.append([])
    gender = torch.cat([gender, torch.tensor([0])])
    country = torch.cat([country, torch.tensor([0])])
    worst_tower = worst_oracle = 0.0
    ulps = []
    steps = 5
    for step in range(steps):
        new = torch.randint(1, V, (5,), generator=g)
        u = sess.append(all_slots, new)
        refilled = [len(h) == L for h in hist]          # full windows shift and go through the whole tower
        for i in range(5):
            hist[i] = (hist[i] + [int(new[i])])[-L:]
        win = torch.zeros(5, L, dtype=torch.long)
        for i, h in enumerate(hist):
            win[i, :len(h)] = torch.tensor(h)
        assert torch.equal(sess.window[torch.tensor(all_slots)].cpu(), win)
        assert sess.lengths[all_slots].tolist() == [len(h) for h in hist]
        want = _tower(model, win, gender, country)
        err = (u - want).abs().max().item()
        worst_tower = max(worst_tower, err)
        assert err <= 3e-3, (step, err)
        if step == 0:
            # the never-opened slot's first append is the tower on a one-item history
            assert (u[4] - want[4]).abs().max().item() <= 3e-3
        if step in (0, steps - 1):
            ref = _oracle(model, win, gender, country)
            e = (u.cpu().double() - ref).abs().max().item()
            worst_oracle = max(worst_oracle, e)
            assert e <= 1e-2, (step, e)
        # layer 0 K / V of the positions appended incrementally (rows that are not full windows)
        ws = model.engine.workspace(5, L)
        kv = ws["qkv_0"].view(5, L, 3, 4, 64)
        for i, s in enumerate(all_slots):
            if refilled[i]:
                continue
            p = len(hist[i]) - 1
            ulps.append(_bf16_ulps(sess.k_cache[0][s, :, p], kv[i, p, 1]))
            ulps.append(_bf16_ulps(sess.v_cache[0][s, :, p], kv[i, p, 2]))
    print("sessions", L, prune, "worst vs tower", worst_tower, "vs oracle", worst_oracle,
          "layer-0 K/V ulps: max", max(ulps), "bit-equal rows", sum(u == 0 for u in ulps), "of", len(ulps))
    assert max(ulps) <= 1


@gpu
def test_session_recommend_matches_oracle():
    """recommend on session embeddings excludes the windows' ids and returns the canonical top 10 of the session
    embedding (oracle.recommend); the same selection replayed over three catalog shards and merged agrees."""
    from mrm_b200 import retrieval, synthetic
    from mrm_b200.sessions import UserSessions
    from oracle import two_tower_oracle as oracle
    from test_recommend_exclusion import _assert_no_excluded, _assert_same_ranking
    V, B, L = 2001, 37, 200
    model = _model(L, seed=4, V=V)
    table = synthetic.make_catalog(V - 1, 256, seed=9)
    index = retrieval.CatalogIndex(table)
    g = torch.Generator().manual_seed(2)
    ids = torch.randint(1, V, (B, L), generator=g)
    lengths = torch.randint(1, L + 1, (B,), generator=g)
    lengths[:3] = L
    ids[torch.arange(L)[None, :] >= lengths[:, None]] = 0
    sess = UserSessions(model, capacity=64)
    slots = torch.randperm(64, generator=g)[:B]
    sess.open(slots, ids)
    for _ in range(2):
        sess.append(slots, torch.randint(1, V, (B,), generator=g))
    idx, score = sess.recommend(slots, index, k=10)
    win = sess.window[slots.cuda()].cpu()
    emb = sess.emb[slots.cuda()].cpu()
    for b in range(B):
        want_s, want_i = oracle.recommend(emb[b], table, [h for h in win[b].tolist() if h], 10)
        _assert_same_ranking(idx[b], score[b], want_i, want_s)
    _assert_no_excluded(idx.cpu(), win)
    # emulated shards: per-shard top 10 with the same exclusions, merged
    u = F.normalize(sess.emb[slots.cuda()], p=2, dim=1, eps=1e-8)
    exclude = retrieval.Exclusions(sess.window[slots.cuda()], index.vocab_size)
    cuts = [0, 555, 1300, V]
    parts_i, parts_s = [], []
    for a, b in zip(cuts[:-1], cuts[1:]):
        i, s, _ = retrieval.retrieve_topk(u, retrieval.CatalogIndex(table, shard=(a, b - a)), 10, exclude=exclude)
        parts_i.append(i)
        parts_s.append(s)
    mi, ms = retrieval.merge_topk(torch.stack(parts_s), torch.stack(parts_i))
    assert torch.equal(mi.long(), idx) and torch.equal(ms, score)


@gpu
def test_session_guards():
    from mrm_b200.sessions import UserSessions
    V, L = 101, 16
    model = _model(L, seed=1, V=V)
    sess = UserSessions(model, capacity=4)
    ids = torch.tensor([[5, 6, 7, 0], [9, 0, 0, 0]])
    sess.open([1, 3], ids)
    with pytest.raises(ValueError):
        sess.append([1, 1], [3, 4])                       # duplicate slot
    with pytest.raises(ValueError):
        sess.append([4], [3])                             # slot outside [0, capacity)
    with pytest.raises(ValueError):
        sess.append([-1], [3])
    with pytest.raises(ValueError):
        sess.append([1], [0])                             # item id outside [1, V)
    with pytest.raises(ValueError):
        sess.append([1], [V])
    with pytest.raises(ValueError):
        sess.open([0], torch.zeros(1, 4, dtype=torch.long))                 # empty history
    with pytest.raises(ValueError):
        sess.open([0], torch.tensor([[1, 0, 2, 0]]))                      # not a right-padded prefix
    with pytest.raises(ValueError):
        sess.open([0], torch.ones(1, L + 1, dtype=torch.long))             # longer than max_seq_len
    with pytest.raises(ValueError):
        sess.open([0], torch.tensor([[1, V]]))                             # id outside the vocabulary
    with pytest.raises(ValueError):
        sess.recommend([0], None)                                          # empty slot
    sess.append([1, 3], [3, 4])
    # stale caches: after an optimizer step and after loading weights
    model.engine.adamw_step(lr=1e-3)
    with pytest.raises(RuntimeError):
        sess.append([1], [3])
    with pytest.raises(RuntimeError):
        sess.recommend([3], None)
    sess.open([1, 3], ids)
    sess.append([1, 3], [3, 4])
    model.load_state_dict(model.state_dict())
    with pytest.raises(RuntimeError):
        sess.append([3], [3])
    sess.reset([3])
    assert sess.lengths[3] == 0
    sess.append([3], [8])                                 # a reset slot starts at position 0
    assert sess.lengths[3] == 1
    # engines whose ID table is row-sharded or on peers
    m2 = _model(L, seed=2, V=V)
    m2.engine.table_rows = torch.zeros(1, 256, device="cuda")
    with pytest.raises(NotImplementedError):
        UserSessions(m2, capacity=2)
    m2.engine.table_rows, m2.engine.peer_table = None, object()
    with pytest.raises(NotImplementedError):
        UserSessions(m2, capacity=2)
    eng = model.engine
    ws = eng.session_workspace(1)
    eng.peer_table = object()
    with pytest.raises(NotImplementedError):
        eng.session_append(ws, None, None, None, None, None, None, None)
    eng.peer_table = None

