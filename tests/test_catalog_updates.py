"""Live catalog updates of a built retrieval index: `CatalogIndex.upsert` / `retire` / `retired_ids`
(tt_index_rows_live, tt_catalog_retire, and the retired bitmap of tt_score_topk_live / tt_exact_topk_live).

Updated rows are compared with `torch.equal` against a from-scratch `index_catalog_device` over the final live set.
Retrieval is compared bit for bit against an fp64 oracle on 2^-7 grid catalogs (every score exact), where retired
songs are columns at -inf, and against the same index without the retired set but with it in every user's
`Exclusions`.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

GRID = 2.0 ** -7
KEYS = ("target_audio", "target_image", "target_input_ids", "target_tabular")


def _oracle(users, table, K, exclude=None, retired=None):
    """canonical top K of the exact scores with item 0, ``exclude`` (U, m) and the ``retired`` ids at -inf"""
    from _lossy_catalogs import exact_scores, oracle_topk
    s = exact_scores(users, table, exclude=exclude)
    if retired is not None and retired.numel():
        s[:, retired.to(s.device)] = -float("inf")
    return oracle_topk(s, K)


def _grid(n_items, n_users, seed):
    from mrm_b200 import synthetic
    table = synthetic.make_catalog(n_items, 256, seed=seed, grid=GRID)
    users, _ = synthetic.make_queries(table, n_users, seed=seed + 1, noise=5.0, grid=GRID)
    return table, users.cuda()


def _model(V, seed=3):
    from mrm_b200 import synthetic
    from mrm_b200.models import TwoTowerModel
    m = TwoTowerModel(vocab_size=V, tabular_input_dim=17, num_genders=3, num_countries=50, max_seq_len=50,
                      user_embedding_dim=256, item_embedding_dim=256, use_lora=True, seed=seed)
    sd = synthetic.make_state_dict(m.engine.cfg, seed=seed)
    synthetic.make_item_features(m.engine.cfg, 1, V, state_dict=sd)        # non-trivial BatchNorm running stats
    m.load_state_dict(sd)
    return m


@pytest.fixture
def world1():
    """A single-rank NCCL group over a HashStore (no ports, no other process), destroyed on teardown."""
    import torch.distributed as dist
    if dist.is_initialized():
        pytest.skip("a process group already exists")
    try:
        dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1,
                                device_id=torch.device("cuda", torch.cuda.current_device()))
    except Exception as exc:       # noqa: BLE001
        pytest.skip(f"single-rank NCCL group unavailable: {exc}")
    try:
        yield dist.group.WORLD
    finally:
        dist.destroy_process_group()


# ---- 1. an updated index equals a rebuilt one, bit for bit ----------------------------------------------------------
def test_updated_index_equals_rebuilt_index():
    from mrm_b200 import retrieval, synthetic
    from mrm_b200.evaluate_metrics import index_catalog_device
    V = 25_001
    m = _model(V)
    cfg = m.engine.cfg
    bank = synthetic.make_item_features(cfg, V - 1, V, seed=72)[0]           # song i's features: row i - 1
    bank2 = synthetic.make_item_features(cfg, V - 1, V, seed=73)[0]          # changed features of re-embedded songs
    cur = {k: bank[k].clone() for k in KEYS}

    def feats(ids):
        return {k: cur[k][ids - 1].cuda() for k in KEYS}

    g = torch.Generator().manual_seed(5)
    first = torch.arange(1, 15_001)
    t32, t16 = index_catalog_device(m, feats(first), first.cuda(), V)
    index = retrieval.CatalogIndex.from_device_tables(t32, t16)
    cuts = [0, 7001, 16_411, V]
    shards = [retrieval.CatalogIndex.from_shard(t32[a:b].clone(), a, V) for a, b in zip(cuts[:-1], cuts[1:])]
    everyone = [index] + shards

    def upsert(ids, bs=131072):
        f = feats(ids)
        for ix in everyone:
            ix.upsert(m, f, ids, batch_size=bs)

    def retire(ids):
        for ix in everyone:
            ix.retire(ids)

    retire(torch.arange(15_001, V))
    assert index.retired_ids().numel() == V - 15_001
    new = torch.arange(15_001, 21_001)
    again = torch.randperm(15_000, generator=g)[:200] + 1
    for k in KEYS:
        cur[k][again - 1] = bank2[k][again - 1]
    rest = torch.cat([new[778:], again])[torch.randperm(6000 - 778 + 200, generator=g)]
    upsert(new[:1])
    upsert(new[1:778])
    upsert(rest, bs=1000)
    live = torch.arange(1, 21_001)
    gone = live[torch.randperm(live.numel(), generator=g)[:500]]
    retire(gone.cuda())
    back = gone[:50]
    upsert(back)
    retired = torch.cat([torch.arange(21_001, V), gone[50:]]).sort().values
    keep = torch.ones(V, dtype=torch.bool)
    keep[retired] = False
    keep[0] = False
    live = torch.nonzero(keep).flatten()

    def compare():
        r32, r16 = index_catalog_device(m, feats(live), live.cuda(), V)
        assert torch.equal(index.table, r32) and torch.equal(index.table_bf16, r16)
        for (a, b), sh in zip(zip(cuts[:-1], cuts[1:]), shards):
            assert torch.equal(sh.table, r32[a:b]) and torch.equal(sh.table_bf16, r16[a:b])
            assert torch.equal(sh.retired_ids().cpu(), retired[(retired >= a) & (retired < b)])
        assert torch.equal(index.retired_ids().cpu(), retired)
        rebuilt = retrieval.CatalogIndex.from_device_tables(r32, r16)
        assert index.de_max >= rebuilt.de_max and index.ne_max >= rebuilt.ne_max
        return r32

    before = compare()
    # a few training steps: upsert must use the weights the model has NOW
    batch = {k: v.cuda() for k, v in synthetic.make_batch(cfg, 32, seed=4).items()}
    opt = torch.optim.AdamW(m.parameters(), lr=2e-3)
    m.train()
    for _ in range(3):
        opt.zero_grad(set_to_none=True)
        m(batch)[0].backward()
        opt.step()
    upsert(live)
    after = compare()
    assert not torch.equal(before[live.cuda()], after[live.cuda()])


# ---- 2. retrieval against the oracle ---------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["own_top", "random", "with_exclusions"])
def test_retired_songs_never_returned_exact(case):
    from mrm_b200 import retrieval
    table, users = _grid(40_000, 300, seed=61)
    V, U = table.shape[0], users.shape[0]
    g = torch.Generator().manual_seed(7)
    full = retrieval.CatalogIndex(table)
    assert full.plan(U, 256).sample_stride > 1
    ex = None
    if case == "own_top":                         # every user's best item: every answer changes
        R = torch.unique(_oracle(users, table, 1)[0].long().flatten()).cpu()
    else:
        R = torch.randperm(V - 1, generator=g)[:2000] + 1
    if case == "with_exclusions":
        ex = torch.randint(1, V, (U, 50), generator=g).cuda()
    index = retrieval.CatalogIndex(table)
    index.retire(R)
    assert index.plan(U, 256).sample_stride > 1
    ex_all = torch.cat([R.cuda().expand(U, -1), ex if ex is not None else torch.zeros(U, 1, dtype=torch.long,
                                                                                         device="cuda")], 1)
    for K in (10, 100):
        want_i, want_s = _oracle(users, table, K, exclude=ex, retired=R)
        got_i, got_s, _ = retrieval.retrieve_topk(users, index, K,
                                                  exclude=None if ex is None else retrieval.Exclusions(ex, V))
        assert torch.equal(got_i, want_i) and torch.equal(got_s, want_s), (case, K)
        alt_i, alt_s, _ = retrieval.retrieve_topk(users, full, K, exclude=retrieval.Exclusions(ex_all, V))
        assert torch.equal(got_i, alt_i) and torch.equal(got_s, alt_s), (case, K)


# ---- 3. zero-row flood -----------------------------------------------------------------------------------------------
def test_retired_unlisted_rows_end_the_zero_row_flood():
    from _lossy_catalogs import on_grid, quantize
    from mrm_b200 import retrieval
    N, U, K = 20_000, 300, 100
    g = torch.Generator().manual_seed(17)
    c = torch.nn.functional.normalize(torch.randn(256, generator=g), dim=0)
    table = torch.zeros(N + 1, 256)
    real = torch.randperm(N, generator=g)[:N // 20] + 1
    table[real] = quantize(torch.nn.functional.normalize(torch.randn(len(real), 256, generator=g) - 2.5 * c, dim=1))
    users = quantize(torch.nn.functional.normalize(c + 0.02 * torch.randn(U, 256, generator=g), dim=1)).cuda()
    assert on_grid(table)
    unlisted = torch.ones(N + 1, dtype=torch.bool)
    unlisted[real] = False
    unlisted[0] = False
    R = torch.nonzero(unlisted).flatten()
    index = retrieval.CatalogIndex(table)
    index.retire(R)
    idx, score, nfb = retrieval.retrieve_topk(users, index, K)
    want_i, want_s = _oracle(users, table, K, retired=R)
    assert torch.equal(idx, want_i) and torch.equal(score, want_s)
    got = set(idx.flatten().tolist())
    assert got <= set(real.tolist()), "only real rows"
    print(f"\n[flood] fallback users: {nfb}")


# ---- 4. the exact fallback honours the retired set ------------------------------------------------------------------
def test_exact_fallback_honours_retired():
    from _lossy_catalogs import near_duplicate_items
    from mrm_b200 import retrieval
    table, users, groups = near_duplicate_items()
    users = users.cuda()
    g = torch.Generator().manual_seed(9)
    R = torch.cat([ids[torch.randperm(len(ids), generator=g)[:len(ids) // 3]] for ids in groups]
                  + [torch.randperm(table.shape[0] - 1, generator=g)[:500] + 1])
    R = torch.unique(R)
    index = retrieval.CatalogIndex(table)
    index.retire(R)
    for K in (10, 100):
        want_i, want_s = _oracle(users, table, K, retired=R)
        idx, score, nfb = retrieval.retrieve_topk(users, index, K)
        assert nfb > 0
        assert torch.equal(idx, want_i) and torch.equal(score, want_s), K
        print(f"\n[fallback K={K}] fallback users: {nfb}")


# ---- 5. fewer live songs than K --------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_items", [2000, 40_000])
def test_fewer_live_songs_than_k(n_items):
    from mrm_b200 import inference, retrieval
    table, users = _grid(n_items, 40, seed=91)
    V, U = table.shape[0], users.shape[0]
    kept = torch.tensor([3, 17, 1000, 1500, n_items])
    R = torch.ones(V, dtype=torch.bool)
    R[kept] = False
    R[0] = False
    index = retrieval.CatalogIndex(table)
    index.retire(torch.nonzero(R).flatten())
    want_i, want_s = _oracle(users, table, 10, retired=torch.nonzero(R).flatten())
    i, s, _ = retrieval.retrieve_topk(users, index, 10)
    assert torch.equal(i, want_i) and torch.equal(s, want_s)
    assert (i[:, 5:] == -1).all() and torch.isneginf(s[:, 5:]).all() and (i[:, :5] > 0).all()
    ex = torch.zeros(U, 1, dtype=torch.long, device="cuda")
    for div in (0.0, 0.5):
        ri, rs = inference.recommend_embeddings(users, index, ex, 10, diversity=div, pool=20)
        assert (ri[:, 5:] == -1).all() and torch.isneginf(rs[:, 5:]).all(), div
        assert set(ri[:, :5].flatten().tolist()) <= set(kept.tolist()), div


# ---- 6. sharded ------------------------------------------------------------------------------------------------------
def test_sharded_bounded_protocol_with_retired_songs():
    from _lossy_catalogs import exact_scores
    from mrm_b200 import retrieval
    table, users = _grid(40_000, 300, seed=111)
    V, U, K, kps = table.shape[0], users.shape[0], 10, 96
    g = torch.Generator().manual_seed(3)
    R1 = torch.unique(_oracle(users, table, 2)[0].long().flatten()).cpu()
    R2 = torch.randperm(V - 1, generator=g)[:3000] + 1
    full = retrieval.CatalogIndex(table)
    cuts = [0, 9001, 27_777, V]
    shards = [retrieval.CatalogIndex(table, shard=(a, b - a)) for a, b in zip(cuts[:-1], cuts[1:])]
    for batch in (R1, R2):
        for ix in [full] + shards:
            ix.retire(batch)
    R = torch.unique(torch.cat([R1, R2]))
    want_i, want_s, _ = retrieval.retrieve_topk(users, full, K)
    oi, os_ = _oracle(users, table, K, retired=R)
    assert torch.equal(want_i, oi) and torch.equal(want_s, os_)
    lists = [retrieval.retrieve_candidates(users, sh, kps) for sh in shards]
    mi, ms, bad = retrieval.merge_bounded(torch.stack([x[1] for x in lists]), torch.stack([x[0] for x in lists]),
                                          torch.stack([x[2] for x in lists]), K)
    assert not bad.any()
    assert torch.equal(mi, want_i) and torch.equal(ms, want_s)
    dead = torch.zeros(V, dtype=torch.bool, device="cuda")
    dead[R.cuda()] = True
    for (a, b), sh, (li, ls, bound, flag) in zip(zip(cuts[:-1], cuts[1:]), shards, lists):
        assert not flag.any()
        s = exact_scores(users, table[a:b], item_base=a)
        s[:, dead[a:b]] = -float("inf")
        assert not torch.isin(li[li >= 0], R.cuda().int()).any()
        listed = torch.zeros_like(s, dtype=torch.bool)
        rows = torch.arange(U, device="cuda")[:, None].expand_as(li)
        listed[rows[li >= 0], (li[li >= 0] - a).long()] = True
        s[listed] = -float("inf")
        assert (s.max(dim=1).values <= bound).all()


def test_sharded_topk_and_diversity_on_a_one_rank_group(world1):
    from mrm_b200 import inference, retrieval
    table, users = _grid(20_000, 300, seed=131)
    V = table.shape[0]
    g = torch.Generator().manual_seed(5)
    ex = torch.randint(1, V, (300, 30), generator=g).cuda()
    R = torch.randperm(V - 1, generator=g)[:1500] + 1
    plain = retrieval.CatalogIndex(table)
    shard = retrieval.CatalogIndex(table, shard=(0, V))
    for ix in (plain, shard):
        ix.retire(R)
    for K in (10, 100):
        wi, ws, _ = retrieval.retrieve_topk(users, plain, K)
        gi, gs = retrieval.sharded_topk(users, shard, K, group=world1)
        assert torch.equal(gi, wi) and torch.equal(gs, ws), K
        for bounded in (True, False):
            gi, gs = retrieval.sharded_topk(users, shard, K, group=world1, bounded=bounded)
            assert torch.equal(gi, wi) and torch.equal(gs, ws), (K, bounded)
    for k, div in ((10, 0.3), (100, 0.8)):
        want_i, want_s = inference.recommend_embeddings(users, plain, ex, k, diversity=div, pool=100)
        got_i, got_s = inference.recommend_embeddings(users, shard, ex, k, diversity=div, pool=100, group=world1)
        assert torch.equal(got_i, want_i) and torch.equal(got_s, want_s), (k, div)
        assert not torch.isin(got_i, R.cuda()).any()


# ---- 7. end to end ---------------------------------------------------------------------------------------------------
def test_end_to_end_never_returns_retired_songs():
    from mrm_b200 import inference, retrieval, synthetic
    from mrm_b200.evaluate_metrics import calculate_metrics_global
    from mrm_b200.sessions import UserSessions
    V, B, L = 3001, 37, 50
    m = _model(V, seed=4)
    cfg = m.engine.cfg
    table = synthetic.make_catalog(V - 1, 256, seed=9)
    g = torch.Generator().manual_seed(6)
    ids = torch.randint(1, V, (B, L), generator=g)
    ids[torch.arange(L)[None, :] >= torch.randint(1, L + 1, (B,), generator=g)[:, None]] = 0
    loader = [synthetic.make_batch(cfg, 64, seed=30 + i) for i in range(3)]
    # the songs these users would get: retired, every answer changes
    index0 = retrieval.CatalogIndex(table)
    top = inference.recommend_batch(m, index0, ids, k=3)[0]
    R = torch.unique(torch.cat([top.flatten().cpu(), torch.randperm(V - 1, generator=g)[:300] + 1]))
    index = retrieval.CatalogIndex(table)
    index.retire(R)
    rebuilt_table = table.clone()
    rebuilt_table[R] = 0
    rebuilt = retrieval.CatalogIndex(rebuilt_table)
    assert torch.equal(index.table.cpu(), rebuilt_table)
    hist = ids * (ids != 0)
    ex_plus = torch.cat([hist, R.expand(B, -1)], 1)
    got = inference.recommend_batch(m, index, ids, k=10)
    want = inference.recommend_batch(m, rebuilt, ids, k=10, exclude_ids=ex_plus)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    assert not torch.isin(got[0].cpu(), R).any()
    sess = UserSessions(m, capacity=64)
    slots = list(range(5, 5 + B))
    sess.open(slots, ids)
    got_s = sess.recommend(slots, index, k=10)
    d = torch.tensor(slots).cuda()
    want_s = sess.recommend(slots, rebuilt, k=10, exclude_ids=torch.cat([sess.window[d], R.cuda().expand(B, -1)], 1))
    assert torch.equal(got_s[0], want_s[0]) and torch.equal(got_s[1], want_s[1])
    assert not torch.isin(got_s[0].cpu(), R).any()
    # global metrics: the same as retrieving from the rebuilt catalog with the retired songs excluded for everyone
    kl = [10, 20, 50]
    got_m = calculate_metrics_global(m, loader, table, torch.device("cuda"), k_list=kl, index=index)
    m.eval()
    with torch.no_grad():
        users = torch.cat([m.get_user_embedding(b["history_ids"].cuda(), b["history_mask"].cuda(),
                                                b["user_gender"].cuda(), b["user_country"].cuda()) for b in loader])
    targets = torch.cat([b["target_id"] for b in loader]).cuda()
    U = users.shape[0]
    wi, _, _ = retrieval.retrieve_topk(users, rebuilt, 50,
                                       exclude=retrieval.Exclusions(R.cuda().expand(U, -1).contiguous(), V))
    gi, _, _ = retrieval.retrieve_topk(users, index, 50)
    assert torch.equal(gi, wi) and not torch.isin(gi.cpu().long(), R).any()
    rec, ndcg = retrieval.rank_metrics(wi, targets, kl)
    for j, k in enumerate(kl):
        assert got_m[f"Recall@{k}"] == rec[j].cpu().mean().item()
        assert got_m[f"NDCG@{k}"] == ndcg[j].cpu().mean().item()


# ---- 8. the path without retire is today's -------------------------------------------------------------------------
def test_without_retire_the_calls_are_todays(monkeypatch):
    from mrm_b200 import _lib, retrieval
    table, users = _grid(40_000, 300, seed=141)
    index = retrieval.CatalogIndex(table)
    calls = []

    class Rec:
        def __getattr__(self, name):
            calls.append(name)
            return getattr(_lib.lib(), name)
    monkeypatch.setattr(retrieval, "lib", lambda: Rec())
    want_i, want_s, _ = retrieval.retrieve_topk(users, index, 100)
    retrieval.retrieve_candidates(users, index, 64)
    assert index.retired_bits is None
    assert "tt_score_topk_excl" in calls and not any(c.endswith("_live") for c in calls), calls
    # an all-zero bitmap retires nothing: bit-identical results through the masked kernels
    calls.clear()
    index.retired_bits = torch.zeros((index.num_rows + 255) // 256 * 8, device="cuda", dtype=torch.int32)
    got_i, got_s, _ = retrieval.retrieve_topk(users, index, 100)
    assert "tt_score_topk_live" in calls and "tt_score_topk_excl" not in calls
    assert torch.equal(got_i, want_i) and torch.equal(got_s, want_s)
    assert index.retired_ids().numel() == 0


def test_all_zero_bitmap_in_the_exact_fallback():
    from _lossy_catalogs import near_duplicate_items
    from mrm_b200 import retrieval
    table, users, _ = near_duplicate_items()
    users = users.cuda()
    index = retrieval.CatalogIndex(table)
    want = retrieval.retrieve_topk(users, index, 100)
    index.retired_bits = torch.zeros((index.num_rows + 255) // 256 * 8, device="cuda", dtype=torch.int32)
    got = retrieval.retrieve_topk(users, index, 100)
    assert want[2] > 0 and got[2] == want[2]
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


# ---- 9. guards -------------------------------------------------------------------------------------------------------
def test_python_guards_raise_before_any_launch():
    from mrm_b200 import _lib, retrieval, synthetic
    V = 1001
    m = _model(V, seed=5)
    feats, ids = synthetic.make_item_features(m.engine.cfg, 20, V, seed=8)
    index = retrieval.CatalogIndex(synthetic.make_catalog(V - 1, 256, seed=2))
    t32, t16 = index.table.clone(), index.table_bf16.clone()
    n0 = _lib.launch_count
    bad_ids = [torch.tensor([0, 5]), torch.tensor([5, V]), torch.tensor([-3, 5]), torch.tensor([7, 9, 7]),
               torch.tensor([1.0, 2.0]), torch.tensor([[1, 2]])]
    for b in bad_ids:
        with pytest.raises(ValueError):
            index.retire(b)
    for b in bad_ids[:4]:
        f = {k: v[:b.numel()] for k, v in feats.items()}
        with pytest.raises(ValueError):
            index.upsert(m, f, b)
    bad_feats = [{k: v[:19] for k, v in feats.items()}, {k: v[:, :64] for k, v in feats.items()},
                 {k: v for k, v in feats.items() if k != "target_audio"},
                 {k: v.long() for k, v in feats.items()}]
    for f in bad_feats:
        with pytest.raises(ValueError):
            index.upsert(m, f, ids)
    assert _lib.launch_count == n0 and index.retired_bits is None
    assert torch.equal(index.table, t32) and torch.equal(index.table_bf16, t16)


def test_c_entry_points_reject_bad_ids_before_launch():
    from mrm_b200 import _lib, retrieval, synthetic
    V = 1001
    index = retrieval.CatalogIndex(synthetic.make_catalog(V - 1, 256, seed=2))
    bits = torch.zeros((V + 255) // 256 * 8, device="cuda", dtype=torch.int32)
    t32, t16 = index.table.clone(), index.table_bf16.clone()
    l = _lib.lib()
    y = torch.randn(3, 256, device="cuda")
    w, b = torch.ones(256, device="cuda"), torch.zeros(256, device="cuda")
    stats = torch.zeros(2, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    for bad in ([0, 5, 6], [5, V, 6], [5, 6, 5], [-1, 2, 3]):
        i = torch.tensor(bad, device="cuda", dtype=torch.int64)
        assert l.tt_catalog_retire(i.data_ptr(), 3, V, 0, V, index.table.data_ptr(), index.table_bf16.data_ptr(),
                                   bits.data_ptr(), s) != 0
        assert l.tt_index_rows_live(y.data_ptr(), 3, w.data_ptr(), b.data_ptr(), i.data_ptr(), V, 0, V,
                                    index.table.data_ptr(), index.table_bf16.data_ptr(), bits.data_ptr(),
                                    stats.data_ptr(), s) != 0
    i = torch.tensor([4, 5, 6], device="cuda", dtype=torch.int64)
    assert l.tt_catalog_retire(i.data_ptr(), 3, V, 10, V, index.table.data_ptr(), index.table_bf16.data_ptr(),
                               bits.data_ptr(), s) != 0               # rows [10, V + 10) outside the catalog
    assert l.tt_catalog_retire(i.data_ptr(), 3, V, 0, V, index.table.data_ptr(), index.table_bf16.data_ptr(),
                               None, s) != 0
    torch.cuda.synchronize()
    assert not bits.any() and not stats.any()
    assert torch.equal(index.table, t32) and torch.equal(index.table_bf16, t16)
    # a good call goes through, and retiring twice changes nothing more
    for _ in range(2):
        assert l.tt_catalog_retire(i.data_ptr(), 3, V, 0, V, index.table.data_ptr(), index.table_bf16.data_ptr(),
                                   bits.data_ptr(), s) == 0
    torch.cuda.synchronize()
    assert bits[0].item() == 0b1110000 and not index.table[4:7].any() and torch.equal(index.table[7:], t32[7:])
