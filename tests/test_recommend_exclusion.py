"""Seen-item exclusion inside the selection kernels (retrieval.Exclusions, tt_score_topk_excl, tt_exact_topk_excl)
and the batched recommendation built on it (inference.recommend_batch).

Oracle: the reference's masking (src/inference.py:296-302), i.e. the fp32 score matrix with column 0 and every excluded
column set to -inf, canonical top K (score descending, item id ascending). Where ids and scores are compared bit for
bit the catalogs are on the 2^-7 grid, on which every dot product is exact in any precision and order.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

GRID = 2.0 ** -7
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _grid_catalog(n_items, n_users, seed):
    from mrm_b200 import synthetic
    table = synthetic.make_catalog(n_items, 256, seed=seed, grid=GRID)
    users, _ = synthetic.make_queries(table, n_users, seed=seed + 1, noise=5.0, grid=GRID)
    return table, users


def _from_top(scores, m, seed, spread=2):
    """(U, m) histories of each user's own best items: its best one plus m - 1 others of its top spread * m
    (canonical order), shuffled — the exclusion changes every answer."""
    from oracle import two_tower_oracle as oracle
    g = torch.Generator().manual_seed(seed)
    _, best = oracle.canonical_topk(scores, spread * m)
    r = torch.rand(best.shape, generator=g)
    r[:, 0] = -1.0
    pick = r.argsort(dim=1)[:, :m]
    pick = torch.gather(pick, 1, torch.rand(pick.shape, generator=g).argsort(dim=1))
    return torch.gather(best, 1, pick)


def _masked_topk(scores, ex, K):
    """Oracle: columns of ``ex`` (0 / out-of-range ids = no entry) and column 0 at -inf, canonical top K; positions
    without an admissible item are id -1, score -inf."""
    from oracle import two_tower_oracle as oracle
    V = scores.shape[1]
    s = scores.clone()
    s[:, 0] = float("-inf")
    ex = torch.where((ex > 0) & (ex < V), ex, torch.zeros_like(ex))
    s.scatter_(1, ex, float("-inf"))
    v, i = oracle.canonical_topk(s, K)
    i = torch.where(torch.isneginf(v), torch.full_like(i, -1), i)
    return i, v


def _assert_no_excluded(idx, ex):
    for u in range(idx.shape[0]):
        got = set(idx[u].tolist())
        assert 0 not in got
        assert not got & (set(ex[u].tolist()) - {0}), u


@pytest.mark.parametrize("m", [50, 300, 512, 4096])
def test_excluded_topk_bit_exact_on_grid(m):
    """20 000-item grid catalog, 300 users (not a multiple of the 256-user tile), histories taken from each user's
    own best items: ids and scores equal the masked oracle bit for bit, for K = 10 and 100. m >= 300 is beyond what
    an exact top-(k + m) post-filter can take (at most 256 candidates per user)."""
    from mrm_b200 import retrieval
    from oracle import two_tower_oracle as oracle
    table, users = _grid_catalog(20_000, 300, seed=11)
    index = retrieval.CatalogIndex(table)
    scores = oracle.retrieval_scores(users, table)
    ex = _from_top(scores, m, seed=m)
    exclude = retrieval.Exclusions(ex.cuda(), index.vocab_size)
    for K in (10, 100):
        idx, score, _ = retrieval.retrieve_topk(users.cuda(), index, K, exclude=exclude)
        torch.cuda.synchronize()
        want_i, want_s = _masked_topk(scores, ex, K)
        assert torch.equal(idx.cpu().long(), want_i), (m, K)
        assert torch.equal(score.cpu(), want_s), (m, K)
        _, plain = oracle.canonical_topk(scores, K)
        assert (want_i != plain).any(dim=1).all(), "the exclusion must change every user's answer"


def test_empty_and_unclean_exclusion_rows():
    """All-zero rows leave the result bit-identical to no exclusion. Rows with duplicates, negative ids, ids >= V and
    empty slots build the same lists and bitmaps, and give the same result, as their cleaned form."""
    from mrm_b200 import retrieval
    from oracle import two_tower_oracle as oracle
    table, users = _grid_catalog(20_000, 300, seed=21)
    V = table.shape[0]
    index = retrieval.CatalogIndex(table)
    u = users.cuda()
    base_i, base_s, _ = retrieval.retrieve_topk(u, index, 100)
    zero = retrieval.Exclusions(torch.zeros(300, 64, dtype=torch.long, device="cuda"), V)
    zi, zs, _ = retrieval.retrieve_topk(u, index, 100, exclude=zero)
    assert torch.equal(zi, base_i) and torch.equal(zs, base_s)

    scores = oracle.retrieval_scores(users, table)
    clean = _from_top(scores, 40, seed=3)
    g = torch.Generator().manual_seed(4)
    junk = torch.cat([clean, clean[:, :15], -torch.randint(1, 1000, (300, 5), generator=g),
                      V + torch.randint(0, 1000, (300, 5), generator=g), torch.zeros(300, 7, dtype=torch.long)], 1)
    junk = torch.gather(junk, 1, torch.rand(junk.shape, generator=g).argsort(dim=1))
    a = retrieval.Exclusions(clean.cuda(), V)
    b = retrieval.Exclusions(junk.cuda(), V)
    assert (a.cnt.cpu() == 40).all() and torch.equal(a.cnt, b.cnt)
    assert torch.equal(a.ids[:, :40].cpu().long(), clean.sort(dim=1).values)
    assert torch.equal(a.ids[:, :40], b.ids[:, :40]) and torch.equal(a.bits, b.bits)
    ai, as_, _ = retrieval.retrieve_topk(u, index, 100, exclude=a)
    bi, bs, _ = retrieval.retrieve_topk(u, index, 100, exclude=b)
    assert torch.equal(ai, bi) and torch.equal(as_, bs)
    want_i, want_s = _masked_topk(scores, clean, 100)
    assert torch.equal(ai.cpu().long(), want_i) and torch.equal(as_.cpu(), want_s)
    with pytest.raises(ValueError):
        retrieval.Exclusions(torch.ones(2, 4097, dtype=torch.long, device="cuda"), V)


def test_excluded_topk_keeps_the_canonical_tie_order():
    """Coarse grid: thousands of exact score ties. With each user's best items excluded, the ties among the
    remaining items still come out in ascending item id."""
    from mrm_b200 import retrieval, synthetic
    from oracle import two_tower_oracle as oracle
    gold = torch.load(os.path.join(GOLDEN, "retrieval_grid_coarse.pt"), weights_only=False)
    table = synthetic.make_catalog(gold["num_items"], 256, seed=gold["seed"], grid=gold["grid"])
    users, _ = synthetic.make_queries(table, gold["num_users"], seed=gold["seed"] + 1, noise=gold["noise"],
                                      grid=gold["grid"])
    index = retrieval.CatalogIndex(table)
    scores = oracle.retrieval_scores(users, table)
    ex = _from_top(scores, 120, seed=9)
    idx, score, _ = retrieval.retrieve_topk(users.cuda(), index, 100,
                                            exclude=retrieval.Exclusions(ex.cuda(), index.vocab_size))
    torch.cuda.synchronize()
    want_i, want_s = _masked_topk(scores, ex, 100)
    assert torch.equal(idx.cpu().long(), want_i) and torch.equal(score.cpu(), want_s)
    ties = (want_s[:, 1:] == want_s[:, :-1]).sum().item()
    assert ties > 1000, ties


def test_excluded_topk_large_catalog_needs_no_fallback():
    """300 001 items (the sample pass seeds the thresholds), 1500 users, 512 excluded ids per user taken from its
    own top 1000: the sample-rank correction keeps every user on the fast path (no exact fallback), and the result
    matches an fp64 torch scoring with the same masking (the property checks of test_large_catalog_properties)."""
    from mrm_b200 import retrieval, synthetic
    N, U, K = 300_001, 1500, 100
    table = synthetic.make_catalog(N, 256, seed=77)
    users, _ = synthetic.make_queries(table, U, seed=78, noise=3.0)
    index = retrieval.CatalogIndex(table)
    ref = users.cuda().double() @ table.cuda().double().t()
    ref[:, 0] = -float("inf")
    top = ref.topk(1000, dim=1).indices
    g = torch.Generator(device="cuda").manual_seed(3)
    ex = torch.gather(top, 1, torch.rand(top.shape, device="cuda", generator=g).argsort(dim=1)[:, :512])
    idx, score, nfb = retrieval.retrieve_topk(users.cuda(), index, K, exclude=retrieval.Exclusions(ex, N + 1))
    torch.cuda.synchronize()
    assert nfb == 0
    assert (idx > 0).all() and (idx <= N).all()
    assert (score[:, 1:] <= score[:, :-1]).all()
    ref.scatter_(1, ex, -float("inf"))
    rv, ri = torch.sort(ref, dim=1, descending=True, stable=True)
    ri, rv = ri[:, :K].int(), rv[:, :K].float()
    assert (idx == ri).float().mean().item() > 0.999
    assert (score - rv).abs().max().item() <= 1e-6
    assert (score >= rv[:, -1:] - 1e-6).all()
    assert not (idx.long().unsqueeze(2) == ex.unsqueeze(1)).any()


def test_exact_fallback_with_exclusions_agrees():
    """tt_exact_topk_excl (the per-user brute-force path) equals the main path for users with exclusions."""
    from mrm_b200 import retrieval
    from mrm_b200._lib import check, lib
    table, users = _grid_catalog(20_000, 300, seed=31)
    index = retrieval.CatalogIndex(table)
    from oracle import two_tower_oracle as oracle
    ex = _from_top(oracle.retrieval_scores(users, table), 300, seed=5)
    exclude = retrieval.Exclusions(ex.cuda(), index.vocab_size)
    K = 100
    u = users.cuda()
    idx, score, _ = retrieval.retrieve_topk(u, index, K, exclude=exclude)
    keys = torch.empty(index.num_rows, device="cuda", dtype=torch.int64)
    for row in (0, 7, 191, 299):
        oi = torch.empty(K, device="cuda", dtype=torch.int32)
        os_ = torch.empty(K, device="cuda")
        check(lib().tt_exact_topk_excl(u[row].data_ptr(), index.table.data_ptr(), index.num_rows, 0, 1, K,
                                       exclude.ids[row].data_ptr(), exclude.cnt[row:].data_ptr(), keys.data_ptr(),
                                       os_.data_ptr(), oi.data_ptr(), torch.cuda.current_stream().cuda_stream),
              "tt_exact_topk_excl")
        torch.cuda.synchronize()
        assert torch.equal(oi, idx[row]), row
        assert torch.equal(os_, score[row]), row


def test_excluded_shards_replayed_on_one_gpu():
    """The sharded protocols with exclusions, 3 ragged shards on one GPU: per-shard candidate lists written into one
    packed buffer and merged in place (as retrieval.sharded_topk exchanges them) — certified users bit-equal to the
    unsharded excluded result, >= 97 % certified; and the per-shard exact top K merged — equal for every user."""
    from mrm_b200 import retrieval
    from oracle import two_tower_oracle as oracle
    table, users = _grid_catalog(20_000, 300, seed=41)
    V, U, K = table.shape[0], 300, 100
    ex = _from_top(oracle.retrieval_scores(users, table), 300, seed=6)
    exclude = retrieval.Exclusions(ex.cuda(), V)
    u = users.cuda()
    full_i, full_s, _ = retrieval.retrieve_topk(u, retrieval.CatalogIndex(table), K, exclude=exclude)
    cuts = [0, 6001, 13777, V]
    G = len(cuts) - 1
    kps = retrieval.shard_kprime(256, G)
    allp = torch.empty(G * U, 2 * kps + 2, device="cuda", dtype=torch.int32)
    parts_i, parts_s = [], []
    for g, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        shard = retrieval.CatalogIndex(table, shard=(a, b - a))
        retrieval.retrieve_candidates(u, shard, kps, pack=allp[g * U:(g + 1) * U], exclude=exclude)
        i, s, _ = retrieval.retrieve_topk(u, shard, K, exclude=exclude)
        parts_i.append(i)
        parts_s.append(s)
    bad = torch.zeros(U, device="cuda", dtype=torch.int32)
    mi, ms = retrieval.merge_packed(allp, G, U, kps, K, bad)
    torch.cuda.synchronize()
    ok = bad == 0
    assert ok.float().mean().item() >= 0.97, ok.float().mean().item()
    assert torch.equal(mi[ok], full_i[ok]) and torch.equal(ms[ok], full_s[ok])
    ei, es = retrieval.merge_topk(torch.stack(parts_s), torch.stack(parts_i))
    assert torch.equal(ei, full_i) and torch.equal(es, full_s)
    _assert_no_excluded(full_i.cpu(), ex)


def test_fewer_admissible_items_than_k():
    """A 30-item catalog with 25 or all 30 items excluded: the tail is id -1 with score -inf."""
    from mrm_b200 import retrieval
    from oracle import two_tower_oracle as oracle
    table, users = _grid_catalog(30, 4, seed=51)
    index = retrieval.CatalogIndex(table)
    ex = torch.zeros(4, 30, dtype=torch.long)
    ex[1, :25] = torch.arange(1, 26)
    ex[2, :25] = torch.arange(6, 31)
    ex[3] = torch.arange(1, 31)
    idx, score, _ = retrieval.retrieve_topk(users.cuda(), index, 10,
                                            exclude=retrieval.Exclusions(ex.cuda(), index.vocab_size))
    torch.cuda.synchronize()
    want_i, want_s = _masked_topk(oracle.retrieval_scores(users, table), ex, 10)
    assert torch.equal(idx.cpu().long(), want_i) and torch.equal(score.cpu(), want_s)
    assert (idx[1:3, 5:] == -1).all() and torch.isneginf(score[1:3, 5:]).all()
    assert (idx[3] == -1).all() and torch.isneginf(score[3]).all()
    assert (idx[0] > 0).all()


def _assert_same_ranking(got_idx, got_score, want_idx, want_score, tol=2e-6):
    """Same ids in the same order, except that items whose exact scores are closer than `tol` may swap (the user
    vector is re-normalised on two different devices, so scores agree to an ulp, not bit for bit)."""
    got_idx, want_idx = got_idx.cpu().tolist(), want_idx.tolist()
    assert torch.allclose(got_score.cpu(), want_score, atol=tol), (got_score, want_score)
    for pos, (a, b) in enumerate(zip(got_idx, want_idx)):
        if a != b:
            assert a in want_idx, (pos, a, want_idx)
            assert abs(want_score[want_idx.index(a)].item() - want_score[pos].item()) <= tol, (pos, a, b)


def test_recommend_batch_end_to_end():
    """Histories -> CUDA user tower (max_seq_len 512) -> in-kernel exclusion -> top 10, for 37 users with full and
    right-padded histories, against get_user_embedding + oracle.recommend per user; then with exclude_ids, one user
    excluding a 700-item listening history (longer than the tower's window)."""
    from mrm_b200 import inference, retrieval, synthetic
    from mrm_b200.models import TwoTowerModel
    from oracle import two_tower_oracle as oracle
    V, B, L = 2001, 37, 512
    model = TwoTowerModel(vocab_size=V, tabular_input_dim=17, num_genders=3, num_countries=50, max_seq_len=L,
                          user_embedding_dim=256, item_embedding_dim=256, use_lora=True, seed=4)
    table = synthetic.make_catalog(V - 1, 256, seed=9)
    index = retrieval.CatalogIndex(table)
    g = torch.Generator().manual_seed(2)
    ids = torch.randint(1, V, (B, L), generator=g)
    lengths = torch.randint(1, L + 1, (B,), generator=g)
    lengths[:5] = L
    ids[torch.arange(L)[None, :] >= lengths[:, None]] = 0                 # right-padded
    gender = torch.randint(0, 3, (B,), generator=g)
    country = torch.randint(0, 50, (B,), generator=g)

    model.eval()
    with torch.no_grad():
        u = model.get_user_embedding(ids.cuda(), (ids != 0).long().cuda(), gender.cuda(), country.cuda()).cpu()
    model.train()

    idx, score = inference.recommend_batch(model, index, ids, user_gender=gender, user_country=country, k=10)
    assert idx.dtype == torch.int64 and idx.shape == (B, 10) and score.shape == (B, 10)
    assert model.training
    for b in range(B):
        hist = [h for h in ids[b].tolist() if h]
        want_s, want_i = oracle.recommend(u[b], table, hist, 10)
        _assert_same_ranking(idx[b], score[b], want_i, want_s)
    _assert_no_excluded(idx.cpu(), ids)

    ex = torch.zeros(B, 700, dtype=torch.long)
    ex[:, :L] = ids
    ex[5] = torch.randperm(V - 1, generator=g)[:700] + 1
    idx, score = inference.recommend_batch(model, index, ids, user_gender=gender, user_country=country, k=10,
                                           exclude_ids=ex)
    for b in range(B):
        want_s, want_i = oracle.recommend(u[b], table, [h for h in ex[b].tolist() if h], 10)
        _assert_same_ranking(idx[b], score[b], want_i, want_s)
    _assert_no_excluded(idx.cpu(), ex)
