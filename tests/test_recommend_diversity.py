"""Diversified recommendations: maximal-marginal-relevance selection from each user's candidate pool
(retrieval.diversify, tt_mmr_select, tt_mmr_gather_rows) and the ``diversity`` / ``pool`` arguments of
inference.recommend_embeddings / recommend_batch and sessions.UserSessions.recommend.

Reference: `mmr_select` below, fp64 on the CPU, following the definition the kernel implements — lam = 1 - diversity,
mu = 1 - lam; sim = fp64 dot product of the fp32 rows rounded once to fp32; m_j = the largest sim to the picks so far
(0 before the first); each step takes the unpicked admissible position with the largest lam * r_j - mu * m_j (two
rounded fp64 products, one subtraction), ties to the smaller position. On 2^-7 grid catalogs every sim is exact in
any summation order, so ids and scores are compared bit for bit.
"""
import math

import pytest
import torch

GRID = 2.0 ** -7


def mmr_select(idx, rel, table, k, diversity, return_gaps=False):
    """fp64 reference: (ids int64 (U, k), scores fp32 (U, k)) in pick order, -1 / -inf where the pool runs out; with
    ``return_gaps`` also each step's objective margin over the runner-up (U, k) fp64 (inf when there is none)."""
    lam = 1.0 - float(diversity)
    mu = 1.0 - lam
    idx, rel, table = idx.long().cpu(), rel.float().cpu(), table.float().cpu()
    U, P = idx.shape
    out_i = torch.full((U, k), -1, dtype=torch.long)
    out_s = torch.full((U, k), float("-inf"), dtype=torch.float32)
    gaps = torch.full((U, k), float("inf"), dtype=torch.float64)
    for u in range(U):
        free = idx[u] >= 0
        rows = table[idx[u].clamp(min=0)].double()
        r = rel[u].double()
        m = torch.zeros(P, dtype=torch.float64)
        for t in range(k):
            if not free.any():
                break
            obj = torch.where(free, lam * r - mu * m, torch.full_like(r, float("-inf")))
            j = int(torch.argmax(obj))                   # the first maximum: ties go to the smaller position
            rest = obj.clone()
            rest[j] = float("-inf")
            if math.isfinite(rest.max().item()):
                gaps[u, t] = (obj[j] - rest.max()).item()
            out_i[u, t], out_s[u, t] = idx[u, j], rel[u, j]
            free[j] = False
            sim = (rows @ rows[j]).float().double()
            m = sim if t == 0 else torch.maximum(m, sim)
    return (out_i, out_s, gaps) if return_gaps else (out_i, out_s)


# ---- 1. the reference on hand-made rows (CPU) ----------------------------------------------------------------------
def _hand_pool():
    """5 items: 1 and 2 are the same direction, 3 orthogonal to them, 4 opposite to 1; pool in canonical order."""
    table = torch.zeros(6, 256)
    table[1, 0] = 1.0
    table[2, 0] = 1.0
    table[3, 1] = 1.0
    table[4, 0] = -1.0
    table[5, 2] = 1.0
    idx = torch.tensor([[1, 2, 3, 4, -1, -1]])
    rel = torch.tensor([[0.9, 0.8, 0.5, 0.4, float("-inf"), float("-inf")]])
    return idx, rel, table


def test_reference_lambda_one_is_the_canonical_top_k():
    idx, rel, table = _hand_pool()
    i, s = mmr_select(idx, rel, table, 4, 0.0)
    assert i.tolist() == [[1, 2, 3, 4]] and torch.equal(s, rel[:, :4])


def test_reference_lambda_zero_picks_farthest_first():
    idx, rel, table = _hand_pool()
    i, _ = mmr_select(idx, rel, table, 4, 1.0)
    # c_0 first; then the smallest max-similarity: item 4 (-1) beats 3 (0) and 2 (+1); then 3; then 2
    assert i.tolist() == [[1, 4, 3, 2]]


def test_reference_tie_goes_to_the_smaller_position():
    table = torch.zeros(4, 256)
    table[1, 0] = table[2, 1] = table[3, 2] = 1.0
    idx = torch.tensor([[3, 1, 2]])
    rel = torch.tensor([[0.5, 0.5, 0.5]])
    i, _ = mmr_select(idx, rel, table, 3, 0.5)
    assert i.tolist() == [[3, 1, 2]]


def test_reference_never_picks_the_minus_one_tail():
    idx, rel, table = _hand_pool()
    i, s = mmr_select(idx, rel, table, 6, 0.7)
    assert sorted(i[0, :4].tolist()) == [1, 2, 3, 4]
    assert i[0, 4:].tolist() == [-1, -1] and torch.isneginf(s[0, 4:]).all()


# ---- GPU helpers -----------------------------------------------------------------------------------------------------
def _grid_setup(n_items, n_users, seed):
    from mrm_b200 import synthetic
    table = synthetic.make_catalog(n_items, 256, seed=seed, grid=GRID)
    users, _ = synthetic.make_queries(table, n_users, seed=seed + 1, noise=5.0, grid=GRID)
    return table, users


def _pool(users, index, P, ex=None):
    """The exact top P admissible candidates from the GPU path: (ids int32, scores fp32) (U, P)."""
    from mrm_b200 import retrieval
    exclude = None if ex is None else retrieval.Exclusions(ex.cuda(), index.vocab_size)
    i, s, _ = retrieval.retrieve_topk(users.cuda(), index, P, exclude=exclude)
    return i, s


# ---- 2. kernel against the reference on grid catalogs ---------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("P", [10, 64, 100, 129, 256])
def test_kernel_matches_reference_on_grid(P):
    from mrm_b200 import retrieval
    from oracle import two_tower_oracle as oracle
    from test_recommend_exclusion import _from_top
    table, users = _grid_setup(20_000, 48, seed=61)
    index = retrieval.CatalogIndex(table)
    ex = _from_top(oracle.retrieval_scores(users, table), 20, seed=P)
    pi, ps = _pool(users, index, P, ex)
    for k in sorted({1, 10, P}):
        if k > P:
            continue
        for div in (0.3, 0.7, 1.0):
            gi, gs = retrieval.diversify(pi, ps, index, k, div)
            torch.cuda.synchronize()
            wi, ws = mmr_select(pi, ps, table, k, div)
            assert torch.equal(gi.cpu().long(), wi), (P, k, div)
            assert torch.equal(gs.cpu(), ws), (P, k, div)
        gi, gs = retrieval.diversify(pi, ps, index, k, 0.0)        # lambda = 1: the pool's first k
        assert torch.equal(gi, pi[:, :k]) and torch.equal(gs, ps[:, :k]), (P, k)


# ---- 3. generic floats -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_kernel_matches_reference_on_generic_floats():
    """Gaussian unit rows, 2 000 users, P = 100, k = 10. Ids equal the reference for every user, except where the
    reference's objective margin at the first differing step is below the fp32 rounding of sim (then the order of the
    fp64 sums may legitimately decide)."""
    from mrm_b200 import retrieval, synthetic
    table = synthetic.make_catalog(50_000, 256, seed=71)
    users, _ = synthetic.make_queries(table, 2000, seed=72, noise=3.0)
    index = retrieval.CatalogIndex(table)
    pi, ps = _pool(users, index, 100)
    gi, gs = retrieval.diversify(pi, ps, index, 10, 0.3)
    wi, ws, gaps = mmr_select(pi, ps, table, 10, 0.3, return_gaps=True)
    gi = gi.cpu().long()
    print(f"smallest objective margin met: {gaps.min().item():.3e}")
    bad = (gi != wi).any(dim=1).nonzero().flatten().tolist()
    for u in bad:
        t = int((gi[u] != wi[u]).nonzero()[0])
        # |sim| <= 1: one fp32 rounding of sim moves mu * m by at most mu * 2^-24
        assert gaps[u, t].item() <= 0.3 * 2.0 ** -23, (u, t, gaps[u, t].item())
    assert len(bad) <= 20, bad
    ok = (gi == wi).all(dim=1)
    assert torch.equal(gs.cpu()[ok], ws[ok])


# ---- 4. near-duplicate versions of songs -----------------------------------------------------------------------------
def _versions_catalog(n_songs=3000, seed=81):
    """Grid rows: each song has 1 to 5 versions that differ from the song's row in 6 entries. Returns (table,
    song of every item id (-1 for id 0), users = a song row plus grid noise)."""
    g = torch.Generator().manual_seed(seed)
    base = torch.randint(-128, 129, (n_songs, 256), generator=g).float() * GRID
    nver = torch.randint(1, 6, (n_songs,), generator=g)
    song = torch.repeat_interleave(torch.arange(n_songs), nver)
    rows = base[song].clone()
    for r in range(rows.shape[0]):
        cols = torch.randperm(256, generator=g)[:6]
        rows[r, cols] = torch.randint(-128, 129, (6,), generator=g).float() * GRID
    table = torch.cat([torch.zeros(1, 256), rows])
    song = torch.cat([torch.tensor([-1]), song])
    pick = torch.randint(0, n_songs, (400,), generator=g)
    users = base[pick] + torch.randint(-96, 97, (400, 256), generator=g).float() * GRID
    return table, song, users


@pytest.mark.gpu
def test_near_duplicate_versions_are_spread_out():
    from mrm_b200 import inference, retrieval
    table, song, users = _versions_catalog()
    index = retrieval.CatalogIndex(table)
    ex = torch.zeros(users.shape[0], 1, dtype=torch.long, device="cuda")
    plain, _ = inference.recommend_embeddings(users.cuda(), index, ex, 10)
    s0 = song[plain.cpu()]
    dup = [len(set(r.tolist())) < 10 for r in s0]
    assert sum(dup) > 0, "no user's plain top 10 holds two versions of one song"
    div, _ = inference.recommend_embeddings(users.cuda(), index, ex, 10, diversity=0.3)
    s1 = song[div.cpu()]
    assert all(len(set(r.tolist())) == 10 for r in s1)
    assert (div > 0).all()
    print(f"plain top 10 with a repeated song: {sum(dup)} of {len(dup)} users; diversified: 0")


# ---- 5. diversity = 0 is today's path --------------------------------------------------------------------------------
def _model(L=50, V=2001, seed=4):
    from mrm_b200.models import TwoTowerModel
    return TwoTowerModel(vocab_size=V, tabular_input_dim=17, num_genders=3, num_countries=50, max_seq_len=L,
                         user_embedding_dim=256, item_embedding_dim=256, use_lora=True, seed=seed)


def _histories(B, L, V, seed):
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1, V, (B, L), generator=g)
    lengths = torch.randint(1, L + 1, (B,), generator=g)
    ids[torch.arange(L)[None, :] >= lengths[:, None]] = 0
    return ids


@pytest.mark.gpu
def test_zero_diversity_makes_todays_calls(monkeypatch):
    from mrm_b200 import inference, ops, retrieval, synthetic
    from mrm_b200.sessions import UserSessions
    V, B, L = 2001, 21, 50
    model = _model(L, V)
    index = retrieval.CatalogIndex(synthetic.make_catalog(V - 1, 256, seed=9))
    ids = _histories(B, L, V, seed=5)
    want = inference.recommend_batch(model, index, ids, k=10)
    sess = UserSessions(model, capacity=32)
    slots = list(range(3, 3 + B))
    sess.open(slots, ids)
    want_s = sess.recommend(slots, index, k=10)

    def boom(*a, **kw):
        raise AssertionError("tt_mmr_select launched at diversity 0")
    monkeypatch.setattr(ops, "mmr_select", boom)
    for got in (inference.recommend_batch(model, index, ids, k=10, diversity=0.0),
                inference.recommend_batch(model, index, ids, k=10, diversity=0, pool=40)):
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    got = sess.recommend(slots, index, k=10, diversity=0.0, pool=10)
    assert torch.equal(got[0], want_s[0]) and torch.equal(got[1], want_s[1])
    with pytest.raises(AssertionError):
        inference.recommend_batch(model, index, ids, k=10, diversity=0.1)


# ---- 6. fewer admissible items than k --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fewer_admissible_items_than_k():
    from mrm_b200 import inference, retrieval
    table, users = _grid_setup(30, 4, seed=91)
    index = retrieval.CatalogIndex(table)
    ex = torch.zeros(4, 30, dtype=torch.long)
    ex[1, :25] = torch.arange(1, 26)
    ex[2, :25] = torch.arange(6, 31)
    ex[3] = torch.arange(1, 31)
    for pool in (10, 20, 100):
        idx, score = inference.recommend_embeddings(users.cuda(), index, ex.cuda(), 10, diversity=0.6, pool=pool)
        pi, ps = _pool(torch.nn.functional.normalize(users.cuda(), dim=1, eps=1e-8), index, pool, ex)
        wi, ws = mmr_select(pi, ps, table, 10, 0.6)
        assert torch.equal(idx.cpu(), wi) and torch.equal(score.cpu(), ws), pool
        assert (idx[0] > 0).all()
        assert (idx[1:3, 5:] == -1).all() and torch.isneginf(score[1:3, 5:]).all()
        assert (idx[3] == -1).all() and torch.isneginf(score[3]).all()
    tiny, tu = _grid_setup(3, 2, seed=93)           # a 3-item catalog, pool and k larger than it
    idx, score = inference.recommend_embeddings(tu.cuda(), retrieval.CatalogIndex(tiny),
                                                torch.zeros(2, 1, dtype=torch.long, device="cuda"), 5, diversity=0.9)
    assert (idx[:, 3:] == -1).all() and torch.isneginf(score[:, 3:]).all()
    assert sorted(idx[0, :3].tolist()) == [1, 2, 3]


# ---- 7. sharded catalogs replayed on one GPU -------------------------------------------------------------------------
@pytest.mark.gpu
def test_sharded_rows_replayed_on_one_gpu():
    """3 ragged shards each write the pool rows they own (zeros elsewhere); their sum is the gathered input, and the
    kernel in that mode is bit-equal to the plain-index result."""
    from mrm_b200 import ops, retrieval
    table, users = _grid_setup(20_000, 300, seed=101)
    V, P, k = table.shape[0], 100, 10
    index = retrieval.CatalogIndex(table)
    pi, ps = _pool(users, index, P)
    want_i, want_s = retrieval.diversify(pi, ps, index, k, 0.4)
    total = torch.zeros(300, P, 256, device="cuda")
    cuts = [0, 6001, 13777, V]
    for a, b in zip(cuts[:-1], cuts[1:]):
        shard = retrieval.CatalogIndex(table, shard=(a, b - a))
        part = torch.full((300, P, 256), float("nan"), device="cuda")
        ops.mmr_gather_rows(pi, shard.table, shard.item_base, part)
        own = (pi >= a) & (pi < b)
        assert (part[~own] == 0).all()
        total += part
    assert torch.equal(total[pi >= 0], table.cuda()[pi[pi >= 0].long()])
    lam = 1.0 - 0.4
    gi, gs = ops.mmr_select(pi, ps, k, lam, 1.0 - lam, ops.MMR_ROWS_GATHERED, total)
    assert torch.equal(gi, want_i) and torch.equal(gs, want_s)


# ---- 8. end to end ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_recommend_batch_diversified_end_to_end():
    """Histories -> CUDA user tower -> exclusion -> top P -> MMR, against get_user_embedding, an fp64 masked top P on
    the CPU and `mmr_select`. The user vector is re-normalised on two devices, so scores agree to an ulp, not bit for
    bit: a user may differ only where two of its pool's scores are within that tolerance."""
    from mrm_b200 import inference, retrieval, synthetic
    from test_recommend_exclusion import _masked_topk
    V, B, L, k, P = 2001, 37, 50, 10, 60
    model = _model(L, V)
    table = synthetic.make_catalog(V - 1, 256, seed=9)
    index = retrieval.CatalogIndex(table)
    ids = _histories(B, L, V, seed=6)
    idx, score = inference.recommend_batch(model, index, ids, k=k, diversity=0.4, pool=P)
    assert idx.dtype == torch.int64 and idx.shape == (B, k) and model.training
    model.eval()
    with torch.no_grad():
        u = model.get_user_embedding(ids.cuda(), (ids != 0).long().cuda(), torch.zeros(B, dtype=torch.long).cuda(),
                                     torch.zeros(B, dtype=torch.long).cuda()).cpu()
    model.train()
    u = torch.nn.functional.normalize(u.double(), dim=1, eps=1e-8)
    scores = u @ table.double().t()
    scores[:, 0] = float("-inf")
    pool_i, pool_s = _masked_topk(scores, ids, P)
    want_i, _ = mmr_select(pool_i, pool_s.float(), table, k, 0.4)
    n_close = 0
    for b in range(B):
        if torch.equal(idx[b].cpu(), want_i[b]):
            continue
        ps = pool_s[b]
        assert (ps[:-1] - ps[1:]).abs().min().item() <= 2e-6, (b, idx[b], want_i[b])
        n_close += 1
    assert n_close <= 3, n_close
    assert torch.allclose(score.cpu().double(), scores.gather(1, idx.cpu()), atol=2e-6)
    from test_recommend_exclusion import _assert_no_excluded
    _assert_no_excluded(idx.cpu(), ids)


@pytest.mark.gpu
def test_sessions_recommend_diversified_equals_recommend_embeddings():
    from mrm_b200 import inference, retrieval, synthetic
    from mrm_b200.sessions import UserSessions
    V, B, L = 2001, 19, 50
    model = _model(L, V)
    index = retrieval.CatalogIndex(synthetic.make_catalog(V - 1, 256, seed=9))
    ids = _histories(B, L, V, seed=7)
    sess = UserSessions(model, capacity=32)
    slots = torch.randperm(32, generator=torch.Generator().manual_seed(1))[:B]
    sess.open(slots, ids)
    sess.append(slots, torch.randint(1, V, (B,), generator=torch.Generator().manual_seed(2)))
    got_i, got_s = sess.recommend(slots, index, k=10, diversity=0.35, pool=80)
    d = slots.cuda()
    want_i, want_s = inference.recommend_embeddings(sess.emb[d], index, sess.window[d], 10, diversity=0.35, pool=80)
    assert torch.equal(got_i, want_i) and torch.equal(got_s, want_s)
    plain_i, _ = sess.recommend(slots, index, k=10)
    assert not torch.equal(got_i, plain_i)


# ---- 9. guards and determinism ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_python_guards():
    from mrm_b200 import inference, retrieval, synthetic
    from mrm_b200.sessions import UserSessions
    V = 2001
    model = _model(50, V)
    index = retrieval.CatalogIndex(synthetic.make_catalog(V - 1, 256, seed=9))
    ids = _histories(3, 50, V, seed=8)
    u = torch.randn(3, 256, device="cuda")
    ex = torch.zeros(3, 1, dtype=torch.long, device="cuda")
    sess = UserSessions(model, capacity=4)
    sess.open([0, 1, 2], ids)
    bad = [dict(diversity=-0.1), dict(diversity=1.5), dict(diversity=float("nan")), dict(diversity=0.3, pool=9),
           dict(diversity=0.3, pool=257), dict(diversity=0.0, pool=9)]
    for kw in bad:
        with pytest.raises(ValueError):
            inference.recommend_embeddings(u, index, ex, 10, **kw)
        with pytest.raises(ValueError):
            inference.recommend_batch(model, index, ids, k=10, **kw)
        with pytest.raises(ValueError):
            sess.recommend([0, 1, 2], index, k=10, **kw)
    pi, ps = _pool(u.cpu(), index, 20)
    for k, div in ((0, 0.3), (21, 0.3), (5, -0.5), (5, float("nan"))):
        with pytest.raises(ValueError):
            retrieval.diversify(pi, ps, index, k, div)


@pytest.mark.gpu
def test_c_guards_reject_before_launch_and_runs_are_bit_identical():
    from mrm_b200 import ops, retrieval
    from mrm_b200._lib import TTError, lib
    table, users = _grid_setup(5000, 64, seed=111)
    index = retrieval.CatalogIndex(table)
    pi, ps = _pool(users, index, 256)
    oi = torch.full((64, 256), 7, device="cuda", dtype=torch.int32)
    os_ = torch.full((64, 256), 7.0, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    T, N = index.table.data_ptr(), index.num_rows

    def call(U=64, P=256, k=10, lam=0.5, mu=0.5, source=0, idx=pi.data_ptr(), sc=ps.data_ptr(), rows=T,
             out_i=oi.data_ptr(), out_s=os_.data_ptr()):
        return lib().tt_mmr_select(idx, sc, U, P, k, lam, mu, source, rows, 0, N, out_i, out_s, st)
    bad = [dict(k=0), dict(k=11, P=10), dict(P=257, k=10), dict(lam=1.5), dict(lam=-0.1), dict(mu=2.0),
           dict(lam=float("nan")), dict(mu=float("nan")), dict(idx=None), dict(sc=None), dict(rows=None),
           dict(out_i=None), dict(out_s=None), dict(source=2), dict(source=-1), dict(U=-1)]
    for kw in bad:
        assert call(**kw) != 0, kw
        assert b"tt_mmr_select" in lib().tt_last_error(), kw
    assert call(U=0) == 0
    torch.cuda.synchronize()
    assert (oi == 7).all() and (os_ == 7.0).all(), "a rejected call wrote its output"
    with pytest.raises(TTError):
        ops.mmr_select(pi, ps, 300, 0.5, 0.5, ops.MMR_ROWS_TABLE, index.table, 0, N)
    a = retrieval.diversify(pi, ps, index, 100, 0.3)
    b = retrieval.diversify(pi, ps, index, 100, 0.3)
    torch.cuda.synchronize()
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
def test_empty_batch_launches_nothing():
    """U = 0: tensors without storage have null data pointers; the call succeeds and launches nothing, also through
    `retrieval.diversify` on both row sources."""
    from mrm_b200 import _lib, ops, retrieval
    table, _ = _grid_setup(500, 1, seed=121)
    index = retrieval.CatalogIndex(table)
    ei = torch.empty(0, 20, device="cuda", dtype=torch.int32)
    es = torch.empty(0, 20, device="cuda")
    assert ei.data_ptr() == 0
    st = torch.cuda.current_stream().cuda_stream
    assert _lib.lib().tt_mmr_select(None, None, 0, 20, 5, 0.5, 0.5, 0, None, 0, 0, None, None, st) == 0
    assert _lib.lib().tt_mmr_gather_rows(None, 0, None, 0, 0, None, st) == 0
    i, s = retrieval.diversify(ei, es, index, 5, 0.4)
    assert i.shape == (0, 5) and s.shape == (0, 5)
    i, s = ops.mmr_select(ei, es, 5, 0.6, 0.4, ops.MMR_ROWS_GATHERED, torch.empty(0, 20, 256, device="cuda"))
    assert i.shape == (0, 5) and s.shape == (0, 5)


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


@pytest.mark.gpu
def test_sharded_index_path_on_a_one_rank_group(world1, monkeypatch):
    """`recommend_embeddings(diversity > 0)` on an index marked sharded (one shard covering the catalog, a one-rank
    NCCL group): the sharded_topk pool, the chunked gather + all-reduce of `diversify` (chunks of 7 users, so 300 users
    take 43 chunks, the last one short) and the gathered-row kernel — bit-equal to the plain index."""
    from mrm_b200 import inference, retrieval
    table, users = _grid_setup(20_000, 300, seed=131)
    V = table.shape[0]
    ex = torch.randint(1, V, (300, 30), generator=torch.Generator().manual_seed(5)).cuda()
    plain = retrieval.CatalogIndex(table)
    shard = retrieval.CatalogIndex(table, shard=(0, V))
    assert shard.is_sharded
    P = 100
    monkeypatch.setattr(retrieval, "_DIVERSIFY_CHUNK_BYTES", 7 * P * 1024)
    for k, div in ((10, 0.3), (100, 0.8)):
        want_i, want_s = inference.recommend_embeddings(users.cuda(), plain, ex, k, diversity=div, pool=P)
        got_i, got_s = inference.recommend_embeddings(users.cuda(), shard, ex, k, diversity=div, pool=P, group=world1)
        assert torch.equal(got_i, want_i) and torch.equal(got_s, want_s), (k, div)
