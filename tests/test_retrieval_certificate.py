"""The exactness certificate of retrieval, on catalogs where bf16 scoring is lossy, against a bit-exact fp64 oracle.

Retrieval scores bf16 operands on the tensor cores and promises the exact fp32 top K in canonical order. That
rests on tt_topk_finalize: it re-scores the candidates in fp64 and certifies that the exact K-th score beats
score(T) + eps, where T is the weakest candidate key and eps = du * ne_max + nu * de_max + nu * ne_max * 2^-18
bounds |bf16-path score - exact score|; users that fail go to the brute-force fallback. The bounded shard protocol
publishes the same score(T) + eps as each shard's completeness bound.

On the 2^-7 grid fixtures elsewhere in the suite bf16 is exact and every branch of that certificate would pass
with eps = 0. Here every entry is on the 2^-20 grid (tests/_lossy_catalogs.py), so the oracle is exact while the
bf16 path misranks on purpose, and every comparison is torch.equal on ids and scores for every user. Each case
asserts that the path it targets ran (flags, fallback, uncertified users) and prints how many users took it
(run pytest with -s to see the counts).
"""
import functools

import pytest
import torch

from _lossy_catalogs import (accumulation_dominated, bf16_exact, emulate_fp32_accumulation, exact_scores,
                             lossy_gaussian, near_duplicate_items, near_duplicate_users, on_grid, oracle_topk, quantize)

pytestmark = pytest.mark.gpu

FIXTURES = {
    "items": near_duplicate_items,
    "users": near_duplicate_users,
    "gaussian": functools.partial(lossy_gaussian, 20_000, 300),
    "accumulation": accumulation_dominated,
}


@functools.lru_cache(maxsize=None)
def _index(name):
    from mrm_b200 import retrieval
    table, _, _ = FIXTURES[name]()
    return retrieval.CatalogIndex(table)


def _check_fixture(name):
    """each fixture's own property: the grid, and on which side bf16 loses information"""
    table, users, groups = FIXTURES[name]()
    assert on_grid(table) and on_grid(users)
    lossy_items, lossy_users = {"items": (True, False), "users": (False, True), "gaussian": (True, True),
                                "accumulation": (False, False)}[name]
    assert bf16_exact(table) != lossy_items and bf16_exact(users) != lossy_users
    for ids in groups:            # all members of a group are one row in bf16 (items) or score alike (users, acc.)
        assert len(ids) >= 300
        if name == "items":
            assert (table[ids].bfloat16() == table[ids[0]].bfloat16()).all()
    if name == "accumulation":
        # the model most favourable to the tensor core cannot tell the members of a group apart
        for u in range(8):
            s = emulate_fp32_accumulation(users[u:u + 1], table[groups[u % len(groups)]])
            assert (s == s[0, 0]).all()
    return table, users, groups


def _assert_rises_with_id(scores, groups, n_users):
    """the adversarial order: for a planted user the exact scores of its group rise strictly with the id"""
    for u in range(n_users):
        s = scores[u, groups[u % len(groups)].to(scores.device)]
        assert (s[1:] > s[:-1]).all(), u


def _assert_equal(idx, score, ref_idx, ref_score, what):
    bad = ((idx != ref_idx) | (score != ref_score)).any(dim=1)
    assert not bad.any(), f"{what}: {int(bad.sum())} users differ from the oracle, first {bad.nonzero()[:5].flatten().tolist()}"


# ---------------------------------------------------------------------------------------------------------------
# A. near-duplicate groups (versions of one song), lossy on the item side or on the user side
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,kprime", [(10, 256), (10, 10), (100, 256), (100, 100), (256, 256)])
@pytest.mark.parametrize("side", ["items", "users"])
def test_near_duplicate_groups_fall_back_to_the_exact_top_k(side, K, kprime):
    from mrm_b200 import retrieval
    table, users, groups = _check_fixture(side)
    index = _index(side)
    for U in (1, 300):
        u = users[:U].cuda()
        s = exact_scores(u, table)
        _assert_rises_with_id(s, groups, U)
        ref_i, ref_s = oracle_topk(s, K)
        idx, score, nfb = retrieval.retrieve_topk(u, index, K, kprime)
        print(f"\n[A {side} K={K} K'={kprime} U={U}] fallback users: {nfb}")
        _assert_equal(idx, score, ref_i, ref_s, f"A {side} U={U}")
        assert nfb > 0, "no user failed the certificate: the case tests nothing"


# ---------------------------------------------------------------------------------------------------------------
# B. generic lossy catalogs: exact for every user, and no needless fallback
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,U", [(20_000, 300), (20_000, 1500), (300_001, 300), (300_001, 1500)])
def test_lossy_random_catalog_is_exact_without_fallback(N, U):
    from mrm_b200 import retrieval
    K = 100
    table, users, _ = lossy_gaussian(N, 1500)
    users = users[:U]
    assert on_grid(table) and on_grid(users) and not bf16_exact(table) and not bf16_exact(users)
    index = retrieval.CatalogIndex(table)
    assert (index.plan(U, 256).sample_stride > 1) == (N > 100_000)      # the larger catalog takes the sample pass
    u = users.cuda()
    idx, score, nfb = retrieval.retrieve_topk(u, index, K)
    ref_i, ref_s = oracle_topk(exact_scores(u, table), K)
    print(f"\n[B N={N} U={U}] fallback users: {nfb}")
    _assert_equal(idx, score, ref_i, ref_s, "B")
    assert nfb == 0, f"{nfb} users fell back on generic data: eps is looser than it needs to be"


# ---------------------------------------------------------------------------------------------------------------
# C. accumulation-dominated catalogs: du = de = 0, eps is the accumulation slack alone
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [10, 100, 256])
def test_accumulation_dominated_catalog_falls_back(K):
    from mrm_b200 import retrieval
    table, users, groups = _check_fixture("accumulation")
    u = users.cuda()
    s = exact_scores(u, table)
    _assert_rises_with_id(s, groups, users.shape[0])
    ref_i, ref_s = oracle_topk(s, K)
    flags = torch.empty(u.shape[0], device="cuda", dtype=torch.int32)
    idx, score, nfb = retrieval.retrieve_topk(u, _index("accumulation"), K, flags_out=flags)
    print(f"\n[C K={K}] flagged users: {int(flags.sum())}, fallback users: {nfb}")
    _assert_equal(idx, score, ref_i, ref_s, "C")
    assert nfb > 0 and nfb == int(flags.sum())


# ---------------------------------------------------------------------------------------------------------------
# D. sampled start threshold above the user's own K-th best (the nsel < K branch)
# ---------------------------------------------------------------------------------------------------------------
def test_start_threshold_above_the_kth_best_falls_back():
    from mrm_b200 import retrieval
    N, U, K = 40_000, 300, 100
    table, users, _ = lossy_gaussian(N, U, seed=15)
    table, users = table.clone(), users.clone()
    index = retrieval.CatalogIndex(table)
    plan = index.plan(U, 256)
    stride, tiles, rank = plan.sample_stride, plan.sample_tiles, plan.sample_rank
    assert stride > 1 and tiles > 0 and rank + 4 < K, (stride, tiles, rank)
    # rank + 4 planted items, each alone in a 32-score chunk of a sampled item step (256 items): every one of them
    # owns a sampled chunk maximum, so the start threshold is the rank-th best of them, while the catalog holds
    # fewer than K such items
    n_p = rank + 4
    ids = [t * stride * 256 + 32 * c + 7 for c in range(8) for t in range(tiles)]
    ids = torch.tensor([i for i in ids if i <= N][:n_p])
    assert ids.unique().numel() == n_p
    g = torch.Generator().manual_seed(16)
    d = torch.nn.functional.normalize(torch.randn(256, generator=g), dim=0)
    table[ids] = quantize(torch.nn.functional.normalize(d + 0.05 * torch.randn(n_p, 256, generator=g), dim=1))
    planted = torch.arange(0, U, 3)
    users[planted] = quantize(torch.nn.functional.normalize(d + 0.05 * torch.randn(len(planted), 256, generator=g), dim=1))
    assert on_grid(table) and on_grid(users)
    index = retrieval.CatalogIndex(table)
    assert index.plan(U, 256).sample_rank == rank
    u = users.cuda()
    s = exact_scores(u, table)
    ref_i, ref_s = oracle_topk(s, K)
    assert (s[planted.cuda()][:, ids.cuda()].min(dim=1).values > ref_s[planted.cuda(), n_p]).all()
    flags = torch.empty(U, device="cuda", dtype=torch.int32)
    idx, _, _ = retrieval.retrieve_topk(u, index, K, flags_out=flags, exact_fallback=False)
    short = (idx[:, K - 1] < 0)            # fewer than K candidates survived the threshold: nsel < K
    print(f"\n[D stride={stride} sample tiles={tiles} rank={rank}] users with nsel < K: {int(short.sum())}, "
          f"flagged: {int(flags.sum())}")
    assert short[planted.cuda()].all() and (flags[short] == 1).all()
    idx, score, nfb = retrieval.retrieve_topk(u, index, K)
    _assert_equal(idx, score, ref_i, ref_s, "D")
    assert nfb >= len(planted)


# ---------------------------------------------------------------------------------------------------------------
# E. sparse vocabulary: unlisted ids are zero rows, a flood of +0.0 ties
# ---------------------------------------------------------------------------------------------------------------
def test_sparse_vocabulary_zero_row_ties_come_out_in_ascending_id():
    from mrm_b200 import retrieval
    N, U, K = 20_000, 300, 100
    g = torch.Generator().manual_seed(17)
    c = torch.nn.functional.normalize(torch.randn(256, generator=g), dim=0)
    table = torch.zeros(N + 1, 256)
    real = torch.randperm(N, generator=g)[:N // 20] + 1                       # 5 % of the ids have a row
    table[real] = quantize(torch.nn.functional.normalize(torch.randn(len(real), 256, generator=g) - 2.5 * c, dim=1))
    users = quantize(torch.nn.functional.normalize(c + 0.02 * torch.randn(U, 256, generator=g), dim=1))
    assert on_grid(table) and on_grid(users) and not bf16_exact(table)
    u = users.cuda()
    s = exact_scores(u, table)
    ref_i, ref_s = oracle_topk(s, K)
    assert (ref_s[:, K - 1] == 0).all(), "every user's top K must reach into the zero rows"
    idx, score, nfb = retrieval.retrieve_topk(u, retrieval.CatalogIndex(table), K)
    print(f"\n[E] fallback users: {nfb}, zero-score entries: {int((ref_s == 0).sum())}")
    _assert_equal(idx, score, ref_i, ref_s, "E")
    zero = ref_s == 0
    assert (idx[:, 1:][zero[:, 1:] & zero[:, :-1]] > idx[:, :-1][zero[:, 1:] & zero[:, :-1]]).all()


# ---------------------------------------------------------------------------------------------------------------
# F. exclusions through the flags: the fallback must honour each user's history
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["items", "users", "accumulation"])
def test_exclusions_reach_the_exact_fallback(name):
    from mrm_b200 import retrieval
    table, users, groups = _check_fixture(name)
    U, K, m = users.shape[0], 100, 64
    g = torch.Generator().manual_seed(18)
    hist = torch.zeros(U, m, dtype=torch.long)
    for u in range(U):
        ids = groups[u % len(groups)]
        own = torch.cat([ids[-5:], ids[torch.randperm(len(ids), generator=g)[:40]]])   # the best five + random members
        other = torch.randint(1, table.shape[0], (10,), generator=g)
        h = torch.cat([own, other])
        hist[u, :len(h)] = h
    u = users.cuda()
    ex = retrieval.Exclusions(hist.cuda(), table.shape[0])
    ref_i, ref_s = oracle_topk(exact_scores(u, table, exclude=hist), K)
    idx, score, nfb = retrieval.retrieve_topk(u, _index(name), K, exclude=ex)
    print(f"\n[F {name}] fallback users: {nfb}")
    _assert_equal(idx, score, ref_i, ref_s, f"F {name}")
    assert nfb > 0
    got = idx.cpu()
    assert not any(set(got[r].tolist()) & set(hist[r].tolist()) for r in range(U))


# ---------------------------------------------------------------------------------------------------------------
# G. the bounded shard contract, item by item, and its merge
# ---------------------------------------------------------------------------------------------------------------
_CUTS = {1: [0], 2: [0, 7001], 3: [0, 1700, 13_333], 8: [0, 900, 2500, 2600, 6000, 9999, 14_000, 17_500]}


@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("name", ["items", "users", "gaussian", "accumulation"])
def test_bounded_candidates_bound_every_unlisted_item(name, G):
    from mrm_b200 import retrieval
    table, users, _ = _check_fixture(name)
    V, U, K = table.shape[0], users.shape[0], 100
    cuts = _CUTS[G] + [V]
    kps = retrieval.shard_kprime(256, G)
    u = users.cuda()
    s = exact_scores(u, table)
    ref_i, ref_s = oracle_topk(s, K)
    allp = torch.empty(G * U, 2 * kps + 2, device="cuda", dtype=torch.int32)
    flooded = 0
    for q, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        shard = retrieval.CatalogIndex(table, shard=(a, b - a))
        i, sc, bound, flag = retrieval.retrieve_candidates(u, shard, kps, pack=allp[q * U:(q + 1) * U])
        listed = i >= 0
        assert ((i[listed] >= a) & (i[listed] < b)).all()
        # listed scores: the exact ones, bit for bit
        assert torch.equal(sc[listed], s.gather(1, i.clamp(min=0).long())[listed]), f"shard {q}: listed scores"
        assert torch.isneginf(sc[~listed]).all()
        # every item of the shard that is not listed: exact score <= bound
        unlisted = torch.ones(U, b - a, device="cuda", dtype=torch.bool)
        r, c = listed.nonzero(as_tuple=True)
        unlisted[r, i[r, c].long() - a] = False
        over = unlisted & (s[:, a:b] > bound[:, None])
        assert not over.any(), (f"shard {q} [{a}, {b}): {int(over.any(dim=1).sum())} users have an unlisted item "
                                f"above the bound, e.g. user {over.any(dim=1).nonzero()[0].item()}")
        flooded += int(flag.sum())
    bad = torch.zeros(U, device="cuda", dtype=torch.int32)
    mi, ms = retrieval.merge_packed(allp, G, U, kps, K, bad)
    ok = bad == 0
    print(f"\n[G {name} shards={G} K'={kps}] uncertified users: {int((~ok).sum())}, tie-flood flags: {flooded}")
    _assert_equal(mi[ok], ms[ok], ref_i[ok], ref_s[ok], f"G {name} certified users")
    if name in ("items", "users", "accumulation"):
        assert not ok.all(), "every user certified on an adversarial catalog: the bound tests nothing"


# ---------------------------------------------------------------------------------------------------------------
# H. the accumulation model behind the slack term
# ---------------------------------------------------------------------------------------------------------------
def test_tensor_core_accumulation_error_within_the_slack_term():
    """|C - C_fp64| <= 2^-18 ||a|| ||b|| for C = A B^T at K = 256 on adversarial bf16 operands.

    This runs tt_gemm_bf16, not tt_score_topk: both issue tcgen05.mma kind::f16 with an fp32 accumulator in tensor
    memory, 16 instructions of K = 16 at K = 256. The test assumes that the summation inside one instruction is the
    same in both kernels, which holds as long as both use that instruction kind and operand type.

    Every 16-wide K group holds one dominant product and fifteen products 2^-22 .. 2^-29 times smaller (just below
    the alignment window of an adder that aligns to the largest product); the dominant products cancel across the
    groups (alternating signs, or eight positive groups then eight negative ones, which also lets the accumulator
    grow before it cancels).

    Measured on an NVIDIA B200 (1000 W power limit): the worst entry reaches 0.086 of the bound, and the worst error
    relative to sum|a_k b_k| is 10.8 x 2^-23 (about 2^-19.6). So products below the alignment window are dropped,
    but the error stays far below the 256 x 2^-23 = 2^-15 of rounding after every product."""
    from mrm_b200 import ops
    M = N = 256
    g = torch.Generator().manual_seed(19)
    mant = lambda *s: 1 + torch.randint(0, 128, s, generator=g).float() / 128        # 8 significant bits
    A = torch.empty(M, 256)
    B = torch.empty(N, 256)
    for r in range(M):
        e = 22 + r % 8
        A[r] = mant(256) * 2.0 ** -e
        A[r, ::16] = mant(16) * (0.5 if r % 3 == 0 else 1.0)
    for r in range(N):
        B[r] = mant(256) * (1 if r % 4 else -1)
        kind = r % 3
        if kind == 0:
            pattern = torch.tensor([(-1.0) ** q for q in range(16)])
        elif kind == 1:
            pattern = torch.tensor([1.0] * 8 + [-1.0] * 8)
        else:
            pattern = torch.sign(torch.randn(16, generator=g))
        B[r, ::16] = mant(16) * pattern
    A16, B16 = A.bfloat16(), B.bfloat16()
    assert torch.equal(A16.float(), A) and torch.equal(B16.float(), B)
    out = torch.empty(M, N, device="cuda")
    ops.gemm(A16.cuda(), B16.cuda(), out_f32=out)
    ref = A.double().cuda() @ B.double().cuda().t()
    bound = 2.0 ** -18 * A.double().norm(dim=1).cuda()[:, None] * B.double().norm(dim=1).cuda()[None, :]
    err = (out.double() - ref).abs()
    ratio = err / bound
    per_abs = err / (2.0 ** -23 * (A.double().abs() @ B.double().abs().t()).cuda())
    print(f"\n[H] worst |C - C_fp64| / (2^-18 ||a|| ||b||) = {ratio.max().item():.4g}; "
          f"worst |C - C_fp64| / (2^-23 sum|a_k b_k|) = {per_abs.max().item():.4g}")
    assert (ratio <= 1).all(), f"accumulation error {ratio.max().item():.3g} x the slack term"
