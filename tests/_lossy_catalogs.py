"""Catalogs on which bf16 scoring is lossy while an fp64 oracle stays bit-exact, and that oracle.

Every entry lies on the 2^-20 grid inside (-1, 1): it has at most 20 significant bits, so it is exact in fp32,
while most such values are not exact in bf16. A product of two entries is a multiple of 2^-40 and every partial
sum of 256 of them stays below 2^8, so a 256-term dot product is exact in fp64 whatever the summation order. The
retrieval kernels' exact re-score (fp64 accumulate, one rounding to fp32), their brute-force fallback and a torch
fp64 matmul therefore agree bit for bit, and the oracle below is the exact answer, not an approximation of it.

The fixtures are adversarial for the exactness certificate of tt_topk_finalize: the bf16 path scores members of
one group identically, breaks the tie by ascending item id, and so keeps the LOWEST ids, while the exact scores
rise with the id. Each builder returns CPU tensors: ``table`` (N + 1, 256) fp32 with row 0 = 0, ``users``
(U, 256) fp32 and ``groups``, a list of id tensors (ascending) of the planted groups, user u planted on
``groups[u % len(groups)]``.
"""
from __future__ import annotations

import functools
from typing import List, Optional, Tuple

import torch

GRID = 2.0 ** -20
D = 256


def on_grid(t: torch.Tensor) -> bool:
    """every entry a multiple of 2^-20 strictly inside (-1, 1)"""
    return bool(torch.equal(torch.round(t / GRID) * GRID, t)) and bool((t.abs() < 1).all())


def bf16_exact(t: torch.Tensor) -> bool:
    return bool(torch.equal(t.bfloat16().float(), t))


def quantize(t: torch.Tensor) -> torch.Tensor:
    return torch.round(t.clamp(-1 + GRID, 1 - GRID) / GRID) * GRID


def _gen(seed: int) -> torch.Generator:
    return torch.Generator().manual_seed(seed)


def _signs(g: torch.Generator, *shape) -> torch.Tensor:
    return torch.randint(0, 2, shape, generator=g).float() * 2 - 1


def _bf16_filler(n: int, g: torch.Generator) -> torch.Tensor:
    """n rows on the 2^-7 grid (at most 7 significant bits: bf16-exact), norm about 1"""
    return torch.round((torch.randn(n, D, generator=g) / 16).clamp(-0.99, 0.99) * 128) / 128


def _lossy_filler(n: int, g: torch.Generator) -> torch.Tensor:
    return quantize(torch.nn.functional.normalize(torch.randn(n, D, generator=g), dim=1))


def _group_ranges(n_items: int, sizes: List[int], g: torch.Generator) -> List[torch.Tensor]:
    """disjoint runs of consecutive ids in [1, n_items], one per size, at random places"""
    gap = (n_items - sum(sizes)) // (len(sizes) + 1)
    out, start = [], 1
    for s in sizes:
        start += int(torch.randint(gap // 2, gap + 1, (1,), generator=g))
        out.append(torch.arange(start, start + s))
        start += s
    assert start <= n_items + 1
    return out


@functools.lru_cache(maxsize=None)
def near_duplicate_items(n_items: int = 20_000, n_users: int = 300, seed: int = 11):
    """Versions of one song, lossy on the ITEM side: member i of a group is one bf16-exact base row plus i * 2^-20
    in four coordinates that hold 0.75 in the base. 599 * 2^-20 is below half a bf16 ulp of 0.75 (2^-9), so every
    member rounds to the base row in bf16 and all members tie on the bf16 path. Users are bf16-exact and weigh
    those coordinates positively: the exact score rises by 3 * 2^-20 per member. Fillers are lossy Gaussian rows.
    Only the nu * de_max term of the certificate's eps covers the gap (du = 0)."""
    g = _gen(seed)
    sizes = [300 + 43 * k for k in range(8)]              # 300 .. 601 members
    table = _lossy_filler(n_items + 1, g)
    groups = _group_ranges(n_items, sizes, g)
    bases = []
    for ids in groups:
        base = _signs(g, D) / 16
        coords = torch.randperm(D, generator=g)[:4]
        base[coords] = 0.75
        bases.append((base, coords))
        rows = base.expand(len(ids), D).clone()
        rows[:, coords] += torch.arange(len(ids)).float()[:, None] * GRID
        table[ids] = rows
    table[0] = 0
    users = torch.empty(n_users, D)
    for u in range(n_users):
        base, coords = bases[u % len(groups)]
        x = base + _signs(g, D) * (torch.rand(D, generator=g) < 0.3).float() / 64     # +-2^-4 +-2^-6: bf16-exact
        x[coords] = 0.75
        users[u] = x
    return table, users, groups


# bf16-exact values in [2^-4, 1), ascending: 128 per binade
_BF16_LADDER = torch.cat([(128 + torch.arange(128).float()) * 2.0 ** (-11 + b) for b in range(4)])


@functools.lru_cache(maxsize=None)
def near_duplicate_users(n_items: int = 20_000, n_users: int = 300, seed: int = 12):
    """Versions of one song, lossy on the USER side: every row is bf16-exact (de_max = 0). Member i of a group is a
    base row with x_i at coordinate c1 and -x_i at c2 (both 0 in the base), x_i the i-th bf16 value of [2^-4, 1).
    A planted user holds 0.75 + rho at c1 and 0.75 - rho at c2, rho in [2^-10, 2^-9): both round to 0.75 in bf16,
    so the bf16 path scores every member alike, while the exact score rises by 2 * rho * x_i. Only the du * ne_max
    term of eps covers the gap."""
    g = _gen(seed)
    sizes = [300 + 30 * k for k in range(8)]              # 300 .. 510 members (<= 512 ladder values)
    table = _bf16_filler(n_items + 1, g)
    groups = _group_ranges(n_items, sizes, g)
    bases = []
    for ids in groups:
        base = _signs(g, D) / 16
        c1, c2 = torch.randperm(D, generator=g)[:2].tolist()
        base[c1] = base[c2] = 0
        bases.append((base, c1, c2))
        rows = base.expand(len(ids), D).clone()
        x = _BF16_LADDER[:len(ids)]
        rows[:, c1], rows[:, c2] = x, -x
        table[ids] = rows
    table[0] = 0
    users = torch.empty(n_users, D)
    for u in range(n_users):
        base, c1, c2 = bases[u % len(groups)]
        x = base + _signs(g, D) * (torch.rand(D, generator=g) < 0.3).float() / 64
        rho = float(torch.randint(256, 512, (1,), generator=g)) * GRID
        x[c1], x[c2] = 0.75 + rho, 0.75 - rho
        users[u] = x
    return table, users, groups


@functools.lru_cache(maxsize=None)
def lossy_gaussian(n_items: int, n_users: int, seed: int = 13):
    """Normalised Gaussian rows and users near a planted target (synthetic.make_queries, noise 3.3), all quantised
    to the 2^-20 grid: generic data, lossy in bf16 on both sides."""
    g = _gen(seed)
    table = _lossy_filler(n_items + 1, g)
    table[0] = 0
    t = torch.randint(1, n_items + 1, (n_users,), generator=g)
    users = quantize(torch.nn.functional.normalize(table[t] + 3.3 * torch.randn(n_users, D, generator=g) / 16, dim=1))
    return table, users, []


# accumulation-dominated catalog: coordinates of group q
def _acc_coords(q: int):
    return q, 240 + q, [16 * j + q for j in range(1, 15)]   # cancel pair in K-groups 0 and 15, one small per 1..14


_ACC_Z = 8            # K-group 0: fillers hold -0.5 here, every user 2^-4 or 2^-5


@functools.lru_cache(maxsize=None)
def accumulation_dominated(n_items: int = 20_000, n_users: int = 300, seed: int = 14):
    """Users and items bf16-exact (du = de = 0: eps is the fp32-accumulation slack alone). Member t of group q holds
    0.75 at coordinate q (K-group 0), -0.75 at 240 + q (K-group 15) and m_j(t) * 2^-20 at 16 j + q (j = 1..14,
    m_j <= 127, sum_j m_j = t); its users hold 0.75 at both ends and 2^-12 or 2^-13 on the smalls. The exact score
    is t * 2^-32 (or t * 2^-33): it rises with the id. On the tensor core's fp32 accumulator every small product
    (< 2^-25) arrives while the accumulator holds 0.5625 (ulp 2^-24) and is lost before K-group 15 cancels it: the
    bf16 path scores all members 0 (`emulate_fp32_accumulation`). Other groups' members score about -0.047 for a
    planted user and fillers -2^-5 or less."""
    g = _gen(seed)
    sizes = [300, 400, 500, 600]
    table = _bf16_filler(n_items + 1, g)
    used = set([_ACC_Z])
    for q in range(len(sizes)):
        a, b, smalls = _acc_coords(q)
        used.update([a, b, *smalls])
    used = sorted(used)
    table[:, used] = 0
    table[:, _ACC_Z] = -0.5
    groups = _group_ranges(n_items, sizes, g)
    for q, ids in enumerate(groups):
        a, b, smalls = _acc_coords(q)
        t = torch.arange(len(ids))
        rows = torch.zeros(len(ids), D)
        rows[:, a], rows[:, b] = 0.75, -0.75
        for j, c in enumerate(smalls):
            rows[:, c] = (t - 127 * j).clamp(0, 127).float() * GRID
        table[ids] = rows
    table[0] = 0
    users = torch.zeros(n_users, D)
    for u in range(n_users):
        q = u % len(groups)
        a, b, smalls = _acc_coords(q)
        for h in range(len(groups)):
            users[u, h] = -1.0 / 16
        users[u, a] = users[u, b] = 0.75
        users[u, smalls] = 2.0 ** -12 if (u // len(groups)) % 2 == 0 else 2.0 ** -13
        users[u, _ACC_Z] = 2.0 ** -4 if (u // len(groups)) % 3 else 2.0 ** -5
    return table, users, groups


def emulate_fp32_accumulation(users: torch.Tensor, rows: torch.Tensor) -> torch.Tensor:
    """Scores of bf16(users) . bf16(rows) with each 16-wide K group summed exactly and added to an fp32 accumulator
    with one rounding: the most favourable model of tcgen05.mma kind::f16 at K = 256 (16 instructions)."""
    u, r = users.bfloat16().double(), rows.bfloat16().double()
    acc = torch.zeros(u.shape[0], r.shape[0], dtype=torch.float32)
    for k in range(0, D, 16):
        acc = (acc.double() + u[:, k:k + 16] @ r[:, k:k + 16].t()).float()
    return acc


def exact_scores(users: torch.Tensor, table: torch.Tensor, item_base: int = 0, mask_item0: bool = True,
                 exclude: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp64 dot products (exact on the grid), rounded once to fp32, of ``users`` against rows item_base.. of
    ``table`` (on the users' device); column of global item 0 and the excluded ids (int64 (U, m), 0 = empty slot,
    global ids) set to -inf"""
    s = (users.double() @ table.to(users.device).double().t()).float()
    if mask_item0 and item_base == 0:
        s[:, 0] = -float("inf")
    if exclude is not None:
        loc = exclude.to(users.device) - item_base
        ok = (exclude.to(users.device) > 0) & (loc >= 0) & (loc < s.shape[1])
        rows = torch.arange(s.shape[0], device=s.device)[:, None].expand_as(loc)
        s[rows[ok], loc[ok]] = -float("inf")
    return s


def oracle_topk(scores: torch.Tensor, K: int, item_base: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """canonical top K (score descending, then id ascending) of an `exact_scores` matrix; -1 / -inf where fewer
    than K items are admissible"""
    v, i = torch.sort(scores, dim=1, descending=True, stable=True)
    v, i = v[:, :K].contiguous(), (i[:, :K] + item_base).int()
    i[torch.isneginf(v)] = -1
    return i, v
