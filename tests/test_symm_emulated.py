"""The cross-GPU kernels of csrc/tt_symm.cu and the team forms of tt_rows_gather / tt_rows_scatter_add, on ONE GPU with
emulated peer ranks (tests/_emulated_team.py: G ordinary allocations laid out as symm.SymmArena lays out its
symmetric memory, ranks launched one after the other with their control blocks pre-stamped).

  tt_symm_allgather    every arena holds rank q's source at dst_off + q * nbytes, byte for byte; nothing else moved
  tt_dp_adamw_step     bit-equal to tt_adamw_step on the rank-order fp32 gradient sum with grad_scale 1 / G (the
                       unicast path sums the peers in rank order and does adamw_kernel's arithmetic), and close to the
                       fp64 AdamW of the oracle; the row-sharded table's shard gets the same treatment
  tt_symm_barrier      control-block invariants, interleaved with the other collectives
  tt_rows_gather / tt_rows_scatter_add (team forms)   round-robin owners: id lives at row id // G of rank id % G
  TrainStepRunner._phase_symm_step, unchanged, on G threads (one engine replica each) against the virtual data-parallel
                       step of tests/_virtual_dp.py followed by tt_adamw_step, and against the fp64 oracle
  symm.SymmArena as shipped at world 1 (single-rank NCCL group)

Real multi-GPU concurrency (spin waits racing across devices, NVLink ordering, the timeout) is left to
tools/symm_check.py and tools/dist_check.py under torchrun.
"""
import ctypes
import dataclasses

import pytest
import torch

from _emulated_team import (DONE, READY, EmulatedGroup, EmulatedWorld, ThreadedEmulatedArena, check_ctrl, make_team,
                            run_collective, run_ranks)

pytestmark = pytest.mark.gpu

WORLDS = [1, 2, 3, 4, 8, 16]
LR, BETAS, EPS, WD = 1e-3, (0.9, 0.999), 1e-8, 0.01
# the hyper-parameters as the kernels receive them (fp32): 1 - fp32(0.999) is 1.3e-5 away from 1e-3
HP32 = tuple(float(torch.tensor(x, dtype=torch.float32)) for x in (LR, BETAS[0], BETAS[1], EPS, WD))


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.uint8)


def _bit_equal(a: torch.Tensor, b: torch.Tensor) -> bool:
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _random_bytes(n: int, gen) -> torch.Tensor:
    return torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=gen)


def _fill_sentinel(arenas, gen) -> None:
    """Random bytes everywhere but the control blocks."""
    for a in arenas:
        a.buf[:a.ctrl_offset].copy_(_random_bytes(a.ctrl_offset, gen))
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------
# tt_symm_allgather
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("G", WORLDS)
def test_allgather_places_every_rank_block(G):
    from mrm_b200._lib import lib
    big = lib().tt_num_sms() * 256 * 16 + 4096 + 48      # more than one pass of the grid-stride loop
    rounds = [  # (segment sizes in bytes, pre_barrier); several collectives in a row on the same arenas
        ([16], 0),
        ([48, 1024, 16, 4080], 1),
        ([big, 32], 0),
        ([208, 640, 96], 1),
        ([big // 2 + 8, 16, 65536], 0),
    ]
    layout = {}
    for i, (sizes, _) in enumerate(rounds):
        for s, nb in enumerate(sizes):
            layout[f"r{i}s{s}"] = G * nb + (16 if (i + s) % 2 else 0)     # some blocks with slack after the last rank
    gen = torch.Generator(device="cuda").manual_seed(G)
    arenas = make_team(G, layout)
    _fill_sentinel(arenas, gen)
    expect = [a.buf[:a.ctrl_offset].clone() for a in arenas]
    for i, (sizes, pre) in enumerate(rounds):
        srcs = [[_random_bytes(nb, gen) for nb in sizes] for _ in range(G)]
        run_collective(arenas, lambda r: arenas[r].allgather(
            [(srcs[r][s], f"r{i}s{s}") for s in range(len(sizes))], pre_barrier=bool(pre)), ready=bool(pre))
        for s, nb in enumerate(sizes):
            off = arenas[0].offset(f"r{i}s{s}")
            for q in range(G):
                for e in expect:
                    e[off + q * nb:off + (q + 1) * nb] = srcs[q][s]
        for a, e in zip(arenas, expect):
            assert torch.equal(a.buf[:a.ctrl_offset], e), f"round {i}: arena {a.rank} differs"
        if i == 1:       # a barrier between two all-gathers: control-block invariants only
            run_collective(arenas, lambda r: arenas[r].barrier(), ready=True)
    for a in arenas:
        assert a.issued == len(rounds) + 1


# ---------------------------------------------------------------------------------------------------------------
# tt_dp_adamw_step
# ---------------------------------------------------------------------------------------------------------------
def _grad(n: int, sign: torch.Tensor, gen, shift: int = 0) -> torch.Tensor:
    """A gradient whose elements keep one sign per element across ranks (``sign``), so the fp32 rank-order sum has
    no cancellation and the fp64 reference is well conditioned. Some float4 groups are -0.0 or +0.0 on every rank,
    others on this rank only (``shift``)."""
    g = sign * (1e-3 + torch.rand(n, device="cuda", generator=gen))
    g4 = g.view(-1, 4)
    g4[0::29] = -0.0
    g4[1::31] = 0.0
    g4[3 + shift::7] = -0.0
    g4[5 + shift::11] = 0.0
    g4[2 + shift::13, 2] = -0.0          # a -0.0 inside an otherwise non-zero group
    return g


def _dp_case(case: str, G: int):
    """(n, shadow_begin, table shard elements per rank)."""
    per4 = 300
    if case == "grid_cap":          # per-rank slice above 4 * num_sms CTAs x 256 threads x 4 (unroll) float4s
        from mrm_b200._lib import lib
        per4 = lib().tt_num_sms() * 4 * 256 * 4 + 12345
    n = 4 * G * per4
    if case == "shadow_at_0":
        return n, 0, 0
    if case == "shadow_at_n":
        return n, n, 0
    if case == "table":             # the shard dwarfs the dense slice: the grid comes from the shard, as at c5
        n = 4 * G * 64
        return n, 4 * (G // 2 * 64 + 17), 4 * 1024 * 300
    return n, 4 * (G // 2 * per4 + 37), 0          # shadow_mid / grid_cap: inside rank G // 2's slice


DP_CASES = [(G, c) for G in WORLDS for c in ("shadow_at_0", "shadow_at_n", "shadow_mid", "table")] + \
           [(1, "grid_cap"), (3, "grid_cap")]


@pytest.mark.parametrize("G,case", DP_CASES)
def test_dp_adamw_step_matches_adamw_kernel_and_fp64(G, case):
    from mrm_b200 import ops
    from oracle import two_tower_oracle as oracle
    n, sb, tn = _dp_case(case, G)
    per = n // G
    gen = torch.Generator(device="cuda").manual_seed(100 * G + len(case))
    arenas = make_team(G, {"flat": n * 4, "grad": n * 4, "shadow": (n - sb) * 2, "guard": 256})
    _fill_sentinel(arenas, gen)
    p0 = 0.05 * torch.randn(n, device="cuda", generator=gen)
    for a in arenas:
        a.view("flat", torch.float32, (n,)).copy_(p0)
    m = [torch.zeros(per, device="cuda") for _ in range(G)]
    v = [torch.zeros(per, device="cuda") for _ in range(G)]
    steps = [torch.zeros((), dtype=torch.long, device="cuda") for _ in range(G)]
    sign = torch.where(torch.rand(n, device="cuda", generator=gen) < 0.5, -1.0, 1.0)
    if tn:
        tsign = torch.where(torch.rand(tn, device="cuda", generator=gen) < 0.5, -1.0, 1.0)
        shards = [[0.05 * torch.randn(tn, device="cuda", generator=gen), torch.zeros(tn, device="cuda"),
                   torch.zeros(tn, device="cuda"), torch.zeros(tn, device="cuda")] for _ in range(G)]
        t_ref = [[t.clone() for t in s] for s in shards]
        t64 = [[s[0].double(), torch.zeros(tn, dtype=torch.float64, device="cuda"),
                torch.zeros(tn, dtype=torch.float64, device="cuda")] for s in shards]
    # reference 1: tt_adamw_step over the whole buffer on the rank-order sum; reference 2: fp64 oracle AdamW
    p_ref, m_ref, v_ref = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    sh_ref = torch.zeros(n - sb, device="cuda", dtype=torch.bfloat16)
    step_ref = torch.zeros((), dtype=torch.long, device="cuda")
    p64, m64, v64 = p0.double(), torch.zeros(n, dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda")
    worst = {"p": 0.0, "m": 0.0, "v": 0.0}
    for step in range(1, 4):
        grads = [_grad(n, sign, gen, r) for r in range(G)]
        for a, g in zip(arenas, grads):
            a.view("grad", torch.float32, (n,)).copy_(g)
        if tn:
            for r, s in enumerate(shards):
                s[1].copy_(_grad(tn, tsign, gen, r))
            for s, r in zip(shards, t_ref):
                r[1].copy_(s[1])
            t_g = [s[1].clone() for s in shards]
        for s in steps:
            s.fill_(step)
        guard = [a.view("guard", torch.uint8, (256,)).clone() for a in arenas]

        run_collective(arenas, lambda r: arenas[r].dp_adamw_step(
            "flat", "grad", "shadow", n, sb, m[r], v[r], steps[r], LR, BETAS, EPS, WD,
            table_shard=shards[r] if tn else None), ready=True)

        gsum = grads[0].clone()
        for g in grads[1:]:
            gsum = gsum + g
        step_ref.fill_(step)
        ops.adamw_step(p_ref, gsum, m_ref, v_ref, step_ref, LR, BETAS[0], BETAS[1], EPS, WD,
                       shadow=sh_ref if sb < n else None, shadow_begin=sb, shadow_end=n, grad_scale=1.0 / G)
        g64 = sum(g.double() for g in grads) / G
        p64, m64, v64 = oracle.adamw_step(p64, g64, m64, v64, step, *HP32)
        torch.cuda.synchronize()
        flat0 = arenas[0].view("flat", torch.float32, (n,))
        for r, a in enumerate(arenas):
            flat, shadow = a.view("flat", torch.float32, (n,)), a.view("shadow", torch.bfloat16, (n - sb,))
            assert _bit_equal(flat, p_ref), f"step {step}: rank {r}'s parameters differ from tt_adamw_step"
            assert _bit_equal(flat, flat0)
            assert _bit_equal(shadow, sh_ref), f"step {step}: rank {r}'s bf16 shadow differs from tt_adamw_step"
            assert _bit_equal(shadow, flat[sb:].to(torch.bfloat16))
            assert _bit_equal(m[r], m_ref[r * per:(r + 1) * per]) and _bit_equal(v[r], v_ref[r * per:(r + 1) * per]), \
                f"step {step}: rank {r}'s moments differ from tt_adamw_step"
            assert _bit_equal(a.view("grad", torch.float32, (n,)), grads[r]), "the dense gradient must stay in place"
            assert torch.equal(a.view("guard", torch.uint8, (256,)), guard[r])
        # fp64: p differs by a few roundings of p * decay and of the step; m and v by the roundings of the G-term
        # same-sign fp32 sum (at most G - 1 of 2^-24 each) and of the moment updates
        err_p = (p_ref.double() - p64).abs()
        assert bool((err_p <= 1e-6 * p64.abs() + 1e-5 * LR).all()), (step, err_p.max().item())
        err_m = ((m_ref.double() - m64).abs() / m64.abs().clamp_min(1e-30))[m64 != 0]
        err_v = ((v_ref.double() - v64).abs() / v64.abs().clamp_min(1e-30))[v64 != 0]
        assert bool((m_ref[m64 == 0] == 0).all()) and bool((v_ref[v64 == 0] == 0).all())
        assert err_m.max().item() <= 2e-6 and err_v.max().item() <= 4e-6, (err_m.max().item(), err_v.max().item())
        worst = {"p": max(worst["p"], err_p.max().item()), "m": max(worst["m"], err_m.max().item()),
                 "v": max(worst["v"], err_v.max().item())}
        if tn:
            for r in range(G):
                ref, s = t_ref[r], shards[r]
                ops.adamw_step(ref[0], ref[1], ref[2], ref[3], step_ref, LR, BETAS[0], BETAS[1], EPS, WD,
                               shadow=None, zero_grad=True, grad_scale=1.0 / G)
                t64[r] = list(oracle.adamw_step(t64[r][0], t_g[r].double() / G, t64[r][1], t64[r][2], step, *HP32))
            torch.cuda.synchronize()
            for r in range(G):
                ref, s = t_ref[r], shards[r]
                for what, got, want in (("p", s[0], ref[0]), ("m", s[2], ref[2]), ("v", s[3], ref[3])):
                    assert _bit_equal(got, want), f"step {step}: rank {r}'s table shard {what} differs from tt_adamw_step"
                assert bool((s[1].view(torch.int32) == 0).all()), "the table shard's gradient must be cleared (+0.0)"
                e = (s[0].double() - t64[r][0]).abs()
                assert bool((e <= 1e-6 * t64[r][0].abs() + 1e-5 * LR).all()), (step, r, e.max().item())
                worst["p"] = max(worst["p"], e.max().item())
    print(f"dp_adamw G={G} {case}: bit-equal to tt_adamw_step; worst vs fp64 oracle: |dp| {worst['p']:.3g}, "
          f"rel m {worst['m']:.3g}, rel v {worst['v']:.3g}")


# ---------------------------------------------------------------------------------------------------------------
# tt_rows_gather / tt_rows_scatter_add with a team (row-sharded ID table)
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("G", [1, 2, 3, 5, 8, 16])
def test_team_rows_gather_and_scatter_add(G):
    from mrm_b200 import ops
    V = 31 * G + (G - 1 if G > 1 else 6)         # not a multiple of G: the last ranks own fewer rows
    per = (V + G - 1) // G
    gen = torch.Generator(device="cuda").manual_seed(7 + G)
    # SymmShardedTable's weight and gradient blocks, behind a leading block so both offsets are non-zero
    arenas = make_team(G, {"head": 768, "weight": per * 1024, "grad": per * 1024})
    _fill_sentinel(arenas, gen)
    full = torch.randn(V, 256, device="cuda", generator=gen)
    for r, a in enumerate(arenas):
        rows = len(range(r, V, G))
        a.view("weight", torch.float32, (per, 256))[:rows].copy_(full[r::G])
    # distinct ids: slot 0 = padding, V - 1, ids owned by every rank, then a random selection
    must = [V - 1] + [q if q > 0 else G for q in range(G)]
    rest = [i for i in torch.randperm(V - 1, generator=torch.Generator().manual_seed(G)).add(1).tolist() if i not in must]
    ids = [0] + list(dict.fromkeys(must)) + rest[:max(8, V // 3)]
    n = len(ids)
    max_rows = n + 37
    uniq = torch.ones(max_rows, dtype=torch.long, device="cuda")    # slots past n hold valid ids the kernels must skip
    uniq[:n] = torch.tensor(ids, device="cuda")
    state = torch.tensor([n + 5, n], dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    before = [a.buf.clone() for a in arenas]
    for r, a in enumerate(arenas):       # every rank's view of the table gives the same rows
        cache = torch.full((max_rows, 256), float("nan"), device="cuda")
        ops.rows_gather(uniq, state, cache, team=a.team, weight_offset=a.offset("weight"))
        torch.cuda.synchronize()
        assert _bit_equal(cache[:n], full[uniq[:n]]), f"rank {r}: gathered rows differ from table[uniq]"
        assert bool(cache[n:].isnan().all()), "rows past n_uniq were written"
    for a, b in zip(arenas, before):
        assert torch.equal(a.buf, b), "the gather wrote into an arena"

    r = G - 1
    gacc = torch.randn(max_rows, 256, device="cuda", generator=gen)
    gacc0 = gacc.clone()
    ops.rows_scatter_add(uniq, state, gacc, team=arenas[r].team, grad_offset=arenas[r].offset("grad"))
    torch.cuda.synchronize()
    expect = [b.clone() for b in before]
    for s in range(1, n):
        i = ids[s]
        q, row = i % G, i // G
        g = expect[q][arenas[q].offset("grad"):arenas[q].offset("grad") + per * 1024].view(torch.float32).view(per, 256)
        g[row] = g[row] + gacc0[s]                   # one fp32 add per element: bit-exact
    for q, (a, e) in enumerate(zip(arenas, expect)):
        assert torch.equal(a.buf, e), f"rank {q}'s arena differs after the scatter-add"
    assert _bit_equal(gacc[0], gacc0[0]), "slot 0 (padding) must be neither added nor cleared"
    assert bool((gacc[1:n].view(torch.int32) == 0).all()), "gacc[1:n] must be cleared"
    assert _bit_equal(gacc[n:], gacc0[n:]), "rows past n_uniq were touched"


# ---------------------------------------------------------------------------------------------------------------
# host-side argument validation (no launch)
# ---------------------------------------------------------------------------------------------------------------
def test_symm_entry_points_reject_bad_arguments():
    from mrm_b200._lib import SymmSegment, SymmTeam, lib
    l = lib()
    stream = torch.cuda.current_stream().cuda_stream
    n = 4 * 2 * 64
    arenas = make_team(2, {"flat": n * 4, "grad": n * 4, "shadow": n * 2, "table": 1024})
    a = arenas[0]
    src = torch.zeros(64, dtype=torch.uint8, device="cuda")
    m = torch.zeros(n // 2, device="cuda")
    v = torch.zeros(n // 2, device="cuda")
    step = torch.ones((), dtype=torch.long, device="cuda")
    tp = torch.zeros(16, device="cuda")

    def team(**kw):
        t = SymmTeam()
        ctypes.memmove(ctypes.byref(t), ctypes.byref(a.team), ctypes.sizeof(SymmTeam))
        for k, val in kw.items():
            if k == "bufs":
                for q, ptr in val.items():
                    t.bufs[q] = ptr
            else:
                setattr(t, k, val)
        return t

    def gather(t, nbytes=64):
        segs = (SymmSegment * 4)()
        segs[0].src, segs[0].dst_offset, segs[0].nbytes = src.data_ptr(), a.offset("table"), nbytes
        return l.tt_symm_allgather(ctypes.byref(t), segs, 1, 0, stream)

    def adamw(t, n_=n, shard=(None, None, None, None), shard_n=0):
        return l.tt_dp_adamw_step(ctypes.byref(t), a.offset("flat"), a.offset("grad"), a.offset("shadow"), n_, 0,
                                  m.data_ptr(), v.data_ptr(), LR, 0.9, 0.999, EPS, WD, step.data_ptr(), *shard, shard_n,
                                  stream)

    def barrier(t):
        return l.tt_symm_barrier(ctypes.byref(t), stream)

    # a launch that slipped through must not wait: every flag of rank 0's block is already far ahead
    a.ctrl()[READY:READY + 16] = 1000
    a.ctrl()[DONE:DONE + 16] = 1000
    p = a.buf.data_ptr()
    bad_teams = {"world 0": team(world=0), "world 17": team(world=17), "rank -1": team(rank=-1),
                 "rank = world": team(rank=2), "misaligned peer": team(bufs={1: arenas[1].buf.data_ptr() + 8}),
                 "null peer": team(bufs={1: None}), "ctrl_offset % 128": team(ctrl_offset=a.ctrl_offset + 64)}
    for what, t in bad_teams.items():
        for name, fn in (("allgather", gather), ("dp_adamw", adamw), ("barrier", barrier)):
            assert fn(t) != 0, f"{name} accepted a team with {what}"
            assert l.tt_last_error(), (name, what)
    good = team()
    assert gather(good, nbytes=24) != 0, "a segment that is not a multiple of 16 bytes"
    assert adamw(good, n_=n + 4) != 0 and adamw(good, n_=n - 4) != 0, "n not divisible by 4 * world"
    for miss in range(4):
        shard = [tp.data_ptr()] * 4
        shard[miss] = None
        assert adamw(good, shard=tuple(shard), shard_n=16) != 0, f"a table shard without pointer {miss}"
    assert p == a.buf.data_ptr()
    # rows gather / scatter-add: team world out of range, misaligned shard offset
    uniq = torch.zeros(4, dtype=torch.long, device="cuda")
    state = torch.zeros(2, dtype=torch.int32, device="cuda")
    cache = torch.zeros(4, 256, device="cuda")
    for t, off in ((team(world=0), 0), (team(world=17), 0), (good, 8)):
        assert l.tt_rows_gather(ctypes.byref(t), off, None, uniq.data_ptr(), state.data_ptr() + 4, 4, cache.data_ptr(),
                                stream) != 0
        assert l.tt_rows_scatter_add(ctypes.byref(t), off, None, uniq.data_ptr(), state.data_ptr() + 4, 4,
                                     cache.data_ptr(), stream) != 0
    torch.cuda.synchronize()
    for x in arenas:            # nothing was launched: no epoch advanced, nobody signalled into rank 1's block
        check_ctrl(x)
    assert int(arenas[1].ctrl().abs().sum()) == 0


# ---------------------------------------------------------------------------------------------------------------
# the real training step on emulated ranks
# ---------------------------------------------------------------------------------------------------------------
_ORACLE = {}
B_RANK, STEPS = 16, 3


def _cfg():
    from mrm_b200 import synthetic
    return synthetic.TwoTowerConfig(vocab_size=2001, max_seq_len=50, dropout=0.0)


def _batches(G):
    from mrm_b200 import synthetic
    cfg = _cfg()
    # few users: the same user id on several ranks exercises the cross-rank collision mask
    return [[synthetic.make_batch(cfg, B_RANK, seed=40 + 10 * s + r, num_users=12) for r in range(G)]
            for s in range(STEPS)]


def _run_emulated_runners(G, sharded, sd, batches, monkeypatch):
    """TrainStepRunner with comm='symm' on G threads; returns per rank a list of per-step snapshots."""
    import torch.distributed as dist
    from mrm_b200 import symm
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.sharding import SymmShardedTable
    from mrm_b200.train import TrainStepRunner
    cfg = _cfg()
    world = EmulatedWorld(G, threaded=True)
    real_rank, real_size = dist.get_rank, dist.get_world_size
    monkeypatch.setattr(symm, "available", lambda group=None: True)
    monkeypatch.setattr(symm, "SymmArena", ThreadedEmulatedArena)
    monkeypatch.setattr(dist, "get_rank", lambda group=None: group.rank if isinstance(group, EmulatedGroup) else real_rank(group))
    monkeypatch.setattr(dist, "get_world_size",
                        lambda group=None: group.size() if isinstance(group, EmulatedGroup) else real_size(group))
    dev_batches = [[{k: v.cuda() for k, v in b.items()} for b in step] for step in batches]

    def rank(r):
        grp = world.group(r)
        table = None
        if sharded:
            eng = TwoTowerEngine(dataclasses.replace(cfg, vocab_size=2))
            table = SymmShardedTable(cfg.vocab_size, cfg.embedding_dim, grp, eng.device)
            eng.peer_table = table
        else:
            eng = TwoTowerEngine(cfg)
        eng.load_state_dict(sd)            # sharded: each owner loads its rows, then the table arena's barrier
        runner = TrainStepRunner(eng, B_RANK, cfg.max_seq_len, world_size=G, lr=LR, use_graph=False, rank=r, group=grp,
                                 sharded_table=table, betas=BETAS, eps=EPS, weight_decay=WD, comm="symm")
        assert runner.arena is not None and isinstance(runner.arena, ThreadedEmulatedArena)
        snaps = []
        for s in range(STEPS):
            loss = runner.step_from_host(dev_batches[s][r])
            torch.cuda.current_stream().synchronize()
            snap = {"loss": loss, "flat": eng.flat.clone(), "shadow": eng.shadow.clone(), "m": eng.exp_avg.clone(),
                    "v": eng.exp_avg_sq.clone(), "step": int(eng.step_dev.item()),
                    "loss_all": runner.arena.view("loss_all", torch.float32, (G, 4)).clone(), "layout": eng.layout,
                    "dense_begin": eng.dense_begin, "grad_zero": bool((eng.grad == 0).all())}
            if sharded:
                snap["table"] = [t.clone() for t in table.shard_tensors()]
                snap["rows"] = table.rows
            snaps.append(snap)
        return snaps

    return run_ranks(world, rank)


def _table_full(snaps, G, V, k):
    """The (V, 256) table of shard tensor k (0 = p, 2 = m, 3 = v) reassembled from the ranks' round-robin shards."""
    out = torch.empty(V, 256, device="cuda")
    for r, s in enumerate(snaps):
        out[r::G] = s["table"][k].view(-1, 256)[:s["rows"]]
    return out


def _by_name(flat, layout, name):
    off, shape = layout[name]
    n = 1
    for d in shape:
        n *= d
    return flat[off:off + n].view(shape)


@pytest.mark.parametrize("sharded", [False, True], ids=["replicated_table", "sharded_table"])
@pytest.mark.parametrize("G", [2, 4])
def test_symm_training_step_on_emulated_ranks(G, sharded, monkeypatch):
    from mrm_b200 import ops, synthetic
    from mrm_b200.engine import TwoTowerEngine
    from oracle import two_tower_oracle as oracle
    from _virtual_dp import virtual_dp_step
    TABLE = "user_tower.item_embedding.weight"
    cfg = _cfg()
    V = cfg.vocab_size
    sd = synthetic.make_state_dict(cfg, seed=3)
    batches = _batches(G)
    runs = _run_emulated_runners(G, sharded, sd, batches, monkeypatch)
    monkeypatch.undo()
    lay = runs[0][0]["layout"]

    # the reference: G replicated engines, torch.cat exchanges, tt_adamw_step on the rank-order gradient sum;
    # every step starts from the runner's state before it (lockstep), so the two gradients differ only by the order
    # fp32 atomics land in
    refs = []
    for _ in range(G):
        e = TwoTowerEngine(cfg)
        e.load_state_dict(sd)
        refs.append(e)
    rl = refs[0].layout
    n_ref = refs[0].numel
    step_dev = torch.zeros((), dtype=torch.long, device="cuda")
    b1 = BETAS[0]

    def runner_full(snaps, key, k_table):
        """A runner state tensor (flat / m / v) in the reference engine's layout."""
        G_ = len(snaps)
        if key == "flat":
            src = snaps[0]["flat"]
        else:
            src = torch.cat([s[key] for s in snaps])
        out = torch.zeros(n_ref, device="cuda")
        for name in rl:
            if name == TABLE and sharded:
                _by_name(out, rl, name).copy_(_table_full(snaps, G_, V, k_table))
            else:
                _by_name(out, rl, name).copy_(_by_name(src, lay, name))
        return out

    p_prev = torch.zeros(n_ref, device="cuda")
    for name in rl:
        _by_name(p_prev, rl, name).copy_(refs[0].p[name])
    m_prev = torch.zeros(n_ref, device="cuda")
    v_prev = torch.zeros(n_ref, device="cuda")
    touched_ever = torch.zeros(V, dtype=torch.bool, device="cuda")
    worst = {"grad_vs_ref": 0.0, "param_vs_ref": 0.0, "oracle_grad": 0.0}
    for s in range(STEPS):
        snaps = [run[s] for run in runs]
        # every rank holds the same parameters and shadow, every rank's loss share, a cleared gradient
        for r, sn in enumerate(snaps):
            assert _bit_equal(sn["flat"], snaps[0]["flat"]) and _bit_equal(sn["shadow"], snaps[0]["shadow"]), (s, r)
            assert _bit_equal(sn["shadow"], sn["flat"][sn["dense_begin"]:].to(torch.bfloat16)), (s, r)
            assert _bit_equal(sn["loss_all"], snaps[0]["loss_all"]), (s, r)
            assert sn["step"] == s + 1 and sn["grad_zero"], (s, r)
        # reference step from the runner's state before this step
        for e in refs:
            for name in rl:
                e.p[name].copy_(_by_name(p_prev, rl, name))
            e.shadow_valid = False
            e.grad.zero_()
        dbs = [{k: v.cuda() for k, v in b.items()} for b in batches[s]]
        total, wss = virtual_dp_step(refs, dbs)
        shares = torch.stack([ws["loss"].view(()) for ws in wss])
        gsum = refs[0].grad.clone()
        for e in refs[1:]:
            gsum = gsum + e.grad
        p_ref, m_ref, v_ref = p_prev.clone(), m_prev.clone(), v_prev.clone()
        step_dev.fill_(s + 1)
        ops.adamw_step(p_ref, gsum, m_ref, v_ref, step_dev, LR, BETAS[0], BETAS[1], EPS, WD, shadow=None,
                       grad_scale=1.0 / G)
        torch.cuda.synchronize()
        la = snaps[0]["loss_all"]
        assert _bit_equal(la[:, 0], shares), (s, la[:, 0].tolist(), shares.tolist())
        assert bool((la[:, 1:] == 0).all())
        assert abs(snaps[0]["loss"] - total) <= 1e-6 * abs(total), (s, snaps[0]["loss"], total)

        p_run, m_run, v_run = (runner_full(snaps, k, j) for k, j in (("flat", 0), ("m", 2), ("v", 3)))
        g_run = (m_run - b1 * m_prev) / (1 - b1)
        g_ref = (m_ref - b1 * m_prev) / (1 - b1)
        for name in rl:
            a, b = _by_name(g_run, rl, name), _by_name(g_ref, rl, name)
            err, ref = (a - b).norm().item(), b.norm().item()
            bound = 1e-2 * ref + 1e-6 * a.numel() ** 0.5
            worst["grad_vs_ref"] = max(worst["grad_vs_ref"], err / bound)
            assert err <= bound, (s, name, err, ref)
        # parameters: the same AdamW from the same state. Wherever the two gradients agree to 0.1 % the updates agree
        # to 1 % of lr; elsewhere (noise-level gradients such as the Linear bias in front of BatchNorm, whose true
        # gradient is zero) an update may flip its sign, which moves the element by at most 2 lr
        agree = (g_run - g_ref).abs() <= 1e-3 * g_ref.abs()
        assert agree.float().mean().item() >= 0.9, (s, agree.float().mean().item())
        dp = (p_run - p_ref).abs()
        worst["param_vs_ref"] = max(worst["param_vs_ref"], dp[agree].max().item())
        assert dp[agree].max().item() <= 1e-2 * LR, (s, dp[agree].max().item())
        assert dp.max().item() <= 2.01 * LR, (s, dp.max().item())
        if sharded:
            # rows no rank's batch has touched so far carry no moments and only decayed
            touched = torch.zeros(V, dtype=torch.bool, device="cuda")
            for b in dbs:
                touched[b["history_ids"].view(-1)] = True
            touched_ever |= touched
            tp, tprev = _by_name(p_run, rl, TABLE), _by_name(p_prev, rl, TABLE)
            quiet = ~touched_ever
            quiet[0] = True
            assert int(quiet.sum()) > 100
            assert _bit_equal(tp[quiet], _by_name(p_ref, rl, TABLE)[quiet])
            assert bool((_by_name(m_run, rl, TABLE)[quiet] == 0).all()) and bool((_by_name(v_run, rl, TABLE)[quiet] == 0).all())
            decayed = tprev[quiet] * (1 - LR * WD)
            assert bool(((tp[quiet] - decayed).abs() <= 1.2e-7 * decayed.abs()).all())
        if s == 0:
            # fp64 oracle: global-batch InfoNCE over per-rank towers, then AdamW (tolerances of
            # tests/test_bench_shapes.py::test_dp_parameter_gradients_match_global_batch_oracle)
            if G not in _ORACLE:
                _ORACLE[G] = oracle.dp_loss_and_grads(sd, batches[0], cfg.temperature, cfg.num_heads, dtype=torch.float64)
            ol, og = _ORACLE[G][0], _ORACLE[G][1]
            worst["oracle_loss"] = abs(snaps[0]["loss"] - ol.item())
            assert worst["oracle_loss"] <= 5e-3, (snaps[0]["loss"], ol.item())
            for name, ref in og.items():
                got = _by_name(g_run, rl, name).cpu().double()
                err = (got - ref).norm().item()
                bound = 0.15 * ref.norm().item() + 5e-5 * ref.numel() ** 0.5
                worst["oracle_grad"] = max(worst["oracle_grad"], err / bound)
                assert err <= bound, (name, err, ref.norm().item())
                p0 = sd[name].double()
                po, _, _ = oracle.adamw_step(p0, ref, torch.zeros_like(p0), torch.zeros_like(p0), 1, LR, BETAS[0],
                                             BETAS[1], EPS, WD)
                # step 1 moves every element by at most lr: the signs may differ where the bf16 gradient is noise
                dp_o = (_by_name(p_run, rl, name).cpu().double() - po).abs().max().item()
                assert dp_o <= 2 * LR + 1e-6 * p0.abs().max().item(), (name, dp_o)
        p_prev, m_prev, v_prev = p_run, m_run, v_run
    print(f"symm step G={G} {'sharded' if sharded else 'replicated'}: loss shares bit-equal; worst gradient error / "
          f"bound {worst['grad_vs_ref']:.3g}; worst |p - p_ref| where the gradients agree {worst['param_vs_ref']:.3g}; "
          f"fp64 oracle: loss {worst['oracle_loss']:.3g}, worst gradient error / bound {worst['oracle_grad']:.3g}")


# ---------------------------------------------------------------------------------------------------------------
# symm.SymmArena as shipped, world 1
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def world1():
    """A single-rank NCCL group over a HashStore: no ports, no other process. Destroyed on teardown, because several
    code paths branch on dist.is_initialized()."""
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


def test_symm_arena_world1(world1):
    from mrm_b200 import ops, symm
    n, sb = 4 * 1000, 4 * 333
    layout = {"flat": n * 4, "grad": n * 4, "shadow": (n - sb) * 2, "odd": 1000, "blk": 4096}
    try:
        a = symm.SymmArena(layout, world1)
    except Exception as exc:       # noqa: BLE001
        pytest.skip(f"symmetric memory at world 1: {type(exc).__name__}: {exc}")
    print(f"SymmArena world 1: multicast mapping {'present' if a.multicast else 'absent'}")
    assert a.rank == 0 and a.world == 1 and a.team.world == 1 and a.team.bufs[0] == a.buf.data_ptr()
    off = 0
    for name, nb in layout.items():
        assert a.offset(name) == off and a.offset(name) % 256 == 0
        assert a.view(name, torch.uint8, (nb,)).data_ptr() == a.buf.data_ptr() + off
        off = (off + nb + 255) // 256 * 256
    assert a.ctrl_offset == off and a.nbytes == off + 4096 and a.buf.numel() == a.nbytes
    assert a.error_word().data_ptr() == a.buf.data_ptr() + a.ctrl_offset + 8
    a.check()
    a.error_word().fill_(1)
    with pytest.raises(RuntimeError):
        a.check()
    a.error_word().zero_()
    with pytest.raises(AssertionError):
        a.allgather([(torch.zeros(8, dtype=torch.uint8, device="cuda"), "blk")])
    ctrl = a.buf[a.ctrl_offset:a.ctrl_offset + 192].view(torch.int32)

    gen = torch.Generator(device="cuda").manual_seed(5)
    a.buf[:a.ctrl_offset].copy_(_random_bytes(a.ctrl_offset, gen))
    expect = a.buf[:a.ctrl_offset].clone()
    src = _random_bytes(2048, gen)
    a.allgather([(src, "blk")], pre_barrier=True)
    torch.cuda.synchronize()
    expect[a.offset("blk"):a.offset("blk") + 2048] = src
    assert torch.equal(a.buf[:a.ctrl_offset], expect)
    assert ctrl[0].item() == 1 and ctrl[1].item() == 0 and ctrl[2].item() == 0
    assert ctrl[READY].item() == 1 and ctrl[DONE].item() == 1

    p0 = 0.05 * torch.randn(n, device="cuda", generator=gen)
    sign = torch.where(torch.rand(n, device="cuda", generator=gen) < 0.5, -1.0, 1.0)
    g = _grad(n, sign, gen)
    a.view("flat", torch.float32, (n,)).copy_(p0)
    a.view("grad", torch.float32, (n,)).copy_(g)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    step = torch.ones((), dtype=torch.long, device="cuda")
    a.dp_adamw_step("flat", "grad", "shadow", n, sb, m, v, step, LR, BETAS, EPS, WD)
    p_ref, m_ref, v_ref = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    sh_ref = torch.zeros(n - sb, device="cuda", dtype=torch.bfloat16)
    ops.adamw_step(p_ref, g.clone(), m_ref, v_ref, step, LR, BETAS[0], BETAS[1], EPS, WD, shadow=sh_ref,
                   shadow_begin=sb, shadow_end=n, grad_scale=1.0)
    torch.cuda.synchronize()
    how = "multimem (multicast)" if a.multicast else "unicast"
    assert _bit_equal(a.view("flat", torch.float32, (n,)), p_ref), how
    assert _bit_equal(a.view("shadow", torch.bfloat16, (n - sb,)), sh_ref), how
    assert _bit_equal(m, m_ref) and _bit_equal(v, v_ref), how
    assert _bit_equal(a.view("grad", torch.float32, (n,)), g)
    assert ctrl[0].item() == 2 and ctrl[1].item() == 0 and ctrl[2].item() == 0
    a.check()
