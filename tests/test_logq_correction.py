"""logQ correction of in-batch negatives (train.LogQCorrection, tt_logq_*, tt_infonce_*_off).

CPU: a numpy restatement of the streaming estimator (hash, once-per-slot update, offset) checked on hand-made
streams, the count-based offsets and every Python guard. GPU: the estimator kernel against the restatement bit for
bit, the corrected loss kernels against fp64 torch, the engine step against an fp64 restatement of the corrected
loss built on oracle.two_tower_forward, the unchanged default path, graph against eager, emulated data-parallel
ranks, checkpoint / restore and train_one_epoch.
"""
import math

import numpy as np
import pytest
import torch

GOLDEN = np.uint64(0x9E3779B97F4A7C15)
LR, BETAS, EPS, WD = 1e-3, (0.9, 0.999), 1e-8, 0.01


# ---------------------------------------------------------------------------------------------------------------
# numpy restatement of the streaming estimator
# ---------------------------------------------------------------------------------------------------------------
def slot(ids, k: int, log2H: int) -> np.ndarray:
    """Low log2H bits of the splitmix64 finaliser of id + (k + 1) * golden ratio (mod 2^64)."""
    with np.errstate(over="ignore"):
        z = np.asarray(ids, dtype=np.int64).astype(np.uint64) + np.uint64(k + 1) * GOLDEN
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z & np.uint64((1 << log2H) - 1)).astype(np.int64)


class Estimator:
    """State A int64 / Bv fp32 [h, H], step t; every fp32 operation rounded once, as the kernel does."""

    def __init__(self, h: int, log2H: int, alpha: float, init: float):
        self.h, self.log2H = h, log2H
        self.a = np.float32(alpha)
        self.om = np.float32(1.0 - alpha)
        self.A = np.zeros((h, 1 << log2H), dtype=np.int64)
        self.Bv = np.full((h, 1 << log2H), np.float32(init), dtype=np.float32)
        self.t = 0

    def step(self, ids) -> np.ndarray:
        self.t += 1
        ids = np.asarray(ids, dtype=np.int64)
        best = np.zeros(len(ids), dtype=np.float32)
        for k in range(self.h):
            s = slot(ids, k, self.log2H)
            u = np.unique(s)                      # a slot is updated once however many ids hit it
            gap = (self.t - self.A[k, u]).astype(np.float32)
            self.Bv[k, u] = (self.om * self.Bv[k, u]) + (self.a * gap)
            self.A[k, u] = self.t
            best = np.maximum(best, self.Bv[k, s])
        return (-np.log(best.astype(np.float64))).astype(np.float32)


def test_interval_of_a_periodic_id_converges():
    est = Estimator(2, 16, alpha=0.2, init=50.0)
    for t in range(1, 601):
        ids = [1000 + t]                          # a fresh id every step keeps the other slots busy
        if t % 7 == 0:
            ids.append(42)
        est.step(ids)
    for k in range(2):
        assert abs(est.Bv[k, slot([42], k, 16)[0]] - 7.0) < 1e-3


def test_duplicates_update_a_slot_once():
    a, b = Estimator(2, 10, 0.1, 10.0), Estimator(2, 10, 0.1, 10.0)
    for t in range(20):
        oa = a.step([5, 5, 5, 9, t + 100])
        ob = b.step([5, 9, t + 100])
        assert np.array_equal(oa[[0, 3, 4]], ob) and oa[0] == oa[1] == oa[2]
    assert np.array_equal(a.Bv, b.Bv) and np.array_equal(a.A, b.A)


def test_forced_collisions_take_the_max_over_arrays():
    log2H = 3
    s0 = slot(np.arange(1, 200), 0, log2H)
    s1 = slot(np.arange(1, 200), 1, log2H)
    # x collides with y in array 0 but not in array 1
    pairs = [(x, y) for x in range(1, 200) for y in range(x + 1, 200) if s0[x - 1] == s0[y - 1] and s1[x - 1] != s1[y - 1]]
    x, y = pairs[0]
    est = Estimator(2, log2H, alpha=0.5, init=10.0)
    for t in range(1, 41):
        off = est.step([y] if t % 2 else [x, y])   # y every step, x every other step
    bx0, bx1 = est.Bv[0, s0[x - 1]], est.Bv[1, s1[x - 1]]
    assert bx0 < 1.01 and bx1 > 1.9                # array 0 sees x's slot every step (shared with y), array 1 every 2
    assert off[0] == np.float32(-np.log(np.float64(max(bx0, bx1))))


def test_initial_state():
    from mrm_b200.train import LogQCorrection
    est = Estimator(1, 4, alpha=0.25, init=8.0)
    assert (est.A == 0).all() and (est.Bv == np.float32(8.0)).all()
    off = est.step([3])
    s = slot([3], 0, 4)[0]
    assert est.A[0, s] == 1 and est.Bv[0, s] == np.float32(np.float32(0.75) * np.float32(8.0) + np.float32(0.25))
    assert off[0] == np.float32(-np.log(np.float64(est.Bv[0, s])))
    c = LogQCorrection.streaming(1000, num_slots=16, device="cpu")
    assert c.init_interval is None
    c.bind(64)
    assert c.init_interval == 1000 / 64 and torch.equal(c.Bv, torch.full((2, 16), 1000 / 64))
    assert int(c.step) == 0 and bool((c.A == 0).all())
    c.bind(8)                                                 # a later runner with another batch keeps the state
    assert c.init_interval == 1000 / 64
    small = LogQCorrection.streaming(10, num_slots=16, device="cpu")
    small.bind(64)
    assert small.init_interval == 1.0
    fixed = LogQCorrection.streaming(10, num_slots=16, init_interval=3.0, device="cpu")
    fixed.bind(64)
    assert fixed.init_interval == 3.0


def test_from_counts_offsets():
    from mrm_b200.train import LogQCorrection
    counts = np.random.default_rng(0).zipf(1.5, size=5000).astype(np.float64)
    counts[::7] = 0
    for s in (1.0, 0.5):
        c = LogQCorrection.from_counts(counts, smoothing=s, device="cpu")
        assert c.table.dtype == torch.float32 and c.table.shape == (5000,)
        assert abs(torch.exp(c.table.double()).sum().item() - 1.0) < 1e-6
        assert bool((c.table[::7] == c.floor).all())
        assert c.floor == float(np.float32(math.log(s / (counts + s).sum())))
    o = LogQCorrection.from_offsets(torch.tensor([-1.0, -2.0, -3.0]), device="cpu")
    assert o.floor == -3.0 and torch.equal(o.table, torch.tensor([-1.0, -2.0, -3.0]))


@pytest.mark.parametrize("kw", [dict(alpha=0.0), dict(alpha=1.5), dict(alpha=-0.1), dict(alpha=float("nan")),
                                dict(num_slots=3), dict(num_slots=2 ** 29), dict(num_slots=0), dict(num_hashes=0),
                                dict(num_hashes=5), dict(init_interval=0.0), dict(init_interval=float("nan"))])
def test_streaming_guards(kw):
    from mrm_b200.train import LogQCorrection
    with pytest.raises(ValueError):
        LogQCorrection.streaming(1000, device="cpu", **kw)


def test_table_guards():
    from mrm_b200.train import LogQCorrection
    bad_counts = [[1.0, -1.0], [1.0, float("nan")], [[1.0, 2.0]], [], [1.0, float("inf")]]
    for c in bad_counts:
        with pytest.raises(ValueError):
            LogQCorrection.from_counts(c, device="cpu")
    for s in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            LogQCorrection.from_counts([1.0, 2.0], smoothing=s, device="cpu")
    for t in ([0.0, float("nan")], [[0.0]], [], [float("-inf")]):
        with pytest.raises(ValueError):
            LogQCorrection.from_offsets(t, device="cpu")
    with pytest.raises(ValueError):
        LogQCorrection.streaming(0, device="cpu")


def test_user_side_needs_user_idx_and_fused_optimizer():
    from mrm_b200.train import LogQCorrection, TrainStepRunner, train_one_epoch
    c = LogQCorrection.from_counts([1.0, 2.0], device="cpu")
    with pytest.raises(ValueError):
        TrainStepRunner(None, 16, 8, with_user_idx=False, logq_users=c)

    class _Model:
        def train(self):
            pass

    opt = torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=0.1)
    for kw in (dict(logq=c), dict(logq_users=c)):
        with pytest.raises(ValueError):
            train_one_epoch(_Model(), [], opt, torch.device("cpu"), 0, **kw)


def test_state_dict_guards():
    from mrm_b200.train import LogQCorrection
    a = LogQCorrection.streaming(100, num_slots=16, device="cpu")
    a.bind(4)
    with pytest.raises(ValueError):
        LogQCorrection.streaming(100, num_slots=32, device="cpu").load_state_dict(a.state_dict())
    with pytest.raises(ValueError):
        LogQCorrection.from_counts([1.0, 2.0], device="cpu").load_state_dict(a.state_dict())


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _zipf_ids(rng, n, num_ids):
    return np.minimum(rng.zipf(1.2, size=n), num_ids).astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 256, 4096])
@pytest.mark.parametrize("log2H,h", [(8, 1), (8, 2), (8, 4), (20, 1), (20, 2), (20, 4)])
def test_stream_update_kernel_matches_restatement(n, log2H, h):
    from mrm_b200 import ops
    steps, alpha, init, num_ids = 300, 0.05, 40.0, 20000
    rng = np.random.default_rng(n * 100 + log2H * 10 + h)
    stream = [_zipf_ids(rng, n, num_ids) for _ in range(steps)]
    ref = Estimator(h, log2H, alpha, init)
    ref_off = np.stack([ref.step(ids) for ids in stream])
    ids_dev = torch.from_numpy(np.stack(stream)).cuda()
    states = []
    for _ in range(2):
        A = torch.zeros(h, 1 << log2H, dtype=torch.int64, device="cuda")
        Bv = torch.full((h, 1 << log2H), init, dtype=torch.float32, device="cuda")
        step = torch.zeros(1, dtype=torch.int64, device="cuda")
        off = torch.empty(steps, n, device="cuda")
        for t in range(steps):
            ops.logq_stream_update(ids_dev[t], A, Bv, step, alpha, float(np.float32(1.0 - alpha)), off[t])
        torch.cuda.synchronize()
        states.append((A, Bv, step, off))
    A, Bv, step, off = states[0]
    assert int(step) == steps
    assert torch.equal(A.cpu(), torch.from_numpy(ref.A)) and torch.equal(Bv.cpu(), torch.from_numpy(ref.Bv))
    for x, y in zip(states[0], states[1]):
        assert torch.equal(x, y)
    err = (off.cpu().double() - torch.from_numpy(ref_off).double()).abs().max().item()
    assert err <= 2.0 ** -20, err


@pytest.mark.gpu
def test_table_gather_kernel():
    from mrm_b200 import ops
    table = torch.randn(1000, device="cuda")
    ids = torch.tensor([0, 999, 1000, -1, 5, 5, 2 ** 40], device="cuda")
    out = torch.empty(7, device="cuda")
    ops.logq_table_gather(ids, table, -7.5, out)
    ref = torch.tensor([table[0], table[999], -7.5, -7.5, table[5], table[5], -7.5], device="cuda")
    assert torch.equal(out, ref)


def _loss_block(R, C, pos0, seed):
    g = torch.Generator().manual_seed(seed)
    S = (torch.randn(R, C, generator=g) * 4.0).cuda()
    uid_cols = torch.randint(0, max(C // 3, 2), (C,), generator=g).cuda()
    uid_rows = uid_cols[pos0:pos0 + R].clone()
    oi = (-torch.rand(C, generator=g) * 8.0).cuda()
    ou = (-torch.rand(C, generator=g) * 8.0).cuda()
    return S, uid_rows, uid_cols, oi, ou


@pytest.mark.gpu
@pytest.mark.parametrize("R,G,r", [(70, 1, 0), (64, 4, 2), (32, 3, 1)], ids=["square", "gathered_G4", "gathered_G3"])
def test_offset_loss_kernels_match_fp64(R, G, r):
    from mrm_b200 import ops
    C, pos0 = R * G, R * r
    S, uid_rows, uid_cols, oi, ou = _loss_block(R, C, pos0, seed=R + G)
    coll = (uid_rows[:, None] == uid_cols[None, :])
    coll[torch.arange(R), pos0 + torch.arange(R)] = False
    Sm = S.masked_fill(coll, -1e4).double()
    x = Sm - oi.double()[None, :]
    lse_ref = torch.logsumexp(x, 1)
    pos_ref = Sm[torch.arange(R), pos0 + torch.arange(R)] - oi.double()[pos0:pos0 + R]
    S1 = S.clone()
    lse, pos = torch.empty(R, device="cuda"), torch.empty(R, device="cuda")
    ops.infonce_rows_off(S1, uid_rows, uid_cols, pos0, oi, lse, pos)
    assert torch.equal(S1, Sm.float())                     # S keeps the uncorrected masked logits
    assert (lse.double() - lse_ref).abs().max().item() < 1e-4
    assert (pos.double() - pos_ref).abs().max().item() < 1e-5
    # gradient: column log-sum-exps of the other direction (any values the kernel must combine exactly as stated)
    col_lse = torch.logsumexp(Sm - ou.double()[pos0:pos0 + R, None], 0).float()
    coef = 0.5 / C
    dS = torch.empty(R, (C + 7) // 8 * 8, device="cuda", dtype=torch.bfloat16)[:, :C]
    ops.infonce_grad_off(S1, lse, col_lse, pos0, coef, oi, ou, dS)
    ref = coef * (torch.exp(Sm - oi.double()[None, :] - lse.double()[:, None])
                  + torch.exp(Sm - ou.double()[pos0:pos0 + R, None] - col_lse.double()[None, :]))
    ref[torch.arange(R), pos0 + torch.arange(R)] -= 2 * coef
    assert (dS.double() - ref).abs().max().item() < 1e-4
    # zero offsets: bit-equal to the plain kernels
    z = torch.zeros(C, device="cuda")
    Sa, Sb = S.clone(), S.clone()
    la, pa, lb, pb = (torch.empty(R, device="cuda") for _ in range(4))
    ops.infonce_rows(Sa, uid_rows, uid_cols, pos0, la, pa)
    ops.infonce_rows_off(Sb, uid_rows, uid_cols, pos0, z, lb, pb)
    assert torch.equal(Sa, Sb) and torch.equal(la, lb) and torch.equal(pa, pb)
    da, db = torch.empty_like(dS), torch.empty_like(dS)
    ops.infonce_grad(Sa, la, col_lse, pos0, coef, da)
    ops.infonce_grad_off(Sa, la, col_lse, pos0, coef, z, z, db)
    assert torch.equal(da, db)


@pytest.mark.gpu
def test_c_entry_points_reject_bad_arguments():
    from mrm_b200 import _lib
    l = _lib.lib()
    x = torch.zeros(64, device="cuda")
    i64 = torch.zeros(64, dtype=torch.long, device="cuda")
    p, q = x.data_ptr(), i64.data_ptr()
    assert l.tt_logq_stream_update(q, 4, q, p, 0, 3, q, 0.1, 0.9, p, None) == 1          # h = 0
    assert l.tt_logq_stream_update(q, 4, q, p, 5, 3, q, 0.1, 0.9, p, None) == 1          # h = 5
    assert l.tt_logq_stream_update(q, 4, q, p, 1, 29, q, 0.1, 0.9, p, None) == 1         # H = 2^29
    assert l.tt_logq_stream_update(q, 4, q, p, 1, 3, q, 0.0, 1.0, p, None) == 1          # alpha = 0
    assert l.tt_logq_stream_update(q, 0, q, p, 1, 3, q, 0.1, 0.9, p, None) == 1          # n = 0
    assert l.tt_logq_stream_update(None, 4, q, p, 1, 3, q, 0.1, 0.9, p, None) == 1
    assert l.tt_logq_table_gather(q, 4, None, 10, 0.0, p, None) == 1
    assert l.tt_logq_table_gather(q, 4, p, 0, 0.0, p, None) == 1
    assert l.tt_infonce_rows_off(p, 4, 8, 8, None, None, 0, None, p, p, None) == 1       # no offsets
    assert l.tt_infonce_rows_off(p, 4, 8, 8, None, None, 5, p, p, p, None) == 1          # positives outside
    assert l.tt_infonce_grad_off(p, 4, 8, 8, p, p, 0, 0.1, p, None, p, 8, None) == 1
    assert l.tt_infonce_grad_off(p, 4, 8, 8, p, p, 0, 0.1, p, p, p, 7, None) == 1        # odd ld_d
    torch.cuda.synchronize()


# ---- engine step against an fp64 restatement of the corrected loss ------------------------------------------
def corrected_infonce(logits, oi, ou):
    """The corrected symmetric InfoNCE on the masked logits (users x items): user rows over x - oi[j], item rows
    (columns of logits) over x - ou[i]."""
    d = logits.diagonal()
    lse_r = torch.logsumexp(logits - oi[None, :], dim=1)
    lse_c = torch.logsumexp(logits - ou[:, None], dim=0)
    return 0.5 * ((lse_r - (d - oi)).mean() + (lse_c - (d - ou)).mean())


def corrected_loss_and_grads(sd, batch, oi, ou, temperature, num_heads):
    from oracle import two_tower_oracle as oracle
    q = {k: (v.clone() if k.endswith(oracle.TRAINABLE_SKIP) else v.detach().double().clone().requires_grad_(True))
         for k, v in sd.items()}
    b64 = {k: (v.double() if v.is_floating_point() else v) for k, v in batch.items()}
    _, logits, u, i, _ = oracle.two_tower_forward(q, b64, temperature, num_heads, training=True)
    loss = corrected_infonce(logits, oi.double(), ou.double())
    loss.backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in q.items()
             if isinstance(v, torch.Tensor) and v.requires_grad}
    grads["user_tower.item_embedding.weight"][0] = 0
    return loss.detach(), logits.detach(), u.detach(), i.detach(), grads


def _small_cfg():
    from mrm_b200 import synthetic
    return synthetic.TwoTowerConfig(vocab_size=2001, max_seq_len=50, dropout=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("users", [False, True], ids=["items", "items_and_users"])
def test_engine_step_matches_fp64_corrected_loss(users):
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import LogQCorrection
    cfg = _small_cfg()
    sd = synthetic.make_state_dict(cfg, seed=0)
    B = 64
    batch = synthetic.make_batch(cfg, B, seed=7, num_users=40)     # same-user collisions
    rng = np.random.default_rng(3)
    items = LogQCorrection.from_counts(rng.zipf(1.3, size=cfg.vocab_size).clip(max=10 ** 6).astype(float))
    ucorr = LogQCorrection.from_counts(rng.zipf(1.5, size=40).astype(float)) if users else None
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(sd)
    db = {k: v.cuda() for k, v in batch.items()}
    oi, ou = torch.zeros(B, device="cuda"), torch.zeros(B, device="cuda")
    items.offsets(db["target_id"], oi)
    if ucorr is not None:
        ucorr.offsets(db["user_idx"], ou)
    ws = eng.forward_towers(db, training=True)
    loss = eng.loss_forward(ws, db["user_idx"], offsets=(oi, ou))
    eng.backward()
    torch.cuda.synchronize()
    assert not torch.equal(oi, torch.zeros_like(oi)) and (users == (not torch.equal(ou, torch.zeros_like(ou))))
    torch.set_num_threads(8)
    rl, rlog, ru, ri, grads = corrected_loss_and_grads(sd, batch, oi.cpu(), ou.cpu(), cfg.temperature, cfg.num_heads)
    assert abs(loss.item() - rl.item()) <= 5e-3, (loss.item(), rl.item())
    assert (ws["un"].cpu().double() - ru).abs().max().item() <= 5e-3
    assert (ws["in"].cpu().double() - ri).abs().max().item() <= 5e-3
    assert (ws["S"].cpu().double() - rlog).abs().max().item() <= 8e-2      # logits stay uncorrected
    # tolerance anchor: the uncorrected step of the same engine against the same fp64 restatement with zero offsets
    # (what test_c2_step_matches_fp64_oracle anchors on the reference's own bf16 error); bound = max(2 x that error,
    # 3e-2 ||g|| + 1e-5 sqrt(n)) per parameter
    plain = TwoTowerEngine(cfg)
    plain.load_state_dict(sd)
    plain.forward(db, training=True)
    plain.backward()
    torch.cuda.synchronize()
    zero = torch.zeros(B)
    pl, _, _, _, pgrads = corrected_loss_and_grads(sd, batch, zero, zero, cfg.temperature, cfg.num_heads)
    bad, worst = [], 0.0
    for k, ref in grads.items():
        err = (eng.g[k].cpu().double() - ref).norm().item()
        anchor = (plain.g[k].cpu().double() - pgrads[k]).norm().item()
        bound = max(2 * anchor, 3e-2 * ref.norm().item() + 1e-5 * ref.numel() ** 0.5)
        worst = max(worst, err / bound)
        if err > bound:
            bad.append((k, err, anchor, ref.norm().item()))
    print(f"corrected engine step ({'items and users' if users else 'items'}): loss {loss.item():.5f} vs "
          f"{rl.item():.5f}; worst gradient error / bound {worst:.3g}")
    assert not bad, bad[:5]
    # the correction changes the objective: the plain loss differs
    assert abs(pl.item() - rl.item()) > 1e-2


# ---- the default path is unchanged ----------------------------------------------------------------------------
def _runner(cfg, sd, B, **kw):
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import TrainStepRunner
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(sd)
    return eng, TrainStepRunner(eng, B, cfg.max_seq_len, lr=LR, betas=BETAS, eps=EPS, weight_decay=WD, **kw)


PLAIN_FIELDS = ["history_ids", "history_mask", "user_gender", "user_country", "target_audio", "target_image",
                "target_input_ids", "target_tabular", "user_idx"]


@pytest.mark.gpu
def test_runner_without_correction_never_calls_the_new_ops(monkeypatch):
    from mrm_b200 import ops, synthetic
    cfg = _small_cfg()
    sd = synthetic.make_state_dict(cfg, seed=0)

    def boom(*a, **k):
        raise AssertionError("a logQ op ran on the default path")

    for name in ("logq_table_gather", "logq_stream_update", "infonce_rows_off", "infonce_grad_off"):
        monkeypatch.setattr(ops, name, boom)
    B = 32
    eng, run = _runner(cfg, sd, B)
    assert [f[0] for f in run._fields] == PLAIN_FIELDS
    off = 0
    for name, shape, dt, o, nb in run._fields:
        assert o == off
        off += (nb + 255) // 256 * 256
    assert run._static_buf.numel() == off and run._offsets is None
    for s in range(3):
        run.step_from_host({k: v.cuda() for k, v in synthetic.make_batch(cfg, B, seed=s).items()})
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_zero_offsets_equal_no_correction():
    """dS / dS2 / log-sum-exps / loss (what the loss kernels write) must be bit-equal; the parameter gradients then
    differ at most by the fp32-atomic ordering noise that two plain runs show."""
    from mrm_b200 import synthetic
    from mrm_b200.train import LogQCorrection
    cfg = _small_cfg()
    sd = synthetic.make_state_dict(cfg, seed=1)
    B = 32
    batch = {k: v.cuda() for k, v in synthetic.make_batch(cfg, B, seed=5, num_users=20).items()}
    outs = []
    for corr in (None, None, LogQCorrection.from_offsets(torch.zeros(cfg.vocab_size)),
                 LogQCorrection.from_offsets(torch.zeros(cfg.vocab_size))):
        eng, run = _runner(cfg, sd, B, use_graph=False, logq=corr,
                           logq_users=None if corr is None else LogQCorrection.from_offsets(torch.zeros(20)))
        loss = run.step_from_host(batch)
        ws = eng.workspace(B, cfg.max_seq_len)
        torch.cuda.synchronize()
        outs.append(dict(loss=loss, m=eng.exp_avg.clone(), **{k: ws[k].clone() for k in
                                                             ("lse_r", "lse_c", "pos_r", "pos_c", "dS", "dS2", "S")}))
    plain, other = outs[0], outs[1]
    noise = (plain["m"] - other["m"]).abs().max().item()
    for o in outs[2:]:
        assert o["loss"] == plain["loss"]
        for k in ("lse_r", "lse_c", "pos_r", "pos_c", "dS", "dS2", "S"):
            assert torch.equal(o[k], plain[k]), k
        d = (o["m"] - plain["m"]).abs().max().item()
        assert d <= 2 * noise + 1e-12, (d, noise)
    print(f"zero offsets: loss-kernel outputs bit-equal; first-moment difference {d:.3g} (plain vs plain {noise:.3g})")


# ---- graph against eager ----------------------------------------------------------------------------------------
def _copy_state(dst, src):
    for a, b in ((dst.flat, src.flat), (dst.shadow, src.shadow), (dst.exp_avg, src.exp_avg),
                 (dst.exp_avg_sq, src.exp_avg_sq), (dst.bn_running_mean, src.bn_running_mean),
                 (dst.bn_running_var, src.bn_running_var)):
        a.copy_(b)


@pytest.mark.gpu
def test_graph_replay_matches_eager_with_streaming_estimator():
    from mrm_b200 import synthetic
    from mrm_b200.train import LogQCorrection
    cfg = _small_cfg()
    sd = synthetic.make_state_dict(cfg, seed=2)
    B = 64
    batches = [{k: v.cuda() for k, v in synthetic.make_batch(cfg, B, seed=20 + s, num_users=50).items()}
               for s in range(5)]
    cors = {}
    runs = {}
    for mode in ("eager", "graph"):
        ci = LogQCorrection.streaming(cfg.vocab_size, num_slots=2 ** 12, alpha=0.1)
        cu = LogQCorrection.streaming(50, num_slots=2 ** 8, num_hashes=1, alpha=0.2)
        cors[mode] = (ci, cu)
        runs[mode] = _runner(cfg, sd, B, use_graph=(mode == "graph"), logq=ci, logq_users=cu)
    (ee, er), (ge, gr) = runs["eager"], runs["graph"]
    for s, b in enumerate(batches):
        m_prev = ee.exp_avg.clone() if ee.exp_avg is not None else torch.zeros(ee.numel, device="cuda")
        le = er.step_from_host(b)
        lg = gr.step_from_host(b)
        torch.cuda.synchronize()
        for ce, cg in zip(cors["eager"], cors["graph"]):
            assert int(ce.step) == s + 1 and torch.equal(ce.step, cg.step)
            assert torch.equal(ce.A, cg.A) and torch.equal(ce.Bv, cg.Bv), s
        assert abs(le - lg) <= 1e-2 * abs(le), (s, le, lg)
        ge_ = (ge.exp_avg - BETAS[0] * m_prev) / (1 - BETAS[0])
        ee_ = (ee.exp_avg - BETAS[0] * m_prev) / (1 - BETAS[0])
        for name, (o, shape) in ee.layout.items():
            n = int(np.prod(shape))
            a, r = ge_[o:o + n], ee_[o:o + n]
            assert (a - r).norm().item() <= 1e-2 * r.norm().item() + 1e-6 * n ** 0.5, (s, name)
        _copy_state(ge, ee)                       # lockstep: the next step starts from the same state


# ---- checkpoint -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_checkpoint_restore_is_bit_equal():
    from mrm_b200.train import LogQCorrection
    rng = np.random.default_rng(9)
    stream = [torch.from_numpy(_zipf_ids(rng, 512, 5000)).cuda() for _ in range(6)]

    def make():
        c = LogQCorrection.streaming(5000, num_slots=2 ** 14, num_hashes=3, alpha=0.05)
        c.bind(512)
        return c

    whole = make()
    out_whole = torch.empty(6, 512, device="cuda")
    for t in range(6):
        whole.offsets(stream[t], out_whole[t])
    first = make()
    out = torch.empty(6, 512, device="cuda")
    for t in range(3):
        first.offsets(stream[t], out[t])
    sd = first.state_dict()
    second = LogQCorrection.streaming(1, num_slots=2 ** 14, num_hashes=3, alpha=0.5, init_interval=1.0)
    second.load_state_dict(sd)
    assert second.alpha == 0.05 and second.num_ids == 5000 and second.init_interval == 5000 / 512
    for t in range(3, 6):
        second.offsets(stream[t], out[t])
    torch.cuda.synchronize()
    assert torch.equal(out, out_whole)
    for k in ("A", "Bv", "step"):
        assert torch.equal(getattr(second, k), getattr(whole, k)), k
    assert int(whole.step) == 6


# ---- train_one_epoch --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_train_one_epoch_with_streaming_estimator(monkeypatch):
    from mrm_b200 import synthetic
    from mrm_b200.models import TwoTowerModel
    from mrm_b200.train import FusedAdamW, LogQCorrection, TrainStepRunner, train_one_epoch
    m = TwoTowerModel(vocab_size=2001, tabular_input_dim=17, num_genders=3, num_countries=50, max_seq_len=50,
                      user_dropout=0.0)
    cfg = m.engine.cfg
    loader = [synthetic.make_batch(cfg, 32, seed=60 + s) for s in range(3)] + [synthetic.make_batch(cfg, 8, seed=70)]
    for b in loader:
        for k in b:
            b[k] = b[k].pin_memory()
    flushed = []
    real_flush = TrainStepRunner.flush_loss

    def flush(self):
        v = real_flush(self)
        if v is not None:
            flushed.append(v)
        return v

    monkeypatch.setattr(TrainStepRunner, "flush_loss", flush)
    ci = LogQCorrection.streaming(cfg.vocab_size, num_slots=2 ** 12)
    cu = LogQCorrection.streaming(850, num_slots=2 ** 12)
    mean = train_one_epoch(m, loader, FusedAdamW(m, lr=1e-3), torch.device("cuda"), 0, is_main_process=False,
                           logq=ci, logq_users=cu)
    assert int(ci.step) == 4 and int(cu.step) == 4
    assert ci.init_interval == cfg.vocab_size / 32          # fixed by the first runner, kept by the partial batch's
    assert len(flushed) == 4 and math.isfinite(mean)
    assert mean == sum(flushed) / 4


# ---- data parallel on emulated ranks ----------------------------------------------------------------------------
def corrected_dp_loss_and_grads(sd, batches, oi, ou, temperature, num_heads):
    """oracle.dp_loss_and_grads with the corrected loss: per-rank towers in fp64, one corrected symmetric InfoNCE
    over the concatenated global batch, per-rank autograd seeded with d loss / d embedding."""
    from oracle import two_tower_oracle as oracle
    q = {k: (v.clone() if k.endswith(oracle.TRAINABLE_SKIP) else v.detach().double()) for k, v in sd.items()}

    def towers(params, b):
        u = oracle.user_tower(params, b["history_ids"], b["user_gender"], b["user_country"], b.get("history_mask"),
                              num_heads)
        i, _ = oracle.item_fusion(params, b["target_audio"].double(), b["target_image"].double(),
                                  b["target_input_ids"].double(), b["target_tabular"].double(), True)
        return oracle.l2_normalize(u), oracle.l2_normalize(i)

    with torch.no_grad():
        embs = [towers(q, b) for b in batches]
    U = torch.cat([e[0] for e in embs]).requires_grad_(True)
    I = torch.cat([e[1] for e in embs]).requires_grad_(True)
    uid = torch.cat([b["user_idx"] for b in batches])
    logits = U @ I.t() / temperature
    coll = (uid[:, None] == uid[None, :]) & ~torch.eye(len(uid), dtype=torch.bool)
    loss = corrected_infonce(logits.masked_fill(coll, -1e4), oi.double(), ou.double())
    loss.backward()
    grads, off = None, 0
    for b in batches:
        n = b["history_ids"].shape[0]
        qr = {k: (v if k.endswith(oracle.TRAINABLE_SKIP) else v.clone().requires_grad_(True)) for k, v in q.items()}
        u, i = towers(qr, b)
        torch.autograd.backward([u, i], [U.grad[off:off + n], I.grad[off:off + n]])
        gr = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in qr.items()
              if isinstance(v, torch.Tensor) and v.requires_grad}
        grads = gr if grads is None else {k: grads[k] + gr[k] for k in gr}
        off += n
    grads["user_tower.item_embedding.weight"][0] = 0
    return loss.detach(), grads


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 4])
def test_symm_step_on_emulated_ranks(G, monkeypatch):
    import torch.distributed as dist
    from _emulated_team import EmulatedGroup, EmulatedWorld, ThreadedEmulatedArena, run_ranks
    from mrm_b200 import symm, synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import LogQCorrection, TrainStepRunner
    cfg = _small_cfg()
    sd = synthetic.make_state_dict(cfg, seed=3)
    B, STEPS, NU = 16, 3, 40
    batches = [[synthetic.make_batch(cfg, B, seed=40 + 10 * s + r, num_users=NU) for r in range(G)]
               for s in range(STEPS)]
    # a warmed-up estimator state, so the first step's offsets differ between ids
    rng = np.random.default_rng(11)
    warm_i = Estimator(2, 10, 0.1, 8.0)
    warm_u = Estimator(1, 6, 0.2, 2.0)
    for _ in range(30):
        warm_i.step(_zipf_ids(rng, G * B, cfg.vocab_size - 1))
        warm_u.step(rng.integers(0, NU, G * B))

    def to_state(est, alpha, num_ids, init):
        return {"kind": "streaming", "A": torch.from_numpy(est.A.copy()), "Bv": torch.from_numpy(est.Bv.copy()),
                "step": torch.tensor([est.t]), "alpha": alpha, "num_ids": num_ids, "init_interval": init}

    si, su = to_state(warm_i, 0.1, cfg.vocab_size, 8.0), to_state(warm_u, 0.2, NU, 2.0)
    world = EmulatedWorld(G, threaded=True)
    real_rank, real_size = dist.get_rank, dist.get_world_size
    monkeypatch.setattr(symm, "available", lambda group=None: True)
    monkeypatch.setattr(symm, "SymmArena", ThreadedEmulatedArena)
    monkeypatch.setattr(dist, "get_rank", lambda group=None: group.rank if isinstance(group, EmulatedGroup) else real_rank(group))
    monkeypatch.setattr(dist, "get_world_size",
                        lambda group=None: group.size() if isinstance(group, EmulatedGroup) else real_size(group))
    dev_batches = [[{k: v.cuda() for k, v in b.items()} for b in step] for step in batches]

    def rank(r):
        eng = TwoTowerEngine(cfg)
        eng.load_state_dict(sd)
        ci = LogQCorrection.streaming(cfg.vocab_size, num_slots=2 ** 10, alpha=0.1)
        cu = LogQCorrection.streaming(NU, num_slots=2 ** 6, num_hashes=1, alpha=0.2)
        ci.load_state_dict(si)
        cu.load_state_dict(su)
        runner = TrainStepRunner(eng, B, cfg.max_seq_len, world_size=G, lr=LR, use_graph=False, rank=r,
                                 group=world.group(r), betas=BETAS, eps=EPS, weight_decay=WD, comm="symm",
                                 logq=ci, logq_users=cu)
        assert runner.arena is not None
        snaps = []
        for s in range(STEPS):
            loss = runner.step_from_host(dev_batches[s][r])
            torch.cuda.current_stream().synchronize()
            snaps.append({"loss": loss, "m": eng.exp_avg.clone(), "oi": runner._offsets[0].clone(),
                          "ou": runner._offsets[1].clone(),
                          "est": [(c.A.clone(), c.Bv.clone(), c.step.clone()) for c in (ci, cu)]})
        return snaps, eng.layout

    runs = run_ranks(world, rank)
    monkeypatch.undo()
    for s in range(STEPS):
        gi = np.concatenate([b["target_id"].numpy() for b in batches[s]])
        gu = np.concatenate([b["user_idx"].numpy() for b in batches[s]])
        ref_oi, ref_ou = warm_i.step(gi), warm_u.step(gu)
        for r in range(G):
            sn = runs[r][0][s]
            for (A, Bv, st), ref in zip(sn["est"], (warm_i, warm_u)):
                assert int(st) == ref.t and torch.equal(A.cpu(), torch.from_numpy(ref.A)), (s, r)
                assert torch.equal(Bv.cpu(), torch.from_numpy(ref.Bv)), (s, r)
            assert torch.equal(sn["oi"], runs[0][0][s]["oi"]) and torch.equal(sn["ou"], runs[0][0][s]["ou"])
            assert (sn["oi"].cpu().double() - torch.from_numpy(ref_oi).double()).abs().max().item() <= 2.0 ** -20
            assert (sn["ou"].cpu().double() - torch.from_numpy(ref_ou).double()).abs().max().item() <= 2.0 ** -20
            assert sn["loss"] == runs[0][0][s]["loss"]
        if s == 0:
            oi, ou = runs[0][0][0]["oi"].cpu(), runs[0][0][0]["ou"].cpu()
            assert oi.unique().numel() > 4 and ou.unique().numel() > 2
            ol, og = corrected_dp_loss_and_grads(sd, batches[0], oi, ou, cfg.temperature, cfg.num_heads)
            loss = runs[0][0][0]["loss"]
            assert abs(loss - ol.item()) <= 5e-3, (loss, ol.item())
            m = torch.cat([runs[r][0][0]["m"] for r in range(G)])
            g = m / (1 - BETAS[0])
            lay = runs[0][1]
            for name, ref in og.items():
                o, shape = lay[name]
                got = g[o:o + ref.numel()].view(shape).cpu().double()
                err = (got - ref).norm().item()
                assert err <= 0.15 * ref.norm().item() + 5e-5 * ref.numel() ** 0.5, (name, err, ref.norm().item())
