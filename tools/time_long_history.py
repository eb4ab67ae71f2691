#!/usr/bin/env python
"""Long listening histories on the GPU, timed with CUDA events, one process:

  * attention forward / backward at dropout 0.1, H = 4: the tiled kernels at L = 1024, 2048, 4096 with
    B * L = 131 072 tokens (B = 128, 64, 32), alternated round by round with the per-item kernels at B = 256,
    L = 512. A 256 MB buffer is overwritten before every timed pass (L2 flushed). Microseconds (median of the
    rounds) and algorithmic causal TFLOP/s: 2 (forward) or 5 (backward) products of 64 * L(L+1)/2 multiply-adds per
    (sequence, head); recomputation does not count;
  * TrainStepRunner (CUDA-graph replay) at B = 64, L = 2048: ms per step and peak device memory;
  * recommend_batch at 10 000 users x 1 M items, L = 2048, K = 100: end-to-end ms, and the user tower alone.

Prints the device name and power limit with the numbers."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def _events(fn, flush=None):
    if flush is not None:
        flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def attention(rounds=15):
    from mrm_b200 import ops
    H, drop = 4, 0.1
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    cases = [(256, 512), (128, 1024), (64, 2048), (32, 4096)]
    bufs = {}
    g = torch.Generator(device="cuda").manual_seed(1)
    for B, L in cases:
        qkv = torch.randn(B * L, 3 * H * 64, device="cuda", generator=g).bfloat16()
        dctx = torch.randn(B * L, H * 64, device="cuda", generator=g).bfloat16()
        ctx = torch.empty(B * L, H * 64, device="cuda", dtype=torch.bfloat16)
        lse = torch.empty(B, H, L, device="cuda")
        dqkv = torch.empty(B * L, 3 * H * 64, device="cuda", dtype=torch.bfloat16)
        fwd = (lambda qkv=qkv, ctx=ctx, lse=lse, B=B, L=L:
               ops.attn_fwd(qkv, ctx, lse, B, L, H, drop_p=drop, drop_seed=5, drop_site=1))
        bwd = (lambda qkv=qkv, ctx=ctx, dctx=dctx, lse=lse, dqkv=dqkv, B=B, L=L:
               ops.attn_bwd(qkv, ctx, dctx, lse, dqkv, B, L, H, drop_p=drop, drop_seed=5, drop_site=1))
        for _ in range(3):
            fwd()
            bwd()
        bufs[(B, L)] = (fwd, bwd)
    torch.cuda.synchronize()
    ts = {(c, k): [] for c in cases for k in ("fwd", "bwd")}
    for _ in range(rounds):
        for c in cases:          # alternated: every round times every case once
            fwd, bwd = bufs[c]
            ts[(c, "fwd")].append(_events(fwd, flush))
            ts[(c, "bwd")].append(_events(bwd, flush))
    print("attention, dropout 0.1, H = 4, L2 flushed before each pass, median of %d alternated rounds" % rounds)
    print(f"{'kernels':9s} {'B':>4s} {'L':>5s} {'fwd us':>9s} {'fwd TFLOP/s':>12s} {'bwd us':>9s} {'bwd TFLOP/s':>12s}")
    for B, L in cases:
        macs = 64 * L * (L + 1) / 2 * B * H
        row = []
        for k, prods in (("fwd", 2), ("bwd", 5)):
            t = sorted(ts[((B, L), k)])[rounds // 2]
            row += [t * 1e3, 2 * prods * macs / (t * 1e-3) / 1e12]
        kind = "per-item" if L <= 512 else "tiled"
        print(f"{kind:9s} {B:4d} {L:5d} {row[0]:9.1f} {row[1]:12.1f} {row[2]:9.1f} {row[3]:12.1f}")
    del bufs, flush
    torch.cuda.empty_cache()


def train_step(B=64, L=2048, steps=10):
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import TrainStepRunner
    cfg = synthetic.TwoTowerConfig(vocab_size=100_001, max_seq_len=L, dropout=0.1)
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(synthetic.make_state_dict(cfg, seed=0))
    runner = TrainStepRunner(eng, B, L, lr=1e-4, use_graph=True)
    runner.load_batch({k: v.cuda() for k, v in synthetic.make_batch(cfg, B, seed=1, full_length=True).items()})
    for _ in range(3):
        runner.step_resident()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t = _events(lambda: [runner.step_resident() for _ in range(steps)])
    print(f"train step (graph replay) B={B} L={L} full-length histories, dropout 0.1: {t / steps:.3f} ms/step, "
          f"peak device memory {torch.cuda.max_memory_allocated() / 2**30:.2f} GiB (torch allocator)")
    del runner, eng
    torch.cuda.empty_cache()


def recommend(users_n=10_000, items_n=1_000_000, L=2048, K=100):
    from mrm_b200 import inference, retrieval
    from mrm_b200.models import TwoTowerModel
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(2)
    table = torch.nn.functional.normalize(torch.randn(items_n + 1, 256, device=dev, generator=g), dim=1)
    table[0] = 0
    index = retrieval.CatalogIndex(table, device=dev)
    model = TwoTowerModel(vocab_size=items_n + 1, max_seq_len=L, seed=0, device=dev)
    ids = torch.randint(1, items_n + 1, (users_n, L), device=dev, generator=g)
    lens = torch.randint(1, L + 1, (users_n,), device=dev, generator=g)
    ids[torch.arange(L, device=dev)[None, :] >= lens[:, None]] = 0
    mask = (ids != 0).long()
    chunk = min(inference._TOWER_CHUNK, inference._TOWER_TOKENS // L)

    def tower():
        model.eval()
        with torch.no_grad():
            for s in range(0, users_n, chunk):
                model.get_user_embedding(ids[s:s + chunk], mask[s:s + chunk])
        model.train()

    run = lambda: inference.recommend_batch(model, index, ids, k=K)   # noqa: E731
    for _ in range(2):
        run()
        tower()
    torch.cuda.synchronize()
    e2e = sorted(_events(run) for _ in range(5))[2]
    tw = sorted(_events(tower) for _ in range(5))[2]
    print(f"recommend_batch {users_n} users x {items_n} items, L={L} (random lengths), K={K}: {e2e:.1f} ms end to end, "
          f"user tower alone {tw:.1f} ms ({chunk} users per tower call), median of 5")


def main():
    import mrm_b200  # noqa: F401
    print(f"device={torch.cuda.get_device_name(0)} power_limit,max_sm_clock={_power_limit()}")
    attention()
    train_step()
    recommend()


if __name__ == "__main__":
    main()
