#!/usr/bin/env python
"""Diversified recommendations on the GPU, timed with CUDA events, one process: 10 000 users x 1 M synthetic unit-norm
items, 50 excluded ids per user, diversity 0.3, (k, P) in {(10, 100), (100, 256)}:

  * tt_mmr_select alone over the users' pools (rows from the index's fp32 table): the median of 5 windows of 10
    launches. Algorithmic work: U * P rows of 1 KB read (the pools' rows, 10 000 x 256 KB = 2.6 GB at P = 256, far
    beyond the 126 MB L2, so they come from HBM; at P = 100, 1 GB) and at most U * (k - 1) * P * 256 fp64
    multiply-adds;
  * `recommend_embeddings` with and without diversity, alternated in the same run (medians of 5 each);
  * single-user latency of `recommend_embeddings` with diversity (host wall clock around a call that ends in a device
    synchronise, median of 11).

Prints the device name and power limit with the numbers, to stdout (nothing is written). With two or more GPUs, run
under `torch.distributed.run --nproc_per_node=2 tools/time_diversity.py --check-sharded` to check that the sharded
result equals the single-GPU result bit for bit."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch  # noqa: E402

from time_long_history import _events, _power_limit  # noqa: E402

USERS, ITEMS, DIVERSITY = 10_000, 1_000_000, 0.3
#: the measured HBM peak DESIGN.md §4 quotes every kernel's bandwidth against
HBM_PEAK = 6.55e12


def _median(xs):
    return sorted(xs)[len(xs) // 2]


def _setup(dev):
    g = torch.Generator(device=dev).manual_seed(2)
    table = torch.nn.functional.normalize(torch.randn(ITEMS + 1, 256, device=dev, generator=g), dim=1)
    table[0] = 0
    users = torch.nn.functional.normalize(table[1:USERS + 1] + 0.7 * torch.randn(USERS, 256, device=dev, generator=g),
                                          dim=1)
    ex = torch.randint(1, ITEMS + 1, (USERS, 50), device=dev, generator=g)
    return table, users, ex


def timings():
    from mrm_b200 import inference, ops, retrieval
    print(f"device={torch.cuda.get_device_name(0)} power_limit,max_sm_clock={_power_limit()}")
    dev = torch.device("cuda", 0)
    table, users, ex = _setup(dev)
    index = retrieval.CatalogIndex(table, device=dev)
    exclude = retrieval.Exclusions(ex, index.vocab_size)
    lam = 1.0 - DIVERSITY
    for k, P in ((10, 100), (100, 256)):
        pi, ps, _ = retrieval.retrieve_topk(users, index, P, exclude=exclude)
        sel = lambda: ops.mmr_select(pi, ps, k, lam, 1.0 - lam, ops.MMR_ROWS_TABLE, index.table, 0,   # noqa: E731
                                     index.num_rows)
        sel()

        def ten():
            for _ in range(10):
                sel()
        t_k = _median([_events(ten) for _ in range(5)]) / 10
        plain = lambda: inference.recommend_embeddings(users, index, ex, k)                          # noqa: E731
        div = lambda: inference.recommend_embeddings(users, index, ex, k, diversity=DIVERSITY, pool=P)  # noqa: E731
        plain()
        div()
        tp, td = [], []
        for _ in range(5):
            tp.append(_events(plain))
            td.append(_events(div))
        one_u, one_x = users[:1].contiguous(), ex[:1].contiguous()
        inference.recommend_embeddings(one_u, index, one_x, k, diversity=DIVERSITY, pool=P)
        torch.cuda.synchronize()
        wall = []
        for _ in range(11):
            t0 = time.perf_counter()
            inference.recommend_embeddings(one_u, index, one_x, k, diversity=DIVERSITY, pool=P)
            torch.cuda.synchronize()
            wall.append((time.perf_counter() - t0) * 1e3)
        nbytes = USERS * P * 1024.0
        fma = USERS * (k - 1) * P * 256.0
        s = t_k * 1e-3
        print(f"k={k} P={P}: {USERS} users x {ITEMS} items, diversity {DIVERSITY}")
        print(f"  tt_mmr_select alone:          {t_k * 1e3:9.1f} us   rows read {nbytes / 1e9:.2f} GB -> "
              f"{nbytes / s / 1e12:.2f} TB/s ({nbytes / s / HBM_PEAK * 100:.0f} % of the measured {HBM_PEAK / 1e12:.2f} "
              f"TB/s HBM peak); <= {fma / 1e9:.2f} G fp64 multiply-adds -> <= {2 * fma / s / 1e12:.2f} TFLOP/s fp64")
        print(f"  recommend_embeddings:         {_median(tp):9.3f} ms plain top {k}   {_median(td):9.3f} ms diversified "
              f"(top {P} + MMR), alternated, medians of 5")
        print(f"  single user, diversified:     {_median(wall):9.3f} ms wall clock incl. synchronise (median of 11)")


def check_sharded():
    """Under torch.distributed.run: every rank holds one contiguous slice of the catalog; the diversified result of
    the sharded index must equal the single-GPU one bit for bit (and be identical on every rank)."""
    import torch.distributed as dist
    from mrm_b200 import inference, retrieval
    dist.init_process_group("nccl")
    rank, ws = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    table, users, ex = _setup(dev)
    V = table.shape[0]
    cuts = [V * r // ws for r in range(ws + 1)]
    shard = retrieval.CatalogIndex.from_shard(table[cuts[rank]:cuts[rank + 1]], cuts[rank], V, device=dev)
    full = retrieval.CatalogIndex(table, device=dev)
    for k, P in ((10, 100), (100, 256)):
        si, ss = inference.recommend_embeddings(users, shard, ex, k, diversity=DIVERSITY, pool=P)
        fi, fs = inference.recommend_embeddings(users, full, ex, k, diversity=DIVERSITY, pool=P)
        same = torch.equal(si, fi) and torch.equal(ss, fs)
        flag = torch.tensor([0 if same else 1], device=dev)
        dist.all_reduce(flag)
        if rank == 0:
            print(f"sharded over {ws} GPUs, k={k} P={P}: "
                  f"{'bit-identical to' if flag.item() == 0 else 'DIFFERENT from'} the single-GPU result")
    dist.destroy_process_group()


if __name__ == "__main__":
    if "--check-sharded" in sys.argv:
        check_sharded()
    else:
        timings()
