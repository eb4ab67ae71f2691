#!/usr/bin/env python
"""Cost of excluding seen items inside the retrieval kernels, timed with CUDA events at the c3 shape
(10 k users x 1 M items, top-100; USERS / ITEMS override):

  * one retrieve_topk pass without exclusions, with m = 50 and m = 512 random ids per user, and with each user's
    512 best items excluded (the worst case: every excluded item would have been a candidate); ms per pass (the
    exclusion lists are built once per batch, timed separately) and users whose certificate failed (exact fallback);
  * single-user latency (B = 1, m = 50 history items): inference.recommend_batch (tower + in-kernel exclusion)
    against the user tower + inference.recommend_topk (exact top-(k + m), exclusion afterwards) on the same inputs,
    and the two retrieval paths alone on the same user embedding.

Prints the device name and power limit with the numbers."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402


def _time(fn, warmup=3, reps=7):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    import mrm_b200  # noqa: F401
    from mrm_b200 import inference, retrieval
    from mrm_b200.models import TwoTowerModel
    users_n, items_n, K = int(os.environ.get("USERS", 10_000)), int(os.environ.get("ITEMS", 1_000_000)), 100
    dev = torch.device("cuda", 0)
    print(f"device={torch.cuda.get_device_name(dev)} power_limit,max_sm_clock={_power_limit()}")
    g = torch.Generator(device=dev).manual_seed(1)
    table = torch.nn.functional.normalize(torch.randn(items_n + 1, 256, device=dev, generator=g), dim=1)
    table[0] = 0
    index = retrieval.CatalogIndex(table, device=dev)
    t = torch.randint(1, items_n, (users_n,), device=dev, generator=g)
    users = torch.nn.functional.normalize(table[t] + 3.3 / 16 * torch.randn(users_n, 256, device=dev, generator=g), dim=1)
    V = items_n + 1

    top = torch.empty(users_n, 512, device=dev, dtype=torch.long)
    for s in range(0, users_n, 1000):                     # fp32 scores of 1000 users at a time (4 GB)
        sc = users[s:s + 1000] @ table.t()
        sc[:, 0] = -float("inf")
        top[s:s + 1000] = sc.topk(512, dim=1).indices
    del sc
    cases = [("none", None),
             ("m=50 random", torch.randint(1, V, (users_n, 50), device=dev, generator=g)),
             ("m=512 random", torch.randint(1, V, (users_n, 512), device=dev, generator=g)),
             ("m=512 top-ranked", top)]
    print(f"users={users_n} items={items_n} K={K}")
    base = None
    for name, ids in cases:
        ex = None if ids is None else retrieval.Exclusions(ids, V)
        med, mn = _time(lambda: retrieval.retrieve_topk(users, index, K, exact_fallback=False, exclude=ex))
        base = med if base is None else base
        _, _, n_fb = retrieval.retrieve_topk(users, index, K, exclude=ex)
        _, _, n_fb10 = retrieval.retrieve_topk(users, index, 10, exclude=ex)
        build = "" if ids is None else f" exclusions_build_ms={_time(lambda: retrieval.Exclusions(ids, V))[0]:.3f}"
        print(f"exclude={name:18s} ms_per_pass median={med:.3f} min={mn:.3f} ratio_to_none={med / base:.3f} "
              f"fallback_users={n_fb} (at K=10: {n_fb10}){build}")

    # single user, m = 50: the same history feeds the tower (max_seq_len 50) and the exclusion of both paths
    model = TwoTowerModel(vocab_size=V, max_seq_len=50, seed=0, device=dev)
    hist = torch.randint(1, V, (1, 50), device=dev, generator=g)
    z = torch.zeros(1, dtype=torch.long, device=dev)

    def tower():
        model.eval()
        with torch.no_grad():
            return model.get_user_embedding(hist, (hist != 0).long(), z, z)

    u1 = tower()
    un = torch.nn.functional.normalize(u1, p=2, dim=1, eps=1e-8)
    a_i, _ = inference.recommend_batch(model, index, hist, k=10)
    b_i, _ = inference.recommend_topk(u1, index, hist, 10)
    same = torch.equal(a_i, b_i)
    rb = _time(lambda: inference.recommend_batch(model, index, hist, k=10), warmup=5, reps=21)
    rt = _time(lambda: inference.recommend_topk(tower(), index, hist, 10), warmup=5, reps=21)
    kb = _time(lambda: retrieval.retrieve_topk(un, index, 10, exclude=retrieval.Exclusions(hist, V)), warmup=5, reps=21)
    kt = _time(lambda: inference.recommend_topk(u1, index, hist, 10), warmup=5, reps=21)
    print(f"single user m=50 k=10 (same ids: {same}): recommend_batch ms median={rb[0]:.3f} min={rb[1]:.3f} | "
          f"tower + recommend_topk ms median={rt[0]:.3f} min={rt[1]:.3f}")
    print(f"single user retrieval only: Exclusions + retrieve_topk(exclude=) ms median={kb[0]:.3f} min={kb[1]:.3f} | "
          f"recommend_topk ms median={kt[0]:.3f} min={kt[1]:.3f}")


if __name__ == "__main__":
    main()
