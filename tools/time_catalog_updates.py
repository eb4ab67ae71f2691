#!/usr/bin/env python
"""Cost of live catalog updates at the c3 shape (10 k users x 1 M items, K = 100, seeded), CUDA events:

  * one retrieve_topk pass (exact_fallback=False) per setting of the retired bitmap: none, all-zero, 1 % and 10 % of
    the songs retired at random, and the 1 000 songs that appear most often in the users' top 100; ms per pass
    (median / min of 7 after 3 warm-up passes) and the users whose certificate failed (exact fallback);
  * CatalogIndex.upsert of 100 / 10 k / 100 k songs into the 1 M-row index against a full index_catalog_device of
    1 M songs, and CatalogIndex.retire of 100 / 10 k ids (host time around calls that end in a synchronise).

PARENT_TREE=<a checkout of the parent commit with its library built>: additionally times the no-bitmap pass of that
tree and of this one in separate processes, alternating three times (two builds cannot share one process).
Prints the device name and power limit with the numbers."""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.environ.get("TREE") or os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

USERS, ITEMS, K = int(os.environ.get("USERS", 10_000)), int(os.environ.get("ITEMS", 1_000_000)), 100


def _events(fn, warmup=3, reps=7):
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


def _host(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def _workload(dev):
    g = torch.Generator(device=dev).manual_seed(1)
    table = torch.nn.functional.normalize(torch.randn(ITEMS + 1, 256, device=dev, generator=g), dim=1)
    table[0] = 0
    t = torch.randint(1, ITEMS, (USERS,), device=dev, generator=g)
    users = torch.nn.functional.normalize(table[t] + 3.3 / 16 * torch.randn(USERS, 256, device=dev, generator=g), dim=1)
    return table, users


def plain_pass():
    """one process: the no-bitmap pass of the tree TREE names (default: this one)"""
    import mrm_b200  # noqa: F401
    from mrm_b200 import retrieval
    dev = torch.device("cuda", 0)
    table, users = _workload(dev)
    index = retrieval.CatalogIndex(table, device=dev)
    med, mn = _events(lambda: retrieval.retrieve_topk(users, index, K, exact_fallback=False))
    print(f"ms_per_pass median={med:.3f} min={mn:.3f}")


def main():
    import mrm_b200  # noqa: F401
    from mrm_b200 import retrieval, synthetic
    from mrm_b200.evaluate_metrics import index_catalog_device
    from mrm_b200.models import TwoTowerModel
    dev = torch.device("cuda", 0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print(f"device,power_limit,max_sm_clock={q}")
    print(f"users={USERS} items={ITEMS} K={K}")
    table, users = _workload(dev)

    def scoring(label, index):
        med, mn = _events(lambda: retrieval.retrieve_topk(users, index, K, exact_fallback=False))
        _, _, nfb = retrieval.retrieve_topk(users, index, K)
        print(f"retired={label:<28} ms_per_pass median={med:.3f} min={mn:.3f} fallback_users={nfb}")
        return med

    base = scoring("none (no bitmap)", retrieval.CatalogIndex(table, device=dev))
    zero = retrieval.CatalogIndex(table, device=dev)
    zero.retired_bits = torch.zeros((zero.num_rows + 255) // 256 * 8, device=dev, dtype=torch.int32)
    r0 = scoring("0 % (all-zero bitmap)", zero)
    del zero
    g = torch.Generator().manual_seed(2)
    ratios = {"0 %": r0 / base}
    for frac in (0.01, 0.10):
        ix = retrieval.CatalogIndex(table, device=dev)
        ix.retire(torch.randperm(ITEMS, generator=g)[:int(frac * ITEMS)] + 1)
        ratios[f"{frac:.0%}"] = scoring(f"{frac:.0%} random", ix) / base
        del ix
    ix = retrieval.CatalogIndex(table, device=dev)
    top, _, _ = retrieval.retrieve_topk(users, ix, K)
    cnt = torch.bincount(top.flatten().long(), minlength=ITEMS + 1)
    cnt[0] = 0
    ix.retire(torch.topk(cnt, 1000).indices)
    ratios["top-1000"] = scoring("1000 most frequent in top 100", ix) / base
    del ix
    print("ratio_to_no_bitmap " + " ".join(f"{k}={v:.3f}" for k, v in ratios.items()))

    # ---- update costs
    V = ITEMS + 1
    m = TwoTowerModel(vocab_size=V, tabular_input_dim=17, num_genders=3, num_countries=50, max_seq_len=50,
                      user_embedding_dim=256, item_embedding_dim=256, use_lora=True, seed=3)
    cfg = m.engine.cfg
    sd = synthetic.make_state_dict(cfg, seed=3)
    m.load_state_dict(sd)
    gd = torch.Generator(device=dev).manual_seed(4)
    feats = {k: torch.randn(ITEMS, cfg.modality_dim, device=dev, generator=gd)
             for k in ("target_audio", "target_image", "target_input_ids", "target_tabular")}
    ids = torch.arange(1, V, device=dev)
    out = (torch.zeros(V, 256, device=dev), torch.zeros(V, 256, device=dev, dtype=torch.bfloat16))
    full_med, full_min = _host(lambda: index_catalog_device(m, feats, ids, V, out=out))
    print(f"index_catalog_device {ITEMS} songs  ms median={full_med:.3f} min={full_min:.3f}")
    index = retrieval.CatalogIndex.from_device_tables(*out)
    for n in (100, 10_000, 100_000):
        sel = torch.randperm(ITEMS, generator=g)[:n]
        f = {k: v[sel.to(dev)] for k, v in feats.items()}
        u_ids = sel + 1
        med, mn = _host(lambda: index.upsert(m, f, u_ids))
        print(f"upsert {n:>7} songs  ms median={med:.3f} min={mn:.3f} fraction_of_rebuild={med / full_med:.4f}")
    for n in (100, 10_000):
        r_ids = torch.randperm(ITEMS, generator=g)[:n] + 1
        med, mn = _host(lambda: index.retire(r_ids))
        print(f"retire {n:>7} ids    ms median={med:.3f} min={mn:.3f}")

    parent = os.environ.get("PARENT_TREE")
    if parent:
        print("# no-bitmap pass, parent tree vs this tree, separate processes, alternating")
        for run in range(1, 4):
            for name, env in (("parent", {"TREE": os.path.abspath(parent)}), ("new   ", {})):
                e = {k: v for k, v in os.environ.items() if k not in ("TREE", "TT_B200_LIB")}
                e.update(env)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--plain"], env=e, capture_output=True,
                                   text=True)
                print(f"{name} run {run}: {r.stdout.strip()}{r.stderr.strip()[-300:] if r.returncode else ''}")


if __name__ == "__main__":
    plain_pass() if "--plain" in sys.argv else main()
