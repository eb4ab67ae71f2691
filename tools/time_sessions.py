#!/usr/bin/env python
"""User sessions on the GPU, timed with CUDA events, one process, at L = 200 and L = 2048:

  * 10 000 sessions opened at random lengths below L - 8 (so the timed appends stay on the incremental path);
  * one `append` for all users, against the user tower on the same windows (get_user_embedding in the chunks
    recommend_batch uses);
  * `append` + `recommend` at K = 100 on 1 M items, against `recommend_batch` on the same windows;
  * single-user `append` latency (host wall clock around a call that ends in a device synchronise);
  * tt_session_attn alone for the 10 000 rows of one layer: microseconds and achieved bytes/s, bytes = the K and V
    rows it must read (positions 0..pos of every (row, head), 128 B each) plus the rows it writes. The caches (4 GB and
    40 GB) exceed the 126 MB L2, so the reads come from HBM.

Medians of 5 (11 for the single user). Prints the device name and power limit with the numbers."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from time_long_history import _events, _power_limit  # noqa: E402


def _median(xs):
    return sorted(xs)[len(xs) // 2]


def run(L, model, index, users_n=10_000, K=100):
    from mrm_b200 import inference, ops
    from mrm_b200.sessions import UserSessions
    dev = model.engine.device
    V = model.engine.cfg.vocab_size
    g = torch.Generator().manual_seed(L)
    lens = torch.randint(1, L - 8, (users_n,), generator=g)
    ids = torch.randint(1, V, (users_n, L), generator=g)
    ids[torch.arange(L)[None, :] >= lens[:, None]] = 0
    sess = UserSessions(model, capacity=users_n)
    slots = np.arange(users_n)
    sess.open(slots, ids)
    torch.cuda.synchronize()
    chunk = min(inference._TOWER_CHUNK, inference._TOWER_TOKENS // L)

    def tower():
        w = sess.window
        model.eval()
        with torch.no_grad():
            for s in range(0, users_n, chunk):
                model.get_user_embedding(w[s:s + chunk], (w[s:s + chunk] != 0).long())
        model.train()

    new = [torch.randint(1, V, (users_n,), generator=g) for _ in range(8)]
    step = iter(range(8))
    append = lambda: sess.append(slots, new[next(step)])                       # noqa: E731
    append()                                                                   # warm-up (workspace, first launches)
    tower()
    t_app = _median([_events(append) for _ in range(3)])
    t_tow = _median([_events(tower) for _ in range(3)])
    rec = lambda: sess.recommend(slots, index, k=K)                            # noqa: E731
    batch = lambda: inference.recommend_batch(model, index, sess.window, k=K)  # noqa: E731
    rec()
    batch()
    t_rec = _median([_events(rec) for _ in range(5)])
    t_batch = _median([_events(batch) for _ in range(5)])
    # the attention kernel alone on the last append's rows (re-writes the same K/V rows: idempotent)
    ws = sess._append_ws(users_n)
    d_slot = torch.from_numpy(slots.astype(np.int32)).to(dev)
    d_pos = torch.from_numpy((sess.lengths - 1).astype(np.int32)).to(dev)
    attn = lambda: ops.session_attn(ws["qkv_0"], sess.k_cache[0], sess.v_cache[0], d_slot, d_pos, ws["ctx_0"])  # noqa
    attn()
    t_attn = _median([_events(attn) for _ in range(5)])
    H = model.engine.cfg.num_heads
    nbytes = float(sess.lengths.sum()) * H * 128 * 2 + users_n * (H * 128 * 2 + 3 * 512 + 512)
    # one user
    one = np.array([int(sess.lengths.argmin())])       # stays below L: the incremental path
    item = torch.tensor([5])
    sess.append(one, item)
    torch.cuda.synchronize()
    wall = []
    for _ in range(11):
        t0 = time.perf_counter()
        sess.append(one, item)
        torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3)
    print(f"L={L}: {users_n} sessions, mean length {sess.lengths.mean():.0f}")
    print(f"  append, all users:            {t_app:8.2f} ms   user tower on the same windows: {t_tow:8.2f} ms "
          f"({t_tow / t_app:.1f}x)")
    print(f"  append + recommend K={K}:     {t_app + t_rec:8.2f} ms   (recommend alone {t_rec:.2f} ms)   "
          f"recommend_batch: {t_batch:8.2f} ms ({t_batch / (t_app + t_rec):.1f}x)")
    print(f"  tt_session_attn, one layer:   {t_attn * 1e3:8.1f} us   {nbytes / 1e9:.2f} GB -> "
          f"{nbytes / (t_attn * 1e-3) / 1e12:.2f} TB/s ({nbytes / (t_attn * 1e-3) / 7.7e12 * 100:.0f} % of the "
          f"7.7 TB/s data-sheet HBM bandwidth)")
    print(f"  single-user append:           {_median(wall):8.3f} ms wall clock incl. synchronise (median of 11)")
    del sess
    torch.cuda.empty_cache()


def main():
    from mrm_b200 import retrieval
    from mrm_b200.models import TwoTowerModel
    print(f"device={torch.cuda.get_device_name(0)} power_limit,max_sm_clock={_power_limit()}")
    dev = torch.device("cuda", 0)
    items_n = 1_000_000
    g = torch.Generator(device=dev).manual_seed(2)
    table = torch.nn.functional.normalize(torch.randn(items_n + 1, 256, device=dev, generator=g), dim=1)
    table[0] = 0
    index = retrieval.CatalogIndex(table, device=dev)
    for L in (200, 2048):
        model = TwoTowerModel(vocab_size=items_n + 1, max_seq_len=L, seed=0, device=dev)
        run(L, model, index)
        del model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
