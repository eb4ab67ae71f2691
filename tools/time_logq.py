#!/usr/bin/env python
"""Cost of the logQ correction on the graph-replayed c2 training step (batch 256, seq_len 200, 100 000 items,
dropout 0.1, AdamW), one GPU, CUDA events:

  * no correction (the default path);
  * static item-side correction (LogQCorrection.from_counts: one table-gather launch beside the towers);
  * streaming correction on both sides (items and users: two tt_logq_stream_update launches beside the towers).

The three runners are timed in rounds that alternate between them; each number is the median over rounds of the
mean step time of a window of 50 replayed steps. Prints the device name and power limit with the numbers, to stdout
(nothing is written)."""
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from time_long_history import _events, _power_limit  # noqa: E402

B, L, V, USERS = 256, 200, 100_001, 1_000_000


def main(rounds: int = 7, window: int = 50):
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import LogQCorrection, TrainStepRunner
    assert torch.cuda.is_available(), "time_logq.py measures on a CUDA device"
    print(f"device={torch.cuda.get_device_name(0)} power_limit,max_sm_clock={_power_limit()}")
    cfg = synthetic.TwoTowerConfig(vocab_size=V, max_seq_len=L, dropout=0.1)
    sd = synthetic.make_state_dict(cfg, seed=0)
    batch = {k: v.cuda() for k, v in synthetic.make_batch(cfg, B, seed=500, full_length=True,
                                                         num_users=USERS).items()}
    counts = np.random.default_rng(0).zipf(1.3, size=V).clip(max=10 ** 7).astype(np.float64)
    variants = {
        "none": {},
        "static items": {"logq": LogQCorrection.from_counts(counts)},
        "streaming items + users": {"logq": LogQCorrection.streaming(V),
                                    "logq_users": LogQCorrection.streaming(USERS)},
    }
    runners = {}
    for name, kw in variants.items():
        eng = TwoTowerEngine(cfg)
        eng.load_state_dict(sd)
        r = TrainStepRunner(eng, B, L, **kw)
        r.load_batch(batch)
        for _ in range(5):                     # eager warm-up, capture, replays
            r.step_resident()
        torch.cuda.synchronize()
        runners[name] = r
        print(f"{name}: {r.kernels_per_step} kernels per step")
    times = {name: [] for name in runners}
    for _ in range(rounds):
        for name, r in runners.items():
            def run(r=r):
                for _ in range(window):
                    r.step_resident()
            times[name].append(_events(run) / window)
    base = statistics.median(times["none"])
    for name, t in times.items():
        med = statistics.median(t)
        print(f"{name:>24}: {med * 1e3:8.1f} us/step (min {min(t) * 1e3:.1f}, max {max(t) * 1e3:.1f}; "
              f"{100 * (med / base - 1):+.2f} % against no correction)")


if __name__ == "__main__":
    main()
