"""bench.py --dump-outputs: dump_train_outputs re-runs the captured train step from the seeded start, so what it
writes does not depend on how many steps ran before it, and equals the first step of a fresh engine."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

B, L, V = 32, 50, 20_001


def _runner(cfg, sd, batch):
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import TrainStepRunner
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(sd)
    runner = TrainStepRunner(eng, B, L)
    runner.load_batch(batch)
    return eng, runner


def test_dump_train_outputs_is_the_seeded_step(tmp_path):
    import bench
    from mrm_b200 import synthetic
    cfg = synthetic.TwoTowerConfig(vocab_size=V, max_seq_len=L, dropout=0.1)
    sd = synthetic.make_state_dict(cfg, seed=0)
    batch = synthetic.make_batch(cfg, B, seed=1, full_length=True)
    eng, runner = _runner(cfg, sd, batch)
    for steps, d in ((3, "a"), (6, "b")):           # eager warm-up, graph capture, replays
        for _ in range(steps):
            runner.step_resident()
        bench.dump_train_outputs(str(tmp_path / d), runner, eng, sd, batch)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= bench.DUMP_MAX_BYTES

    def load(d, name):
        a = np.load(tmp_path / d / (name + ".npy"))
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        return a

    for f in names:
        a, b = load("a", f[:-4]), load("b", f[:-4])
        if f.startswith("grad."):        # fp32 atomics: the summation order varies
            assert np.abs(a - b).max() <= 1e-5 * np.abs(a).max() + 1e-12, f
        else:
            assert np.array_equal(a, b), f
    # forward + backward of a fresh engine from the same state, batch and dropout seed: the same forward outputs bit
    # for bit, the same gradients up to the summation order of their fp32 atomics
    from mrm_b200.engine import TwoTowerEngine
    ref = TwoTowerEngine(cfg)
    ref.load_state_dict(sd)
    loss, logits, u, i = ref.forward({k: v.cuda() for k, v in batch.items()}, training=True)
    ref.backward()
    torch.cuda.synchronize()
    assert load("a", "loss").tolist() == [loss.item()]
    assert load("a", "logits").shape == (B, B) and np.array_equal(load("a", "logits"), logits.cpu().numpy())
    assert np.array_equal(load("a", "user_emb"), u.cpu().numpy())
    assert np.array_equal(load("a", "item_emb"), i.cpu().numpy())
    key = "user_tower.item_embedding.weight"
    rows = load("a", f"grad.{key}.row_ids")
    assert rows.shape == (bench.DUMP_TABLE_ROWS,)
    for name, g in ref.g.items():
        if name == key:
            g = g[torch.from_numpy(rows).long().cuda()]
        g = g.cpu().double().numpy()
        assert np.abs(load("a", f"grad.{name}") - g).max() <= 1e-5 * np.abs(g).max() + 1e-12, name
    assert len(names) == 4 + len(ref.g) + 1
