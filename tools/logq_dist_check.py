#!/usr/bin/env python
"""Real multi-GPU check of the streaming logQ estimator (run under torch.distributed.run on >= 2 GPUs):

  python -m torch.distributed.run --nproc_per_node=N tools/logq_dist_check.py [--nccl]

Every rank trains 20 steps with gathered negatives and streaming correction on both sides (items by target_id,
users by user_idx). Every rank updates its own estimator replica from the all-gathered ids, so after the run the
replicas must be bit-identical: rank 0 all-gathers A, Bv and the step counter of both sides and compares them.
--nccl uses the library exchanges (the target id rides in the packed embedding all-gather); the default uses the
symmetric-arena step (the target ids are one more block of its first all-gather)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
from mrm_b200 import synthetic  # noqa: E402
from mrm_b200.engine import TwoTowerEngine  # noqa: E402
from mrm_b200.train import LogQCorrection, TrainStepRunner  # noqa: E402


def main():
    comm = "nccl" if "--nccl" in sys.argv else "auto"
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = synthetic.TwoTowerConfig(vocab_size=3001, max_seq_len=50, dropout=0.1)
    sd = synthetic.make_state_dict(cfg, seed=7)
    B, steps, users = 32, 20, 200
    eng = TwoTowerEngine(cfg)
    eng.load_state_dict(sd)
    ci = LogQCorrection.streaming(cfg.vocab_size, num_slots=2 ** 12, alpha=0.05)
    cu = LogQCorrection.streaming(users, num_slots=2 ** 10, num_hashes=1, alpha=0.05)
    runner = TrainStepRunner(eng, B, cfg.max_seq_len, world_size=world, lr=1e-3, use_graph=True, comm=comm,
                             logq=ci, logq_users=cu)
    if rank == 0:
        print(f"world {world}, device {torch.cuda.get_device_name(local)}, "
              f"{'symmetric arena' if runner.arena is not None else 'NCCL'} exchanges:", runner.comm_description())
    losses = []
    for s in range(steps):
        b = synthetic.make_batch(cfg, B, seed=100 + 10 * s + rank, num_users=users)
        losses.append(runner.step_from_host({k: v.cuda() for k, v in b.items()}))
    torch.cuda.synchronize()
    ok = True
    for side, c in (("items", ci), ("users", cu)):
        for name in ("A", "Bv", "step"):
            mine = getattr(c, name).contiguous()
            got = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(got, mine)
            if rank == 0:
                same = all(torch.equal(g, got[0]) for g in got[1:])
                ok &= same
                print(f"{side} {name}: {'bit-identical on all ranks' if same else 'DIFFERS between ranks'}")
    if rank == 0:
        ok &= int(ci.step) == steps and int(cu.step) == steps
        print(f"estimator steps {int(ci.step)} / {int(cu.step)}; losses first {losses[0]:.4f} last {losses[-1]:.4f}")
        print("OK" if ok else "FAILED")
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
