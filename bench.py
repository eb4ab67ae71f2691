#!/usr/bin/env python
"""Benchmark of the two-tower hot path on B200 (one JSON line on rank 0).

Headline metric (BASELINE.json configs[1]): two-tower train samples/sec — one step = forward +
backward + InfoNCE + dense AdamW on batch 256/GPU, seq len 200, 100k-item ID table, dropout 0.1,
all histories full length, synthetic precomputed modality embeddings.
  value : device-resident inputs, the whole step replayed as one CUDA graph, CUDA-event timing.
  e2e   : through the public train_one_epoch-style call with HOST (pinned) batches: H2D of every
          step's batch and D2H of its loss inside the timed region.
  roofline     : the tcgen05 GEMM (dominant kernel): algorithmic FLOPs / event-timed duration of
                 the step's own GEMM launches, against MEASURED_PEAKS.json bf16 sustained.
  cpu_baseline : the reference's OWN train_one_epoch / calculate_metrics_global (baseline/_ref) on this box's host
                 cores, bounded sample, rank 0 at N=1.
  parity       : loss / embeddings of the bench batch (dropout 0) against the oracle; top-100 of 512 bench users
                 against an fp64 canonical sort; sharded == single-GPU retrieval result.
  retrieval    : evaluate_metrics workload (BASELINE.json configs[2]): 10k users x 1M items,
                 top-100 + Recall/NDCG, ONE seeded catalog sharded over the N GPUs.
  indexing     : catalog indexing of those 1M items (item list split over the N GPUs), GB/s vs 3 KB/item.
  c4, c5       : (8 GPUs) BASELINE.json configs[3] and [4]: global batch 4096 with all-gathered negatives; 10M-item
                 row-sharded ID table at seq len 512 (train step) and 10k x 10M retrieval.
`--impl reference` runs the UNMODIFIED reference (baseline/_ref, installed by __graft_entry__.build()) for the same
metric and config on the host cores; rank 0 only.
`--dump-outputs DIR` (one GPU) runs the timed c2 step once more from the seeded start and writes what it computed as
DIR/<name>.npy (dump_train_outputs): the same every run, so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

C2 = dict(batch=256, seq_len=200, vocab=100_001)      # BASELINE.json configs[1]
C3 = dict(users=10_000, items=1_000_000, k=100, hist_len=50)  # BASELINE.json configs[2]
CPU_SAMPLE_BATCH = 64
C2_WORKLOAD = ("c2: two-tower train step (fwd+bwd+InfoNCE+dense AdamW), batch 256/GPU, seq_len 200 (all positions valid), "
               "100k-item ID table, dropout 0.1")
C4 = dict(batch=512, seq_len=200, vocab=100_001)                 # BASELINE.json configs[3]: 8 x 512 = 4096 global
C5 = dict(batch=512, seq_len=512, vocab=10_000_001, users=10_000, k=100)   # BASELINE.json configs[4]
DUMP_TABLE_ROWS = 16_384      # --dump-outputs: seeded row sample of the ID table (all 100k rows are 102 MB)
DUMP_MAX_BYTES = 64 << 20


def flops_per_sample_fwd(L, B_neg, D=256, FF=1024, NL=2):
    """SURVEY.md §8d algorithmic work per sample (all positions valid)."""
    return (L * NL * (2 * D * 3 * D + 2 * D * D + 4 * D * FF + 4 * ((L + 1) / 2) * D)
            + (2 * 304 * 256 + 2 * 256 * 256) + (2 * 512 * 512 + 2 * 512 * 256) + 2 * B_neg * D)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.samples, self.stop_flag = gpu_index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                parts = [x.strip() for x in out.stdout.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.01)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(s[0])) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for j, n in enumerate(names) if any(s[2 + j].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.samples[0][1])), "reasons": reasons,
                "samples": len(sm)}


def pin(batch):
    return {k: v.pin_memory() for k, v in batch.items()}


# ------------------------------------------------------------------------------------------
# CPU arm: the UNMODIFIED reference (baseline/_ref, installed by __graft_entry__.build()) on the host cores;
# the oracle port only when that install is missing
# ------------------------------------------------------------------------------------------
def _c2_cfg(dropout):
    from mrm_b200 import synthetic
    return synthetic.TwoTowerConfig(vocab_size=C2["vocab"], max_seq_len=C2["seq_len"], dropout=dropout)


def reference_train_samples_per_s(steps, warmup, batch_size):
    """The reference's own train_one_epoch (src/train.py:41-76: TwoTowerModel.forward, backward, torch.optim.AdamW
    lr 1e-4 as train.py:302, dropout 0.1 as shipped) on `steps` c2 batches, on the CPU. autocast / GradScaler
    disable themselves without CUDA, so this is the reference's fp32 path (SURVEY.md App. A).
    Returns (samples/s, ms/step, kind, detail)."""
    from mrm_b200 import synthetic
    from oracle import ref_loader
    if ref_loader.reference_location() is None:
        sps, ms = port_train_samples_per_s(steps, warmup, min(batch_size, CPU_SAMPLE_BATCH))
        return sps, ms, "port", f"oracle port (baseline/_ref absent), batch {min(batch_size, CPU_SAMPLE_BATCH)}"
    import logging
    import warnings
    warnings.filterwarnings("ignore")
    two_tower, _, train, where = ref_loader.import_reference("installed")
    logging.disable(logging.WARNING)
    cfg = _c2_cfg(0.1)
    model = ref_loader.build_reference_model(two_tower, cfg, synthetic.make_state_dict(cfg, seed=0), torch.float32,
                                             dropout=0.1)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4)
    dev = torch.device("cpu")

    def batches(n, seed0):
        return [synthetic.make_batch(cfg, batch_size, seed=seed0 + i, full_length=True, num_users=1_000_000)
                for i in range(n)]

    def run(loader):
        if train is not None:
            train.train_one_epoch(model, loader, opt, dev, 0, is_main_process=False)
            return
        model.train()                              # src.train not importable (tqdm/joblib): same body by hand
        for b in loader:
            opt.zero_grad(set_to_none=True)
            loss, _, _, _ = model(b)
            loss.backward()
            opt.step()
            loss.item()

    if warmup > 0:
        run(batches(warmup, 100))
    timed = batches(steps, 200)
    t0 = time.perf_counter()
    run(timed)
    dt = time.perf_counter() - t0
    logging.disable(logging.NOTSET)
    api = "train_one_epoch" if train is not None else "TwoTowerModel.forward/backward + AdamW loop"
    return batch_size * steps / dt, dt / steps * 1e3, "reference", f"reference {api} from {where}"


def port_train_samples_per_s(steps, warmup, batch_size):
    from mrm_b200 import synthetic
    from oracle import two_tower_oracle as oracle
    cfg = _c2_cfg(0.0)
    sd = synthetic.make_state_dict(cfg, seed=0)
    batch = synthetic.make_batch(cfg, batch_size, seed=1, full_length=True, num_users=1_000_000)
    p = {k: v.clone() for k, v in sd.items()}
    m = {k: torch.zeros_like(v) for k, v in p.items() if v.is_floating_point()}
    v2 = {k: torch.zeros_like(v) for k, v in p.items() if v.is_floating_point()}
    times = []
    for t in range(1, warmup + steps + 1):
        t0 = time.perf_counter()
        _, _, _, _, grads, _ = oracle.loss_and_grads(p, batch, cfg.temperature, cfg.num_heads)
        for k, g in grads.items():
            p[k], m[k], v2[k] = oracle.adamw_step(p[k], g, m[k], v2[k], t)
        dt = time.perf_counter() - t0
        if t > warmup:
            times.append(dt)
    total = sum(times)
    return batch_size * len(times) / total, total / len(times) * 1e3


class _PrecomputedUsers(torch.nn.Module):
    """calculate_metrics_global only calls .eval() and .get_user_embedding(): feeding it precomputed user embeddings
    times the scoring / top-K / metric part (the c3 metric) of the reference's own function."""

    def __init__(self, users):
        super().__init__()
        self.users, self.pos = users, 0

    def get_user_embedding(self, history_ids, history_mask=None, user_gender=None, user_country=None):
        n = history_ids.shape[0]
        u = self.users[self.pos:self.pos + n]
        self.pos += n
        return u


def reference_retrieval_users_per_s(num_users=128):
    """The reference's calculate_metrics_global (src/evaluate_metrics.py:106-192; val batch 64, :203) on
    `num_users` users against the 1M-item table, k_list [10, 20, 50, 100], on the CPU."""
    from mrm_b200 import synthetic
    from oracle import ref_loader
    table = synthetic.make_catalog(C3["items"], 256, seed=2)
    users, targets = synthetic.make_queries(table, num_users, seed=3)
    kl = [10, 20, 50, 100]
    if ref_loader.reference_location() is None:
        from oracle import two_tower_oracle as oracle
        t0 = time.perf_counter()
        oracle.calculate_metrics_global(users, table, targets, kl)
        return num_users / (time.perf_counter() - t0), "port"
    import logging
    _, evalm, _, _ = ref_loader.import_reference("installed")
    logging.disable(logging.WARNING)
    loader = []
    for s0 in range(0, num_users, 64):
        n = min(64, num_users - s0)
        z = torch.zeros(n, dtype=torch.long)
        loader.append({"history_ids": torch.ones((n, 4), dtype=torch.long), "history_mask": torch.ones((n, 4), dtype=torch.long),
                       "user_gender": z, "user_country": z, "target_id": targets[s0:s0 + n]})
    t0 = time.perf_counter()
    evalm.calculate_metrics_global(_PrecomputedUsers(users), loader, table, torch.device("cpu"), k_list=kl)
    dt = time.perf_counter() - t0
    logging.disable(logging.NOTSET)
    return num_users / dt, "reference"


def run_reference(args, rank, world):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    B = C2["batch"]
    sps, ms, kind, detail = reference_train_samples_per_s(args.steps, args.warmup, B)
    sample = (f"{detail}: fp32 torch CPU, fwd+bwd+InfoNCE+AdamW, {args.steps} timed steps of batch {B} "
              f"(L={C2['seq_len']}, V={C2['vocab']}, dropout 0.1) after {args.warmup} warm-up steps")
    line = {
        "impl": "reference", "metric": "two-tower train samples/sec", "value": sps, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": C2_WORKLOAD, "global_batch": B, "seq_len": C2["seq_len"], "vocab_size": C2["vocab"],
                   "reference_step_batch": B},
        "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": sample},
        "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def time_gemm_roofline(eng, static_batch, peaks, iters=5):
    """Event-time every tcgen05 GEMM launch of the training step (the step's own operands, fused epilogues
    and launch arguments, on the launching stream). The step is issued eagerly on ONE stream behind a
    ~15 ms device-side sleep, so the whole launch sequence is already queued when the GPU starts it and
    the events bracket kernel execution, not host launch latency. Per launch the roofline time is
    max(flops / bf16 peak, algorithmic bytes / HBM peak); d=256 makes the encoder GEMMs HBM-bound.
    Returns (all launches, the encoder-sized launches (>= 4096 rows or a >= 4096-deep reduction), n)."""
    peak_f = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")) * 1e12
    peak_b = peaks["hbm_gbs"] * 1e9
    zero = dict(flops=0.0, bytes=0.0, secs=0.0, roof_secs=0.0, flop_secs=0.0, byte_secs=0.0, n=0.0)
    acc, big = dict(zero), dict(zero)
    n_launch = 0
    eng.serialize = True
    for it in range(iters + 1):
        eng.gemm_log = []
        torch.cuda._sleep(30_000_000)
        eng.forward(static_batch, training=True)
        eng.backward()
        torch.cuda.synchronize()
        if it > 0:       # first pass warms the eager path
            for e0, e1, f, b, (M, N, K) in eng.gemm_log:
                for d in ((acc, big) if max(M, K) >= 4096 else (acc,)):
                    d["flops"] += f
                    d["bytes"] += b
                    d["secs"] += e0.elapsed_time(e1) * 1e-3
                    d["roof_secs"] += max(f / peak_f, b / peak_b)
                    d["flop_secs"] += f / peak_f
                    d["byte_secs"] += b / peak_b
                    d["n"] += 1
        n_launch = len(eng.gemm_log)
        eng.gemm_log = None
        eng.grad.zero_()
    eng.serialize = False
    return {k: v / iters for k, v in acc.items()}, {k: v / iters for k, v in big.items()}, n_launch


def run_ours(args, rank, world, local_rank):
    import mrm_b200
    from mrm_b200 import _lib, retrieval, synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import TrainStepRunner, make_dp_engine

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    peaks, peak_src = load_peaks()
    B, L, V = C2["batch"], C2["seq_len"], C2["vocab"]
    cfg = synthetic.TwoTowerConfig(vocab_size=V, max_seq_len=L, dropout=0.1)
    eng, table = make_dp_engine(cfg, world, dev)
    eng.load_state_dict(synthetic.make_state_dict(cfg, seed=0))
    runner = TrainStepRunner(eng, B, L, world_size=world, sharded_table=table)
    host_batches = [pin(synthetic.make_batch(cfg, B, seed=100 + rank * 17 + i, full_length=True,
                                             num_users=1_000_000)) for i in range(4)]
    h2d_bytes = sum(v.numel() * v.element_size() for k, v in host_batches[0].items() if k in runner.static)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (includes graph capture) -------------------------------------------------
    sampler = ClockSampler(local_rank)     # samples clocks / throttle reasons from here to the end of the e2e loop
    sampler.start()
    runner.load_batch(host_batches[0])
    for _ in range(max(args.warmup, 3)):
        runner.step_resident()
    torch.cuda.synchronize()

    # ---- value: device-resident inputs ----------------------------------------------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = _lib.launch_count
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    e0.record()
    for i in range(args.steps):
        runner.step_resident()
        marks[i].record()
    e1.record()
    barrier()
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = ms_total.item() / args.steps
    per_step = sorted([e0.elapsed_time(marks[0])] + [marks[i - 1].elapsed_time(marks[i]) for i in range(1, args.steps)])
    pct = {f"p{q}": per_step[min(len(per_step) - 1, int(q / 100.0 * len(per_step)))] for q in (10, 50, 90)}
    value = world * B * 1e3 / ms_step
    launches = runner.kernels_per_step * args.steps + (_lib.launch_count - l0)
    kernels_per_step, runner_comm = runner.kernels_per_step, runner.comm_description()
    id_table_desc = "replicated on every rank" if table is None else table.describe()

    # ---- e2e: host batches, H2D + step + D2H of the loss every step -----------------------
    # Every step's batch crosses PCIe from pinned memory inside the timed region; the copy of batch i+1 is
    # issued while step i computes (double-buffered staging, TrainStepRunner.stage_batch), the loss of every
    # step is read back to the host — one step behind: the host enqueues step i + 1, then waits for loss i
    # (what train.train_one_epoch does between the reference's log lines).
    for i in range(3):
        runner.step_from_host(host_batches[i % 4])
    packed = [runner.pack_host(b) for b in host_batches]      # one pinned buffer per batch: one H2D copy
    runner.stage_batch(packed[0])
    barrier()
    t0 = time.perf_counter()
    e2e_losses = []
    for i in range(args.steps):
        # K copies for K steps; the loss of step i - 1 is returned while step i is already enqueued
        e2e_losses.append(runner.step_from_host(None, prefetch=packed[(i + 1) % 4], defer_loss=True))
    e2e_losses.append(runner.flush_loss())          # the last step's loss: K losses on the host inside the region
    assert sum(l is not None for l in e2e_losses) == args.steps
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / e2e_s.item()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs:
        dump_train_outputs(args.dump_outputs, runner, eng, synthetic.make_state_dict(cfg, seed=0), host_batches[0])

    # ---- forward + backward only (no optimizer step; SURVEY.md §8d) -------------------------
    fb = None
    if world == 1:
        eng2 = TwoTowerEngine(cfg, dev)
        eng2.load_state_dict(synthetic.make_state_dict(cfg, seed=0))
        r2 = TrainStepRunner(eng2, B, L, with_optimizer=False)
        r2.load_batch(host_batches[0])
        for _ in range(4):
            r2.step_resident()
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            r2.step_resident()
        f1.record()
        torch.cuda.synchronize()
        fb_ms = f0.elapsed_time(f1) / args.steps
        fb = {"ms_per_step": fb_ms, "samples_per_s": B * 1e3 / fb_ms,
              "what": "forward + backward + InfoNCE, gradient buffer cleared instead of the AdamW step"}
        del r2, eng2

    # ---- roofline of the dominant kernel (tcgen05 GEMM) -----------------------------------
    g_all, g, gemm_launches = time_gemm_roofline(eng, runner.static, peaks)
    if table is not None:        # those eager passes added gradient rows into the owners' shards: discard them
        torch.cuda.synchronize()
        dist.barrier()
        table.grad.zero_()
        table.barrier()
    peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    hbm_bound = g["byte_secs"] >= g["flop_secs"]
    if hbm_bound:
        roof = {"bound": "hbm", "achieved": g["bytes"] / g["secs"] / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s"}
    else:
        roof = {"bound": "tensor", "achieved": g["flops"] / g["secs"] / 1e12, "peak": peak_tf, "unit": "TFLOP/s"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    traffic = None
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "gemm_dram_traffic.json")
    if os.path.exists(tpath):      # written by tools/ncu_summary.py from the committed `ncu --set full` capture
        with open(tpath) as f:
            traffic = json.load(f).get("encoder_gemm_dram_bytes_per_launch")
    roof.update({
        "kernel": "tt::gemm_bf16_kernel (tcgen05), the encoder-sized launches (51200-row operands)",
        "traffic": traffic, "peak_source": f"{peak_src}",
        "launches_per_step": g["n"], "avg_launch_us": g["secs"] * 1e6 / max(g["n"], 1),
        "algorithmic_bytes_per_launch": g["bytes"] / max(g["n"], 1),
        "frac_of_per_launch_roofline": g["roof_secs"] / g["secs"],
        "tensor_tflops": g["flops"] / g["secs"] / 1e12, "tensor_frac": g["flops"] / g["secs"] / 1e12 / peak_tf,
        "us_per_step": g["secs"] * 1e6, "share_of_step": g["secs"] * 1e3 / ms_step,
        "flops_per_step": g["flops"], "bytes_per_step": g["bytes"],
        "all_gemm_launches": {"launches_per_step": gemm_launches, "us_per_step": g_all["secs"] * 1e6,
                              "flops_per_step": g_all["flops"], "bytes_per_step": g_all["bytes"],
                              "hbm_gbs": g_all["bytes"] / g_all["secs"] / 1e9},
        "how": "CUDA events around each tt_gemm_bf16 launch of the step issued on one stream behind a device-side "
               "sleep (launch queue full, so events bracket execution only; same operands and fused epilogues as "
               "the timed step); algorithmic bytes = operands + outputs + residual/gate per launch"})
    step_flops = 3.0 * flops_per_sample_fwd(L, B) * B

    # ---- parity of the benchmarked step with the oracle (dropout 0 on the bench batch) -------
    parity = bench_parity_train(cfg, host_batches[0], dev) if rank == 0 else None

    # ---- retrieval (configs[2]) -----------------------------------------------------------
    retr = None if args.skip_retrieval else bench_retrieval(eng, rank, world, dev, peaks)
    if retr is not None and parity is not None:
        parity["retrieval"] = retr.pop("parity")

    # ---- catalog indexing (SURVEY.md §8f-2 / §8e item-sharded) ------------------------------
    indexing = None if args.skip_retrieval else bench_indexing(eng, rank, world, dev, peaks)

    # ---- configs[3] / configs[4]: data-parallel at 512/rank, row-sharded 10M-item table ------
    c4 = c5 = None
    want_c45 = world == 8 or (world > 1 and os.environ.get("TT_BENCH_C45", "") == "1")
    if want_c45 and not args.skip_c45:
        del runner
        eng.release_workspaces()
        torch.cuda.empty_cache()
        c4 = bench_c4(rank, world, dev, peaks, args)
        torch.cuda.empty_cache()
        c5 = bench_c5(rank, world, dev, peaks, args)

    cpu = None
    if rank == 0 and world == 1 and not args.skip_cpu:
        torch.set_num_threads(os.cpu_count() or 1)
        sps, ms_cpu, kind, detail = reference_train_samples_per_s(3, 1, B)
        rps, rkind = reference_retrieval_users_per_s(128)
        cpu = {"value": sps, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind,
               "sample": f"{detail}: 3 timed steps of batch {B} of the c2 workload after 1 warm-up ({ms_cpu:.0f} ms/step)",
               "retrieval_users_per_s": rps, "retrieval_kind": rkind,
               "retrieval_sample": "calculate_metrics_global, 128 users x 1M items, k_list [10, 20, 50, 100] (cost is "
                                   "linear in users)"}

    if rank == 0:
        line = {
            "metric": "two-tower train samples/sec", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": C2_WORKLOAD,
                       "global_batch": world * B, "seq_len": L, "vocab_size": V,
                       "parallelism": f"dp{world}" if world > 1 else "single",
                       "negatives": ("all-gathered across ranks" if world > 1 else "in-batch"),
                       "id_table": id_table_desc,
                       "comm": runner_comm,
                       "last_layer": "exact single-row form (only out[b, len-1] of the last encoder layer is ever "
                                     "read: K/V for all positions, query/out_proj/FFN for one row per sequence)",
                       "l2": "per-step working set (~1.2 GB activations + 410 MB optimizer state) exceeds the 126 MB L2"},
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
            "ms_per_step_percentiles": pct,
            "fwd_bwd_only": fb,
            "gpu_launches": launches,
            "kernels_per_step": kernels_per_step,
            "step_tflops": step_flops / (ms_step * 1e-3) / 1e12,
            "step_tflops_note": "reference-algorithm FLOPs of the step (SURVEY.md §8d formula, every layer on every "
                                "position) per second; the executed GEMM FLOPs are roofline.flops_per_step",
            "roofline": roof,
            "clocks": sampler.summary(),
            "parity": parity,
            "retrieval": retr,
            "indexing": indexing,
        }
        if c4 is not None:
            line["c4"] = c4
        if c5 is not None:
            line["c5"] = c5
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)


def dump_train_outputs(out_dir, runner, eng, state, batch):
    """--dump-outputs: the timed step (the runner's captured graph) once more from the benchmark's seeded start —
    parameters and BatchNorm statistics `state`, zero AdamW moments, step and dropout counters, input `batch` — and
    what it computed, as out_dir/<name>.npy in float32: `loss`, `logits`, `user_emb` and `item_emb` as
    TwoTowerEngine.forward returns them, and `grad.<parameter name>` for every parameter gradient (of the ID table a
    fixed seeded sample of DUMP_TABLE_ROWS rows, with their ids as float64 `grad.<name>.row_ids`).
    Gradients are summed with fp32 atomics, so their last bits vary from run to run (on one B200 at 1000 W, by at
    most 7e-7 of each array's largest element); everything else is the same every run. That is why the step starts from the seeded state and not from where the timed loop left the model,
    and why the updated parameters are not written: AdamW turns that rounding noise into updates of up to lr
    wherever the exact gradient is zero (the biases ahead of BatchNorm, the key bias), and over many steps the
    whole state drifts apart. The gradient is read back from AdamW's first moment, which after the first step is
    (1 - beta1) * gradient. Leaves the model in the state after that one step."""
    import numpy as np
    eng.load_state_dict(state)
    eng.refresh_shadow()
    for t in (eng.grad, eng.exp_avg, eng.exp_avg_sq, eng.step_dev, eng.seed_dev):
        t.zero_()
    runner.load_batch(batch)
    runner.step_resident()
    torch.cuda.synchronize()
    ws = eng.workspace(runner.B, runner.L)
    out = {"loss": ws["loss"].view(1), "logits": ws["S"], "user_emb": ws["un"], "item_emb": ws["in"]}
    grad = eng.exp_avg / (1.0 - runner.betas[0])
    for name, (o, shape) in eng.layout.items():
        g = grad[o:o + torch.Size(shape).numel()].view(shape)
        if name == "user_tower.item_embedding.weight":
            rows = torch.randperm(shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_TABLE_ROWS].sort().values
            out[f"grad.{name}.row_ids"] = rows
            g = g[rows.to(g.device)]
        out[f"grad.{name}"] = g
    arrays = {k: v.detach().cpu().numpy().astype(np.float32 if v.is_floating_point() else np.float64)
              for k, v in out.items()}
    nbytes = sum(a.nbytes for a in arrays.values())
    assert nbytes <= DUMP_MAX_BYTES, f"--dump-outputs would write {nbytes} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def bench_parity_train(cfg, host_batch, dev):
    """The bench batch through a fresh engine with dropout 0 against the oracle's fp32 CPU forward."""
    import dataclasses
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    from oracle import two_tower_oracle as oracle
    cfg0 = dataclasses.replace(cfg, dropout=0.0)
    sd = synthetic.make_state_dict(cfg0, seed=0)
    e = TwoTowerEngine(cfg0, dev)
    e.load_state_dict(sd)
    loss, logits, u, i = e.forward({k: v.to(dev) for k, v in host_batch.items()}, training=True)
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        rl, rlog, ru, ri, _ = oracle.two_tower_forward(sd, {k: v.clone() for k, v in host_batch.items()},
                                                       cfg0.temperature, cfg0.num_heads, training=True)
    out = {"train": {"what": "c2 bench batch, dropout 0, forward: CUDA path vs oracle (fp32 CPU)",
                     "loss": loss.item(), "oracle_loss": rl.item(), "loss_abs_err": abs(loss.item() - rl.item()),
                     "user_emb_abs_err": (u.cpu() - ru).abs().max().item(),
                     "item_emb_abs_err": (i.cpu() - ri).abs().max().item(),
                     "logits_abs_err": (logits.cpu() - rlog).abs().max().item(),
                     "tol": {"loss": 5e-3, "emb": 5e-3, "logits": 8e-2}}}
    t = out["train"]
    t["ok"] = bool(t["loss_abs_err"] <= 5e-3 and t["user_emb_abs_err"] <= 5e-3 and t["item_emb_abs_err"] <= 5e-3
                   and t["logits_abs_err"] <= 8e-2)
    del e
    return out


def _timed(fn, iters, dev, world):
    """CUDA-event time of `iters` calls of fn (barrier + synchronize on both sides, max over ranks) in ms per call."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return ms.item()


def _time_train(runner, host_batches, steps, warmup, dev, world):
    runner.load_batch(host_batches[0])
    for _ in range(max(warmup, 3)):
        runner.step_resident()
    return _timed(runner.step_resident, steps, dev, world)


def bench_c4(rank, world, dev, peaks, args):
    """BASELINE.json configs[3]: data parallel, 512 samples per rank (global 4096 on 8 GPUs), L=200, 100k items,
    every rank's positives against the all-gathered items of all ranks."""
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.train import TrainStepRunner, make_dp_engine
    B, L, V = C4["batch"], C4["seq_len"], C4["vocab"]
    cfg = synthetic.TwoTowerConfig(vocab_size=V, max_seq_len=L, dropout=0.1)
    eng, table = make_dp_engine(cfg, world, dev)
    eng.load_state_dict(synthetic.make_state_dict(cfg, seed=0))
    runner = TrainStepRunner(eng, B, L, world_size=world, sharded_table=table)
    hb = [pin(synthetic.make_batch(cfg, B, seed=500 + rank * 17 + i, full_length=True, num_users=1_000_000)) for i in range(2)]
    ms = _time_train(runner, hb, args.steps, args.warmup, dev, world)
    flops = 3.0 * flops_per_sample_fwd(L, world * B) * B            # per rank
    peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    out = {"workload": f"c4: data-parallel train step, {B}/rank x {world} ranks = global batch {world * B}, seq_len {L}, "
                       f"{V - 1} items, all-gathered negatives",
           "global_batch": world * B, "ms_per_step": ms, "samples_per_s": world * B * 1e3 / ms,
           "step_tflops_per_gpu": flops / (ms * 1e-3) / 1e12, "roofline_frac_tensor": flops / (ms * 1e-3) / 1e12 / peak_tf,
           "roofline_ms_tensor_per_rank": flops / (peak_tf * 1e12) * 1e3,
           "id_table": "replicated" if table is None else table.describe(),
           "kernels_per_step": runner.kernels_per_step, "comm": runner.comm_description()}
    del runner, eng, table
    return out


def bench_c5(rank, world, dev, peaks, args):
    """BASELINE.json configs[4]: 10M-item catalog, ID table row-sharded over the ranks (id/row exchange per step),
    seq_len 512, 512 samples per rank; and retrieval of 10k users against the 10M-item table sharded over the ranks."""
    import dataclasses
    from mrm_b200 import retrieval, synthetic
    from mrm_b200.engine import TwoTowerEngine
    from mrm_b200.sharding import RowShardedTable, SymmShardedTable
    from mrm_b200.train import TrainStepRunner
    from mrm_b200 import symm
    B, L, V = C5["batch"], C5["seq_len"], C5["vocab"]
    cfg = synthetic.TwoTowerConfig(vocab_size=V, max_seq_len=L, dropout=0.1)
    eng = TwoTowerEngine(dataclasses.replace(cfg, vocab_size=2), dev)
    use_symm = symm.available() and os.environ.get("TT_COMM", "") != "nccl"
    table = SymmShardedTable(V, 256, device=dev) if use_symm else RowShardedTable(V, 256, rank, world, dev)
    small = dataclasses.replace(cfg, vocab_size=2)
    eng.load_state_dict(synthetic.make_state_dict(small, seed=0))
    g = torch.Generator(device=dev).manual_seed(777 + rank)
    table.weight[:table.rows].copy_(torch.randn(table.rows, 256, device=dev, generator=g) * (2.0 / (V + 256)) ** 0.5)
    runner = TrainStepRunner(eng, B, L, world_size=world, sharded_table=table)
    hb = [pin(synthetic.make_batch(cfg, B, seed=600 + rank * 17 + i, full_length=True, num_users=1_000_000)) for i in range(2)]
    ms = _time_train(runner, hb, args.steps, args.warmup, dev, world)
    flops = 3.0 * flops_per_sample_fwd(L, world * B) * B
    peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    train = {"workload": f"c5 train: {V - 1} items, ID table row-sharded over {world} ranks ({table.rows} rows/rank), "
                         f"seq_len {L}, {B}/rank, all-gathered negatives, dense AdamW on the local rows",
             "ms_per_step": ms, "samples_per_s": world * B * 1e3 / ms,
             "step_tflops_per_gpu": flops / (ms * 1e-3) / 1e12, "roofline_frac_tensor": flops / (ms * 1e-3) / 1e12 / peak_tf,
             "roofline_ms_tensor_per_rank": flops / (peak_tf * 1e12) * 1e3,
             "table_optimizer_bytes_per_rank": table.rows * 256 * 4 * 7,
             "roofline_ms_hbm_table_optimizer": table.rows * 256 * 4 * 7 / (peaks["hbm_gbs"] * 1e9) * 1e3,
             "exchange": table.describe(), "comm": runner.comm_description(), "kernels_per_step": runner.kernels_per_step}
    del runner, eng, table
    torch.cuda.empty_cache()
    # ---- retrieval: 10k users x 10M items, catalog rows sharded contiguously over the ranks
    U, N, K = C5["users"], V - 1, C5["k"]
    index, users, targets = _sharded_catalog(N, U, rank, world, dev, seed=4321)
    kl = [10, 20, 50, 100]
    for _ in range(2):
        m = retrieval.metrics_from_embeddings(users, targets, index, kl)
    res5 = {}

    def pass5():      # certificate flags stay on the device during the timed passes; read (and repaired) afterwards
        res5["i"], res5["s"], res5["bad"] = retrieval.sharded_topk(users, index, K, defer_check=True)

    ms_r = _timed(pass5, 3, dev, world)
    nfb5 = retrieval.finish_sharded_topk(users, index, K, res5["i"], res5["s"], res5["bad"])
    rflops = 2.0 * U * (N + 1) * 256 / world
    retr = {"workload": f"c5 retrieval: {U} users x {N} items, top-{K}, catalog sharded over {world} GPUs",
            "ms_per_pass": ms_r, "users_per_s": U / (ms_r * 1e-3), "scoring_tflops_per_gpu": rflops / (ms_r * 1e-3) / 1e12,
            "roofline_frac_tensor": rflops / (ms_r * 1e-3) / 1e12 / peak_tf, "recall_at_10": m["Recall@10"],
            "fallback_users": int(nfb5)}
    return {"train": train, "retrieval": retr}


def _catalog_rows(lo, hi, dev, seed, chunk=1 << 18):
    """Rows [lo, hi) of THE seeded global catalog (unit-norm rows, row 0 = padding zeros): generated in fixed chunks
    of 2^18 rows, each from its own seed, so every rank count slices the same table without materialising it."""
    out = torch.empty(hi - lo, 256, device=dev)
    c0 = lo // chunk
    while c0 * chunk < hi:
        a, b = c0 * chunk, (c0 + 1) * chunk
        g = torch.Generator(device=dev).manual_seed(seed * 100_003 + c0)
        rows = torch.nn.functional.normalize(torch.randn(chunk, 256, device=dev, generator=g), dim=1)
        s0, s1 = max(a, lo), min(b, hi)
        out[s0 - lo:s1 - lo] = rows[s0 - a:s1 - a]
        c0 += 1
    if lo == 0:
        out[0] = 0
    return out


def _sharded_catalog(N, U, rank, world, dev, seed):
    """(index over this rank's contiguous shard, users, targets): the SAME catalog, users and targets for every
    world size. Targets are planted so Recall@10 is ~0.6-0.7 (the reference's reported regime)."""
    from mrm_b200 import retrieval
    from mrm_b200.sharding import shard_bounds
    first, rows = shard_bounds(N + 1, world, rank)
    shard = _catalog_rows(first, first + rows, dev, seed)
    index = retrieval.CatalogIndex.from_shard(shard, first, N + 1, device=dev) if world > 1 else retrieval.CatalogIndex(shard, device=dev)
    gu = torch.Generator(device=dev).manual_seed(seed + 99)
    targets = torch.randint(1, N + 1, (U,), device=dev, generator=gu)
    noise = torch.randn(U, 256, device=dev, generator=gu)
    # the planted row may live on another rank: every rank contributes the target rows it owns
    trow = torch.zeros(U, 256, device=dev)
    mine = (targets >= first) & (targets < first + rows)
    trow[mine] = shard[targets[mine] - first]
    if world > 1:
        dist.all_reduce(trow, op=dist.ReduceOp.SUM)
    users = torch.nn.functional.normalize(trow + 3.3 / 16.0 * noise, dim=1)
    return index, users, targets


def bench_indexing(eng, rank, world, dev, peaks):
    """Catalog indexing (src/evaluate_metrics.py:24-104) of the c3 catalog's 1M items, item list split over the
    ranks: item tower (eval) -> NaN->0 -> renormalise -> scatter by id into the dense fp32 table + bf16 copy."""
    from mrm_b200.evaluate_metrics import index_catalog_device
    N = C3["items"]
    per = (N + world - 1) // world
    lo, hi = min(rank * per, N), min(N, (rank + 1) * per)
    n = hi - lo
    g = torch.Generator(device=dev).manual_seed(55 + rank)
    feats = {k: torch.randn(n, 128, device=dev, generator=g)
             for k in ("target_audio", "target_image", "target_input_ids", "target_tabular")}
    ids = torch.arange(lo + 1, hi + 1, device=dev)
    ids = ids[torch.randperm(n, device=dev, generator=g)]

    class _M:                      # the functions only need .engine / .eval()
        engine = eng

        def eval(self):
            return self

    table = torch.zeros(N + 1, 256, device=dev)
    table16 = torch.zeros(N + 1, 256, device=dev, dtype=torch.bfloat16)
    m = _M()
    for _ in range(2):
        index_catalog_device(m, feats, ids, N + 1, out=(table, table16))
    ms = _timed(lambda: index_catalog_device(m, feats, ids, N + 1, out=(table, table16)), 5, dev, world)
    bytes_alg = n * (4 * 128 * 4 + 256 * 4)                      # 2 KB of features in, 1 KB of embedding out
    bytes_moved = n * (2048 + 1024 + 1024 + 1024 + 1024 + 1024 + 1024 + 1536)
    gbs = bytes_alg / (ms * 1e-3) / 1e9
    return {"workload": f"f2: catalog indexing, {N} items over {world} GPU(s) ({n} per rank), eval-mode item tower + "
                        "NaN->0 + renormalise + scatter by id (fp32 table + bf16 copy)",
            "ms_per_pass": ms, "items_per_s": N / (ms * 1e-3),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"],
                         "algorithmic_bytes_per_item": 3072, "moved_bytes_per_item": bytes_moved // max(n, 1),
                         "moved_gbs": bytes_moved / (ms * 1e-3) / 1e9},
            "rows_nonzero": int((table.abs().sum(1) > 0).sum().item()) if world == 1 else None}


def _fp64_canonical_topk(users, table, K, chunk=32):
    """Checker (plain torch on the GPU): fp64 scores rounded once to fp32, column 0 masked, stable descending sort
    = the canonical order (score descending, item index ascending)."""
    idx, val = [], []
    t64 = table.double()
    for s0 in range(0, users.shape[0], chunk):
        sc = (users[s0:s0 + chunk].double() @ t64.t()).float()
        sc[:, 0] = float("-inf")
        v, i = torch.sort(sc, dim=1, descending=True, stable=True)
        idx.append(i[:, :K].clone())
        val.append(v[:, :K].clone())
    return torch.cat(idx), torch.cat(val)


def bench_retrieval(eng, rank, world, dev, peaks):
    """10k users x 1M items, top-100 + Recall/NDCG; ONE seeded catalog for every world size, rows sharded
    contiguously over the ranks."""
    from mrm_b200 import retrieval
    U, N, K = C3["users"], C3["items"], C3["k"]
    index, users, targets = _sharded_catalog(N, U, rank, world, dev, seed=1234)
    host_users = users.cpu().pin_memory()
    host_targets = targets.cpu().pin_memory()
    kl = [10, 20, 50, 100]
    for _ in range(2):
        m = retrieval.metrics_from_embeddings(users, targets, index, kl)
    torch.cuda.synchronize()
    iters = 5
    flags = torch.zeros(U, device=dev, dtype=torch.int32)
    res = {}

    def one_pass():
        if world > 1:    # the whole sharded pass: per-shard candidates, exchange, merge + certificate on the device
            res["idx"], res["score"], res["bad"] = retrieval.sharded_topk(users, index, K, defer_check=True)
        else:            # certificate flags are written by every pass and read AFTER the timed region
            res["idx"], res["score"], _ = retrieval.retrieve_topk(users, index, K, exact_fallback=False, flags_out=flags)

    for _ in range(2):      # the timed call itself, warm: scratch of this exact call sequence exists, ranks are in step
        one_pass()
    ms = _timed(one_pass, 2 * iters if world > 1 else iters, dev, world)
    if world > 1:    # certificate read AFTER the timed region; uncertified users (if any) repaired by the exact protocol
        nfb = retrieval.finish_sharded_topk(users, index, K, res["idx"], res["score"], res["bad"])
    else:
        nfb = int(flags.sum().item())
    if world == 1 and nfb:    # the timed pass left uncertified users: finish them exactly (untimed) for the checks below
        res["idx"], res["score"], _ = retrieval.retrieve_topk(users, index, K)
    # e2e: host user embeddings -> device, retrieval, merge, metrics -> host (one untimed call first: the 10 MB
    # device buffer of the host copy comes from the allocator's pool afterwards)
    def e2e_call():
        return retrieval.metrics_from_embeddings(host_users.to(dev, non_blocking=True),
                                                 host_targets.to(dev, non_blocking=True), index, kl)

    e2e_call()
    torch.cuda.synchronize()
    anatomy = None
    if os.environ.get("TT_BENCH_ANATOMY", "") == "1":      # diagnostic: where one e2e call spends its host time
        marks = []

        def mark(name):
            torch.cuda.synchronize()
            marks.append((name, time.perf_counter()))

        if world > 1:
            dist.barrier()
        mark("start")
        du, dt = host_users.to(dev, non_blocking=True), host_targets.to(dev, non_blocking=True)
        mark("h2d")
        if world > 1:
            ai, as_, ab = retrieval.sharded_topk(du, index, K, defer_check=True)
        else:
            ai, as_, _ = retrieval.retrieve_topk(du, index, K)
        mark("topk")
        rec, nd = retrieval.rank_metrics(ai, dt, kl)
        mark("rank_metrics")
        torch.cat([rec.flatten(), nd.flatten()]).cpu()
        mark("readback")
        anatomy = {b[0]: 1e3 * (b[1] - a[1]) for a, b in zip(marks[:-1], marks[1:])}
        # the same statements as metrics_from_embeddings, host clock only (no added synchronisation)
        hm = [("start", time.perf_counter())]
        du, dt = host_users.to(dev, non_blocking=True), host_targets.to(dev, non_blocking=True)
        hm.append(("h2d_enqueue", time.perf_counter()))
        if world > 1:
            ai, as_, ab = retrieval.sharded_topk(du, index, K, 256, None, defer_check=True)
        else:
            ai, as_, _ = retrieval.retrieve_topk(du, index, K)
            ab = torch.zeros(U, device=dev, dtype=torch.int32)
        hm.append(("topk_enqueue", time.perf_counter()))
        rec, nd = retrieval.rank_metrics(ai, dt, kl)
        hm.append(("rank_metrics_enqueue", time.perf_counter()))
        bm = ab.max().float().view(1)
        hm.append(("bad_max", time.perf_counter()))
        pk = torch.cat([rec.flatten(), nd.flatten(), bm])
        hm.append(("cat", time.perf_counter()))
        pk = pk.cpu()
        hm.append(("cpu", time.perf_counter()))
        _ = pk[-1].item()
        rr = pk[:rec.numel()].view(rec.shape)
        _ = [rr[j].mean().item() for j in range(rr.shape[0])]
        hm.append(("means", time.perf_counter()))
        anatomy["host_only"] = {b[0]: 1e3 * (b[1] - a[1]) for a, b in zip(hm[:-1], hm[1:])}
    if world > 1:
        dist.barrier()
    e2e_calls = []
    t0 = time.perf_counter()
    for _ in range(iters):
        t1 = time.perf_counter()
        m = e2e_call()
        e2e_calls.append((time.perf_counter() - t1) * 1e3)
        if os.environ.get("TT_RETRIEVAL_TRACE", "") == "1":
            print(f"[rank {rank}] e2e call done at {time.time() % 100:.4f} took {e2e_calls[-1]:.2f} ms", file=sys.stderr, flush=True)
    torch.cuda.synchronize()
    e2e = torch.tensor([(time.perf_counter() - t0) / iters], device=dev)
    if world > 1:
        dist.all_reduce(e2e, op=dist.ReduceOp.MAX)

    # ---- parity on the bench data ----------------------------------------------------------
    # (a) rank 0 holds the whole catalog once more and checks a 512-user sample against an fp64 canonical sort;
    # (b) for world > 1 the sharded result must EQUAL the single-GPU result on the same catalog (independent of G).
    parity = None
    if rank == 0:
        full = _catalog_rows(0, N + 1, dev, 1234) if world > 1 else index.table
        sel = torch.arange(0, U, max(1, U // 512), device=dev)[:512]
        ri, rv = _fp64_canonical_topk(users[sel], full, K)
        got_i, got_s = res["idx"][sel].long(), res["score"][sel]
        mism = int((got_i != ri).sum().item())
        parity = {"what": f"top-{K} of {sel.numel()} sampled users vs fp64 canonical sort (torch, GPU) of the whole catalog",
                  "index_mismatches": mism, "score_max_abs_err": (got_s - rv).abs().max().item(),
                  "ok": bool(mism == 0)}
        if world > 1:
            single = retrieval.CatalogIndex(full, device=dev)
            si, ss, _ = retrieval.retrieve_topk(users, single, K)
            parity["sharded_equals_single_gpu"] = bool(torch.equal(si, res["idx"]) and torch.equal(ss, res["score"]))
            parity["ok"] = parity["ok"] and parity["sharded_equals_single_gpu"]
            del single, si, ss
        del full
        from oracle import two_tower_oracle as oracle
        om = oracle.rank_metrics(res["idx"].cpu().long(), targets.cpu(), kl)
        parity["metrics_equal_oracle_on_same_lists"] = bool(all(m[k] == om[k].mean().item() for k in m))
        parity["ok"] = parity["ok"] and parity["metrics_equal_oracle_on_same_lists"]
    torch.cuda.empty_cache()

    # ---- the same pass with the user embeddings produced by the CUDA user tower (eval mode) from HOST
    # histories (L = 50, the reference default): H2D ids -> SASRec forward -> retrieval -> merge -> metrics.
    # With several ranks the USERS are split over the ranks for the tower and the 10 MB of embeddings all-gathered.
    from mrm_b200 import synthetic
    from mrm_b200.engine import TwoTowerEngine
    Lh = C3["hist_len"]
    tcfg = synthetic.TwoTowerConfig(vocab_size=4096, max_seq_len=Lh, dropout=0.0)   # small ID table: ids are synthetic
    teng = TwoTowerEngine(tcfg, dev)
    teng.load_state_dict(synthetic.make_state_dict(tcfg, seed=0))
    hb = synthetic.make_batch(tcfg, U, seed=7, full_length=True)
    per = (U + world - 1) // world
    u0, u1 = min(rank * per, U), min(U, (rank + 1) * per)
    UB = min(2000, per)
    h_ids, h_mask = hb["history_ids"][u0:u1].pin_memory(), hb["history_mask"][u0:u1].pin_memory()
    h_g, h_c = hb["user_gender"][u0:u1].pin_memory(), hb["user_country"][u0:u1].pin_memory()
    uemb = torch.zeros(world * per, 256, device=dev)

    def tower_pass():
        if not teng.shadow_valid:
            teng.refresh_shadow()
        for s0 in range(0, u1 - u0, UB):
            n = min(UB, u1 - u0 - s0)
            sl = slice(s0, s0 + n)
            ws = teng.workspace(n, Lh)
            u = teng.user_forward(ws, h_ids[sl].to(dev, non_blocking=True), h_mask[sl].to(dev, non_blocking=True),
                                  h_g[sl].to(dev, non_blocking=True), h_c[sl].to(dev, non_blocking=True), training=False)
            uemb[u0 + s0:u0 + s0 + n].copy_(u)
        if world > 1:
            dist.all_gather_into_tensor(uemb, uemb[rank * per:(rank + 1) * per].clone())
        return retrieval.metrics_from_embeddings(uemb[:U], host_targets.to(dev, non_blocking=True), index, kl)

    for _ in range(2):
        tower_pass()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(iters):
        tower_pass()
    torch.cuda.synchronize()
    e2e_tower = torch.tensor([(time.perf_counter() - t0) / iters], device=dev)
    if world > 1:
        dist.all_reduce(e2e_tower, op=dist.ReduceOp.MAX)
    del teng

    # single-user recommendation latency (src/inference.py:283-306): one user, 50 history items excluded, top-10
    rec_ms = None
    if world == 1:
        from mrm_b200 import inference
        g1 = torch.Generator(device=dev).manual_seed(9)
        hist = torch.randint(1, N, (1, 50), device=dev, generator=g1)
        one = users[:1].contiguous()
        for _ in range(3):
            inference.recommend_topk(one, index, hist, 10)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(20):
            ridx, _ = inference.recommend_topk(one, index, hist, 10)
            ridx.cpu()                      # the caller reads the ids: one sync per query
        rec_ms = (time.perf_counter() - t0) / 20 * 1e3

    flops = 2.0 * U * (N + 1) * 256 / world
    peak_tf = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    return {"metric": "top-100 retrieval users/sec @1M items", "recommend_1user_ms": rec_ms, "users_per_s": U / (ms * 1e-3),
            "ms_per_pass": ms, "e2e_users_per_s": U / e2e.item(), "e2e_ms_per_call_rank0": e2e_calls, "e2e_anatomy_ms": anatomy,
            "e2e_users_per_s_incl_user_tower": U / e2e_tower.item(),
            "scoring_tflops_per_gpu": flops / (ms * 1e-3) / 1e12,
            "roofline_frac_tensor": flops / (ms * 1e-3) / 1e12 / peak_tf,
            "config": {"workload": f"c3: {U} users x {N} items, top-{K}, Recall/NDCG@10/20/50/100, catalog sharded "
                                   f"over {world} GPU(s); the same seeded catalog, users and targets for every world size",
                       "users_per_s": "device-resident user embeddings: scoring + top-K + exact re-score + certificate "
                                      "(events)" + ("; sharded: per-shard pass, exchange, merge, certificate, fallback "
                                                    "(retrieval.sharded_topk)" if world > 1 else
                                                    "; certificate flags read after the timed region"),
                       "e2e_users_per_s": "host user embeddings -> device, retrieval, cross-shard merge, metrics -> host",
                       "e2e_users_per_s_incl_user_tower": f"host histories (L={Lh}) -> CUDA user tower (eval, users split "
                                                          f"over the ranks, embeddings all-gathered) -> same",
                       "kprime": 256},
            "recall_at_10": m["Recall@10"], "fallback_users": nfb, "parity": parity}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--skip-retrieval", action="store_true", help="skip the c3 retrieval section (A/B timing runs)")
    ap.add_argument("--skip-c45", action="store_true", help="skip the c4 / c5 blocks of multi-GPU runs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed c2 step computes from the seeded start to DIR/<name>.npy (one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        ap.error("--dump-outputs runs on one GPU")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1 and dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
