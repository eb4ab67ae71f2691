"""Training-loop entry points with the reference's signatures (src/train.py:41-111) plus the
graph-replayed step runner bench.py and the fast path use.

  train_one_epoch(model, dataloader, optimizer, device, epoch, is_main_process=True, log_interval=50)
  evaluate(model, dataloader, device, k=10)

With a ``FusedAdamW`` optimizer the step is forward + hand-written backward + fused AdamW, captured
once as a CUDA graph and replayed; batches go host -> static device buffers with non-blocking
copies and the loss comes back through a pinned scalar. With any other torch optimizer the model's
autograd node is used (reference-compatible, slower). bf16 needs no GradScaler.
"""
from __future__ import annotations

import logging
import math
import os
from typing import Dict, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _lib
from .engine import TwoTowerEngine

logger = logging.getLogger(__name__)

_BATCH_KEYS = ("history_ids", "history_mask", "user_gender", "user_country", "user_idx", "target_audio",
               "target_image", "target_input_ids", "target_tabular")


class LogQCorrection:
    """logQ correction of in-batch negatives (Yi et al., RecSys 2019) for ONE side of the symmetric InfoNCE.

    Every negative of a batch is another row's positive, so an entity is drawn as a negative with its in-batch
    sampling probability q, and the plain loss learns roughly log p(item | user) - log q(item): retrieval ends up
    biased against what users play most. The correction subtracts log q_j from every logit of column j in the
    training loss only (the logits `forward` returns, evaluation and serving are unchanged). One object per side:
    ``TrainStepRunner(..., logq=<items>, logq_users=<users>)``; the item side reads each row's ``target_id``, the
    user side its ``user_idx``.

    Sources of log q (all produce the offsets on the device, inside the captured step):
      * ``from_offsets(table)``: a fixed fp32 log q per id;
      * ``from_counts(counts, smoothing=1.0)``: log((c + s) / sum(c + s)), computed in fp64 and stored as fp32;
      * ``streaming(num_ids, ...)``: the paper's streaming frequency estimator over the training ids (no pass over
        the dataset): h hash arrays of H slots hold the last step each slot was seen (A) and the estimated
        interval between sightings (Bv); each step updates every slot its ids hit once, then log q = -log(max Bv).
    Ids outside [0, N) of a table get the offset of the rarest id (a zero count with ``from_counts``).

    The object owns its device state, allocated once: a captured step graph keeps pointing at it, so it survives
    runner rebuilds (a trailing partial batch) and is restored in place by ``load_state_dict``. With data-parallel
    gathered negatives every rank updates its replica from the same all-gathered ids (replicas stay bit-identical);
    with negatives="local" each rank estimates from its own batch, which is what its softmax samples from."""

    def __init__(self, kind: str, device=None):
        self.kind = kind
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.table: Optional[torch.Tensor] = None
        self.floor = 0.0
        self.A: Optional[torch.Tensor] = None
        self.Bv: Optional[torch.Tensor] = None
        self.step: Optional[torch.Tensor] = None
        self.alpha = self.num_ids = self.init_interval = None

    @staticmethod
    def _vector(x, what: str) -> torch.Tensor:
        t = torch.as_tensor(x)
        if t.dim() != 1 or t.numel() == 0:
            raise ValueError(f"{what} must be a non-empty 1-D table indexed by id, got shape {tuple(t.shape)}")
        if not (t.is_floating_point() or t.dtype in (torch.int32, torch.int64)):
            raise ValueError(f"{what} must be numeric, got {t.dtype}")
        t = t.detach().cpu().double()
        if not torch.isfinite(t).all():
            raise ValueError(f"{what} contains NaN or infinite values")
        return t

    @classmethod
    def from_offsets(cls, table, device=None) -> "LogQCorrection":
        """A fixed log q per id: ``table[id]`` (fp32)."""
        t = cls._vector(table, "offsets").float()
        self = cls("offsets", device)
        self.table = t.to(self.device)
        self.floor = float(t.min())
        return self

    @classmethod
    def from_counts(cls, counts, smoothing: float = 1.0, device=None) -> "LogQCorrection":
        """log q[id] = log((counts[id] + smoothing) / sum(counts + smoothing)), in fp64, stored as fp32."""
        c = cls._vector(counts, "counts")
        if (c < 0).any():
            raise ValueError("counts must be >= 0")
        if not (math.isfinite(smoothing) and smoothing > 0):
            raise ValueError(f"smoothing must be a finite positive number, got {smoothing}")
        total = float((c + smoothing).sum())
        self = cls("offsets", device)
        self.table = torch.log((c + smoothing) / total).float().to(self.device)
        self.floor = float(np.float32(math.log(smoothing / total)))
        return self

    @classmethod
    def streaming(cls, num_ids: int, num_slots: int = 2 ** 20, num_hashes: int = 2, alpha: float = 0.01,
                  init_interval: Optional[float] = None, device=None) -> "LogQCorrection":
        """The streaming estimator. ``init_interval``: the starting Bv of every slot; None takes
        max(1, num_ids / global batch) (the interval of a uniformly sampled id) when a runner first binds it."""
        if not (isinstance(num_ids, (int, np.integer)) and num_ids >= 1):
            raise ValueError(f"num_ids must be a positive integer, got {num_ids!r}")
        if not (isinstance(num_slots, (int, np.integer)) and 1 <= num_slots <= 2 ** 28
                and num_slots & (num_slots - 1) == 0):
            raise ValueError(f"num_slots must be a power of two in [1, 2^28], got {num_slots!r}")
        if not (isinstance(num_hashes, (int, np.integer)) and 1 <= num_hashes <= 4):
            raise ValueError(f"num_hashes must be in [1, 4], got {num_hashes!r}")
        if not 0.0 < float(alpha) <= 1.0:                                     # also rejects NaN
            raise ValueError(f"alpha must be in (0, 1], got {alpha!r}")
        if init_interval is not None and not (math.isfinite(init_interval) and init_interval > 0):
            raise ValueError(f"init_interval must be a finite positive number, got {init_interval!r}")
        self = cls("streaming", device)
        self.alpha, self.num_ids = float(alpha), int(num_ids)
        self.A = torch.zeros(num_hashes, num_slots, dtype=torch.int64, device=self.device)
        self.Bv = torch.empty(num_hashes, num_slots, dtype=torch.float32, device=self.device)
        self.step = torch.zeros(1, dtype=torch.int64, device=self.device)
        self.init_interval = None
        if init_interval is not None:
            self._init_state(float(init_interval))
        return self

    def _init_state(self, interval: float) -> None:
        self.init_interval = interval
        self.A.zero_()
        self.Bv.fill_(interval)
        self.step.zero_()

    def bind(self, global_batch: int) -> None:
        """Called by the runner before its first step: fixes the default initial interval of a streaming estimator
        from the number of ids each step sees."""
        if self.kind == "streaming" and self.init_interval is None:
            self._init_state(max(1.0, self.num_ids / global_batch))

    def offsets(self, ids: torch.Tensor, out: torch.Tensor) -> None:
        """out[i] = log q of ids[i], on the current stream (one kernel; the streaming estimator also advances)."""
        from . import ops
        if self.kind == "offsets":
            ops.logq_table_gather(ids, self.table, self.floor, out)
        else:
            if self.init_interval is None:
                raise RuntimeError("streaming LogQCorrection used before bind(global_batch)")
            ops.logq_stream_update(ids, self.A, self.Bv, self.step, self.alpha,
                                   float(np.float32(1.0 - self.alpha)), out)

    def state_dict(self) -> Dict[str, object]:
        """Arrays, step counter and hyper-parameters (CPU copies); separate from the model's state_dict."""
        if self.kind == "offsets":
            return {"kind": self.kind, "table": self.table.cpu().clone(), "floor": self.floor}
        return {"kind": self.kind, "A": self.A.cpu().clone(), "Bv": self.Bv.cpu().clone(),
                "step": self.step.cpu().clone(), "alpha": self.alpha, "num_ids": self.num_ids,
                "init_interval": self.init_interval}

    def load_state_dict(self, sd: Dict[str, object]) -> None:
        """Restores in place (a captured graph keeps its pointers); the shapes must be this object's."""
        if sd.get("kind") != self.kind:
            raise ValueError(f"state of a {sd.get('kind')!r} correction loaded into a {self.kind!r} one")
        if self.kind == "offsets":
            if tuple(sd["table"].shape) != tuple(self.table.shape):
                raise ValueError(f"offset table of shape {tuple(sd['table'].shape)}, expected {tuple(self.table.shape)}")
            self.table.copy_(sd["table"])
            self.floor = float(sd["floor"])
            return
        for k in ("A", "Bv", "step"):
            if tuple(sd[k].shape) != tuple(getattr(self, k).shape) or sd[k].dtype != getattr(self, k).dtype:
                raise ValueError(f"estimator state {k} of shape {tuple(sd[k].shape)} / {sd[k].dtype}, expected "
                                 f"{tuple(getattr(self, k).shape)} / {getattr(self, k).dtype}")
        self.A.copy_(sd["A"])
        self.Bv.copy_(sd["Bv"])
        self.step.copy_(sd["step"])
        self.alpha, self.num_ids, self.init_interval = float(sd["alpha"]), int(sd["num_ids"]), sd["init_interval"]


class FusedAdamW:
    """Marker optimizer: AdamW(lr, betas, eps, weight_decay) applied by the engine's fused kernel over the
    whole flat parameter buffer (torch.optim.AdamW defaults, src/train.py:302)."""

    def __init__(self, model, lr: float = 1e-4, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01):
        self.engine: TwoTowerEngine = model.engine if hasattr(model, "engine") else model
        self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay

    def zero_grad(self, set_to_none: bool = True) -> None:
        self.engine.grad.zero_()

    def step(self) -> None:
        self.engine.adamw_step(self.lr, self.betas, self.eps, self.weight_decay)


def make_dp_engine(cfg, world_size: int, device=None, group=None, table: str = "auto"):
    """(engine, table) for data-parallel training on ``world_size`` GPUs of one NVLink domain.

    table="sharded" (what "auto" picks whenever a symmetric arena can be built): the ID table — 92 % of the
    parameters at 100k items — is row-sharded over the ranks (sharding.SymmShardedTable) instead of replicated:
    rows are gathered from / gradient rows added into the owner's memory over NVLink inside the embedding kernels
    and each owner runs AdamW over its V / world rows. Per step and rank that moves B * L rows each way (52 MB at
    batch 256 x 200) where the replicated table needs the whole 102 MB gradient reduced and the whole table
    re-broadcast, and the optimizer touches 1 / world of the rows. Same arithmetic as the replicated step
    (mean of the ranks' gradients, dense AdamW on every row). table="replicated": the reference's DDP layout."""
    import dataclasses
    from . import symm
    from .sharding import SymmShardedTable
    if table == "auto":
        env = os.environ.get("TT_TABLE", "")
        table = env if env in ("sharded", "replicated") else \
            ("sharded" if world_size > 1 and symm.available(group) and os.environ.get("TT_COMM", "") != "nccl" else "replicated")
    if table == "replicated" or world_size == 1:
        return TwoTowerEngine(cfg, device), None
    eng = TwoTowerEngine(dataclasses.replace(cfg, vocab_size=2), device)
    try:
        eng.peer_table = SymmShardedTable(cfg.vocab_size, cfg.embedding_dim, group, eng.device)
    except Exception as exc:      # no peer access / symmetric allocator refused (same outcome on every rank)
        if table == "sharded" and os.environ.get("TT_TABLE", "") == "sharded":
            raise
        logger.warning(f"symmetric arena for the ID table unavailable ({exc}); keeping the table replicated")
        del eng
        return TwoTowerEngine(cfg, device), None
    return eng, eng.peer_table


class TrainStepRunner:
    """One training step (src/train.py:54-65) over static device buffers, replayed as CUDA graphs.

    Data parallel (world_size > 1), one process per GPU:
      negatives="gathered" (default; BASELINE.json config 4): the normalised user / item embeddings
        and user ids of all ranks are all-gathered (3 small NCCL calls), every rank forms its
        (B x G*B) logit blocks, the row log-sum-exps are all-gathered (2 tiny calls) so each rank can
        form the exact gradient of the GLOBAL symmetric InfoNCE for its own rows;
      negatives="local": the reference's DDP semantics (per-rank in-batch negatives, src/train.py:300).
    In both cases BatchNorm statistics are per rank (the reference uses no SyncBatchNorm) and the flat
    gradient buffer is averaged with ONE all-reduce between the backward and optimizer graphs.

    ``logq`` / ``logq_users`` (LogQCorrection): logQ correction of the item / user negatives. The item side adds
    ``target_id`` to the input buffer; the user side needs ``with_user_idx``. The offsets are computed inside the
    step, from the global batch's ids when negatives are gathered."""

    def __init__(self, engine: TwoTowerEngine, B: int, L: int, world_size: int = 1, lr: float = 1e-4,
                 use_graph: bool = True, with_user_idx: bool = True, negatives: str = "gathered",
                 rank: Optional[int] = None, group=None, shard_optimizer: bool = True,
                 with_optimizer: bool = True, sharded_table=None, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.01, comm: str = "auto", logq: Optional[LogQCorrection] = None,
                 logq_users: Optional[LogQCorrection] = None):
        self.eng, self.B, self.L, self.world, self.lr, self.use_graph = engine, B, L, world_size, lr, use_graph
        if logq_users is not None and not with_user_idx:
            raise ValueError("logq_users corrects the user negatives by user_idx: it needs with_user_idx=True")
        for c in (logq, logq_users):
            if c is not None and (not isinstance(c, LogQCorrection)
                                  or c.device != torch.empty(0, device=engine.device).device):
                raise ValueError(f"logq / logq_users must be LogQCorrection objects on {engine.device}")
        self.logq, self.logq_users = logq, logq_users
        self.betas, self.eps, self.weight_decay = tuple(betas), eps, weight_decay
        self.group = group
        #: False = forward + backward only (the gradient buffer is cleared instead of consumed): the
        #: "without optimizer step" timing SURVEY.md §8d asks for; parameters do not change
        self.with_optimizer = with_optimizer
        #: sharding.RowShardedTable: the item-ID table lives row-sharded across the ranks (config 5); every step
        #: starts with the id/row all-to-all and ends with the gradient-row all-to-all + the local-row AdamW
        self.table = sharded_table
        from .sharding import RowShardedTable
        if isinstance(sharded_table, RowShardedTable) and engine.table_rows is None:
            engine.use_external_table(B, L)
        self.rank = (dist.get_rank(group) if world_size > 1 else 0) if rank is None else rank
        self.gathered = world_size > 1 and negatives == "gathered"
        # comm = "symm": every exchange of the step is one of this repo's kernels over a symmetric NVLink arena
        # (csrc/tt_symm.cu) and the whole step is ONE CUDA graph; "nccl": the library collectives between
        # sub-graphs; "auto": symm whenever the process group can build an arena (NCCL group, <= 16 ranks) and the
        # step is the standard one (gathered negatives, optimizer on, replicated table).
        self.arena = None
        if comm not in ("auto", "symm", "nccl"):
            raise ValueError(f"comm={comm!r}")
        from .sharding import SymmShardedTable
        peer_table = isinstance(sharded_table, SymmShardedTable)
        if peer_table:
            engine.peer_table = sharded_table
        want_symm = comm != "nccl" and world_size > 1 and self.gathered and with_optimizer \
            and (sharded_table is None or peer_table) \
            and engine.numel % (4 * world_size) == 0 and os.environ.get("TT_COMM", "") != "nccl"
        if peer_table and not want_symm:
            raise ValueError("a SymmShardedTable needs the symmetric-arena step (gathered negatives, optimizer on)")
        if want_symm:
            from . import symm
            if symm.available(group):
                try:
                    self._setup_symm(engine, B, world_size, group)
                except Exception as exc:          # no peer access / symmetric allocator refused: library path
                    if comm == "symm":
                        raise
                    logger.warning(f"symmetric arena unavailable ({exc}); using the NCCL exchanges")
                    self.arena = None
            elif comm == "symm":
                raise RuntimeError("comm='symm' needs an NCCL process group on one NVLink domain")
        # ZeRO-1 style: reduce-scatter the gradient, AdamW on this rank's 1/world shard (moments are
        # held for the shard only), all-gather the updated parameters. Same bytes on NVLink as one
        # all-reduce, 1/world of the optimizer's HBM traffic.
        # The flat buffer is padded to a multiple of 2048 elements (engine.py), i.e. it splits into equal 16-byte
        # aligned shards for 1/2/4/8 ranks; any other world size keeps the replicated optimizer (one all-reduce).
        self.shard_opt = world_size > 1 and shard_optimizer and engine.numel % (4 * world_size) == 0
        if self.arena is not None:
            self.shard_opt = False           # the arena path shards the optimizer inside its own kernel
        if self.shard_opt:
            self._grad_shard = torch.empty(engine.numel // world_size, device=engine.device)
        # packed exchange buffers: one all-gather for (user emb | item emb | user id), one for the two LSE vectors
        # (+ 8 bytes of target id per row when the item side of the logQ correction is on)
        if self.gathered and self.arena is None:
            D = engine.cfg.embedding_dim
            w = 2 * D * 2 + 8 + (8 if logq is not None else 0)
            self._pack_emb = torch.empty(B, w, device=engine.device, dtype=torch.uint8)
            self._pack_emb_all = torch.empty(world_size * B, w, device=engine.device, dtype=torch.uint8)
            if logq is not None:
                self._tid_all = torch.zeros(world_size * B, device=engine.device, dtype=torch.long)
            self._pack_lse = torch.empty(B, 2, device=engine.device)
            self._pack_lse_all = torch.empty(world_size * B, 2, device=engine.device)
        dev, m = engine.device, engine.cfg.modality_dim
        # One device buffer holds every input of a step (each field 256-byte aligned); the `static` tensors the
        # graph reads are views into it, so a batch packed the same way on the host (`pack_host`) arrives with
        # ONE host->device copy.
        fields = [("history_ids", (B, L), torch.long), ("history_mask", (B, L), torch.long),
                  ("user_gender", (B,), torch.long), ("user_country", (B,), torch.long),
                  ("target_audio", (B, m), torch.float32), ("target_image", (B, m), torch.float32),
                  ("target_input_ids", (B, m), torch.float32), ("target_tabular", (B, m), torch.float32)]
        if with_user_idx:
            fields.append(("user_idx", (B,), torch.long))
        if logq is not None:
            fields.append(("target_id", (B,), torch.long))
        self._fields, off = [], 0
        for name, shape, dt in fields:
            n = 1
            for d in shape:
                n *= d
            nbytes = n * torch.empty((), dtype=dt).element_size()
            self._fields.append((name, shape, dt, off, nbytes))
            off += (nbytes + 255) // 256 * 256
        self._static_buf = torch.zeros(off, device=dev, dtype=torch.uint8)
        self.static: Dict[str, torch.Tensor] = {
            name: self._static_buf[o:o + nb].view(dt).view(shape) for name, shape, dt, o, nb in self._fields}
        # two pinned read-back slots: the loss of step i is copied while step i + 1 is being enqueued (step_from_host)
        self._loss_slots = [{"loss": torch.zeros((), dtype=torch.float32).pin_memory(),
                             "all": torch.zeros(max(world_size, 1), 4).pin_memory(),
                             "err": torch.zeros(1, dtype=torch.int32).pin_memory(),
                             "ev": torch.cuda.Event()} for _ in range(2)]
        self._loss_turn, self._loss_pending = 0, None
        self._graphs = None
        self._cap_stream = None
        self._stage = None
        self._staged = False
        self.kernels_per_step = 0
        self._warm = False
        # logQ offsets over the columns of the logit blocks (global batch when gathered); a side that is off stays 0
        self._offsets = None
        if logq is not None or logq_users is not None:
            n = world_size * B if self.gathered else B
            self._offsets = (torch.zeros(n, device=dev), torch.zeros(n, device=dev))
            for c in (logq, logq_users):
                if c is not None:
                    c.bind(n)
            self._logq_stream = torch.cuda.Stream(device=dev)

    # ---- symmetric-arena path -----------------------------------------------------------------
    def _setup_symm(self, eng: TwoTowerEngine, B: int, G: int, group) -> None:
        from .symm import SymmArena
        D = eng.cfg.embedding_dim
        layout = {"flat": eng.numel * 4, "grad": eng.numel * 4, "shadow": eng.shadow.numel() * 2,
                  "U_all": G * B * D * 2, "I_all": G * B * D * 2, "uid_all": G * B * 8,
                  "lse_r_all": G * B * 4, "lse_c_all": G * B * 4, "loss_all": G * 16}
        if self.logq is not None:
            layout["tid_all"] = G * B * 8
        self.arena = a = SymmArena(layout, group, eng.device)
        eng.rebind_storage(a.view("flat", torch.float32, (eng.numel,)), a.view("grad", torch.float32, (eng.numel,)),
                           a.view("shadow", torch.bfloat16, (eng.shadow.numel(),)))
        eng.release_workspaces()
        self._loss_pad = torch.zeros(4, device=eng.device)            # 16-byte slot: [loss share, 0, 0, 0]
        n = eng.numel // G
        if eng.exp_avg is None or eng.exp_avg.numel() != n:
            eng.exp_avg = torch.zeros(n, device=eng.device)
            eng.exp_avg_sq = torch.zeros(n, device=eng.device)

    def _symm_gathered(self, ws):
        """The gathered workspace of the engine with its exchanged members living in the arena."""
        eng, a, G, B = self.eng, self.arena, self.world, self.B
        key = f"_gath{G}"
        if key not in ws:
            D, dev = eng.cfg.embedding_dim, eng.device
            Cp = (G * B + 7) // 8 * 8
            ws[key] = {
                "U_all": a.view("U_all", torch.bfloat16, (G * B, D)), "I_all": a.view("I_all", torch.bfloat16, (G * B, D)),
                "uid_all": a.view("uid_all", torch.long, (G * B,)),
                "lse_r_all": a.view("lse_r_all", torch.float32, (G * B,)),
                "lse_c_all": a.view("lse_c_all", torch.float32, (G * B,)),
                "S": torch.empty(B, Cp, device=dev)[:, :G * B], "S2": torch.empty(B, Cp, device=dev)[:, :G * B],
                "dS": torch.zeros(B, Cp, device=dev, dtype=torch.bfloat16)[:, :G * B],
                "dS2": torch.zeros(B, Cp, device=dev, dtype=torch.bfloat16)[:, :G * B],
            }
        return ws[key]

    def _phase_symm_step(self):
        """The whole data-parallel step, every exchange a kernel of this repo: capturable as ONE graph."""
        from . import ops
        eng, a = self.eng, self.arena
        # (row-sharded ID table: the owners' rows were made final by the barrier that ended the previous step's
        # optimizer kernel, so the gathers below need no barrier of their own)
        ws = self._ws = eng.forward_towers(self.static, training=True)
        g = self._symm_gathered(ws)
        uid = self.static.get("user_idx")
        # no leading barrier: the peers' last reads of these blocks (previous step's backward) precede the
        # barrier that ended the previous step's optimizer kernel
        blocks = [(ws["un_bf"], "U_all"), (ws["in_bf"], "I_all")] + ([(uid, "uid_all")] if uid is not None else [])
        if self.logq is not None:
            blocks.append((self.static["target_id"], "tid_all"))
        a.allgather(blocks)
        if self._offsets is not None:
            tid_all = a.view("tid_all", torch.long, (self.world * self.B,)) if self.logq is not None else None
            self._compute_offsets(tid_all, g["uid_all"])
        eng.loss_forward(ws, uid, gathered=g, rank=self.rank, offsets=self._offsets)
        eng.loss_value(ws, self.world * self.B)
        self._loss_pad[:1].copy_(ws["loss"].view(1))
        a.allgather([(ws["lse_r"], "lse_r_all"), (ws["lse_c"], "lse_c_all"), (self._loss_pad, "loss_all")])
        eng.backward()
        ops.step_counters_advance(eng.step_dev, eng.seed_dev)
        # one kernel: barrier (every rank's backward done, all gradient rows landed) -> reduce-scatter + AdamW +
        # all-gather of the replicated parameters and AdamW of this rank's ID-table rows -> barrier
        a.dp_adamw_step("flat", "grad", "shadow", eng.numel, eng.dense_begin, eng.exp_avg, eng.exp_avg_sq, eng.step_dev,
                        self.lr, self.betas, self.eps, self.weight_decay,
                        table_shard=None if self.table is None else self.table.shard_tensors())
        eng.grad.zero_()
        eng.shadow_valid = True

    def load_batch(self, batch: Dict[str, torch.Tensor]) -> None:
        for k, dst in self.static.items():
            dst.copy_(batch[k], non_blocking=True)

    # ---- step phases (each is graph-capturable; NCCL calls stay between the graphs) ----------
    def _compute_offsets(self, item_ids, user_ids):
        """log q of every column entity into self._offsets (item side, user side)."""
        if self.logq is not None:
            self.logq.offsets(item_ids, self._offsets[0])
        if self.logq_users is not None:
            self.logq_users.offsets(user_ids, self._offsets[1])

    def _phase_towers(self):
        if self._offsets is not None and not self.gathered:
            # local negatives: the offsets need only this batch's ids, so they run beside the towers
            main, side = torch.cuda.current_stream(), self._logq_stream
            side.wait_stream(main)
            with torch.cuda.stream(side):
                self._compute_offsets(self.static.get("target_id"), self.static.get("user_idx"))
            self._ws = self.eng.forward_towers(self.static, training=True)
            main.wait_stream(side)
            return
        self._ws = self.eng.forward_towers(self.static, training=True)

    def _phase_loss_rows(self):
        eng, ws = self.eng, self._ws
        g = eng.gathered_workspace(ws, self.world) if self.gathered else None
        if self._offsets is not None and self.gathered:
            self._compute_offsets(self._tid_all if self.logq is not None else None, g["uid_all"])
        eng.loss_forward(ws, self.static.get("user_idx"), gathered=g, rank=self.rank, offsets=self._offsets)

    def _phase_backward(self):
        if self.gathered:
            self.eng.loss_value(self._ws, self.world * self.B)
        self.eng.backward()

    def _phase_opt(self):
        if self.shard_opt:
            self.eng.adamw_step_sharded(self.rank, self.world, self._grad_shard, lr=self.lr, betas=self.betas,
                                        eps=self.eps, weight_decay=self.weight_decay)
        else:
            self.eng.adamw_step(lr=self.lr, betas=self.betas, eps=self.eps, weight_decay=self.weight_decay)

    def _phase_drop_grad(self):
        from . import ops
        self.eng.grad.zero_()
        ops.step_counters_advance(None, self.eng.seed_dev)     # dropout masks still change from step to step

    def _phase_post_opt(self):
        """After the parameter all-gather: zero the local gradient buffer, refresh the bf16 operand shadow."""
        self.eng.grad.zero_()
        self.eng.refresh_shadow()

    # -- packed all-gathers (byte views; every piece is copied by a small device-to-device copy) --
    def _phase_pack_emb(self):
        ws, D, B = self._ws, self.eng.cfg.embedding_dim, self.B
        pk = self._pack_emb
        pk[:, :2 * D].copy_(ws["un_bf"].view(torch.uint8).view(B, 2 * D))
        pk[:, 2 * D:4 * D].copy_(ws["in_bf"].view(torch.uint8).view(B, 2 * D))
        if "user_idx" in self.static:
            pk[:, 4 * D:4 * D + 8].copy_(self.static["user_idx"].view(torch.uint8).view(B, 8))
        if self.logq is not None:
            pk[:, 4 * D + 8:].copy_(self.static["target_id"].view(torch.uint8).view(B, 8))

    def _phase_unpack_emb(self):
        ws, D, B, G = self._ws, self.eng.cfg.embedding_dim, self.B, self.world
        g = self.eng.gathered_workspace(ws, G)
        pk = self._pack_emb_all
        g["U_all"].view(torch.uint8).view(G * B, 2 * D).copy_(pk[:, :2 * D])
        g["I_all"].view(torch.uint8).view(G * B, 2 * D).copy_(pk[:, 2 * D:4 * D])
        if "user_idx" in self.static:
            g["uid_all"].view(torch.uint8).view(G * B, 8).copy_(pk[:, 4 * D:4 * D + 8])
        if self.logq is not None:
            self._tid_all.view(torch.uint8).view(G * B, 8).copy_(pk[:, 4 * D + 8:])

    def _comm_embeddings(self):
        dist.all_gather_into_tensor(self._pack_emb_all, self._pack_emb, group=self.group)

    def _phase_pack_lse(self):
        ws = self._ws
        self._pack_lse[:, 0].copy_(ws["lse_r"])
        self._pack_lse[:, 1].copy_(ws["lse_c"])

    def _phase_unpack_lse(self):
        g = self.eng.gathered_workspace(self._ws, self.world)
        g["lse_r_all"].copy_(self._pack_lse_all[:, 0])
        g["lse_c_all"].copy_(self._pack_lse_all[:, 1])

    def _comm_lse(self):
        dist.all_gather_into_tensor(self._pack_lse_all, self._pack_lse, group=self.group)

    def _comm_grads(self):
        if self.shard_opt:
            dist.reduce_scatter_tensor(self._grad_shard, self.eng.grad, op=dist.ReduceOp.AVG, group=self.group)
        else:
            dist.all_reduce(self.eng.grad, op=dist.ReduceOp.AVG, group=self.group)

    def _comm_params(self):
        n = self.eng.numel // self.world
        dist.all_gather_into_tensor(self.eng.flat, self.eng.flat[self.rank * n:(self.rank + 1) * n], group=self.group)

    def _comm_lookup(self):
        rows = self.table.lookup(self.static["history_ids"].view(-1))
        self.eng.table_rows[1:].copy_(rows)

    def _comm_table_grad(self):
        g = self.eng.table_rows_grad
        self.table.backward(g[1:], scale=1.0 / self.world)      # same averaging as the dense gradient
        g.zero_()

    def _phase_table_opt(self):
        self.table.adamw_step(self.eng.step_dev, lr=self.lr, betas=self.betas, eps=self.eps,
                              weight_decay=self.weight_decay)    # step counter already advanced by the engine

    def _sequence(self):
        """[(callable, is_communication)] of one step."""
        if self.arena is not None:
            return [(self._phase_symm_step, False)]
        seq = [(self._comm_lookup, True)] if self.table is not None else []
        seq += [(self._phase_towers, False)]
        if self.gathered:
            seq += [(self._phase_pack_emb, False), (self._comm_embeddings, True), (self._phase_unpack_emb, False),
                    (self._phase_loss_rows, False), (self._phase_pack_lse, False), (self._comm_lse, True),
                    (self._phase_unpack_lse, False)]
        else:
            seq += [(self._phase_loss_rows, False)]
        seq += [(self._phase_backward, False)]
        if self.table is not None:
            seq += [(self._comm_table_grad, True)]
        if not self.with_optimizer:
            return seq + [(self._phase_drop_grad, False)]
        if self.world > 1:
            seq += [(self._comm_grads, True)]
        seq += [(self._phase_opt, False)]
        if self.table is not None:
            seq += [(self._phase_table_opt, False)]
        if self.shard_opt:
            seq += [(self._comm_params, True), (self._phase_post_opt, False)]
        return seq

    def _eager(self):
        for fn, _ in self._sequence():
            fn()

    def comm_description(self):
        """The cross-rank exchanges of one step, in order (what bench.py prints next to the timing)."""
        if self.world == 1:
            return []
        if self.arena is not None:
            how = "NVLS multicast (multimem.ld_reduce / multimem.st)" if self.arena.multicast else "peer loads / stores"
            pre = [] if self.table is None else [
                "tt_ids_dedup + tt_rows_gather / tt_rows_scatter_add: the step's distinct ID-table rows read from / "
                "combined gradient rows added into the owners' memory over NVLink (no exchange between ranks)"]
            return pre + [f"tt_symm_allgather (user emb | item emb | user id), {how}",
                    "tt_symm_allgather (row log-sum-exps of both directions | loss share)",
                    f"tt_dp_adamw_step: gradient reduce-scatter -> AdamW -> parameter + bf16 shadow all-gather in one "
                    f"kernel over {self.eng.numel * 4} B, {how}; no library collective, the step is one CUDA graph"]
        n = self.eng.numel * 4
        names = {
            "_comm_lookup": "NCCL all_to_all x3 (token ids -> owner ranks, rows back): row-sharded ID table lookup",
            "_comm_embeddings": f"NCCL all_gather_into_tensor (user emb | item emb | user id), {self._pack_emb.numel()} B/rank"
                                if self.gathered else "",
            "_comm_lse": "NCCL all_gather_into_tensor (row log-sum-exps of both directions), 8 B/sample",
            "_comm_table_grad": "NCCL all_to_all (gradient rows -> owner ranks)",
            "_comm_grads": (f"NCCL reduce_scatter_tensor AVG (flat fp32 gradient, {n} B)" if self.shard_opt
                            else f"NCCL all_reduce AVG (flat fp32 gradient, {n} B)"),
            "_comm_params": f"NCCL all_gather_into_tensor (updated fp32 parameter shards, {n} B total)",
        }
        return [names.get(fn.__name__, fn.__name__) for fn, is_comm in self._sequence() if is_comm]

    def _loss_tensor(self) -> torch.Tensor:
        return self.eng.workspace(self.B, self.L)["loss"]

    def step_resident(self) -> torch.Tensor:
        """One step on whatever is in the static buffers; returns the device loss scalar (with gathered
        negatives: this rank's share of the global loss; step_from_host sums it over ranks)."""
        self.eng.weights_epoch += 1            # a replayed graph updates the parameters without adamw_step's Python
        if not self._warm:
            c0 = _lib.launch_count
            self._eager()                      # allocates workspaces / moments, sets func attributes
            self.kernels_per_step = _lib.launch_count - c0
            self._warm = True
            torch.cuda.synchronize()
            return self._loss_tensor()
        if not self.use_graph:
            self._eager()
            return self._loss_tensor()
        if self._graphs is None:
            # consecutive compute phases are fused into one graph; communication stays eager
            plan, cur = [], []
            for fn, is_comm in self._sequence():
                if is_comm:
                    if cur:
                        plan.append(("graph", cur))
                        cur = []
                    plan.append(("comm", fn))
                else:
                    cur.append(fn)
            if cur:
                plan.append(("graph", cur))
            graphs = []
            for kind, item in plan:
                if kind == "comm":
                    item()                     # keeps the buffers consistent while capturing the rest
                    graphs.append(("comm", item))
                else:
                    g = torch.cuda.CUDAGraph()
                    # captured on a high-priority stream: the kernel nodes of the main chain inherit it, the
                    # engine's side streams (weight gradients, item tower) stay at the default priority, so
                    # the block scheduler serves the critical path first
                    if self._cap_stream is None:
                        self._cap_stream = torch.cuda.Stream(device=self.eng.device, priority=-1)
                    with torch.cuda.graph(g, stream=self._cap_stream):
                        for fn in item:
                            fn()
                    g.replay()
                    graphs.append(("graph", g))
            self._graphs = graphs
            return self._loss_tensor()
        for kind, item in self._graphs:
            if kind == "comm":
                item()
            else:
                item.replay()
        return self._loss_tensor()

    # -- double-buffered input: the NEXT batch crosses PCIe while the current step computes ----------
    def pack_host(self, batch: Dict[str, torch.Tensor]) -> torch.Tensor:
        """A batch as ONE pinned uint8 buffer in the layout of the device input buffer (a collate function
        would write this directly); `stage_batch` / `step_from_host` move it with a single copy."""
        out = torch.empty(self._static_buf.numel(), dtype=torch.uint8).pin_memory()
        for name, shape, dt, o, nb in self._fields:
            out[o:o + nb].view(dt).view(shape).copy_(batch[name])
        return out

    def stage_batch(self, host_batch) -> None:
        """Start the host->device copy of a (pinned) batch — a dict or a `pack_host` buffer — into the staging
        buffer on the copy stream. The following ``step_from_host(None)`` consumes it with one device copy."""
        if self._stage is None:
            self._stage_buf = torch.empty_like(self._static_buf)
            self._stage = {name: self._stage_buf[o:o + nb].view(dt).view(shape)
                           for name, shape, dt, o, nb in self._fields}
            self._copy_stream = torch.cuda.Stream(device=self.eng.device)
            self._staged_ev = torch.cuda.Event()
            self._consumed_ev = torch.cuda.Event()
            self._consumed_ev.record()
        self._copy_stream.wait_event(self._consumed_ev)      # the previous staged batch has been picked up
        with torch.cuda.stream(self._copy_stream):
            if isinstance(host_batch, torch.Tensor):
                self._stage_buf.copy_(host_batch, non_blocking=True)
            else:
                for k, dst in self._stage.items():
                    dst.copy_(host_batch[k], non_blocking=True)
            self._staged_ev.record()
        self._staged = True

    def step_from_host(self, host_batch, prefetch=None, defer_loss: bool = False):
        """Host batch -> device -> step -> loss on the host (one sync, like the reference's loss.item()).
        ``host_batch=None`` takes the batch announced by ``stage_batch`` / the previous call's ``prefetch``;
        ``prefetch`` (the next batch, pinned) is copied while this step runs.
        ``defer_loss=True`` pipelines the read-back: the call enqueues this step and its loss copy, then returns the
        loss of the PREVIOUS deferred step (None on the first call) — every step's loss still crosses to the host, but
        the host stays one step ahead of the GPU instead of draining it every step; `flush_loss()` returns the last one."""
        if isinstance(host_batch, torch.Tensor):
            self._static_buf.copy_(host_batch, non_blocking=True)
        elif host_batch is not None:
            self.load_batch(host_batch)
        else:
            assert self._staged, "step_from_host(None) needs a staged batch (stage_batch / prefetch=)"
            main = torch.cuda.current_stream()
            main.wait_event(self._staged_ev)
            self._static_buf.copy_(self._stage_buf, non_blocking=True)
            self._consumed_ev.record()
            self._staged = False
        loss = self.step_resident()
        if prefetch is not None:
            self.stage_batch(prefetch)
        if self.arena is None and self.gathered:
            loss = loss.clone()
            dist.all_reduce(loss, op=dist.ReduceOp.SUM, group=self.group)
        # this step's loss (and, with the NVLink arena, every rank's share + the arena's error word) -> pinned slot
        slot = self._loss_slots[self._loss_turn]
        if self.arena is not None:
            # every rank's loss share came with the log-sum-exp exchange: one small D2H, no collective
            slot["all"].copy_(self.arena.view("loss_all", torch.float32, (self.world, 4)), non_blocking=True)
            slot["err"].copy_(self.arena.error_word(), non_blocking=True)
        else:
            slot["loss"].copy_(loss, non_blocking=True)
        slot["ev"].record()
        prev = self.flush_loss()          # the previous deferred step's loss (None if nothing is pending)
        self._loss_pending = self._loss_turn
        self._loss_turn ^= 1
        if defer_loss:
            return prev
        assert prev is None, "flush_loss() before switching from deferred to immediate loss reads"
        return self.flush_loss()

    def flush_loss(self):
        """Wait for and return the loss of the most recent step whose read-back is still pending (None if none)."""
        if self._loss_pending is None:
            return None
        slot = self._loss_slots[self._loss_pending]
        self._loss_pending = None
        slot["ev"].synchronize()
        if self.arena is not None:
            if int(slot["err"][0]) != 0:
                raise RuntimeError("a cross-GPU wait timed out (peer rank missing or stalled)")
            return float(slot["all"][:, 0].sum())
        return float(slot["loss"])


def train_one_epoch(model, dataloader, optimizer, device, epoch, is_main_process=True, log_interval=50,
                    logq: Optional[LogQCorrection] = None, logq_users: Optional[LogQCorrection] = None):
    """Reference signature and return value (mean loss), src/train.py:41-76. ``logq`` / ``logq_users``: logQ
    correction of the item / user negatives (LogQCorrection; needs a FusedAdamW optimizer). A streaming estimator
    keeps its state across epochs and across the runner rebuilt for a batch of another shape."""
    model.train()
    total_loss, num_batches = 0.0, len(dataloader)
    runner: Optional[TrainStepRunner] = None
    fused = isinstance(optimizer, FusedAdamW)
    if (logq is not None or logq_users is not None) and not fused:
        raise ValueError("the logQ correction runs in the fused training step only: use a FusedAdamW optimizer")
    keys = _BATCH_KEYS + (("target_id",) if logq is not None else ())
    staged = False
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    it = iter(dataloader)
    batch = next(it, None)
    i = -1
    while batch is not None:
        i += 1
        nxt = next(it, None)
        if fused:
            B, L = batch["history_ids"].shape
            if runner is None or (runner.B, runner.L) != (B, L):
                if runner is not None:          # a loss of the previous shape's runner may still be on its way
                    pending = runner.flush_loss()
                    if pending is not None:
                        total_loss += pending
                runner = TrainStepRunner(model.engine, B, L, world_size=world, lr=optimizer.lr,
                                         betas=optimizer.betas, eps=optimizer.eps,
                                         weight_decay=optimizer.weight_decay, with_user_idx="user_idx" in batch,
                                         logq=logq, logq_users=logq_users)
                staged = False
            cur = None if staged else {k: v for k, v in batch.items() if k in keys}
            # the next batch goes over PCIe during this step when it is pinned and has the same shape
            pre = None
            if nxt is not None and tuple(nxt["history_ids"].shape) == (B, L) and \
                    all(v.is_pinned() for k, v in nxt.items() if k in keys and isinstance(v, torch.Tensor)):
                pre = {k: v for k, v in nxt.items() if k in keys}
            # the loss is read one step behind (the host enqueues step i + 1 while step i runs) except where the
            # reference logs it, so the GPU is not drained every step; every step's loss still reaches the host
            prev_loss = runner.step_from_host(cur, prefetch=pre, defer_loss=True)
            staged = pre is not None
            if prev_loss is not None:
                total_loss += prev_loss
            if (is_main_process and (i + 1) % log_interval == 0) or nxt is None:
                loss_val = runner.flush_loss()
                total_loss += loss_val
                if is_main_process and (i + 1) % log_interval == 0:
                    logger.info(f"Epoch {epoch} [{i+1}/{num_batches}] | Loss: {loss_val:.4f}")
            batch = nxt
            continue
        else:
            for k, v in batch.items():
                if isinstance(v, torch.Tensor):
                    batch[k] = v.to(device)
            optimizer.zero_grad(set_to_none=True)
            loss, _, _, _ = model(batch)
            loss.backward()
            optimizer.step()
            model.engine.shadow_valid = False     # the fp32 masters changed behind the bf16 shadow
            loss_val = loss.item()
        total_loss += loss_val
        if is_main_process and (i + 1) % log_interval == 0:
            logger.info(f"Epoch {epoch} [{i+1}/{num_batches}] | Loss: {loss_val:.4f}")
        batch = nxt
    return total_loss / max(num_batches, 1)


def evaluate(model, dataloader, device, k=10):
    """In-batch Recall@k (src/train.py:78-111): the positive must be among the k best logits of its row under the
    canonical order (logit descending, column ascending). Forward in eval mode on the CUDA engine, the rank of the
    diagonal counted by `tt_inbatch_recall` into a device (hits, total) pair — no top-k list, no per-batch host
    sync; hits / total are summed over ranks when a process group exists (:106-109) and read back once."""
    from . import ops
    model.eval()
    eng = model.engine
    if hasattr(model, "_sync_shadow"):
        model._sync_shadow()
    acc = torch.zeros(2, device=eng.device)
    with torch.no_grad():
        for batch in dataloader:
            b = model._batch(batch)
            _, logits, _, _ = eng.forward(b, training=False)
            ops.inbatch_recall(logits, 0, k, acc)
    if dist.is_available() and dist.is_initialized():
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    hits, total = acc.tolist()
    return hits / total if total > 0 else 0.0
