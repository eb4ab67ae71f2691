"""Test helper: G emulated ranks of a symmetric arena on ONE GPU.

The cross-GPU kernels of csrc/tt_symm.cu (and the team forms of tt_rows_gather / tt_rows_scatter_add) reach the
other ranks only through the pointers in ``tt_symm_team``. Here those pointers are G ordinary allocations on one
device, one per emulated rank, laid out exactly as symm.SymmArena lays out its symmetric allocation. The only
cross-rank dependency left is the epoch flags of the control blocks: ranks run their kernel of a collective one
after the other, in rank order, and before rank r's launch of collective e every ``ready`` / ``done`` slot of
rank r's own control block is stamped with e. No wait of the kernel can then spin, whatever the kernel signals,
and what it did signal is checked in the other ranks' blocks right after its launch.

``EmulatedArena``: driven by the test, one rank at a time (``run_collective``).
``ThreadedEmulatedArena``: one Python thread per rank (the real TrainStepRunner on G engine replicas); each
collective method synchronises, meets the other threads, takes its turn in rank order and meets them again, which
is what the real kernels promise when they complete (every rank's blocks visible, every peer done with mine).
"""
import threading

import torch

from mrm_b200 import symm
from mrm_b200._lib import SymmTeam, lib

# SymmCtrl (csrc/tt_symm.cu) as int32 words
EPOCH, DONE_CTAS, ERROR, READY, DONE = 0, 1, 2, 16, 32


class EmulatedWorld:
    """The shared state of G emulated ranks: which arenas belong together, and (threaded) the meeting point."""

    def __init__(self, world: int, threaded: bool = False, timeout: float = 120.0):
        assert 1 <= world <= 16
        self.world = world
        self._meet = threading.Barrier(world, timeout=timeout) if threaded else None
        self._lock = threading.Lock()
        self._made = [0] * world              # arenas constructed so far, per rank
        self._teams = {}                      # construction number -> [arena of rank 0, ...]

    def group(self, rank: int) -> "EmulatedGroup":
        return EmulatedGroup(self, rank)

    def meet(self) -> None:
        if self._meet is not None:
            self._meet.wait()

    def abort(self) -> None:
        if self._meet is not None:
            self._meet.abort()

    def register(self, arena) -> list:
        """Arena number k of every rank forms one team; its members' team pointers are filled once all have come."""
        with self._lock:
            k = self._made[arena.rank]
            self._made[arena.rank] += 1
            members = self._teams.setdefault(k, [None] * self.world)
            members[arena.rank] = arena
            if all(m is not None for m in members):
                for m in members:
                    for q, peer in enumerate(members):
                        m.team.bufs[q] = peer.buf.data_ptr()
        return members


class EmulatedGroup:
    """Stand-in for a process group handle of emulated rank ``rank``."""

    def __init__(self, world: EmulatedWorld, rank: int):
        self.world, self.rank = world, rank

    def size(self) -> int:
        return self.world.world


class EmulatedArena(symm.SymmArena):
    """symm.SymmArena over an ordinary device allocation: only the constructor differs, every method runs as
    shipped. ``group`` is an EmulatedGroup; the team pointers are complete once every rank built its arena."""

    def __init__(self, layout, group=None, device=None):
        w = group.world
        self.group = group
        self.rank, self.world = group.rank, w.world
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        self.offsets = {}
        off = 0
        for name, nbytes in layout.items():
            self.offsets[name] = (off, nbytes)
            off = symm._round_up(off + nbytes, symm._ALIGN)
        self.ctrl_offset = off
        self.nbytes = off + lib().tt_symm_ctrl_bytes()
        self.buf = torch.zeros(self.nbytes, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        self.hdl = None
        self.team = SymmTeam()
        self.team.rank, self.team.world = self.rank, self.world
        self.team.multicast = None
        self.team.ctrl_offset = self.ctrl_offset
        self.multicast = False
        self.issued = 0                       # collectives issued on this arena so far
        self.peers = w.register(self)         # every rank's arena of this team (filled in by the last to come)
        w.meet()
        self._err_host = torch.zeros(1, dtype=torch.int32).pin_memory()

    def ctrl(self) -> torch.Tensor:
        """The control block's first 48 int32 words (epoch, done_ctas, error, ..., ready[16], done[16])."""
        return self.buf[self.ctrl_offset:self.ctrl_offset + 4 * 48].view(torch.int32)


def make_team(world: int, layout, device=None):
    """G emulated arenas of one team, constructed in one thread."""
    w = EmulatedWorld(world)
    return [EmulatedArena(layout, w.group(r), device) for r in range(world)]


def pre_stamp(arena: EmulatedArena, e: int) -> None:
    """Every ready / done slot of ``arena``'s own control block at epoch e: no wait of its next kernel can spin."""
    c = arena.ctrl()
    c[READY:READY + arena.world] = e
    c[DONE:DONE + arena.world] = e


def check_signals(arenas, r: int, e: int, ready: bool) -> None:
    """Rank r's kernel of collective e stamped its slot of every other rank's control block (done, and ready when
    the collective has a leading barrier). Checked before anybody pre-stamps those blocks again."""
    for q, a in enumerate(arenas):
        if q == r:
            continue
        c = a.ctrl().cpu()
        assert int(c[DONE + r]) == e, f"rank {r} did not stamp done[{r}] = {e} into rank {q}'s block: {int(c[DONE + r])}"
        if ready:
            assert int(c[READY + r]) == e, \
                f"rank {r} did not stamp ready[{r}] = {e} into rank {q}'s block: {int(c[READY + r])}"


def check_ctrl(arena: EmulatedArena) -> None:
    """After a collective completed: the epoch counts the collectives issued, the last-CTA counter is back at 0 and
    no wait timed out."""
    c = arena.ctrl().cpu()
    assert int(c[EPOCH]) == arena.issued, (arena.rank, int(c[EPOCH]), arena.issued)
    assert int(c[DONE_CTAS]) == 0, (arena.rank, int(c[DONE_CTAS]))
    assert int(c[ERROR]) == 0, (arena.rank, int(c[ERROR]))
    assert int(arena.error_word().item()) == 0
    arena.check()


def run_collective(arenas, launch, ready: bool) -> None:
    """One collective of every emulated rank, in rank order: pre-stamp, ``launch(r)`` (which calls the arena's
    method as shipped), synchronise, check rank r's stamps; then the control-block invariants of every arena.
    ``ready``: the collective signals the ready flags too (dp_adamw, barrier, all-gather with pre_barrier)."""
    e = arenas[0].issued + 1
    assert all(a.issued + 1 == e for a in arenas)
    for r, a in enumerate(arenas):
        pre_stamp(a, e)
        launch(r)
        torch.cuda.synchronize()
        check_signals(arenas, r, e, ready)
    for a in arenas:
        a.issued = e
        check_ctrl(a)


class ThreadedEmulatedArena(EmulatedArena):
    """An EmulatedArena whose collectives are called from one thread per rank (each thread on its own stream)."""

    def _collective(self, launch, ready: bool) -> None:
        w = self.group.world
        torch.cuda.current_stream().synchronize()      # this rank's inputs are complete
        w.meet()
        e = self.issued + 1
        for turn in range(self.world):
            if turn == self.rank:
                pre_stamp(self, e)
                launch()
                torch.cuda.current_stream().synchronize()
                check_signals(self.peers, self.rank, e, ready)
            w.meet()                                   # after the last turn: every peer is done with my memory
        self.issued = e
        check_ctrl(self)

    # (super(), not symm.SymmArena: the tests put this class in symm.SymmArena's place)
    def allgather(self, blocks, pre_barrier: bool = False) -> None:
        self._collective(lambda: super(ThreadedEmulatedArena, self).allgather(blocks, pre_barrier), bool(pre_barrier))

    def barrier(self) -> None:
        self._collective(lambda: super(ThreadedEmulatedArena, self).barrier(), True)

    def dp_adamw_step(self, *args, **kwargs) -> None:
        self._collective(lambda: super(ThreadedEmulatedArena, self).dp_adamw_step(*args, **kwargs), True)


def run_ranks(world: EmulatedWorld, fn, timeout: float = 300.0):
    """fn(rank) on one thread per rank of ``world``, each with its own CUDA stream; re-raises the first failure (the
    other threads are released from their meeting point by aborting it). Returns [fn(0), ...]."""
    results, errors = [None] * world.world, []
    dev = torch.cuda.current_device()

    def body(r):
        try:
            torch.cuda.set_device(dev)
            with torch.cuda.stream(torch.cuda.Stream()):
                results[r] = fn(r)
                torch.cuda.current_stream().synchronize()
        except BaseException as exc:          # noqa: BLE001 - reported by the caller
            errors.append((r, exc))
            world.abort()

    threads = [threading.Thread(target=body, args=(r,), daemon=True) for r in range(world.world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout)
    assert not any(t.is_alive() for t in threads), "an emulated rank did not finish"
    if errors:
        errors.sort(key=lambda x: isinstance(x[1], threading.BrokenBarrierError))
        raise errors[0][1]
    return results
