"""Data parallelism over the GPUs of one box: one process per GPU, trials sharded by rank, gradients averaged with
NCCL all-reduce over NVLink 5 / NVSwitch, overlapped with the backward pass.

The reference has no working data-parallel path (SURVEY.md section 2.1: only the model is passed to
``accelerator.prepare``); what it *would* do under ``accelerate launch`` is DistributedDataParallel: bucketed
``ncclAllReduce(SUM) / world``.  This module implements exactly that semantics on the engine's flat gradient buffer:
the buffer is laid out in reverse execution order, so a bucket is a contiguous range that is final as soon as the
backward schedule passes the matching mark; its all-reduce is enqueued right there and runs on NCCL's stream while
the remaining backward kernels run on the compute stream.

Bucket plan and partitioning are pure host logic (tested on CPU with the gloo backend, world size 2).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def shard_range(n_trials: int, rank: int, world: int) -> Tuple[int, int]:
    """Trials [lo, hi) of a global batch that rank ``rank`` processes (contiguous, balanced)."""
    base, rem = divmod(n_trials, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def plan_buckets(marks: Sequence[Tuple[int, int]], total: int, target_elems: int) -> List[Tuple[int, int, int]]:
    """Group the backward schedule's completion marks into buckets.

    ``marks`` = [(call_index, grad_offset)], increasing in both: after call ``call_index`` of the backward
    schedule every gradient element below ``grad_offset`` is final.  Returns [(call_index, lo, hi)]: all-reduce
    range [lo, hi) after ``call_index`` calls.  Buckets are at least ``target_elems`` long except the last."""
    out: List[Tuple[int, int, int]] = []
    lo = 0
    for ci, off in marks:
        if off - lo >= target_elems and off < total:
            out.append((ci, lo, off))
            lo = off
    last_call = marks[-1][0] if marks else 0
    out.append((last_call, lo, total))
    return out


def core_buckets(marks: Sequence[Tuple[int, int]], core: Tuple[int, int], target_elems: int
                 ) -> List[Tuple[int, int, int]]:
    """plan_buckets over the shared core [lo, hi) of a multi-session flat gradient only: the marks clipped to that
    span.  The core parameters and their marks' offsets are the same for every session, so every session's plan
    gets the same ranges (its call indices may differ)."""
    lo, hi = core
    clipped = [(ci, min(max(off, lo), hi) - lo) for ci, off in marks]
    return [(ci, a + lo, b + lo) for ci, a, b in plan_buckets(clipped, hi - lo, target_elems)]


def all_reduce_mean(t: torch.Tensor, group=None, async_op: bool = False):
    """Mean over ranks, in place (DDP semantics).  NCCL averages inside the collective; gloo (CPU tests) sums and
    divides."""
    if dist.get_backend(group) == "nccl":
        return dist.all_reduce(t, op=dist.ReduceOp.AVG, group=group, async_op=async_op)
    w = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group, async_op=False)
    t.div_(dist.get_world_size(group))
    return w


class SessionExchange:
    """Session gradients of a multi-session model under data parallelism, where every rank may run another session.

    Only the shared core goes through the all-reduce buckets.  A rank's own session gradient (its head range and its
    embedder range of the flat gradient) travels as two fixed-size all-gathers instead: the head slab, padded to the
    widest session's head range, and the embedder slab, padded likewise; the session ids travel with the head slab.
    The sizes depend on the engine only, so every rank issues the same collectives with the same counts in the same
    order, whichever session it ran, and plans of different sessions can be captured and replayed side by side.
    mmfm_session_grad_combine then writes, on every rank alike, the rank mean of each session some rank ran; the
    ranges of the other sessions keep the zero the backward left there."""

    def __init__(self, store, world: int, group=None):
        dev = store.device
        self.world, self.pg = world, group
        self.ranges = store.session_ranges
        self.head_len = max(h1 - h0 for h0, h1, _, _ in self.ranges)
        self.emb_len = max(e1 - e0 for _, _, e0, e1 in self.ranges)
        # the combine kernel's range tables: one range per session each (the second one empty)
        self.head_tab = torch.tensor([[h0, h1, 0, 0] for h0, h1, _, _ in self.ranges], dtype=torch.int64, device=dev)
        self.emb_tab = torch.tensor([[e0, e1, 0, 0] for _, _, e0, e1 in self.ranges], dtype=torch.int64, device=dev)
        self.ids = torch.zeros(world, dtype=torch.int32, device=dev)
        self.send_head = torch.zeros(self.head_len, device=dev)
        self.send_emb = torch.zeros(self.emb_len, device=dev)
        self.recv_head = torch.zeros(world, self.head_len, device=dev)
        self.recv_emb = torch.zeros(world, self.emb_len, device=dev)

    def bytes_per_step(self) -> Tuple[int, int]:
        """(sent, received) bytes of one rank's session exchange per step (ids included)."""
        n = 4 * (1 + self.head_len + self.emb_len)
        return n, n * self.world

    def _send(self, pl, grad: torch.Tensor, lo: int, hi: int, send: torch.Tensor, recv: torch.Tensor):
        from . import ops
        ops.scale_inplace(grad[lo:hi], pl.gscale)
        send[:hi - lo].copy_(grad[lo:hi])                 # cudaMemcpyAsync; the pad past hi - lo is never read
        return dist.all_gather_into_tensor(recv.view(-1), send, group=self.pg, async_op=True)

    def send_heads(self, pl, grad: torch.Tensor) -> list:
        """Enqueued once the head wgrads are done: the ids and the head slab."""
        h0, h1, _, _ = self.ranges[pl.session_index]
        return [dist.all_gather_into_tensor(self.ids, pl.session_id, group=self.pg, async_op=True),
                self._send(pl, grad, h0, h1, self.send_head, self.recv_head)]

    def send_embedders(self, pl, grad: torch.Tensor) -> list:
        """Enqueued after the last embedder launch: the embedder slab."""
        _, _, e0, e1 = self.ranges[pl.session_index]
        return [self._send(pl, grad, e0, e1, self.send_emb, self.recv_emb)]

    def combine(self, grad: torch.Tensor) -> None:
        """After the gathers are waited for: every ran session's ranges = the rank mean of its gathered slabs."""
        from . import ops
        ops.session_grad_combine(grad, self.recv_head, self.ids, self.head_tab, 1.0 / self.world)
        ops.session_grad_combine(grad, self.recv_emb, self.ids, self.emb_tab, 1.0 / self.world)


class DataParallel:
    """Attach to a ``MultiModal`` (B200 path) so that ``loss.backward()`` leaves rank-averaged gradients in
    ``Parameter.grad`` -- DDP semantics (mean over ranks of the per-rank gradients, SURVEY.md section 8e).

    A ``MultiSessionMultiModal`` rank may feed any session in any step: the shared core is all-reduced in buckets and
    the session gradients go through a SessionExchange, so each session's gradient is the sum of the gradients of the
    ranks that ran it, over the world size, and a session no rank ran stays zero."""

    xchg: Optional[SessionExchange] = None       # set for a multi-session model on more than one rank

    def __init__(self, model, process_group=None, bucket_mb: float = 8.0, broadcast: bool = True):
        self.model = model
        self.pg = process_group
        self.world = dist.get_world_size(process_group)
        self.rank = dist.get_rank(process_group)
        self.bucket_elems = int(bucket_mb * 1024 * 1024 / 4)
        eng = model.engine()
        eng.ddp = self
        self.eng = eng
        multi = eng.store.session_ranges is not None and self.world > 1
        self.xchg = SessionExchange(eng.store, self.world, process_group) if multi else None
        if broadcast and self.world > 1:
            dist.broadcast(eng.store.flat, src=0, group=process_group)   # same initial weights on every rank
        self._graphs = []            # per-plan capture states (held here only so close() can drop the graphs)
        import atexit
        import os
        import weakref
        self.graph_ddp = os.environ.get("MMFM_DDP_GRAPH", "1") != "0"
        # captured graphs hold NCCL work: they must be gone before the process group is torn down.  Call close() before
        # dist.destroy_process_group(); the exit hook covers a plain interpreter exit.
        ref = weakref.ref(self)
        atexit.register(lambda: ref() is not None and ref().close())

    def close(self) -> None:
        """Drop the captured graphs (they hold NCCL work) -- call before ``destroy_process_group``."""
        if not any(st["graph"] is not None for st in self._graphs):
            return
        torch.cuda.synchronize()
        for st in self._graphs:
            st["graph"] = None
            st["runs"] = 0
        import gc
        gc.collect()
        torch.cuda.synchronize()

    def _segments(self, pl):
        """(skipped wgrad calls, (backward call list, n_calls, buckets, tail)) for the plan's current frozen set
        (engine.Plan.backward_schedule)."""
        skip, calls, grad_marks = pl.backward_schedule()
        # cached on the plan object itself (an id()-keyed table could hand a new plan the entry of a freed one)
        cache = pl.__dict__.setdefault("_ddp_segments", {})
        seg = cache.get(skip)
        if seg is None:
            # the whole-buffer scale right after the last mark is replaced by per-bucket scaling before each
            # all-reduce; calls after it (input gradients, no parameter gradient) run once the buckets are enqueued
            n_calls = grad_marks[-1][0] if grad_marks else len(calls)
            tail = n_calls + 1 if n_calls < len(calls) and calls[n_calls][2] == "mmfm_scale_inplace" else n_calls
            marks = [(min(ci, n_calls), off) for ci, off in grad_marks]
            if self.xchg is None:
                buckets = plan_buckets(marks, self.eng.store.total, self.bucket_elems)
            else:
                buckets = core_buckets(marks, self.eng.store.core_range, self.bucket_elems)
            seg = cache[skip] = (calls, n_calls, buckets, tail)
        return skip, seg

    def run_backward(self, pl) -> None:
        """Backward schedule with the bucket all-reduces enqueued at their completion marks.  The first call per plan
        runs eagerly (NCCL communicator set-up, kernel attributes); afterwards the whole sequence -- kernels, per-bucket
        scaling and the NCCL all-reduces on their side stream -- is captured once into a CUDA graph and replayed, so the
        multi-GPU step has the same launch-gap-free backward as the single-GPU one."""
        skip, _ = self._segments(pl)
        graphs = pl.__dict__.setdefault("_ddp_graph", {})       # one per frozen set
        st = graphs.get(skip)
        if st is None:
            st = graphs[skip] = {"runs": 0, "graph": None}
            self._graphs.append(st)
        if self.eng.use_graphs and self.graph_ddp and st["graph"] is None and st["runs"] >= 1 and self.world > 1:
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._run_backward_eager(pl)
                st["graph"] = g
            except Exception:          # capture of collectives unsupported in this build: stay eager, loudly once
                import warnings
                warnings.warn("mmfm DataParallel: CUDA-graph capture of the backward + all-reduce failed; running eagerly")
                self.graph_ddp = False
                torch.cuda.synchronize()
        st["runs"] += 1
        if st["graph"] is not None:
            st["graph"].replay()
        else:
            self._run_backward_eager(pl)

    def _run_backward_eager(self, pl) -> None:
        from . import ops
        _, (calls, n_calls, buckets, tail) = self._segments(pl)
        grad = self.eng.store.grad
        grad.zero_()
        works = []
        done = 0
        xchg = self.xchg
        if xchg is not None:
            # at the first gradient mark, after the last decoder layer: the heads are final from there on
            done = min(pl.backward_schedule()[2][0][0], n_calls)
            ops.run_recorded(calls[:done])
            works += xchg.send_heads(pl, grad)
        for ci, lo, hi in buckets:
            if ci > done:
                ops.run_recorded(calls[done:ci])
                done = ci
            view = grad[lo:hi]
            ops.scale_inplace(view, pl.gscale)
            if self.world > 1:
                works.append(all_reduce_mean(view, self.pg, async_op=True))
        assert done == n_calls, "bucket plan must end at the end of the backward schedule"
        if xchg is not None:       # right behind the last core bucket, after the last embedder launch
            works += xchg.send_embedders(pl, grad)
        if tail < len(calls):
            ops.run_recorded(calls[tail:])
        for w in works:
            if w is not None:
                w.wait()
        if xchg is not None:
            xchg.combine(grad)
