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


def all_reduce_mean(t: torch.Tensor, group=None, async_op: bool = False):
    """Mean over ranks, in place (DDP semantics).  NCCL averages inside the collective; gloo (CPU tests) sums and
    divides."""
    if dist.get_backend(group) == "nccl":
        return dist.all_reduce(t, op=dist.ReduceOp.AVG, group=group, async_op=async_op)
    w = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group, async_op=False)
    t.div_(dist.get_world_size(group))
    return w


class DataParallel:
    """Attach to a ``MultiModal`` (B200 path) so that ``loss.backward()`` leaves rank-averaged gradients in
    ``Parameter.grad`` -- DDP semantics (mean over ranks of the per-rank gradients, SURVEY.md section 8e)."""

    def __init__(self, model, process_group=None, bucket_mb: float = 8.0, broadcast: bool = True):
        self.model = model
        self.pg = process_group
        self.world = dist.get_world_size(process_group)
        self.rank = dist.get_rank(process_group)
        self.bucket_elems = int(bucket_mb * 1024 * 1024 / 4)
        eng = model.engine()
        eng.ddp = self
        self.eng = eng
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
            buckets = plan_buckets(marks, self.eng.store.total, self.bucket_elems)
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
        for ci, lo, hi in buckets:
            if ci > done:
                ops.run_recorded(calls[done:ci])
                done = ci
            view = grad[lo:hi]
            ops.scale_inplace(view, pl.gscale)
            if self.world > 1:
                works.append(all_reduce_mean(view, self.pg, async_op=True))
        assert done == n_calls, "bucket plan must end at the end of the backward schedule"
        if tail < len(calls):
            ops.run_recorded(calls[tail:])
        for w in works:
            if w is not None:
                w.wait()
