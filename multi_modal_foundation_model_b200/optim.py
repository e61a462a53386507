"""Fused AdamW for the B200 path (SURVEY.md section 8f rank 1).

Drop-in for ``torch.optim.AdamW``: the reference's ``AdamW(model.parameters(), lr=..., weight_decay=..., eps=...)``
(``train_multi_modal.py:197-202``) and the fine-tuning idioms on top of it -- a subset of the parameters
(``p for p in model.parameters() if p.requires_grad``), several parameter groups with their own ``lr`` / ``betas`` /
``eps`` / ``weight_decay`` (``OneCycleLR`` with per-group ``max_lr`` keeps driving them), ``add_param_group``,
``state_dict()`` / ``load_state_dict()`` that interoperate with torch's, per-parameter step counts.

The engine keeps every parameter and gradient of the model in two flat fp32 buffers (engine.ParamStore), so one
``mmfm_adamw_multi`` launch updates all the groups: the parameters to update form segments of the flat buffers (adjacent
parameters of one class coalesced), each pointing to a class = one (group, step count) pair whose hyper-parameters
travel by value in the kernel's parameter space.  Parameters in no group, and parameters whose ``.grad`` is None, are
outside every segment and never read or written.  The segment table lives on the device and is rebuilt only when the
groups, the set of parameters with a gradient or the step classes change.  The bf16 shadow weights are refreshed by the
forward schedule's multi-tensor cast, which reads the updated masters.

There is no fallback: parameters that do not live in one engine's flat buffer raise.
"""
from __future__ import annotations

from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib, ops
from ._lib import ADAMW_CHUNK4, ADAMW_MAX_CLASSES, MmfmError


def _pad64(n: int) -> int:
    return (n + 63) // 64 * 64


def segment_table(offsets: Sequence[int], sizes: Sequence[int], cls: Sequence[Optional[int]]):
    """Segments of the flat buffers for the parameters of one store, in flat order (``offsets`` increasing, each
    parameter padded to 64 elements).  ``cls[i]`` is parameter i's class, or None when it is not updated.  Consecutive
    parameters of the same class share one segment, which then spans the zero pad between them; a segment ends at
    the last element of its last parameter.  Returns ``(segments, n_chunks)`` with ``segments`` =
    ``[(lo, hi, class, chunk0)]`` and ``chunk0`` the first work chunk of the segment (the kernel's layout)."""
    n_cls = len({c for c in cls if c is not None})
    if n_cls > ADAMW_MAX_CLASSES:
        raise MmfmError(f"{n_cls} (group, step count) classes: the fused AdamW takes at most {ADAMW_MAX_CLASSES} per "
                        "step (parameters of one group whose step counts drifted apart through skipped steps form one "
                        "class each)")
    segs: List[List[int]] = []
    prev = None
    for i, (o, n, c) in enumerate(zip(offsets, sizes, cls)):
        if c is None:
            prev = None
            continue
        if o % 4:
            raise MmfmError(f"parameter at flat offset {o} is not 16-byte aligned")
        if prev is not None and prev == c and offsets[i - 1] + _pad64(sizes[i - 1]) == o:
            segs[-1][1] = o + n
        else:
            segs.append([o, o + n, c, 0])
        prev = c
    chunk = 0
    for s in segs:
        s[3] = chunk
        chunk += max(1, -(-((s[1] >> 2) - (s[0] >> 2)) // ADAMW_CHUNK4))
    return [tuple(s) for s in segs], chunk


class AdamW(torch.optim.Optimizer):
    def __init__(self, params: Iterable, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 1e-2, amsgrad: bool = False, *, maximize: bool = False, **unused):
        if amsgrad or maximize:
            raise NotImplementedError("the fused AdamW implements amsgrad=False, maximize=False")
        self._store = None
        self._m: Optional[torch.Tensor] = None
        self._v: Optional[torch.Tensor] = None
        self._steps: Optional[torch.Tensor] = None     # per-parameter step counts (store order); state 'step' views
        self._gsig = None        # group structure the entries below were built for
        self._entries: List[Tuple[int, int, torch.nn.Parameter, torch.Tensor]] = []   # (group, store pos, p, grad view)
        self._key = None         # active pattern the segment table was built for
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    def add_param_group(self, param_group):
        if torch.is_tensor(param_group.get("lr", self.defaults.get("lr"))):
            raise NotImplementedError("the fused AdamW takes a float lr (a tensor lr is not supported)")
        super().add_param_group(param_group)

    # -----------------------------------------------------------------------------------------------------
    def _bind(self):
        """Locate the engine store that owns the parameters (created lazily by the first forward pass)."""
        from .engine import live_stores
        p0 = self.param_groups[0]["params"][0]
        for st in live_stores():
            if not st.adopted():
                st.adopt()
            lo, hi = st.flat.data_ptr(), st.flat.data_ptr() + st.flat.numel() * 4
            if lo <= p0.data_ptr() < hi:
                self._store = st
                self._pos = {id(q): i for i, q in enumerate(st.params.values())}
                self._names = list(st.params)
                self._m = torch.zeros_like(st.flat)
                self._v = torch.zeros_like(st.flat)
                st.moments.update((self._m, self._v))      # the engine's plan sizing no longer reserves room for them
                self._steps = torch.zeros(len(self._names), dtype=torch.float32)
                return
        raise MmfmError("parameters are not owned by a B200 engine: move the model to CUDA and run one forward pass "
                        "(model(mod_dict)) before optimizer.step(); there is no fallback optimizer")

    def _home(self, p, i: int) -> None:
        """torch-style per-parameter state as views: moments of the flat buffers, step of the step-count tensor;
        state already there (load_state_dict) is copied in."""
        st, n = self._store, self._names[i]
        m, v = st.view(self._m, n), st.view(self._v, n)
        s = self.state.get(p)
        if s and "exp_avg" in s:
            m.copy_(s["exp_avg"])
            v.copy_(s["exp_avg_sq"])
            self._steps[i] = float(s["step"])
        else:
            m.zero_()
            v.zero_()
            self._steps[i] = 0.0
        self.state[p] = {"step": self._steps[i], "exp_avg": m, "exp_avg_sq": v}

    def _layout(self, gsig) -> None:
        st = self._store
        gv = st.grad_views()
        entries = []
        for gi, g in enumerate(self.param_groups):
            for p in g["params"]:
                i = self._pos.get(id(p))
                if i is None:
                    raise MmfmError("every parameter of the fused AdamW must live in the flat buffer of ONE engine: "
                                    "foreign parameters and parameters of two engines are not supported")
                s = self.state.get(p)
                if not (s and s.get("exp_avg") is not None and s["exp_avg"].data_ptr() == st.view(self._m,
                                                                                             self._names[i]).data_ptr()):
                    self._home(p, i)
                entries.append((gi, i, p, gv[self._names[i]]))
        self._entries, self._gsig, self._key = entries, gsig, None

    def _rebuild(self, key) -> None:
        """Segment table + classes for the parameters that have a gradient this step."""
        st = self._store
        steps = self._steps.tolist()
        cls: List[Optional[int]] = [None] * len(self._names)
        classes = {}
        for (gi, i, _, _), a in zip(self._entries, key):
            if a:
                cls[i] = classes.setdefault((gi, int(steps[i]) + 1), len(classes))
        segs, n_chunks = segment_table([st.offset[n] for n in self._names],
                                       [st.shape[n].numel() for n in self._names], cls)
        self._classes = sorted(classes, key=classes.get)        # [(group, step after this update)]
        self._n_segs, self._n_chunks = len(segs), n_chunks
        self._n_elems = sum(hi - lo for lo, hi, _, _ in segs)
        if segs:
            arr = (_lib.AdamwSeg * len(segs))(*[_lib.AdamwSeg(*s) for s in segs])
            # pageable source: the copy has completed when .to() returns, so nothing is left in flight
            self._segs_dev = torch.from_numpy(np.frombuffer(bytes(arr), dtype=np.uint8).copy()).to(st.device)
        act = [i for (_, i, _, _), a in zip(self._entries, key) if a]
        self._all_active = len(act) == len(self._names)
        self._active = torch.tensor(act, dtype=torch.long)
        self._ones = torch.ones(len(act))
        self._key = key

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if self._store is None:
            self._bind()
        st = self._store
        if not st.adopted():
            st.adopt()
        gsig = tuple((id(g["params"]), len(g["params"])) for g in self.param_groups)
        if gsig != self._gsig:
            self._layout(gsig)
        # gradients must be the flat buffer's views (engine.backward installs them); anything else is copied in.
        # A parameter without a gradient is skipped as by torch.optim.AdamW: weights, moments and step stay.
        key = []
        for _, _, p, v in self._entries:
            gr = p.grad
            if gr is None:
                key.append(False)
                continue
            if gr is not v:
                v.copy_(gr)
            key.append(True)
        key = tuple(key)
        if key != self._key:
            self._rebuild(key)
        if not self._classes:
            return loss
        classes = []
        for gi, s in self._classes:
            g = self.param_groups[gi]
            if torch.is_tensor(g["lr"]):
                raise NotImplementedError("the fused AdamW takes a float lr (a tensor lr is not supported)")
            if g.get("amsgrad") or g.get("maximize"):
                raise NotImplementedError("the fused AdamW implements amsgrad=False, maximize=False")
            b1, b2 = g["betas"]
            classes.append(_lib.AdamwClass(float(g["lr"]), float(b1), float(b2), float(g["eps"]),
                                           float(g["weight_decay"]), 0, s))
        ops.adamw_multi(st.flat, st.grad, self._m, self._v, self._segs_dev, self._n_segs, self._n_chunks, classes,
                        self._n_elems)
        if self._all_active:
            self._steps += 1
        else:
            self._steps.index_add_(0, self._active, self._ones)
        self._classes = [(gi, s + 1) for gi, s in self._classes]
        return loss

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        if self._store is not None:          # re-home the loaded state into the flat moments and the step tensor
            for g in self.param_groups:
                for p in g["params"]:
                    i = self._pos.get(id(p))
                    if i is not None:
                        self._home(p, i)
        self._gsig = self._key = None
