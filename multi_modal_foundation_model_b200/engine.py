"""Step engine: the forward + backward pass of ``MultiModal`` (reference mm.py:242-308 + autograd of
trainer/base.py:194-195) as a pre-bound schedule of sm_100a kernel launches through the C ABI.

Data layout in HBM (all buffers are torch tensors owned by the plan; the library allocates nothing):
  * tokens of all modalities live in ONE packed residual stream (B, S = n_mod*T, H) fp32 -- the torch.cat of
    mm.py:98-108 never happens: the embedding GEMM epilogue writes modality k at token offset k*T;
  * every GEMM operand is bf16 (activations produced in bf16 by the LayerNorm / GEMM epilogues; weights shadowed in
    bf16 -- natural and transposed -- by one multi-tensor cast per step from the fp32 master parameters);
  * master parameters and gradients are two flat fp32 buffers with identical offsets, ordered in reverse execution
    order so that data-parallel gradient buckets are contiguous ranges that complete early in the backward;
    ``Parameter.data`` / ``Parameter.grad`` are views into them (the optimizer keeps working on the same objects).

There is no PyTorch fallback: every arithmetic step is a kernel of libmmfm_b200.so.
"""
from __future__ import annotations

import ctypes as C
import os
import warnings
import weakref
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import adapter, masker as _masker, ops
from ._lib import (ACT_DSOFTSIGN, ACT_GELU, ACT_GELU_DG, ACT_MULAUX, ACT_NONE, ACT_ROWDOT_DROP, ACT_SOFTSIGN, LOSS_CE, LOSS_MSE, LOSS_POISSON, MASK_CAUSAL,
                   MASK_KEY, MASK_KEY_OR_DIAG, MAX_LN, CastItem, MmfmError, lib)
from .ops import NO_DROP, DropSpec

bf16 = torch.bfloat16
SMALL_C = 8

# dropout site ids -- must match oracle/philox_ref.py
SITE_EMBED, SITE_ATTN_PROB, SITE_ATTN_OUT, SITE_XATTN_PROB, SITE_XATTN_OUT, SITE_MLP = 0, 1, 2, 3, 4, 5
SIDE_ENC, SIDE_DEC = 0, 1


def site_id(kind: int, layer: int, side: int) -> int:
    return kind + 16 * layer + 4096 * side


def _pad(n: int, m: int = 8) -> int:
    return (n + m - 1) // m * m


class ModSpec:
    def __init__(self, name: str, index: int, channels: int, loss_kind: str):
        self.name, self.index, self.C = name, index, channels
        if loss_kind not in ("poisson", "mse", "ce"):
            raise NotImplementedError(f"loss kind {loss_kind!r} of modality {name!r}")
        self.loss_kind = {"poisson": LOSS_POISSON, "mse": LOSS_MSE, "ce": LOSS_CE}[loss_kind]
        self.small = channels <= SMALL_C


_STORES = weakref.WeakSet()


def embedding_groups(model):
    """[(parameter-name prefix, encoder_embeddings, decoder_embeddings)]: one group for the reference's single-session
    model, one per session for model.MultiSessionMultiModal (BASELINE configs[3])."""
    sess = getattr(model, "session_embeddings", None)
    if sess is None:
        return [("", model.encoder_embeddings, model.decoder_embeddings)]
    return [(f"session_embeddings.{k}.", v["encoder_embeddings"], v["decoder_embeddings"]) for k, v in sess.items()]


def live_stores():
    """Flat parameter stores of the engines alive in this process (optim.AdamW finds its parameters' owner here)."""
    return list(_STORES)


def fuse_context_norms(named, n_dec: int) -> bool:
    """The `context_norm` of every decoder layer normalises the same encoder context (decoder_embeddings.py:141-145):
    one launch computes all of them from one read of the context (mmfm_layernorm_fwd_multi), and one backward launch
    normalises the gamma-weighted sum of their upstream gradients (mmfm_layernorm_bwd_multi) instead of n passes over the
    context with n read-modify-writes of its gradient.  Their gamma / beta gradients then become final after the LAST
    decoder layer of the backward, so they move behind the decoder layers in the flat gradient order.
    ScaleNorm, widths the fused kernels do not take and more than MAX_LN decoder layers keep the per-layer kernels."""
    if n_dec < 2 or n_dec > MAX_LN:
        return False
    w = named.get("decoder.0.context_norm.weight")
    if w is None:
        return False
    H = w.numel()
    return H in (128, 256, 512) and (H // 128) * n_dec <= 12


def memory_for_plan(free: int, total: int, reserved: int, allocated: int, fraction: float, margin: int) -> int:
    """Bytes a new plan may take: what torch's caching allocator can still obtain from the device without exceeding its
    per-process memory fraction, plus what it holds unused, less ``margin`` (the step's own allocations)."""
    return min(free, int(fraction * total) - reserved) + (reserved - allocated) - margin


def step_margin(transient: int, flat_bytes: int, moments: bool) -> int:
    """Device bytes a training step allocates besides its plan: the output / input-gradient tensors (``transient``),
    the flat-gradient copy of gradient accumulation and, until the fused AdamW has allocated them at its first step,
    its two moment buffers."""
    return transient + flat_bytes + (0 if moments else 2 * flat_bytes)


def _round_alloc(n: int) -> int:
    return (n + 511) // 512 * 512          # the caching allocator's block granularity


def flat_layout(order: Sequence[str], named) -> Tuple[Dict[str, str], Dict[str, int], Dict[str, torch.Size], int]:
    """(alias, offset, shape, total) of the flat buffers: parameters in ``order``, each at a 64-element aligned offset;
    a parameter met again under another name (shared mod_emb) is an alias of the first name."""
    uniq: Dict[int, str] = {}
    alias: Dict[str, str] = {}
    offset: Dict[str, int] = {}
    shape: Dict[str, torch.Size] = {}
    off = 0
    for name in order:
        p = named[name]
        if id(p) in uniq:
            alias[name] = uniq[id(p)]
            continue
        uniq[id(p)] = name
        alias[name] = name
        offset[name] = off
        shape[name] = p.shape
        off += _pad(p.numel(), 64)
    return alias, offset, shape, off


def session_ranges(offset: Dict[str, int], shape: Dict[str, torch.Size], prefixes: Sequence[str]
                   ) -> Tuple[Tuple[int, int], List[Tuple[int, int, int, int]]]:
    """((core_lo, core_hi), [(head_lo, head_hi, emb_lo, emb_hi)] per session prefix) of a multi-session flat layout.

    A session's heads are its ``decoder_embeddings.<m>.out`` parameters, its embedders the rest of its prefix; the shared
    core is every parameter outside all prefixes.  Each range covers its parameters and their pads exactly, starts and
    ends on the 64-element pad (16-byte aligned), and no session range overlaps the core or another session's."""
    def span(names, what):
        names = sorted(names, key=offset.__getitem__)
        if not names:
            raise MmfmError(f"empty {what} range")
        lo = offset[names[0]]
        hi = lo
        for n in names:       # contiguous: each parameter starts where the previous one's pad ends
            if offset[n] != hi:
                raise MmfmError(f"{what} range is not contiguous at {n}")
            hi += _pad(shape[n].numel(), 64)
        assert lo % 64 == 0 and hi % 64 == 0
        return lo, hi

    owned = set()
    out = []
    for prefix in prefixes:
        mine = [n for n in offset if n.startswith(prefix)]
        parts = {n: n[len(prefix):].split(".") for n in mine}        # decoder_embeddings.<m>.out.<weight|bias>
        heads = [n for n in mine if parts[n][0] == "decoder_embeddings" and parts[n][2] == "out"]
        h = span(heads, f"{prefix} head")
        e = span([n for n in mine if n not in heads], f"{prefix} embedder")
        out.append(h + e)
        owned.update(mine)
    core = span([n for n in offset if n not in owned], "shared core")
    spans = sorted([(lo, hi) for r in out for lo, hi in (r[:2], r[2:])] + [core])
    for (_, hi0), (lo1, _) in zip(spans, spans[1:]):
        if lo1 < hi0:
            raise MmfmError("session ranges overlap each other or the shared core")
    return core, out


# ------------------------------------------------------------------------------------------------------------
class ParamStore:
    """Flat fp32 master-parameter and gradient buffers + bf16 shadows."""

    def __init__(self, model, device):
        _STORES.add(self)
        self.device = device
        named = dict(model.named_parameters(remove_duplicate=False))
        order = self._execution_reverse_order(model, named)
        # alias: name -> canonical name (shared mod_emb)
        self.alias, self.offset, self.shape, off = flat_layout(order, named)
        missing = set(named) - set(order)
        if missing:
            raise MmfmError(f"parameters outside the step schedule: {sorted(missing)[:5]} ...")
        self.total = off
        # multi-session model: the shared core's range and, per session (in embedding_groups order), its head and
        # embedder ranges (the data-parallel session exchange); None for the single-session model
        self.core_range: Optional[Tuple[int, int]] = None
        self.session_ranges: Optional[List[Tuple[int, int, int, int]]] = None
        if getattr(model, "session_embeddings", None) is not None:
            self.core_range, self.session_ranges = session_ranges(
                self.offset, self.shape, [prefix for prefix, _, _ in embedding_groups(model)])
        self.flat = torch.zeros(off, device=device, dtype=torch.float32)
        self.grad = torch.zeros(off, device=device, dtype=torch.float32)
        self.params = {n: named[n] for n in self.offset}
        self.bucket_order = [n for n in order if self.alias[n] == n]
        self._grad_views: Optional[Dict[str, torch.Tensor]] = None
        self.moments: "weakref.WeakSet[torch.Tensor]" = weakref.WeakSet()    # optim.AdamW's moment buffers, once bound
        self.adopt()

    @staticmethod
    def _execution_reverse_order(model, named) -> List[str]:
        def lin(prefix):
            # Linear / LayerNorm: weight + bias; ScaleNorm (use_scalenorm, mm_utils.py:31-39): one scalar `scale`
            return [f"{prefix}.weight", f"{prefix}.bias", f"{prefix}.scale"]

        def attn(prefix, fused_q: bool):
            o = lin(f"{prefix}.out_proj")
            if fused_q:
                w = [f"{prefix}.{k}.weight" for k in ("query", "key", "value")]
                b = [f"{prefix}.{k}.bias" for k in ("query", "key", "value")]
            else:  # cross attention: key/value fused, query apart
                w = [f"{prefix}.key.weight", f"{prefix}.value.weight", f"{prefix}.query.weight"]
                b = [f"{prefix}.key.bias", f"{prefix}.value.bias", f"{prefix}.query.bias"]
            return o + w + b

        groups = embedding_groups(model)
        order: List[str] = []
        for prefix, _, dec in reversed(groups):
            for m in reversed(list(dec.keys())):
                order += lin(f"{prefix}decoder_embeddings.{m}.out")
        order += lin("decoder_norm")
        fuse_ctx = fuse_context_norms(named, model.n_dec_layers)
        for i in reversed(range(model.n_dec_layers)):
            p = f"decoder.{i}"
            order += lin(f"{p}.mlp.down_proj") + lin(f"{p}.mlp.up_proj") + lin(f"{p}.ln2")
            order += attn(f"{p}.cross_attn", False) + ([] if fuse_ctx else lin(f"{p}.context_norm")) + lin(f"{p}.query_norm")
            order += attn(f"{p}.attn", True) + lin(f"{p}.ln1")
        if fuse_ctx:   # their gradients come out of ONE launch after the last decoder layer of the backward
            for i in reversed(range(model.n_dec_layers)):
                order += lin(f"decoder.{i}.context_norm")
        order += lin("decoder_proj_context") + lin("encoder_norm")
        for i in reversed(range(model.n_enc_layers)):
            p = f"encoder.{i}"
            order += lin(f"{p}.mlp.down_proj") + lin(f"{p}.mlp.up_proj") + lin(f"{p}.ln2")
            order += attn(f"{p}.attn", True) + lin(f"{p}.ln1")
        for prefix, enc, dec in reversed(groups):
            for side, md in (("decoder_embeddings", dec), ("encoder_embeddings", enc)):
                for m in reversed(list(md.keys())):
                    p = f"{prefix}{side}.{m}.embedder"
                    order += lin(f"{p}.projection") + lin(f"{p}.token_embed") + [f"{p}.pos_embed.weight",
                                                                                  f"{p}.mod_emb.weight"]
        return [n for n in order if n in named]

    def view(self, buf: torch.Tensor, name: str) -> torch.Tensor:
        name = self.alias[name]
        o = self.offset[name]
        shp = self.shape[name]
        return buf[o:o + shp.numel()].view(shp)

    def has(self, name: str) -> bool:
        return name in self.alias

    def p(self, name: str) -> torch.Tensor:
        return self.view(self.flat, name)

    def g(self, name: str) -> torch.Tensor:
        return self.view(self.grad, name)

    def grad_views(self) -> Dict[str, torch.Tensor]:
        """One gradient view per parameter, the same objects every call: engine.backward installs them as
        ``Parameter.grad`` and optim.AdamW recognises them by identity."""
        if self._grad_views is None:
            self._grad_views = {n: self.g(n) for n in self.params}
        return self._grad_views

    def adopted(self) -> bool:
        for n in (self.bucket_order[0], self.bucket_order[-1]):
            if self.params[n].data_ptr() != self.p(n).data_ptr():
                return False
        return True

    @torch.inference_mode(False)
    @torch.no_grad()
    def adopt(self) -> None:
        """Re-home every Parameter's storage into the flat buffer (values preserved)."""
        for n, p in self.params.items():
            v = self.p(n)
            if p.data_ptr() != v.data_ptr():
                v.copy_(p.data.to(self.device, torch.float32))
                p.data = v


# ------------------------------------------------------------------------------------------------------------
class Shadows:
    """bf16 copies (natural and transposed) of the GEMM weights, refreshed by one multi-tensor cast launch."""

    def __init__(self, store: ParamStore, model, sessions: Dict[Any, Tuple[str, List[ModSpec]]]):
        dev = store.device
        self.nat: Dict[str, torch.Tensor] = {}
        self.tr: Dict[str, torch.Tensor] = {}
        items: List[CastItem] = []
        tile = 0

        def add(key: str, names: List[str], want_t: bool = True):
            nonlocal tile
            ws = [store.p(n) for n in names]
            rows = sum(w.shape[0] for w in ws)
            cols = ws[0].shape[1]
            nat = torch.zeros(rows, _pad(cols), device=dev, dtype=bf16)
            tr = torch.zeros(cols, _pad(rows), device=dev, dtype=bf16) if want_t else None
            self.nat[key] = nat[:, :cols]
            if want_t:
                self.tr[key] = tr[:, :rows]
            r0 = 0
            for w in ws:
                it = CastItem()
                it.src, it.ld_src = w.data_ptr(), cols
                it.dst, it.ld_dst = nat[r0:].data_ptr(), nat.stride(0)
                if want_t:
                    it.dst_t, it.ld_dst_t = tr[:, r0:].data_ptr(), tr.stride(0)
                else:
                    it.dst_t, it.ld_dst_t = None, 0
                it.rows, it.cols = w.shape[0], cols
                it.tile_start = tile
                tile += ((w.shape[0] + 31) // 32) * ((cols + 31) // 32)
                items.append(it)
                r0 += w.shape[0]

        for i in range(model.n_enc_layers):
            p = f"encoder.{i}"
            add(f"{p}.attn.qkv", [f"{p}.attn.{k}.weight" for k in ("query", "key", "value")])
            add(f"{p}.attn.out_proj", [f"{p}.attn.out_proj.weight"])
            add(f"{p}.mlp.up_proj", [f"{p}.mlp.up_proj.weight"])
            add(f"{p}.mlp.down_proj", [f"{p}.mlp.down_proj.weight"])
        add("decoder_proj_context", ["decoder_proj_context.weight"])
        for i in range(model.n_dec_layers):
            p = f"decoder.{i}"
            add(f"{p}.attn.qkv", [f"{p}.attn.{k}.weight" for k in ("query", "key", "value")])
            add(f"{p}.attn.out_proj", [f"{p}.attn.out_proj.weight"])
            add(f"{p}.cross_attn.query", [f"{p}.cross_attn.query.weight"])
            add(f"{p}.cross_attn.kv", [f"{p}.cross_attn.key.weight", f"{p}.cross_attn.value.weight"])
            add(f"{p}.cross_attn.out_proj", [f"{p}.cross_attn.out_proj.weight"])
            add(f"{p}.mlp.up_proj", [f"{p}.mlp.up_proj.weight"])
            add(f"{p}.mlp.down_proj", [f"{p}.mlp.down_proj.weight"])
        for prefix, mods in sessions.values():
            for m in mods:
                if m.small:
                    continue
                for side in ("encoder_embeddings", "decoder_embeddings"):
                    p = f"{prefix}{side}.{m.name}.embedder"
                    add(f"{p}.token_embed", [f"{p}.token_embed.weight"], want_t=False)
                    add(f"{p}.projection", [f"{p}.projection.weight"])
                add(f"{prefix}decoder_embeddings.{m.name}.out", [f"{prefix}decoder_embeddings.{m.name}.out.weight"])
        arr = (CastItem * len(items))(*items)
        self.items_dev = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
        self.n_items = len(items)
        self.total_tiles = tile

    def refresh(self) -> None:
        ops.cast_bf16_multi(self.items_dev, self.n_items, self.total_tiles)


class Arena:
    """Bump allocator over one device buffer.  Plans of different sessions (model.MultiSessionMultiModal) never run
    concurrently, so their activation / saved-tensor buffers alias the same arena instead of multiplying the
    footprint by the number of sessions; saved tensors of a plan stay valid until another plan's forward runs."""

    ALIGN = 256

    def __init__(self, nbytes: int, device):
        self.buf = torch.empty(nbytes, device=device, dtype=torch.uint8)
        self.off = 0

    def reset(self):
        self.off = 0

    def take(self, nbytes: int) -> torch.Tensor:
        n = (nbytes + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        if self.off + n > self.buf.numel():
            raise MmfmError("activation arena exhausted (sized from the widest session)")
        t = self.buf[self.off:self.off + nbytes]
        self.off += n
        return t


class PinnedStage:
    """Pinned host buffer feeding an asynchronous H2D copy (a pageable source would make the copy a sync point).  The
    DMA reads the buffer when the copy executes, not when it is enqueued, so a host running steps ahead of the device
    would ship a later step's values; a rewrite therefore waits for the event recorded after the previous copy."""

    def __init__(self, shape, dtype):
        self.host = torch.zeros(*shape, dtype=dtype).pin_memory()
        self.copied = torch.cuda.Event()

    def copy_to(self, dst: torch.Tensor, src: torch.Tensor) -> None:
        self.copied.synchronize()
        self.host.copy_(src)
        dst.copy_(self.host, non_blocking=True)
        self.copied.record()


# ------------------------------------------------------------------------------------------------------------
class Plan:
    """All buffers + the recorded forward / backward launch lists for one (batch size, train/eval) shape.

    ``recompute``: the plan saves only the fp32 residual stream at every layer boundary (plus the embedders, the context,
    the final norms and the heads); each layer's other activations live in scratch buffers every layer reuses, and the
    backward records that layer's forward again from its checkpoint before the layer's own backward.  Engine._plan picks
    it when the plan that saves everything does not fit in device memory.

    ``dry``: size the plan without allocating it -- every buffer is a meta tensor, the launches are recorded and dropped;
    ``arena_bytes`` and ``nbytes`` come out as they would for the plan built."""

    fwd_only = False

    def __init__(self, eng: "Engine", B: int, training: bool, session=None, arena: Optional[Arena] = None,
                 u8_mods: Tuple[str, ...] = (), grad_inputs: Tuple[str, ...] = (), recompute: bool = False,
                 dry: bool = False):
        self.eng, self.B, self.training = eng, B, training
        self.u8_mods = tuple(u8_mods)      # modalities whose inputs / targets arrive as uint8 counts (wire format)
        self.grad_inputs = tuple(grad_inputs)   # modalities whose inputs get a gradient (recorded after the last mark)
        self.recompute = bool(recompute) and not self.fwd_only
        self.arena_bytes = 0               # bytes of the activation buffers (taken from `arena` when one is given)
        self.nbytes = 0                    # every device buffer of the plan: arena_bytes + the rest + det workspace
        if arena is not None and not dry:
            arena.reset()
        self.prefix, self.mods = eng.sessions[session]
        dev = self._dev = torch.device("meta") if dry else eng.device
        # the session's index in eng.sessions (= in store.session_ranges), also as an int32 device scalar: the id this
        # plan contributes to the data-parallel session exchange
        self.session_index = list(eng.sessions).index(session)
        self.session_id = self._new(1, dtype=torch.int32).fill_(self.session_index)
        mods, T, H = self.mods, eng.T, eng.H
        S = T * len(mods)
        R, BT = B * S, B * T
        self.S, self.R, self.BT = S, R, BT

        self._keep: List[Any] = []
        # deterministic mode (torch.use_deterministic_algorithms): the cross-CTA reductions of the backward go through
        # the *_det kernels on this one workspace, sized after recording to the largest call (one stream: shared)
        self.det_ws = ops.DetWorkspace() if ops.deterministic() and not self.fwd_only else None
        self._bufs: Dict[Any, torch.Tensor] = {}     # scratch buffers every layer reuses (_scratch)

        def raw(shape, dtype, esize):
            n = int(np.prod(shape)) * esize
            a = (n + Arena.ALIGN - 1) // Arena.ALIGN * Arena.ALIGN
            self.arena_bytes += a
            self.nbytes += a
            if arena is not None and not dry:
                t = arena.take(n).view(dtype).view(*shape)
            else:
                t = self._new(*shape, dtype=dtype, count=False)
            self._keep.append(t)      # recorded launches hold raw pointers: the plan owns (or pins) every buffer
            return t

        def f32(*s):
            return raw(tuple(s), torch.float32, 4)

        def b16(r, c):
            return raw((r, _pad(c)), bf16, 2)[:, :c]

        def i64(*s):
            return self._new(*s, dtype=torch.int64, zero=True)

        def u8(*s):
            return self._new(*s, dtype=torch.uint8, zero=True)

        self._f32, self._b16 = f32, b16
        # ---- static inputs -------------------------------------------------------------------------------
        self.inp = {m.name: f32(B, T, m.C) for m in mods}
        self.tgt = {m.name: f32(B, T, m.C) for m in mods}
        # byte staging of the uint8 wire format: expanded on the device (inputs -> bf16 GEMM operand, targets -> fp32)
        self.inp_u8 = {m.name: u8(B, T, m.C) for m in mods if m.name in self.u8_mods}
        self.tgt_u8 = {m.name: u8(B, T, m.C) for m in mods if m.name in self.u8_mods}
        self.attn = {m.name: i64(B, T) for m in mods}
        self.ts = {m.name: i64(B, T) for m in mods}
        self.mask = {m.name: i64(B, T) for m in mods}
        self.seed = eng.seed               # ONE device seed per engine: every plan's launches capture the same pointer
        self.gscale = self._new(1).fill_(1.0)
        self.one = self._new(1).fill_(1.0)
        self._dpreds_dirty = False         # dpreds overwritten by head_grad since the last forward
        # per-modality 32-bit Bernoulli thresholds of the device-side mask sampler (0 = read the mask buffer); a device
        # array so that the captured graph sees per-step changes, staged through pinned host memory
        self.sample_thresh = self._new(len(mods), dtype=torch.int32, zero=True)
        self._thresh_stage = None if dry else PinnedStage((len(mods),), torch.int32)
        self._thresh_cur = [0] * len(mods)
        self._mask_stage = {} if dry else {m.name: PinnedStage((B, T), torch.int64) for m in mods}
        # ---- mask products -------------------------------------------------------------------------------
        self.zero, self.kvalid, self.tmask = u8(S), u8(B, S), u8(B, S)
        self.nex, self.inv_n = i64(len(mods)), f32(1)
        self.mod_ids = self._new(S, dtype=torch.int16)
        self.mod_ids.copy_(torch.repeat_interleave(torch.tensor([m.index for m in mods], dtype=torch.int16), T))
        # ---- outputs -------------------------------------------------------------------------------------
        self.preds = {m.name: f32(B, T, m.C) for m in mods}
        self.n_partials = 2 * max(1, lib().mmfm_sm_count())
        self.partials = self._new(len(mods) * self.n_partials, zero=True)
        self.mod_loss, self.loss = f32(len(mods)), f32(1)

        self.wgrad_writes: List[Tuple[int, Tuple[str, ...]]] = []   # (wgrad call index, parameters it writes)
        rec_f, rec_b = ops.Recorder(), ops.Recorder()
        ops.set_recorder(rec_f)
        try:
            self._build_forward(f32, b16)
            if not self.fwd_only:
                ops.set_recorder(rec_b)
                self._build_backward(f32, b16)
        finally:
            ops.set_recorder(None)
            del self._f32, self._b16      # they hold the plan: a dropped plan must free its buffers right away
        self._g_fwd = self._g_bwd = None
        self._n_fwd_runs = self._n_bwd_runs = 0
        self.fwd_calls, self.bwd_calls = rec_f.calls, rec_b.calls
        # frozen parameters: the wgrad launches that write only frozen parameters are left out of the backward; one
        # call list (and captured graph) per such set, derived from the recorded one (same buffers, same plan)
        params = eng.store.params
        self._wgrad_params = [(ci, tuple(params[n] for n in names)) for ci, names in self.wgrad_writes]
        self._skip_of: Dict[Tuple[bool, ...], Tuple[int, ...]] = {}
        self._variants: Dict[Tuple[int, ...], Dict[str, Any]] = {}
        self._keep += rec_f.keep + rec_b.keep
        if self.det_ws is not None:
            ws = self.det_ws       # materialize allocates max(16, bytes) and max(1, tickets) int32 for a new workspace
            self.nbytes += _round_alloc(max(16, ws.want_bytes)) + _round_alloc(4 * max(1, ws.want_tickets))
            if not dry:
                ws.materialize(dev)
        self.n_fwd, self.n_bwd = len(self.fwd_calls), len(self.bwd_calls)

    # ---------------------------------------------------------------------------------------------------
    def _new(self, *shape, dtype=torch.float32, zero: bool = False, count: bool = True) -> torch.Tensor:
        """A device buffer of the plan (a meta tensor in a dry plan), counted in nbytes."""
        t = (torch.zeros if zero else torch.empty)(*shape, device=self._dev, dtype=dtype)
        if count:
            self.nbytes += _round_alloc(t.numel() * t.element_size())
        return t

    def _drop(self, kind: int, layer: int, side: int, p: float) -> DropSpec:
        if not self.training or p <= 0.0:
            return NO_DROP
        return DropSpec(self.seed, site_id(kind, layer, side), p)

    def _scratch(self, key, make, role=None, save: bool = False):
        """A buffer the forward writes.  The training plan takes a new one per call: the backward reads each.  The
        forward-only plan takes one per key and reuses it in every layer: the next layer overwrites it after its last
        reader has run.  The recompute plan takes one per (key, role) -- `role` tells apart the buffers of one key that
        a layer's backward reads together -- and a new one per call for what its backward reads unrecomputed (`save`)."""
        if self.recompute and not save:
            key = (key, role)
        elif not self.fwd_only:
            return make()
        t = self._bufs.get(key)
        if t is None:
            t = self._bufs[key] = make()
        return t

    def _act(self, key, r, c, role=None, save: bool = False):
        """bf16 activation [r, c] (see _scratch)."""
        return self._scratch((key, c), lambda: self._b16(r, c), role, save)

    def _ln_fwd(self, x, name, y, role=None, save: bool = False, modmajor=False):
        st = self.eng.store
        new = lambda: self._new(self.R)
        mean, rstd = self._scratch("ln_mean", new, role, save), self._scratch("ln_rstd", new, role, save)
        self._keep += [mean, rstd]
        self.stats[name] = (mean, rstd)
        if st.has(name + ".scale"):       # ScaleNorm: `mean` unused, `rstd` holds 1 / max(||x||, eps)
            assert not modmajor
            ops.scalenorm_fwd(x, st.p(name + ".scale"), y, rstd, R=self.R, H=self.eng.H)
            return
        ops.layernorm_fwd(x, st.p(name + ".weight"), st.p(name + ".bias"), y, mean, rstd, R=self.R, H=self.eng.H,
                          modmajor_T=self.eng.T if modmajor else 0, S=self.S if modmajor else 0)

    def _ln_bwd(self, dy, x, name, dres, dx, dxb, drop, modmajor=False):
        st = self.eng.store
        mean, rstd = self.stats[name]
        if st.has(name + ".scale"):
            ops.scalenorm_bwd(dy, x, rstd, st.p(name + ".scale"), dres, dx, dxb, drop, st.g(name + ".scale"), R=self.R,
                              H=self.eng.H, ws=self.det_ws)
            return
        ops.layernorm_bwd(dy, x, mean, rstd, st.p(name + ".weight"), dres, dx, dxb, drop, st.g(name + ".weight"),
                          st.g(name + ".bias"), R=self.R, H=self.eng.H, modmajor_T=self.eng.T if modmajor else 0,
                          S=self.S if modmajor else 0, ws=self.det_ws)

    def _bias(self, names: List[str], buf: str = "p") -> Optional[torch.Tensor]:
        """fp32 bias (possibly the concatenation of adjacent biases in the flat buffer)."""
        st = self.eng.store
        if not st.has(names[0]):
            return None
        base = st.flat if buf == "p" else st.grad
        o0 = st.offset[st.alias[names[0]]]
        n = 0
        for nm in names:
            assert st.offset[st.alias[nm]] == o0 + n, "fused biases must be adjacent in the flat buffer"
            n += st.shape[nm].numel()
            assert st.shape[nm].numel() % 64 == 0 or nm == names[-1], "fused biases need 64-element multiples"
        return base[o0:o0 + n]

    def _wgrad_dst(self, names: List[str]) -> torch.Tensor:
        st = self.eng.store
        o0 = st.offset[names[0]]
        n = 0
        for nm in names:
            assert st.offset[nm] == o0 + n, "fused weights must be adjacent in the flat buffer"
            n += st.shape[nm].numel()
            assert len(names) == 1 or st.shape[nm].numel() % 64 == 0
        cols = st.shape[names[0]][1]
        return st.grad[o0:o0 + n].view(n // cols, cols)

    # ---------------------------------------------------------------------------------------------------
    def _attention(self, fwd: bool, tag: str, q, k, v, o, mode, nh, p_drop, kind_p, kind_o, layer, side, sep,
                   grads=None, prep_done=False):
        B, S, H = self.B, self.S, self.eng.H
        d = H // nh
        if fwd:
            self.lse[tag] = self._scratch(("lse", nh), lambda: self._new(B, nh, S), kind_p)
            dp = self._drop(kind_p, layer, side, p_drop)
            if dp.thresh:
                self.pkeep[tag] = self._scratch(("pkeep", nh), lambda: self._new(B * nh * S * ((S + 63) // 64) * 4,
                                                                                 dtype=torch.int16, zero=True), kind_p)
        dp = self._drop(kind_p, layer, side, p_drop)
        do = self._drop(kind_o, layer, side, p_drop)
        kw = dict(B=B, n_heads=nh, Sq=S, Sk=S, d_head=d, mask_mode=mode, mod_q=self.mod_ids if sep else None,
                  mod_k=self.mod_ids if sep else None, drop_p=dp, drop_o=do, p_keep=self.pkeep.get(tag))
        if fwd:
            ops.attention_fwd(q, k, v, o, self.lse[tag], self.kvalid, **kw)
        else:
            d_o, dq, dk, dv = grads
            ops.attention_bwd(q, k, v, o, self.lse[tag], self.kvalid, d_o=d_o, delta=self.delta, dq=dq, dk=dk, dv=dv,
                              prep_done=prep_done, **kw)

    # ---------------------------------------------------------------------------------------------------
    def _build_forward(self, f32, b16):
        eng = self.eng
        st, sh, mods = eng.store, eng.shadows, self.mods
        B, T, H, S, R, BT = self.B, eng.T, eng.H, self.S, self.R, self.BT
        self.stats: Dict[str, Tuple[torch.Tensor, torch.Tensor]] = {}
        self.lse: Dict[str, torch.Tensor] = {}
        self.pkeep: Dict[str, torch.Tensor] = {}
        self.act: Dict[str, torch.Tensor] = {}   # saved bf16 activations by name
        A = self.act
        fo = self.fwd_only

        act = self._act

        def resid(prev, pair, mid=None):
            """Output of a residual sub-layer whose input is `prev`: a buffer of its own in the training plan (the backward
            reads every one); in the forward-only plan the other buffer of `pair` (the residual GEMM never runs in place).
            The recompute plan owns the layer boundaries (its checkpoints) and reuses one buffer per mid-layer position
            `mid` in every layer."""
            if fo:
                return pair[1] if prev is pair[0] else pair[0]
            if mid is not None:
                return self._scratch("resid", lambda: f32(R, H), mid)
            return f32(R, H)

        sh.refresh()
        ops.mask_prep([self.mask[m.name] for m in mods], [self.attn[m.name] for m in mods], [m.C for m in mods],
                      self.zero, self.kvalid, self.tmask, self.nex, self.inv_n, sample_thresh=self.sample_thresh,
                      seed=self.seed)

        # ---- embeddings (encoder_embeddings.py:44-61, decoder_embeddings.py:43-61, mm.py:141-175,289,293) ----
        self.emb = {SIDE_ENC: f32(R, H), SIDE_DEC: f32(R, H)}
        self.xs = [f32(R, H)]
        self.ys = [f32(R, H)]
        self.inb: Dict[str, torch.Tensor] = {}
        for side, sname, x0, p_emb in ((SIDE_ENC, "encoder_embeddings", self.xs[0], eng.hp["embed_dropout"]),
                                       (SIDE_DEC, "decoder_embeddings", self.ys[0], eng.hp["dec_embed_dropout"])):
            for k, m in enumerate(mods):
                pre = f"{self.prefix}{sname}.{m.name}.embedder"
                off = k * T
                pos = st.p(pre + ".pos_embed.weight") if st.has(pre + ".pos_embed.weight") else None
                ops.embed_assemble(st.p(pre + ".mod_emb.weight")[m.index], pos, self.ts[m.name], self.emb[side], B=B,
                                   T=T, S=S, off=off, H=H)
                drop = self._drop(SITE_EMBED, m.index, side, p_emb)
                b1 = st.p(pre + ".token_embed.bias") if st.has(pre + ".token_embed.bias") else None
                if m.small:
                    A[pre + ".hid"] = f32(BT, 2 * m.C)
                    ops.smallc_embed_fwd(self.inp[m.name], st.p(pre + ".token_embed.weight"), b1,
                                         st.p(pre + ".projection.weight"), st.p(pre + ".projection.bias"),
                                         self.emb[side], x0, A[pre + ".hid"], self.zero, drop, eng.embed_scale,
                                         eng.embed_act, B=B, T=T, S=S, off=off, Cc=m.C, H=H)
                else:
                    if m.name not in self.inb:
                        self.inb[m.name] = b16(BT, m.C)
                        if m.name in self.u8_mods:
                            ops.u8_expand(self.inp_u8[m.name].view(BT, m.C), None, self.inb[m.name], R=BT, Cc=m.C)
                            ops.u8_expand(self.tgt_u8[m.name].view(BT, m.C), self.tgt[m.name].view(BT, m.C), None,
                                          R=BT, Cc=m.C)
                        else:
                            ops.cast_bf16(self.inp[m.name].view(BT, m.C), self.inb[m.name])
                    A[pre + ".hid"] = b16(BT, 2 * m.C)
                    ops.gemm_tn(self.inb[m.name], sh.nat[pre + ".token_embed"], A[pre + ".hid"], bias=b1,
                                act=eng.embed_act, act_scale=eng.embed_scale)
                    ops.gemm_tn(A[pre + ".hid"], sh.nat[pre + ".projection"], x0, bias=st.p(pre + ".projection.bias"),
                                drop=drop, remap=(T, S, off), row_zero=self.zero, res=self.emb[side])

        # ---- encoder (encoder_embeddings.py:106-116; mm.py:197-204) ----------------------------------------
        # forward-only: the encoder alternates between its embedding output and the decoder's embedding sum (dead once
        # the embedders have run); it ends where it started, so the decoder then alternates with that buffer
        pair = (self.xs[0], self.emb[SIDE_DEC])
        for i in range(eng.Le):
            self.xs.append(resid(self.xs[-1], pair, 1))
            self.xs.append(resid(self.xs[-1], pair))
            self._enc_layer(i)
        A["encoder_norm"] = act("ln", R, H, save=True)
        self._ln_fwd(self.xs[-1], "encoder_norm", A["encoder_norm"], save=True)
        # context = decoder_proj_context(x) + encoder_emb (mm.py:292)
        self.ctx = f32(R, H)
        ops.gemm_tn(A["encoder_norm"], sh.nat["decoder_proj_context"], self.ctx,
                    bias=st.p("decoder_proj_context.bias"), res=self.emb[SIDE_ENC])

        # ---- decoder (decoder_embeddings.py:133-147; mm.py:207-214) ----------------------------------------
        if eng.fuse_ctx:   # every layer's context_norm(context) from one read of the context
            names = [f"decoder.{i}.context_norm" for i in range(eng.Ld)]
            for n in names:
                A[n] = b16(R, H)
            cmean, crstd = self._new(R), self._new(R)
            self._keep += [cmean, crstd]
            for n in names:
                self.stats[n] = (cmean, crstd)
            ops.layernorm_fwd_multi(self.ctx, [st.p(n + ".weight") for n in names], [st.p(n + ".bias") for n in names],
                                    [A[n] for n in names], cmean, crstd, R=R, H=H)
        pair = (self.ys[0], self.xs[-1])
        for i in range(eng.Ld):
            for mid in (1, 2, None):
                self.ys.append(resid(self.ys[-1], pair, mid))
            self._dec_layer(i)
        # decoder_norm, written modality-major so that every head reads a contiguous [B*T, H] block
        A["decoder_norm"] = act("ln", R, H, save=True)
        self._ln_fwd(self.ys[-1], "decoder_norm", A["decoder_norm"], save=True, modmajor=True)

        # ---- heads + fused masked loss / gradient (decoder_embeddings.py:95-109; mm.py:217-239) -------------
        self.dpreds: Dict[str, torch.Tensor] = {}
        for k, m in enumerate(mods):
            pre = f"{self.prefix}decoder_embeddings.{m.name}.out"
            ym = A["decoder_norm"][k * BT:(k + 1) * BT]
            pr = self.preds[m.name].view(BT, m.C)
            if m.small:
                ops.smallc_head_fwd(ym, st.p(pre + ".weight"), st.p(pre + ".bias"), pr, R=BT, H=H, Cc=m.C)
            else:
                ops.gemm_tn(ym, sh.nat[pre], pr, bias=st.p(pre + ".bias"))
            self.dpreds[m.name] = act("dpreds", BT, m.C, save=True)      # forward-only: written, never read
            ops.loss_fwd_bwd(pr, self.tgt[m.name].view(BT, m.C), self.tmask, self.inv_n, m.loss_kind,
                             self.partials[k * self.n_partials:(k + 1) * self.n_partials], self.dpreds[m.name], B=B,
                             T=T, Cc=m.C, S=S, off=k * T)
        ops.loss_finalize(self.partials, self.n_partials, len(mods), self.inv_n, self.mod_loss, self.loss)

    # -- one layer's forward: recorded by the forward, and again by the recompute plan's backward (replay=True) ----
    def _attn_block(self, pre, x_in, x_out, ln_name, mode, nh, p_drop, layer, side, sep):
        A, sh, R, H = self.act, self.eng.shadows, self.R, self.eng.H
        A[ln_name] = self._act("ln", R, H, "ln1")
        self._ln_fwd(x_in, ln_name, A[ln_name], "ln1")
        A[pre + ".qkv"] = self._act("qkv", R, 3 * H)
        ops.gemm_tn(A[ln_name], sh.nat[pre + ".qkv"], A[pre + ".qkv"],
                    bias=self._bias([f"{pre}.{k}.bias" for k in ("query", "key", "value")]))
        qkv = A[pre + ".qkv"]
        A[pre + ".ao"] = self._act("ao", R, H, "self")
        self._attention(True, pre, qkv[:, :H], qkv[:, H:2 * H], qkv[:, 2 * H:], A[pre + ".ao"], mode, nh, p_drop,
                        SITE_ATTN_PROB, SITE_ATTN_OUT, layer, side, sep)
        ops.gemm_tn(A[pre + ".ao"], sh.nat[pre + ".out_proj"], x_out, bias=self._bias([pre + ".out_proj.bias"]),
                    res=x_in)

    def _mlp_block(self, pre, x_in, x_out, ln_name, p_drop, layer, side, inter, replay):
        A, sh, R, H = self.act, self.eng.shadows, self.R, self.eng.H
        A[ln_name] = self._act("ln", R, H, "ln2")
        self._ln_fwd(x_in, ln_name, A[ln_name], "ln2")
        up_bias = self._bias([pre + ".up_proj.bias"])
        if (self.fwd_only or (self.recompute and not replay)) and inter > 64 and inter % 4 == 0:
            # no backward reads this call's outputs: gelu(u) alone, from the TMA-store kernel's TS_GELU epilogue (the
            # evaluation of its TS_GELU_DG flavour, which the call below takes at these widths: the same bits)
            A[pre + ".g"] = self._act("g", R, inter)
            ops.gemm_tn(A[ln_name], sh.nat[pre + ".up_proj"], A[pre + ".g"], bias=up_bias, act=ACT_GELU)
        else:
            # saved for backward: gelu(u) (operand of the down projection and of its wgrad) and gelu'(u) -- the
            # derivative instead of the pre-activation, so the backward epilogue is a single multiply
            A[pre + ".dg"], A[pre + ".g"] = self._act("dg", R, inter), self._act("g", R, inter)
            ops.gemm_tn(A[ln_name], sh.nat[pre + ".up_proj"], A[pre + ".g"], bias=up_bias, act=ACT_GELU_DG,
                        D2=A[pre + ".dg"])
        if not replay:     # the down projection's output is the next layer's checkpoint: never recomputed
            ops.gemm_tn(A[pre + ".g"], sh.nat[pre + ".down_proj"], x_out, bias=self._bias([pre + ".down_proj.bias"]),
                        drop=self._drop(SITE_MLP, layer, side, p_drop), res=x_in)

    def _enc_layer(self, i, replay=False):
        """Encoder layer i from xs[2i] to xs[2i+2]; replay stops before the down projection."""
        eng, hp = self.eng, self.eng.hp
        pre = f"encoder.{i}"
        x0, x1, x2 = self.xs[2 * i: 2 * i + 3]
        self._attn_block(pre + ".attn", x0, x1, pre + ".ln1", MASK_KEY_OR_DIAG, hp["enc_heads"], hp["enc_dropout"], i,
                         SIDE_ENC, False)
        self._mlp_block(pre + ".mlp", x1, x2, pre + ".ln2", hp["enc_dropout"], i, SIDE_ENC, eng.enc_inter, replay)

    def _dec_layer(self, i, replay=False):
        """Decoder layer i from ys[3i] to ys[3i+3]; replay stops before the down projection."""
        eng, hp, A, sh, R, H = self.eng, self.eng.hp, self.act, self.eng.shadows, self.R, self.eng.H
        pre = f"decoder.{i}"
        y0, y1, y2, y3 = self.ys[3 * i: 3 * i + 4]
        self._attn_block(pre + ".attn", y0, y1, pre + ".ln1", MASK_CAUSAL if eng.causal else MASK_KEY, hp["dec_heads"],
                         hp["dec_dropout"], i, SIDE_DEC, eng.sep)
        # cross attention: q from query_norm(y), k/v from context_norm(context), mask = ENCODER mask
        xa = pre + ".cross_attn"
        A[pre + ".query_norm"] = self._act("ln", R, H, "query_norm")
        self._ln_fwd(y1, pre + ".query_norm", A[pre + ".query_norm"], "query_norm")
        if not eng.fuse_ctx:
            A[pre + ".context_norm"] = self._act("context_norm", R, H)
            self._ln_fwd(self.ctx, pre + ".context_norm", A[pre + ".context_norm"], "context_norm")
        A[xa + ".q"], A[xa + ".kv"] = self._act("xq", R, H), self._act("xkv", R, 2 * H)
        ops.gemm_tn(A[pre + ".query_norm"], sh.nat[xa + ".query"], A[xa + ".q"], bias=self._bias([xa + ".query.bias"]))
        ops.gemm_tn(A[pre + ".context_norm"], sh.nat[xa + ".kv"], A[xa + ".kv"],
                    bias=self._bias([xa + ".key.bias", xa + ".value.bias"]))
        A[xa + ".ao"] = self._act("ao", R, H, "cross")
        self._attention(True, xa, A[xa + ".q"], A[xa + ".kv"][:, :H], A[xa + ".kv"][:, H:], A[xa + ".ao"],
                        MASK_KEY_OR_DIAG, hp["dec_heads"], hp["dec_dropout"], SITE_XATTN_PROB, SITE_XATTN_OUT, i,
                        SIDE_DEC, False)
        ops.gemm_tn(A[xa + ".ao"], sh.nat[xa + ".out_proj"], y2, bias=self._bias([xa + ".out_proj.bias"]), res=y1)
        self._mlp_block(pre + ".mlp", y2, y3, pre + ".ln2", hp["dec_dropout"], i, SIDE_DEC, eng.dec_inter, replay)

    # ---------------------------------------------------------------------------------------------------
    def _build_backward(self, f32, b16):
        eng = self.eng
        st, sh, mods, hp = eng.store, eng.shadows, self.mods, eng.hp
        B, T, H, S, R, BT = self.B, eng.T, eng.H, self.S, self.R, self.BT
        A = self.act
        G, Genc, Gctx = f32(R, H), f32(R, H), f32(R, H)       # fp32 residual-stream gradients
        Gb, Gcb = b16(R, H), b16(R, H)                         # bf16 (dropout-masked) copies feeding the dgrad GEMMs
        d_ao, dh = b16(R, H), b16(R, H)
        dqkv = b16(R, 3 * H)
        du = b16(R, max(eng.enc_inter, eng.dec_inter))
        self.delta = f32(B, max(hp["enc_heads"], hp["dec_heads"]), S)
        ddec = b16(R, H)                                       # gradient wrt decoder_norm output (modality-major)
        self.grad_marks: List[Tuple[int, int]] = []           # (calls issued, flat-gradient offset that is final)

        def mark(next_param: Optional[str]):
            rec = ops._REC
            off = st.total if next_param is None else st.offset[st.alias[next_param]]
            self.grad_marks.append((len(rec.calls), off))

        def lin_bwd(dY, X, wname, shadow_key, dX, *, act=ACT_NONE, aux=None, act_scale=1.0, wnames=None, bnames=None,
                    **extra):
            """dX = dY . W ; dW += dY^T X ; db += colsum(dY)"""
            if dX is not None:
                ops.gemm_tn(dY, sh.tr[shadow_key], dX, act=act, aux=aux, act_scale=act_scale, **extra)
            bn = bnames or [wname + ".bias"]
            wn = wnames or [wname + ".weight"]
            ops.gemm_wgrad(dY, X, self._wgrad_dst(wn), dbias=self._bias(bn, "g") if st.has(bn[0]) else None,
                           ws=self.det_ws)
            writes = wn + ([st.alias[n] for n in bn] if st.has(bn[0]) else [])
            self.wgrad_writes.append((len(ops._REC.calls) - 1, tuple(writes)))

        def mlp_bwd(pre, x_in, ln_name, Gs, inter, dxb, drop_prev):
            duv = du[:, :inter]
            lin_bwd(Gb, A[pre + ".g"], pre + ".down_proj", pre + ".down_proj", duv,
                    act=ACT_MULAUX, aux=A[pre + ".dg"])
            lin_bwd(duv, A[ln_name], pre + ".up_proj", pre + ".up_proj", dh)
            self._ln_bwd(dh, x_in, ln_name, Gs, Gs, dxb, drop_prev)

        def out_proj_bwd(pre, nh, p_drop, kind_o, layer, side):
            """out-projection dgrad (+ wgrad).  At d_head 32 its epilogue also does the attention-backward preparation
            (delta = rowsum(dO * O) per head, output-dropout mask on dO): one launch and one pass over dO / O less per
            attention call.  Returns True when the attention kernel may skip its own preparation.  The TMA-store GEMM,
            the only one with this epilogue, takes it for H > 64."""
            fuse = H > 64 and H % 32 == 0 and H // nh == 32
            if fuse:
                lin_bwd(Gb, A[pre + ".ao"], pre + ".out_proj", pre + ".out_proj", d_ao, act=ACT_ROWDOT_DROP,
                        aux=A[pre + ".ao"], rowdot=self.delta, rowdot_S=S, drop=self._drop(kind_o, layer, side, p_drop))
            else:
                lin_bwd(Gb, A[pre + ".ao"], pre + ".out_proj", pre + ".out_proj", d_ao)
            return fuse

        def attn_bwd(pre, x_in, ln_name, Gs, mode, nh, p_drop, layer, side, sep, dxb, drop_prev):
            fused = out_proj_bwd(pre, nh, p_drop, SITE_ATTN_OUT, layer, side)
            qkv = A[pre + ".qkv"]
            self._attention(False, pre, qkv[:, :H], qkv[:, H:2 * H], qkv[:, 2 * H:], A[pre + ".ao"], mode, nh, p_drop,
                            SITE_ATTN_PROB, SITE_ATTN_OUT, layer, side, sep,
                            grads=(d_ao, dqkv[:, :H], dqkv[:, H:2 * H], dqkv[:, 2 * H:]), prep_done=fused)
            lin_bwd(dqkv, A[ln_name], None, pre + ".qkv", dh,
                    wnames=[f"{pre}.{k}.weight" for k in ("query", "key", "value")],
                    bnames=[f"{pre}.{k}.bias" for k in ("query", "key", "value")])
            self._ln_bwd(dh, x_in, ln_name, Gs, Gs, dxb, drop_prev)

        # ---- heads (reverse order = gradient-bucket order) -------------------------------------------------
        for k, m in reversed(list(enumerate(mods))):
            pre = f"{self.prefix}decoder_embeddings.{m.name}.out"
            ym = A["decoder_norm"][k * BT:(k + 1) * BT]
            dym = ddec[k * BT:(k + 1) * BT]
            if m.small:
                ops.smallc_head_bwd(ym, st.p(pre + ".weight"), self.dpreds[m.name], dym, st.g(pre + ".weight"),
                                    st.g(pre + ".bias"), R=BT, H=H, Cc=m.C, ws=self.det_ws)
            else:
                lin_bwd(self.dpreds[m.name], ym, pre, pre, dym)
        last_dec_drop = self._drop(SITE_MLP, eng.Ld - 1, SIDE_DEC, hp["dec_dropout"])
        self._ln_bwd(ddec, self.ys[-1], "decoder_norm", None, G, Gb, last_dec_drop, modmajor=True)

        # ---- decoder layers --------------------------------------------------------------------------------
        dec_mode = MASK_CAUSAL if eng.causal else MASK_KEY
        dqx, dkvx = b16(R, H), b16(R, 2 * H)
        dctx: List[torch.Tensor] = []
        for i in reversed(range(eng.Ld)):
            pre = f"decoder.{i}"
            y0, y1, y2, y3 = self.ys[3 * i: 3 * i + 4]
            if self.recompute:
                self._dec_layer(i, replay=True)
            mlp_bwd(pre + ".mlp", y2, pre + ".ln2", G, eng.dec_inter, Gb, NO_DROP)
            xa = pre + ".cross_attn"
            fused = out_proj_bwd(xa, hp["dec_heads"], hp["dec_dropout"], SITE_XATTN_OUT, i, SIDE_DEC)
            self._attention(False, xa, A[xa + ".q"], A[xa + ".kv"][:, :H], A[xa + ".kv"][:, H:], A[xa + ".ao"],
                            MASK_KEY_OR_DIAG, hp["dec_heads"], hp["dec_dropout"], SITE_XATTN_PROB, SITE_XATTN_OUT, i,
                            SIDE_DEC, False, grads=(d_ao, dqx, dkvx[:, :H], dkvx[:, H:]), prep_done=fused)
            lin_bwd(dqx, A[pre + ".query_norm"], xa + ".query", xa + ".query", dh)
            self._ln_bwd(dh, y1, pre + ".query_norm", G, G, Gb, NO_DROP)
            if eng.fuse_ctx:    # the layer's gradient wrt its normalised context is kept until the last layer is through
                dctx.append(b16(R, H))
                lin_bwd(dkvx, A[pre + ".context_norm"], None, xa + ".kv", dctx[-1],
                        wnames=[xa + ".key.weight", xa + ".value.weight"], bnames=[xa + ".key.bias", xa + ".value.bias"])
            else:
                lin_bwd(dkvx, A[pre + ".context_norm"], None, xa + ".kv", dh,
                        wnames=[xa + ".key.weight", xa + ".value.weight"], bnames=[xa + ".key.bias", xa + ".value.bias"])
                first = i == eng.Ld - 1
                self._ln_bwd(dh, self.ctx, pre + ".context_norm", None if first else Gctx, Gctx, Gcb if i == 0 else None,
                             NO_DROP)
            prev = self._drop(SITE_MLP, i - 1, SIDE_DEC, hp["dec_dropout"]) if i > 0 else NO_DROP
            attn_bwd(pre + ".attn", y0, pre + ".ln1", G, dec_mode, hp["dec_heads"], hp["dec_dropout"], i, SIDE_DEC,
                     eng.sep, Gb if i > 0 else None, prev)
            if i > 0:
                mark(f"decoder.{i - 1}.mlp.down_proj.weight")
            elif eng.fuse_ctx:
                mark(f"decoder.{eng.Ld - 1}.context_norm.weight")
        if eng.fuse_ctx:   # gradient of the context through every layer's context_norm: one launch
            names = [f"decoder.{i}.context_norm" for i in reversed(range(eng.Ld))]      # the order of dctx
            cmean, crstd = self.stats[names[0]]
            ops.layernorm_bwd_multi(dctx, self.ctx, cmean, crstd, [st.p(n + ".weight") for n in names], Gctx, Gcb,
                                    [st.g(n + ".weight") for n in names], [st.g(n + ".bias") for n in names], R=R, H=H,
                                    ws=self.det_ws)
        mark("decoder_proj_context.weight")

        # ---- context projection + encoder ------------------------------------------------------------------
        lin_bwd(Gcb, A["encoder_norm"], "decoder_proj_context", "decoder_proj_context", dh)
        last_enc_drop = self._drop(SITE_MLP, eng.Le - 1, SIDE_ENC, hp["enc_dropout"])
        self._ln_bwd(dh, self.xs[-1], "encoder_norm", None, Genc, Gb, last_enc_drop)
        for i in reversed(range(eng.Le)):
            pre = f"encoder.{i}"
            if self.recompute:
                self._enc_layer(i, replay=True)
            mlp_bwd(pre + ".mlp", self.xs[2 * i + 1], pre + ".ln2", Genc, eng.enc_inter, Gb, NO_DROP)
            prev = self._drop(SITE_MLP, i - 1, SIDE_ENC, hp["enc_dropout"]) if i > 0 else NO_DROP
            attn_bwd(pre + ".attn", self.xs[2 * i], pre + ".ln1", Genc, MASK_KEY_OR_DIAG, hp["enc_heads"],
                     hp["enc_dropout"], i, SIDE_ENC, False, Gb if i > 0 else None, prev)
            if i > 0:
                mark(f"encoder.{i - 1}.mlp.down_proj.weight")

        # ---- embeddings ------------------------------------------------------------------------------------
        dtok = b16(BT, H)
        self.dhid: Dict[Tuple[int, str], torch.Tensor] = {}
        for side, sname, Gs, G2, p_emb in ((SIDE_DEC, "decoder_embeddings", G, None, hp["dec_embed_dropout"]),
                                           (SIDE_ENC, "encoder_embeddings", Genc, Gctx, hp["embed_dropout"])):
            for k, m in reversed(list(enumerate(mods))):
                pre = f"{self.prefix}{sname}.{m.name}.embedder"
                off = k * T
                dpos = st.g(pre + ".pos_embed.weight") if st.has(pre + ".pos_embed.weight") else None
                ops.embed_assemble_bwd(Gs, G2, self.ts[m.name], dpos, st.g(pre + ".mod_emb.weight")[m.index], B=B, T=T,
                                       S=S, off=off, H=H, ws=self.det_ws)
                drop = self._drop(SITE_EMBED, m.index, side, p_emb)
                if m.small:
                    has_b1 = st.has(pre + ".token_embed.bias")
                    db1 = st.g(pre + ".token_embed.bias") if has_b1 else f32(2 * m.C)
                    ops.smallc_embed_bwd(self.inp[m.name], A[pre + ".hid"], st.p(pre + ".projection.weight"), Gs,
                                         self.zero, drop, eng.embed_scale, eng.embed_act,
                                         st.g(pre + ".token_embed.weight"), db1, st.g(pre + ".projection.weight"),
                                         st.g(pre + ".projection.bias"), B=B, T=T, S=S, off=off, Cc=m.C, H=H,
                                         ws=self.det_ws)
                else:
                    ops.embed_grad_prep(Gs, dtok, self.zero, drop, B=B, T=T, S=S, off=off, H=H)
                    dhid = self.dhid[(side, m.name)] = b16(BT, 2 * m.C)
                    back = ACT_DSOFTSIGN if eng.embed_act == ACT_SOFTSIGN else ACT_NONE
                    lin_bwd(dtok, A[pre + ".hid"], pre + ".projection", pre + ".projection", dhid, act=back,
                            aux=A[pre + ".hid"] if back else None, act_scale=eng.embed_scale)
                    lin_bwd(dhid, self.inb[m.name], pre + ".token_embed", None, None)
        mark(None)
        ops.scale_inplace(st.grad, self.gscale)

        # ---- input gradients (plans whose inputs require grad; they always run with gscale = 1) --------------
        # Both embedders read the inputs: decoder side first, the encoder side adds to it.  Spike streams: the dgrad of
        # token_embed through the GEMM (dX = dhid . W1) on a transposed bf16 copy cast here, so the shared shadow cast
        # of the default schedule stays as it is; the second GEMM adds the first one's output as its residual.
        self.dinp: Dict[str, torch.Tensor] = {}
        sides = ((SIDE_DEC, "decoder_embeddings", G, hp["dec_embed_dropout"]),
                 (SIDE_ENC, "encoder_embeddings", Genc, hp["embed_dropout"]))
        for k, m in enumerate(mods):
            if m.name not in self.grad_inputs:
                continue
            dX = None
            for i, (side, sname, Gs, p_emb) in enumerate(sides):
                pre = f"{self.prefix}{sname}.{m.name}.embedder"
                if m.small:
                    dX = f32(BT, m.C) if dX is None else dX
                    ops.smallc_embed_dx(A[pre + ".hid"], st.p(pre + ".token_embed.weight"),
                                        st.p(pre + ".projection.weight"), Gs, self.zero,
                                        self._drop(SITE_EMBED, m.index, side, p_emb), eng.embed_scale, eng.embed_act, dX,
                                        accumulate=i > 0, B=B, T=T, S=S, off=k * T, Cc=m.C, H=H)
                else:
                    w1t = b16(m.C, 2 * m.C)
                    ops.cast_bf16(st.p(pre + ".token_embed.weight"), None, w1t)
                    out = f32(BT, _pad(m.C, 4))[:, :m.C]          # fp32 rows at a 16-byte pitch
                    ops.gemm_tn(self.dhid[(side, m.name)], w1t, out, res=dX)
                    dX = out
            self.dinp[m.name] = dX

    # ---------------------------------------------------------------------------------------------------
    # -- execution: eager the first time (module load, kernel attributes), CUDA-graph replay afterwards ------
    def _fwd_body(self):
        # every step advances the stream (dropout sites in train(), the device-side mask sampler in either mode)
        self.seed.add_(0x632BE59BD9B4E019)
        ops.run_recorded(self.fwd_calls)

    def head_grad(self, g_loss: Optional[torch.Tensor], g_mod: Optional[torch.Tensor],
                  g_preds: Sequence[Optional[torch.Tensor]]) -> None:
        """Overwrite dpreds with the head gradient of arbitrary upstream gradients of loss (scalar), mod_loss (vector)
        and preds (one per modality); None = absent.  The backward schedule then runs with gscale = 1."""
        restore = g_loss is self.one and g_mod is None and not any(g is not None for g in g_preds)
        g_loss = g_loss.reshape(1).float() if g_loss is not None else None
        g_mod = g_mod.float() if g_mod is not None else None
        B, T = self.B, self.eng.T
        for k, m in enumerate(self.mods):
            gp = g_preds[k] if k < len(g_preds) else None
            ops.loss_grad(self.preds[m.name], self.tgt[m.name], self.tmask, self.inv_n, m.loss_kind,
                          self.dpreds[m.name], g_loss=g_loss, g_mod=g_mod[k:k + 1] if g_mod is not None else None,
                          g_preds=gp.float() if gp is not None else None, B=B, T=T, Cc=m.C, S=self.S, off=k * T)
        self._dpreds_dirty = not restore       # g_loss = 1 alone gives the forward's dpreds bit for bit

    def set_sample_thresh(self, thresh: List[int]) -> None:
        if thresh != self._thresh_cur:
            bits = [v - (1 << 32) if v >= (1 << 31) else v for v in thresh]       # uint32 bit pattern in an int32
            self._thresh_stage.copy_to(self.sample_thresh, torch.tensor(bits, dtype=torch.int32))
            self._thresh_cur = list(thresh)

    def backward_schedule(self) -> Tuple[Tuple[int, ...], List[Any], List[Tuple[int, int]]]:
        """(skipped wgrad call indices, backward call list, gradient marks) for the parameters' current requires_grad
        flags.  A wgrad launch is skipped when every parameter it writes is frozen; its gradient range stays zero.  The
        marks keep their flat-gradient offsets (so data-parallel buckets are unchanged) with call indices counted in
        the filtered list.  Nothing frozen: the recorded list itself."""
        rg = tuple(p.requires_grad for p in self.eng.store.params.values())
        skip = self._skip_of.get(rg)
        if skip is None:
            skip = self._skip_of[rg] = tuple(ci for ci, ps in self._wgrad_params
                                             if not any(p.requires_grad for p in ps))
        if not skip:
            return skip, self.bwd_calls, self.grad_marks
        v = self._variants.get(skip)
        if v is None:
            drop = set(skip)
            kept_before = np.cumsum([0] + [i not in drop for i in range(len(self.bwd_calls))])
            v = self._variants[skip] = {
                "calls": [c for i, c in enumerate(self.bwd_calls) if i not in drop],
                "marks": [(int(kept_before[ci]), off) for ci, off in self.grad_marks], "graph": None, "runs": 0}
        return skip, v["calls"], v["marks"]

    def _bwd_body(self, calls=None):
        self.eng.store.grad.zero_()
        ops.run_recorded(self.bwd_calls if calls is None else calls)

    def _capture(self, body):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            body()
        return g

    def run_forward(self):
        if self.eng.use_graphs and self._g_fwd is None and self._n_fwd_runs >= 1:
            self._g_fwd = self._capture(self._fwd_body)
        self._n_fwd_runs += 1
        if self._g_fwd is not None:
            self._g_fwd.replay()
        else:
            self._fwd_body()
        self._dpreds_dirty = False

    def run_backward(self):
        """Zeroes the flat gradient buffer and runs the backward schedule (without the wgrad launches of frozen
        parameters)."""
        skip, calls, _ = self.backward_schedule()
        if skip:
            v = self._variants[skip]
            if self.eng.use_graphs and v["graph"] is None and v["runs"] >= 1:
                v["graph"] = self._capture(lambda: self._bwd_body(calls))
            v["runs"] += 1
            if v["graph"] is not None:
                v["graph"].replay()
            else:
                self._bwd_body(calls)
            return
        if self.eng.use_graphs and self._g_bwd is None and self._n_bwd_runs >= 1:
            self._g_bwd = self._capture(self._bwd_body)
        self._n_bwd_runs += 1
        if self._g_bwd is not None:
            self._g_bwd.replay()
        else:
            self._bwd_body()


class ForwardPlan(Plan):
    """The forward schedule alone, for steps that run with gradients disabled (torch.no_grad / inference_mode): no
    backward launches, nothing saved for one.  Buffers are allocated by liveness: two fp32 residual-stream buffers used
    in turn (plus the two embedding sums and the context), one bf16 buffer per activation role reused by every layer,
    and one LN-statistics / LSE / dropout-keep / head-gradient buffer that the kernels write and nothing reads.  The
    footprint does not grow with depth, and the MLP-up epilogue stores gelu(u) without its derivative.  Launch for
    launch the training plan's forward otherwise: same kernels, seed advance, masks and dropout sites, same results."""

    fwd_only = True


# ------------------------------------------------------------------------------------------------------------
class _StepFn(torch.autograd.Function):
    """Autograd node of one step: forward = the plan's forward schedule; backward = its backward schedule, writing
    into the flat gradient buffer that ``Parameter.grad`` views (trainer/base.py:194-195 semantics).

    Outputs: loss, the mod_loss vector and one preds tensor per modality, all differentiable.  Extra inputs: the
    modality inputs that require grad (``plan.grad_inputs``, in that order); their gradients are returned."""

    @staticmethod
    def forward(ctx, anchor, eng, plan, *inputs):
        plan.run_forward()
        ctx.eng, ctx.plan = eng, plan
        ctx.in_meta = [(x.shape, x.dtype) for x in inputs]
        ctx.set_materialize_grads(False)        # unused outputs arrive as None: their terms are skipped
        preds = [plan.preds[m.name].clone() for m in plan.mods]
        return (plan.loss.clone().reshape(()), plan.mod_loss.clone(), *preds)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_loss, grad_mod, *grad_preds):
        ctx.eng.backward(ctx.plan, grad_loss, grad_mod, grad_preds)
        pl = ctx.plan
        dinp = []
        for name, (shape, dtype) in zip(pl.grad_inputs, ctx.in_meta):
            g = torch.empty(shape, device=pl.eng.device, dtype=dtype)
            g.copy_(pl.dinp[name].reshape(shape))             # fresh tensor: the plan buffer is reused next step
            dinp.append(g)
        return (None, None, None, *dinp)


class Engine:
    _created = 0

    # the engine's buffers (flat parameters, seed, plans) are never inference tensors, even when the first step runs
    # under torch.inference_mode(): training steps write them in place afterwards
    @torch.inference_mode(False)
    def __init__(self, model):
        self.model = model
        p0 = next(model.parameters())
        if p0.device.type != "cuda":
            raise MmfmError("the B200 path runs on a CUDA device only (move the model with .cuda() / .to('cuda') "
                            "first); there is no CPU fallback")
        lib()  # fail loudly now if the extension is missing
        self.device = p0.device
        groups = embedding_groups(model)
        hp = adapter.hyper_params(model, groups)
        self.hp = hp
        loss_kind = adapter.loss_kinds(model)
        self.H = model.hidden_size
        self.Le, self.Ld = model.n_enc_layers, model.n_dec_layers
        self.fuse_ctx = fuse_context_norms(dict(model.named_parameters(remove_duplicate=False)), self.Ld)
        self.causal, self.sep = bool(model.decoder_causal_mask), bool(model.decoder_sep_mask)
        if hp["enc_act"] != "gelu" or hp["dec_act"] != "gelu":
            raise NotImplementedError("only act='gelu' (mm.yaml:44) is built for the transformer MLP")
        act = hp["embed_act"]
        if act not in ("softsign", "identity"):
            raise NotImplementedError(f"embedder act {act!r}: only 'softsign' (mm.yaml:33) and 'identity' are built")
        self.embed_act = ACT_SOFTSIGN if act == "softsign" else ACT_NONE
        # one (prefix, modality list) per session; the reference's single-session model is the session None
        self.sessions: Dict[Any, Tuple[str, List[ModSpec]]] = {}
        self.multi_session = getattr(model, "session_embeddings", None) is not None
        for prefix, enc, dec in groups:
            names = list(dec.keys())
            if names != list(enc.keys()):
                raise NotImplementedError("encoder and decoder must embed the same modalities in the same order")
            key = prefix.split(".")[1] if self.multi_session else None
            self.sessions[key] = (prefix, [ModSpec(n, model.mod_to_indx[n], enc[n].n_channel,
                                                   loss_kind.get(n, "mse")) for n in names])
        self.mods = next(iter(self.sessions.values()))[1]
        self.embed_scale = float(hp["embed_scale"])
        if self.embed_act == ACT_NONE and self.embed_scale != 1.0:
            raise NotImplementedError("identity embedder activation needs scale == 1")
        self.enc_inter = model.encoder[0].mlp.up_proj.out_features
        self.dec_inter = model.decoder[0].mlp.up_proj.out_features
        for nh in (hp["enc_heads"], hp["dec_heads"]):
            if self.H // nh not in (32, 64):
                raise NotImplementedError(f"head size {self.H // nh}: the attention kernels are built for 32 and 64")
        self.T: Optional[int] = None
        # the step's Philox key (dropout sites + device-side mask sampler): derived from the seed of torch's global
        # generator, so torch.manual_seed / the trainer's set_seed (utils/utils.py:20-29) select the stream, WITHOUT
        # drawing from it (the reference Masker's CPU stream must stay untouched for bit-exact masks); engines created
        # later in the same process get different keys.  Advanced once per step; reseed with engine.reseed(value).
        Engine._created += 1
        key = (torch.initial_seed() * 0x9E3779B97F4A7C15 + Engine._created * 0xD1B54A32D192ED03) & 0x3FFFFFFFFFFFFFFF
        self.seed = torch.tensor([key], dtype=torch.int64, device=self.device)
        self.store = ParamStore(model, self.device)
        self.shadows = Shadows(self.store, model, self.sessions)
        self.plans: Dict[Tuple[int, bool, Any, Tuple[str, ...], bool], Plan] = {}
        self.arenas: Dict[Tuple[int, bool], Arena] = {}
        # steps with gradients disabled: forward-only plans, and the arenas they share across sessions
        self.fwd_plans: Dict[Tuple[int, bool, Any, Tuple[str, ...], bool], ForwardPlan] = {}
        self.fwd_arenas: Dict[Tuple[int, bool], Arena] = {}
        self.ddp = None          # set by parallel.DataParallel
        self.use_graphs = os.environ.get("MMFM_CUDA_GRAPHS", "1") != "0"
        self.last_plan: Optional[Plan] = None
        from .model import MultiModalOutput
        self.output_cls = MultiModalOutput      # dropin.install() swaps in the reference's own dataclass

    # ---------------------------------------------------------------------------------------------------
    @torch.inference_mode(False)
    def _plan(self, B: int, T: int, training: bool, session=None, u8_mods: Tuple[str, ...] = (),
              grad_inputs: Tuple[str, ...] = (), fwd_only: bool = False) -> Plan:
        if self.T is None:
            self.T = T
        elif self.T != T:
            for d in (self.plans, self.arenas, self.fwd_plans, self.fwd_arenas):
                d.clear()
            self.T = T
        plans, arenas, cls = (self.fwd_plans, self.fwd_arenas, ForwardPlan) if fwd_only else (self.plans, self.arenas, Plan)
        # deterministic mode selects other kernels: its own plan (and graphs), never a change to a captured one
        # input-gradient plans record extra launches after the default schedule: their own plan, like the two above
        key = (B, training, session, u8_mods, ops.deterministic(), grad_inputs)
        pl = plans.get(key)
        if pl is None:
            recompute = False if fwd_only else self._choose_recompute(B, training, session, u8_mods, grad_inputs)
            arena = None
            if self.multi_session:
                akey = (B, training, bool(grad_inputs), recompute)
                arena = arenas.get(akey)
                if arena is None:
                    arena = arenas[akey] = Arena(self._arena_bytes(cls, B, training, grad_inputs, recompute),
                                                 self.device)
            pl = cls(self, B, training, session, arena, u8_mods, grad_inputs, recompute=recompute)
            plans[key] = pl
        return pl

    def _arena_bytes(self, cls, B: int, training: bool, grad_inputs, recompute: bool) -> int:
        """Size of the activation arena the sessions' plans share: the widest session's (buffers grow monotonically
        with the channels; with input gradients, every modality's), from a dry plan."""
        widest = max(self.sessions, key=lambda k: sum(m.C for m in self.sessions[k][1]))
        gi = tuple(m.name for m in self.sessions[widest][1]) if grad_inputs else ()
        return cls(self, B, training, widest, grad_inputs=gi, recompute=recompute, dry=True).arena_bytes + (1 << 20)

    def _plan_need(self, B: int, training: bool, session, u8_mods, grad_inputs, recompute: bool) -> int:
        """Device bytes that building this training plan allocates: the dry plan's nbytes, with the shared arena of a
        multi-session model in place of the plan's share of it (nothing when that arena exists already)."""
        dry = Plan(self, B, training, session, None, u8_mods, grad_inputs, recompute=recompute, dry=True)
        if not self.multi_session:
            return dry.nbytes
        have = (B, training, bool(grad_inputs), recompute) in self.arenas
        arena = 0 if have else _round_alloc(self._arena_bytes(Plan, B, training, grad_inputs, recompute))
        return dry.nbytes - dry.arena_bytes + arena

    def _step_transient_bytes(self, B: int, session, grad_inputs) -> int:
        """Device bytes a training step allocates outside its plan: the loss / mod_loss / preds clones, the returned
        masks and example counts, and the input gradients."""
        mods, T = self.sessions[session][1], self.T
        n = _round_alloc(4) + _round_alloc(4 * len(mods)) + _round_alloc(8 * len(mods)) + _round_alloc(8 * B * len(mods) * T)
        n += sum(_round_alloc(4 * B * T * m.C) * (2 if m.name in grad_inputs else 1) for m in mods)
        return n

    def _choose_recompute(self, B: int, training: bool, session, u8_mods, grad_inputs) -> bool:
        """True when the training plan that saves every activation does not fit in the memory torch may still use on
        this device; it then records a recompute plan (Plan.recompute) instead, once, for this plan key."""
        full = self._plan_need(B, training, session, u8_mods, grad_inputs, False)
        free, total = torch.cuda.mem_get_info(self.device)
        flat = _round_alloc(4 * self.store.total)
        margin = step_margin(self._step_transient_bytes(B, session, grad_inputs), flat, len(self.store.moments) > 0)
        avail = memory_for_plan(free, total, torch.cuda.memory_reserved(self.device),
                                torch.cuda.memory_allocated(self.device),
                                torch.cuda.get_per_process_memory_fraction(self.device), margin)
        if full <= avail:
            return False
        rec = self._plan_need(B, training, session, u8_mods, grad_inputs, True)
        warnings.warn(f"batch size {B}: the training plan needs {full} bytes of device memory, {avail} are available; "
                      f"recomputing each layer's activations in the backward instead (plan of {rec} bytes)")
        return True

    def reseed(self, value: int) -> None:
        """Set the step seed (the Philox key of the dropout / mask streams); the next step uses value + one increment."""
        self.seed.fill_(int(value) & 0x3FFFFFFFFFFFFFFF)

    def step(self, mod_dict: Dict[str, Dict[str, Any]]):
        model = self.model
        MultiModalOutput = self.output_cls
        if not self.store.adopted():
            self.store.adopt()
        session = None
        if self.multi_session:
            # one session per batch (trainer/base.py:65); the batch's eid selects its embedders and heads
            eid = next(iter(mod_dict.values())).get("eid")
            session = model.session_key(eid)
            if session not in self.sessions:
                raise MmfmError(f"unknown session {eid!r}: the model holds {sorted(self.sessions)[:4]} ...")
        mods = self.sessions[session][1]
        names = [m.name for m in mods]
        if list(mod_dict.keys()) != names:
            raise MmfmError(f"mod_dict must hold exactly the modalities {names} in this order")
        d0 = mod_dict[names[0]]
        if d0["inputs"].dim() == 2:
            raise MmfmError("first modality must be (B,T,C)")
        B, T = d0["inputs"].shape[:2]
        training = bool(model.training)
        # uint8 wire format (spike counts as bytes): only for modalities that take the GEMM embedder path
        u8_mods = tuple(m.name for m in mods if not m.small and mod_dict[m.name]["inputs"].dtype == torch.uint8)
        for m in mods:
            if mod_dict[m.name]["inputs"].dtype == torch.uint8 and m.name not in u8_mods:
                raise MmfmError(f"modality {m.name}: uint8 inputs are only supported for spike-count modalities (C > {SMALL_C})")
        grad_on = torch.is_grad_enabled()
        if grad_on:
            for m in mods:
                tg = mod_dict[m.name]["targets"]
                if torch.is_tensor(tg) and tg.requires_grad:
                    raise NotImplementedError(f"modality {m.name}: targets that require grad are not supported (the "
                                              "targets are data here; only inputs and parameters get gradients)")
        # modalities whose (floating-point) inputs require grad: extra inputs of the autograd node
        grad_inputs = tuple(m.name for m in mods if grad_on and mod_dict[m.name]["inputs"].requires_grad)
        pl = self._plan(B, T, training, session, u8_mods, grad_inputs, fwd_only=not grad_on)
        thresh = [0] * len(mods)
        for k, m in enumerate(mods):
            d = mod_dict[m.name]
            if d["inputs"].dim() == 2:                                   # mm.py:248-250
                d["inputs"] = d["inputs"].unsqueeze(-1)
                d["targets"] = d["targets"].unsqueeze(-1)
            if d.get("masking_mode"):
                raise NotImplementedError("mask_type 'input' (mm.py:256-263) is broken in the reference itself "
                                          "(UnboundLocalError at mm.py:272); only masking_mode=None is supported")
            if tuple(d["inputs"].shape) != (B, T, m.C):
                raise MmfmError(f"modality {m.name}: inputs shape {tuple(d['inputs'].shape)} != {(B, T, m.C)}")
            if m.name in u8_mods:
                if d["targets"].dtype != torch.uint8:
                    raise MmfmError(f"modality {m.name}: uint8 inputs need uint8 targets")
                pl.inp_u8[m.name].copy_(d["inputs"], non_blocking=True)
                pl.tgt_u8[m.name].copy_(d["targets"], non_blocking=True)
            else:
                pl.inp[m.name].copy_(d["inputs"].detach(), non_blocking=True)
                pl.tgt[m.name].copy_(d["targets"], non_blocking=True)
            pl.attn[m.name].copy_(d["inputs_attn_mask"], non_blocking=True)
            pl.ts[m.name].copy_(d["inputs_timestamp"], non_blocking=True)
            im = d.get("inputs_modality")
            if not (torch.is_tensor(im) and im.is_cuda) and im is not None and int(im) != m.index:   # no D2H sync
                raise MmfmError(f"modality {m.name}: inputs_modality {int(im)} != {m.index}")
            em = d.get("eval_mask")
            if em is None:                                               # mm.py:266-267
                mk = model.masker
                stream = adapter.mask_stream(model)
                if _masker.inactive(mk):
                    pl.mask[m.name].zero_()
                elif stream == "device" and _masker.device_samplable(mk):
                    thresh[k] = max(1, min(0xFFFFFFFF, int(float(mk.ratio) * 4294967296.0)))
                else:
                    regions = d.get("inputs_regions") if m.name == "ap" else None          # mm.py:254
                    col = _masker.sample_mask_column(mk, (B, T, m.C), regions,
                                                     "fast" if stream == "device" else stream)
                    pl._mask_stage[m.name].copy_to(pl.mask[m.name], col)
            elif isinstance(em, (bool, int)):
                # compact form (SURVEY 8f rank 3): the trainer's encoding / decoding masks are all-ones or all-zeros
                # (trainer/base.py:85-96); a scalar says so without a dense (B,T,N) int64 tensor
                pl.mask[m.name].fill_(int(bool(em)))
            elif em.dim() == 2:                                          # compact form: the (B,T) column the model reads
                pl.mask[m.name].copy_(em, non_blocking=True)
            else:                                                        # mm.py:269-270: only column 0 matters
                pl.mask[m.name].copy_(em[:, :, 0], non_blocking=True)
        pl.set_sample_thresh(thresh)
        self.last_plan = pl
        anchor = None
        if grad_on:
            anchor = next((p for p in self.store.params.values() if p.requires_grad), None)
        if anchor is not None or grad_inputs:
            loss, mod_loss, *preds = _StepFn.apply(anchor, self, pl, *[mod_dict[n]["inputs"] for n in grad_inputs])
        else:
            pl.run_forward()
            loss = pl.loss.clone().reshape(())
            mod_loss = pl.mod_loss.clone()
            # fresh tensors, like the reference: the plan's buffers are overwritten by the next step
            preds = [pl.preds[m.name].clone() for m in mods]
        out_loss, out_n, out_p, out_t = {}, {}, {}, {}
        nex = pl.nex.clone()
        tmask = pl.tmask.view(B, len(mods), T).to(torch.int64)
        for k, m in enumerate(mods):
            d = mod_dict[m.name]
            out_loss[m.name] = mod_loss[k]
            out_n[m.name] = nex[k]
            out_p[m.name] = preds[k]
            out_t[m.name] = d["targets"]
            # the reference leaves these keys in the caller's dict (mm.py:272-275, decoder_embeddings.py:91,107)
            d["preds"] = out_p[m.name]
            d["gt"] = d["targets"]
            d["inputs_mask"] = d["targets_mask"] = tmask[:, k]
            d["encoder_attn_mask"] = d["decoder_attn_mask"] = d["inputs_attn_mask"]
        return MultiModalOutput(loss=loss, mod_loss=out_loss, mod_n_examples=out_n, mod_preds=out_p, mod_targets=out_t)

    # ---------------------------------------------------------------------------------------------------
    def backward(self, pl: Plan, grad_loss: Optional[torch.Tensor], grad_mod: Optional[torch.Tensor] = None,
                 grad_preds: Sequence[Optional[torch.Tensor]] = ()) -> None:
        """Backward of the plan's last forward for upstream gradients of loss, mod_loss and preds (None = absent).
        A gradient of loss alone runs the default schedule with gscale = grad_loss; anything else first rewrites the
        head gradient dpreds (Plan.head_grad) and runs the same schedule with gscale = 1."""
        st = self.store
        fresh = all(p.grad is None for p in st.params.values())
        prev = None
        if not fresh:
            # gradient accumulation: keep what is there, compute this step into a clean buffer, then add
            if all(p.grad is None or p.grad.data_ptr() == st.g(n).data_ptr() for n, p in st.params.items()):
                prev = st.grad.clone()
            else:
                prev = torch.zeros_like(st.grad)
                for n, p in st.params.items():
                    if p.grad is not None:
                        st.view(prev, n).copy_(p.grad)
        if grad_loss is not None and grad_mod is None and all(g is None for g in grad_preds) and not pl.grad_inputs:
            if pl._dpreds_dirty:
                pl.head_grad(pl.one, None, ())
            pl.gscale.copy_(grad_loss.reshape(1).to(torch.float32))
        else:
            pl.head_grad(grad_loss, grad_mod, grad_preds)
            pl.gscale.fill_(1.0)
        if self.ddp is not None:
            self.ddp.run_backward(pl)
        else:
            pl.run_backward()
        if prev is not None:
            st.grad.add_(prev)
        gv = st.grad_views()
        for n, p in st.params.items():
            if p.grad is not gv[n] and p.requires_grad:
                p.grad = gv[n]
