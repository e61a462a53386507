"""Thin tensor-level wrappers over the C ABI (one Python function per entry point of ``include/mmfm_b200.h``).

Every wrapper takes CUDA tensors the caller allocated, checks dtype/contiguity, and launches on torch's current
stream.  Nothing here computes anything on its own -- there is no fallback when the library is missing.
The ``record`` hook lets :mod:`engine` pre-bind a whole step into a flat list of ``(cfunc, args)`` pairs.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import (ACT_DGELU, ACT_DSOFTSIGN, ACT_GELU, ACT_NONE, ACT_SOFTSIGN, LOSS_MSE, LOSS_POISSON, MASK_CAUSAL,
                   MASK_KEY, MASK_KEY_OR_DIAG, AttnArgs, CastItem, Dropout, GemmArgs, MaskArgs, check, lib)

bf16 = torch.bfloat16


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class DropSpec:
    """Dropout site description: probability quantised to 1/256 (see oracle/philox_ref.py)."""

    __slots__ = ("seed", "site", "thresh", "scale")

    def __init__(self, seed: Optional[torch.Tensor], site: int, p: float):
        t = int(round(float(p) * 256.0))
        t = max(0, min(255, t))
        if seed is None:
            t = 0
        self.seed = seed
        self.site = int(site)
        self.thresh = t
        self.scale = 256.0 / (256.0 - t)

    def c(self) -> Dropout:
        return Dropout(_p(self.seed) if self.thresh else None, self.site, self.thresh, self.scale)


NO_DROP = DropSpec(None, 0, 0.0)


class Recorder:
    """Collects launches instead of issuing them (used to pre-bind a step; see engine.py)."""

    def __init__(self):
        self.calls: List[Tuple[Callable, tuple, str]] = []
        self.keep: List[object] = []   # ctypes structs must outlive the recorded calls

    def add(self, fn, args, what, meta=None):
        self.calls.append((fn, args, what, meta or {}))


_REC: Optional[Recorder] = None


def set_recorder(r: Optional[Recorder]) -> None:
    global _REC
    _REC = r


def _launch(name: str, *args, keep=(), meta=None):
    fn = getattr(lib(), name)
    if _REC is not None:
        _REC.keep.extend(keep)
        _REC.add(fn, args, name, meta)
        return
    check(fn(*args, _stream()), name)


# ------------------------------------------------------------------------------------------------------------
# deterministic mode: on exactly when torch.are_deterministic_algorithms_enabled()
# ------------------------------------------------------------------------------------------------------------
def deterministic() -> bool:
    return torch.are_deterministic_algorithms_enabled()


def det_ws_need(kind: int, d0: int, d1: int = 1, d2: int = 0) -> Tuple[int, int]:
    """(bytes, tickets) of the workspace one *_det call of `kind` needs at these sizes (host only)."""
    nb, nt = C.c_longlong(0), C.c_int(0)
    check(lib().mmfm_det_ws_bytes(kind, int(d0), int(d1), int(d2), C.byref(nb), C.byref(nt)), "mmfm_det_ws_bytes")
    return nb.value, nt.value


class DetWorkspace:
    """Workspace of the *_det entry points: a byte buffer and zeroed tickets, shared by calls on one stream.  The C
    struct is passed by reference, so a recorded schedule can be sized after recording (``materialize``)."""

    def __init__(self):
        self.c = _lib.DetWs(None, 0, None, 0)
        self.want_bytes, self.want_tickets = 0, 0
        self.buf: Optional[torch.Tensor] = None
        self.tickets: Optional[torch.Tensor] = None

    def require(self, nbytes: int, n_tickets: int) -> None:
        self.want_bytes = max(self.want_bytes, int(nbytes))
        self.want_tickets = max(self.want_tickets, int(n_tickets))

    def materialize(self, device) -> None:
        """(Re)allocate when the recorded needs outgrow the buffers; the tickets start at zero."""
        if self.buf is None or self.buf.numel() < self.want_bytes:
            self.buf = torch.empty(max(16, self.want_bytes), dtype=torch.uint8, device=device)
        if self.tickets is None or self.tickets.numel() < self.want_tickets:
            self.tickets = torch.zeros(max(1, self.want_tickets), dtype=torch.int32, device=device)
        self.c.buf, self.c.bytes = self.buf.data_ptr(), self.buf.numel()
        self.c.tickets, self.c.n_tickets = self.tickets.data_ptr(), self.tickets.numel()


def _launch_det(name: str, ws: Optional[DetWorkspace], need: Tuple[int, int], device, *args, keep=(), meta=None):
    """Launch the *_det twin of `name` on `ws` (a private workspace when None)."""
    if ws is None:
        ws = DetWorkspace()
    ws.require(*need)
    if _REC is None:
        ws.materialize(device)
    _launch(name + "_det", *args, C.byref(ws.c), keep=(*keep, ws), meta=meta)


def run_recorded(calls) -> None:
    st = _stream()
    for c in calls:
        rc = c[0](*c[1], st)
        if rc != 0:
            check(rc, c[2])


def count_kernels(calls) -> int:
    """Kernels launched by a recorded schedule (a C call is one kernel unless its meta says otherwise)."""
    return sum(int(c[3].get("kernels", 1)) for c in calls)


def run_recorded_timed(calls):
    """One eager pass with ONE CUDA event at every launch boundary; returns [(name, meta, ms)] where ms spans from the
    boundary before the call to the boundary after it (so the times sum to the pass; profiling aid for bench.py: events
    on the launching stream, never used for the headline number)."""
    st = _stream()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(calls) + 1)]
    evs[0].record()
    for i, c in enumerate(calls):
        rc = c[0](*c[1], st)
        evs[i + 1].record()
        if rc != 0:
            check(rc, c[2])
    torch.cuda.synchronize()
    return [(c[2], c[3], evs[i].elapsed_time(evs[i + 1])) for i, c in enumerate(calls)]


# ------------------------------------------------------------------------------------------------------------
def gemm_tn(A: torch.Tensor, B: torch.Tensor, D: torch.Tensor, *, M: Optional[int] = None, N: Optional[int] = None,
            K: Optional[int] = None, bias: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None,
            D2: Optional[torch.Tensor] = None, aux: Optional[torch.Tensor] = None, act: int = ACT_NONE,
            act_scale: float = 1.0, drop: DropSpec = NO_DROP, remap: Tuple[int, int, int] = (0, 0, 0),
            row_zero: Optional[torch.Tensor] = None, lda: Optional[int] = None, ldb: Optional[int] = None,
            ldd: Optional[int] = None, ldr: Optional[int] = None, ldaux: Optional[int] = None,
            rowdot: Optional[torch.Tensor] = None, rowdot_S: int = 0) -> None:
    """D = epilogue(A . B^T); A [M,K] bf16, B [N,K] bf16 (row pitches from the tensors unless given)."""
    assert A.dtype == bf16 and B.dtype == bf16 and D.dtype in (bf16, torch.float32)
    a = GemmArgs()
    a.A, a.lda = A.data_ptr(), (lda if lda is not None else A.stride(0))
    a.B, a.ldb = B.data_ptr(), (ldb if ldb is not None else B.stride(0))
    a.M = M if M is not None else A.shape[0]
    a.N = N if N is not None else B.shape[0]
    a.K = K if K is not None else A.shape[1]
    a.D, a.ldd = D.data_ptr(), (ldd if ldd is not None else D.stride(0))
    a.d_fp32 = 1 if D.dtype == torch.float32 else 0
    a.D2 = _p(D2)
    if bias is not None:
        assert bias.dtype == torch.float32
    a.bias = _p(bias)
    if res is not None:
        assert res.dtype == torch.float32
    a.res, a.ldr = _p(res), (ldr if ldr is not None else (res.stride(0) if res is not None else 0))
    a.aux, a.ldaux = _p(aux), (ldaux if ldaux is not None else (aux.stride(0) if aux is not None else 0))
    a.act, a.act_scale = act, act_scale
    a.drop = drop.c()
    a.remap_T, a.remap_S, a.remap_off = remap
    a.row_zero = _p(row_zero)
    if rowdot is not None:
        assert rowdot.dtype == torch.float32 and rowdot_S > 0
    a.rowdot, a.rowdot_S = _p(rowdot), int(rowdot_S)
    mn = float(a.M) * a.N
    nbytes = 2.0 * a.M * a.K + 2.0 * a.N * a.K + mn * (4 if a.d_fp32 else 2)      # algorithmic: A + B + D ...
    nbytes += (2.0 * mn if D2 is not None else 0.0) + (4.0 * mn if res is not None else 0.0) + (2.0 * mn if aux is not None else 0.0)
    _launch("mmfm_gemm_tn", C.byref(a), keep=(a,),
            meta={"flops": 2.0 * a.M * a.N * a.K, "bytes": nbytes, "tag": f"gemm_tn {a.M}x{a.N}x{a.K}"})


def gemm_wgrad(dY: torch.Tensor, X: torch.Tensor, dW: torch.Tensor, *, R: Optional[int] = None,
               NO: Optional[int] = None, KI: Optional[int] = None, ldw: Optional[int] = None,
               dbias: Optional[torch.Tensor] = None, ws: Optional[DetWorkspace] = None) -> None:
    """dW[NO,KI] += dY[R,NO]^T . X[R,KI] ; dbias[NO] += colsum(dY) (optional)"""
    assert dY.dtype == bf16 and X.dtype == bf16 and dW.dtype == torch.float32
    R = R if R is not None else dY.shape[0]
    NO = NO if NO is not None else dY.shape[1]
    KI = KI if KI is not None else X.shape[1]
    args = (dY.data_ptr(), dY.stride(0), X.data_ptr(), X.stride(0), R, NO, KI, dW.data_ptr(),
            ldw if ldw is not None else KI, _p(dbias))
    meta = {"flops": 2.0 * R * NO * KI, "bytes": 2.0 * R * (NO + KI) + 4.0 * NO * KI, "tag": f"wgrad {R}x{NO}x{KI}"}
    if deterministic():
        _launch_det("mmfm_gemm_wgrad", ws, det_ws_need(_lib.DET_WGRAD, R, NO, KI), dW.device, *args, meta=meta)
        return
    _launch("mmfm_gemm_wgrad", *args, meta=meta)


def colsum_bf16(dY: torch.Tensor, out: torch.Tensor, *, R: Optional[int] = None, NO: Optional[int] = None,
                ws: Optional[DetWorkspace] = None) -> None:
    R = R if R is not None else dY.shape[0]
    NO = NO if NO is not None else dY.shape[1]
    args = (dY.data_ptr(), dY.stride(0), R, NO, out.data_ptr())
    if deterministic():
        _launch_det("mmfm_colsum_bf16", ws, det_ws_need(_lib.DET_COLSUM, R, NO), out.device, *args)
        return
    _launch("mmfm_colsum_bf16", *args)


def cast_bf16(x: torch.Tensor, y: Optional[torch.Tensor], yt: Optional[torch.Tensor] = None, *, R: Optional[int] = None,
              Cc: Optional[int] = None, ldx: Optional[int] = None) -> None:
    assert x.dtype == torch.float32
    R = R if R is not None else x.shape[0]
    Cc = Cc if Cc is not None else x.shape[1]
    _launch("mmfm_cast_bf16", x.data_ptr(), ldx if ldx is not None else x.stride(0), _p(y),
            y.stride(0) if y is not None else 0, _p(yt), yt.stride(0) if yt is not None else 0, R, Cc,
            meta={"bytes": float(R) * Cc * (4 + 2 * (y is not None) + 2 * (yt is not None))})


def cast_bf16_multi(items_dev: torch.Tensor, n_items: int, total_tiles: int) -> None:
    _launch("mmfm_cast_bf16_multi", items_dev.data_ptr(), n_items, total_tiles)


def scale_inplace(x: torch.Tensor, scale_dev: torch.Tensor) -> None:
    _launch("mmfm_scale_inplace", x.data_ptr(), x.numel(), scale_dev.data_ptr())


def csr_to_dense_u8(data: torch.Tensor, indices: torch.Tensor, row_ptr: torch.Tensor, out: torch.Tensor, *,
                    n_rows: int, n_cols: int) -> None:
    assert out.dtype == torch.uint8 and out.is_contiguous() and out.numel() == n_rows * n_cols
    _launch("mmfm_csr_to_dense_u8", _p(data) if data.numel() else None, _p(indices) if indices.numel() else None,
            row_ptr.data_ptr(), n_rows, n_cols, out.data_ptr(), meta={"bytes": float(n_rows) * n_cols + 5.0 * data.numel()})


def u8_expand(x: torch.Tensor, y32: Optional[torch.Tensor], y16: Optional[torch.Tensor], *, R: int, Cc: int) -> None:
    """uint8 [R, Cc] (dense) -> fp32 [R, *] and / or bf16 [R, *] (row pitches from the tensors)."""
    assert x.dtype == torch.uint8 and x.is_contiguous()
    _launch("mmfm_u8_expand", x.data_ptr(), R, Cc, _p(y32), y32.stride(0) if y32 is not None else 0, _p(y16),
            y16.stride(0) if y16 is not None else 0, meta={"bytes": float(R) * Cc * (1 + (4 if y32 is not None else 0) + (2 if y16 is not None else 0))})


def column_stats(pred: torch.Tensor, y: torch.Tensor, out: torch.Tensor, *, log_rate: bool,
                 ws: Optional[DetWorkspace] = None) -> None:
    R, Cc = pred.shape
    args = (pred.data_ptr(), y.data_ptr(), R, Cc, 1 if log_rate else 0, out.data_ptr())
    if deterministic():
        _launch_det("mmfm_column_stats", ws, det_ws_need(_lib.DET_COLUMN_STATS, R, Cc), out.device, *args,
                    meta={"bytes": 8.0 * R * Cc})
        return
    _launch("mmfm_column_stats", *args, meta={"bytes": 8.0 * R * Cc})


def adamw_step(p: torch.Tensor, g: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, *, lr: float,
               beta1: float, beta2: float, eps: float, weight_decay: float, step: int) -> None:
    n = p.numel()
    _launch("mmfm_adamw_step", p.data_ptr(), g.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), n, float(lr),
            float(beta1), float(beta2), float(eps), float(weight_decay), int(step), meta={"bytes": 28.0 * n})


def adamw_multi(p: torch.Tensor, g: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor,
                segs_dev: torch.Tensor, n_segs: int, n_chunks: int, classes, n_elems: int) -> None:
    """AdamW over the segments of an uploaded table (``segs_dev``: bytes of ``_lib.AdamwSeg[n_segs]`` on the device),
    one ``_lib.AdamwClass`` per class; ``n_elems`` = elements the segments cover (traffic accounting only)."""
    arr = (_lib.AdamwClass * len(classes))(*classes)
    _launch("mmfm_adamw_multi", p.data_ptr(), g.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), p.numel(),
            segs_dev.data_ptr(), int(n_segs), int(n_chunks), arr, len(classes), keep=(arr,),
            meta={"bytes": 28.0 * n_elems})


def layernorm_fwd(x, gamma, beta, y, mean, rstd, *, R: int, H: int, eps: float = 1e-5, modmajor_T: int = 0,
                  S: int = 0) -> None:
    _launch("mmfm_layernorm_fwd", x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), mean.data_ptr(),
            rstd.data_ptr(), R, H, eps, modmajor_T, S, meta={"bytes": 6.0 * R * H})


def layernorm_bwd(dy, x, mean, rstd, gamma, dres, dx, dxb, drop: DropSpec, dgamma, dbeta, *, R: int, H: int,
                  modmajor_T: int = 0, S: int = 0, ws: Optional[DetWorkspace] = None) -> None:
    d = drop.c()
    args = (dy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(), _p(dres), _p(dx), _p(dxb),
            C.byref(d), _p(dgamma), _p(dbeta), R, H, modmajor_T, S)
    meta = {"bytes": float(R) * H * (2 + 4 + (4 if dres is not None else 0) + (4 if dx is not None else 0)
                                     + (2 if dxb is not None else 0))}
    if deterministic():
        _launch_det("mmfm_layernorm_bwd", ws, det_ws_need(_lib.DET_LN_BWD, R, H), x.device, *args, keep=(d,), meta=meta)
        return
    _launch("mmfm_layernorm_bwd", *args, keep=(d,), meta=meta)


def layernorm_fwd_multi(x, gammas, betas, ys, mean, rstd, *, R: int, H: int, eps: float = 1e-5) -> None:
    """Several LayerNorms over one input (the decoder layers' context_norm): x is read once, len(ys) bf16 outputs."""
    a = _lib.LnMultiArgs()
    a.x, a.R, a.H, a.n, a.eps = x.data_ptr(), R, H, len(ys), eps
    for l, (g, b, y) in enumerate(zip(gammas, betas, ys)):
        a.gamma[l], a.beta[l], a.y[l] = g.data_ptr(), b.data_ptr(), y.data_ptr()
    a.mean, a.rstd = mean.data_ptr(), rstd.data_ptr()
    _launch("mmfm_layernorm_fwd_multi", C.byref(a), keep=(a,), meta={"bytes": float(R) * H * (4 + 2 * len(ys))})


def layernorm_bwd_multi(dys, x, mean, rstd, gammas, dx, dxb, dgammas, dbetas, *, R: int, H: int,
                        ws: Optional[DetWorkspace] = None) -> None:
    """dx = LN'(sum_l dy_l . gamma_l) (written, not accumulated) + optional bf16 copy; dgamma_l / dbeta_l accumulate."""
    a = _lib.LnMultiArgs()
    a.x, a.R, a.H, a.n, a.eps = x.data_ptr(), R, H, len(dys), 0.0
    for l, (dy, g, dg, db) in enumerate(zip(dys, gammas, dgammas, dbetas)):
        a.dy[l], a.gamma[l], a.dgamma[l], a.dbeta[l] = dy.data_ptr(), g.data_ptr(), _p(dg), _p(db)
    a.mean, a.rstd, a.dx, a.dxb = mean.data_ptr(), rstd.data_ptr(), dx.data_ptr(), _p(dxb)
    meta = {"bytes": float(R) * H * (4 + 2 * len(dys) + 4 + (2 if dxb is not None else 0))}
    if deterministic():
        _launch_det("mmfm_layernorm_bwd_multi", ws, det_ws_need(_lib.DET_LN_BWD_MULTI, R, H, len(dys)), x.device,
                    C.byref(a), keep=(a,), meta=meta)
        return
    _launch("mmfm_layernorm_bwd_multi", C.byref(a), keep=(a,), meta=meta)


def scalenorm_fwd(x, g, y, rnorm, *, R: int, H: int, eps: float = 1e-5) -> None:
    _launch("mmfm_scalenorm_fwd", x.data_ptr(), g.data_ptr(), y.data_ptr(), rnorm.data_ptr(), R, H, eps,
            meta={"bytes": 6.0 * R * H})


def scalenorm_bwd(dy, x, rnorm, g, dres, dx, dxb, drop: DropSpec, dg, *, R: int, H: int, eps: float = 1e-5,
                  ws: Optional[DetWorkspace] = None) -> None:
    d = drop.c()
    args = (dy.data_ptr(), x.data_ptr(), rnorm.data_ptr(), g.data_ptr(), _p(dres), _p(dx), _p(dxb), C.byref(d), _p(dg),
            R, H, eps)
    meta = {"bytes": float(R) * H * (2 + 4 + (4 if dres is not None else 0) + (4 if dx is not None else 0)
                                     + (2 if dxb is not None else 0))}
    if deterministic():
        _launch_det("mmfm_scalenorm_bwd", ws, det_ws_need(_lib.DET_SCALENORM_BWD, R, H), x.device, *args, keep=(d,),
                    meta=meta)
        return
    _launch("mmfm_scalenorm_bwd", *args, keep=(d,), meta=meta)


def _attn_args(q, k, v, o, lse, key_valid, *, B, n_heads, Sq, Sk, d_head, mask_mode, mod_q=None, mod_k=None,
               drop_p: DropSpec = NO_DROP, drop_o: DropSpec = NO_DROP, p_keep=None, d_o=None, delta=None, dq=None,
               dk=None, dv=None, prep_done: bool = False) -> AttnArgs:
    a = AttnArgs()
    a.q, a.ldq = q.data_ptr(), q.stride(0)
    a.k, a.ldk = k.data_ptr(), k.stride(0)
    a.v, a.ldv = v.data_ptr(), v.stride(0)
    a.o, a.ldo = o.data_ptr(), o.stride(0)
    a.lse = lse.data_ptr()
    a.key_valid = key_valid.data_ptr()
    a.mod_q, a.mod_k = _p(mod_q), _p(mod_k)
    a.B, a.n_heads, a.Sq, a.Sk, a.d_head = B, n_heads, Sq, Sk, d_head
    a.mask_mode = mask_mode
    a.scale = float(d_head) ** -0.5
    a.drop_p, a.drop_o = drop_p.c(), drop_o.c()
    a.p_keep = _p(p_keep)
    if d_o is not None:
        a.d_o, a.lddo = d_o.data_ptr(), d_o.stride(0)
        a.delta = delta.data_ptr()
        a.dq, a.lddq = dq.data_ptr(), dq.stride(0)
        a.dk, a.lddk = dk.data_ptr(), dk.stride(0)
        a.dv, a.lddv = dv.data_ptr(), dv.stride(0)
    a.prep_done = 1 if prep_done else 0
    return a


def attention_fwd(q, k, v, o, lse, key_valid, **kw) -> None:
    """q/k/v/o: 2-D bf16 views [B*S, h*d] (row pitch = stride(0)); see include/mmfm_b200.h."""
    a = _attn_args(q, k, v, o, lse, key_valid, **kw)
    _launch("mmfm_attention_fwd", C.byref(a), keep=(a,),
            meta={"flops": 4.0 * a.B * a.n_heads * a.Sq * a.Sk * a.d_head})


def attention_bwd(q, k, v, o, lse, key_valid, **kw) -> None:
    a = _attn_args(q, k, v, o, lse, key_valid, **kw)
    # kernels behind the call: prep + one fused kernel (d_head 32, S <= 256, no modality-separation mask), else
    # prep + dq + dkv (mirrors the dispatch in csrc/attention.cu)
    fused = a.d_head == 32 and a.Sq <= 256 and a.Sk <= 256 and not a.mod_q
    _launch("mmfm_attention_bwd", C.byref(a), keep=(a,),
            meta={"flops": 8.0 * a.B * a.n_heads * a.Sq * a.Sk * a.d_head,   # algorithmic: 2x forward
                  "kernels": (2 if fused else 3) - (1 if a.prep_done else 0)})


def mask_prep(masks: Sequence[Optional[torch.Tensor]], attns: Sequence[torch.Tensor], channels: Sequence[int],
              zero_flags, key_valid, tok_mask, n_examples, inv_n, sample_thresh: Optional[torch.Tensor] = None,
              seed: Optional[torch.Tensor] = None) -> None:
    """masks[m]: (B,T) int64 view (any strides) or None; attns[m]: (B,T) int64 view.  sample_thresh: optional device
    int32/uint32 [n_mod]; a non-zero entry makes the kernel draw that modality's Bernoulli mask itself (see the header)."""
    a = MaskArgs()
    if sample_thresh is not None:
        assert sample_thresh.element_size() == 4 and sample_thresh.numel() >= len(attns) and seed is not None
    a.sample_thresh, a.seed = _p(sample_thresh), _p(seed)
    a.n_mod = len(attns)
    a.B, a.T = attns[0].shape
    for m, (mk, at) in enumerate(zip(masks, attns)):
        assert at.dtype == torch.int64 and (mk is None or mk.dtype == torch.int64)
        if mk is not None:
            a.mask[m], a.mask_sb[m], a.mask_st[m] = mk.data_ptr(), mk.stride(0), mk.stride(1)
        else:
            a.mask[m] = None
        a.attn[m], a.attn_sb[m], a.attn_st[m] = at.data_ptr(), at.stride(0), at.stride(1)
        a.channels[m] = int(channels[m])
    _launch("mmfm_mask_prep", C.byref(a), zero_flags.data_ptr(), key_valid.data_ptr(), tok_mask.data_ptr(),
            n_examples.data_ptr(), inv_n.data_ptr(), keep=(a,))


def embed_assemble(mod_row, pos, ts, emb, *, B, T, S, off, H) -> None:
    _launch("mmfm_embed_assemble", mod_row.data_ptr(), _p(pos), _p(ts), emb.data_ptr(), B, T, S, off, H,
            meta={"bytes": 4.0 * B * T * H})                       # emb rows written (the tables stay in cache)


def embed_assemble_bwd(g, g2, ts, dpos, dmod, *, B, T, S, off, H, ws: Optional[DetWorkspace] = None) -> None:
    args = (g.data_ptr(), _p(g2), _p(ts), _p(dpos), dmod.data_ptr(), B, T, S, off, H)
    meta = {"bytes": 4.0 * B * T * H * (2 if g2 is not None else 1)}   # gradient rows read
    if deterministic():
        n_pos = dpos.shape[0] if dpos is not None else 0
        _launch_det("mmfm_embed_assemble_bwd", ws, det_ws_need(_lib.DET_EMBED_ASM_BWD, B, T, H), g.device, *args, n_pos,
                    meta={**meta, "kernels": 2 if dpos is not None else 1})
        return
    _launch("mmfm_embed_assemble_bwd", *args, meta=meta)


def embed_grad_prep(dx, dtok, row_zero, drop: DropSpec, *, B, T, S, off, H) -> None:
    d = drop.c()
    _launch("mmfm_embed_grad_prep", dx.data_ptr(), dtok.data_ptr(), _p(row_zero), C.byref(d), B, T, S, off, H,
            keep=(d,), meta={"bytes": 6.0 * B * T * H})            # fp32 rows in, bf16 rows out


def smallc_embed_fwd(inp, W1, b1, W2, b2, emb, x, hid, row_zero, drop: DropSpec, act_scale, act, *, B, T, S, off, Cc,
                     H) -> None:
    d = drop.c()
    _launch("mmfm_smallc_embed_fwd", inp.data_ptr(), W1.data_ptr(), _p(b1), W2.data_ptr(), _p(b2), emb.data_ptr(),
            x.data_ptr(), hid.data_ptr(), _p(row_zero), C.byref(d), float(act_scale), act, B, T, S, off, Cc, H,
            keep=(d,), meta={"bytes": float(B) * T * (8.0 * H + 4.0 * Cc + 8.0 * Cc)})   # emb rows in, x rows out


def smallc_embed_bwd(inp, hid, W2, dx, row_zero, drop: DropSpec, act_scale, act, dW1, db1, dW2, db2, *, B, T, S, off,
                     Cc, H, ws: Optional[DetWorkspace] = None) -> None:
    d = drop.c()
    args = (inp.data_ptr(), hid.data_ptr(), W2.data_ptr(), dx.data_ptr(), _p(row_zero), C.byref(d), float(act_scale), act,
            dW1.data_ptr(), db1.data_ptr(), dW2.data_ptr(), db2.data_ptr(), B, T, S, off, Cc, H)
    meta = {"bytes": float(B) * T * (4.0 * H + 12.0 * Cc)}   # dx rows in
    if deterministic():
        _launch_det("mmfm_smallc_embed_bwd", ws, det_ws_need(_lib.DET_SMALLC_EMBED_BWD, B * T, Cc, H), dx.device, *args,
                    keep=(d,), meta=meta)
        return
    _launch("mmfm_smallc_embed_bwd", *args, keep=(d,), meta=meta)


def smallc_head_fwd(y, W, b, preds, *, R, H, Cc) -> None:
    _launch("mmfm_smallc_head_fwd", y.data_ptr(), W.data_ptr(), _p(b), preds.data_ptr(), R, H, Cc,
            meta={"bytes": float(R) * (2.0 * H + 4.0 * Cc)})


def smallc_head_bwd(y, W, dpreds, dy, dW, db, *, R, H, Cc, ws: Optional[DetWorkspace] = None) -> None:
    args = (y.data_ptr(), W.data_ptr(), dpreds.data_ptr(), dpreds.stride(0), dy.data_ptr(), dW.data_ptr(), db.data_ptr(),
            R, H, Cc)
    meta = {"bytes": float(R) * (4.0 * H + 2.0 * Cc)}
    if deterministic():
        _launch_det("mmfm_smallc_head_bwd", ws, det_ws_need(_lib.DET_SMALLC_HEAD_BWD, R, H, Cc), dW.device, *args,
                    meta=meta)
        return
    _launch("mmfm_smallc_head_bwd", *args, meta=meta)


def loss_fwd_bwd(preds, targets, tok_mask, inv_n, kind, partials, dpreds, *, B, T, Cc, S, off) -> None:
    _launch("mmfm_loss_fwd_bwd", preds.data_ptr(), targets.data_ptr(), tok_mask.data_ptr(), S, off, inv_n.data_ptr(),
            kind, B, T, Cc, partials.data_ptr(), partials.numel(), dpreds.data_ptr(), dpreds.stride(0),
            meta={"bytes": 10.0 * B * T * Cc})


def loss_finalize(partials, n_partials, n_mod, inv_n, mod_loss, loss) -> None:
    _launch("mmfm_loss_finalize", partials.data_ptr(), n_partials, n_mod, inv_n.data_ptr(), mod_loss.data_ptr(),
            loss.data_ptr())


def loss_grad(preds, targets, tok_mask, inv_n, kind, dpreds, *, g_loss=None, g_mod=None, g_preds=None, B, T, Cc, S,
              off) -> None:
    """dpreds = mask * ell' * (g_loss * inv_n + g_mod) + g_preds: the head gradient for any upstream gradients of the
    step outputs.  g_loss / g_mod: fp32 device scalars or None; g_preds: fp32 (B, T, Cc) of any strides or None."""
    for g in (g_loss, g_mod, g_preds):
        assert g is None or (g.dtype == torch.float32 and g.is_cuda)
    if g_preds is not None:
        assert tuple(g_preds.shape) == (B, T, Cc)
    sb, st, sc = g_preds.stride() if g_preds is not None else (0, 0, 0)
    _launch("mmfm_loss_grad", preds.data_ptr(), targets.data_ptr(), tok_mask.data_ptr(), S, off, inv_n.data_ptr(),
            _p(g_loss), _p(g_mod), _p(g_preds), sb, st, sc, kind, B, T, Cc, dpreds.data_ptr(), dpreds.stride(0),
            meta={"bytes": float(B) * T * Cc * (10 + (4 if g_preds is not None else 0))})


def smallc_embed_dx(hid, W1, W2, dx, row_zero, drop: DropSpec, act_scale, act, dX, *, accumulate: bool, B, T, S, off,
                    Cc, H) -> None:
    """dX (fp32 [B*T, Cc], pitch from the tensor) (+)= input gradient of the small-channel embedder."""
    assert dX.dtype == torch.float32
    d = drop.c()
    _launch("mmfm_smallc_embed_dx", hid.data_ptr(), W1.data_ptr(), W2.data_ptr(), dx.data_ptr(), _p(row_zero),
            C.byref(d), float(act_scale), act, dX.data_ptr(), dX.stride(0), 1 if accumulate else 0, B, T, S, off, Cc, H,
            keep=(d,), meta={"bytes": float(B) * T * (4.0 * H + 8.0 * Cc)})
