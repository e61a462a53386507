"""ctypes binding of ``libmmfm_b200.so`` (the C ABI declared in ``include/mmfm_b200.h``).

The library is built in-tree by :func:`build` (``nvcc -gencode arch=compute_100a,code=sm_100a``); there is no
CPU fallback: :func:`lib` raises if the shared object is missing or cannot be loaded.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
from typing import List, Optional

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_PKG_DIR, "csrc")
# MMFM_LIB_PATH: load another build of the library (A/B measurements of a kernel change against a saved build)
LIB_PATH = os.environ.get("MMFM_LIB_PATH") or os.path.join(_PKG_DIR, "libmmfm_b200.so")
SOURCES = ["host_util.cu", "gemm.cu", "gemm_ts.cu", "norm.cu", "attention.cu", "attention_pipe.cu", "attention_bwd_stream.cu", "attention_bwd_ws.cu", "glue.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-Xptxas", "-v"]

MAX_MOD = 8
ABI_VERSION = 8
MASK_SITE = 8192


def _nvcc() -> str:
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if p and (os.path.isabs(p) and os.path.exists(p) or not os.path.isabs(p)):
            return p
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
    deps.append(os.path.join(os.path.dirname(_PKG_DIR), "include", "mmfm_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source for sm_100a into one shared library next to this file."""
    if not force and not needs_build():
        return LIB_PATH
    objs: List[str] = []
    build_dir = os.path.join(_PKG_DIR, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        extra = os.environ.get("MMFM_NVCC_EXTRA", "").split()      # e.g. -DMMFM_DBG_TIMING for tools/micro probes
        cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-c", os.path.join(_CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [_nvcc(), "-shared", "-o", LIB_PATH, *objs, "-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link of libmmfm_b200.so failed")
    return LIB_PATH


# ------------------------------------------------------------------------------------------------------------
# struct mirrors (include/mmfm_b200.h)
# ------------------------------------------------------------------------------------------------------------
class Dropout(C.Structure):
    _fields_ = [("seed", C.c_void_p), ("site", C.c_uint32), ("thresh", C.c_uint32), ("scale", C.c_float)]


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("lda", C.c_longlong),
        ("B", C.c_void_p), ("ldb", C.c_longlong),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("D", C.c_void_p), ("ldd", C.c_longlong),
        ("d_fp32", C.c_int),
        ("D2", C.c_void_p),
        ("bias", C.c_void_p),
        ("res", C.c_void_p), ("ldr", C.c_longlong),
        ("aux", C.c_void_p), ("ldaux", C.c_longlong),
        ("act", C.c_int), ("act_scale", C.c_float),
        ("drop", Dropout),
        ("remap_T", C.c_int), ("remap_S", C.c_int), ("remap_off", C.c_int),
        ("row_zero", C.c_void_p),
        ("rowdot", C.c_void_p), ("rowdot_S", C.c_int),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("ldq", C.c_longlong),
        ("k", C.c_void_p), ("ldk", C.c_longlong),
        ("v", C.c_void_p), ("ldv", C.c_longlong),
        ("o", C.c_void_p), ("ldo", C.c_longlong),
        ("lse", C.c_void_p),
        ("key_valid", C.c_void_p),
        ("mod_q", C.c_void_p), ("mod_k", C.c_void_p),
        ("B", C.c_int), ("n_heads", C.c_int), ("Sq", C.c_int), ("Sk", C.c_int), ("d_head", C.c_int),
        ("mask_mode", C.c_int),
        ("scale", C.c_float),
        ("drop_p", Dropout), ("drop_o", Dropout),
        ("p_keep", C.c_void_p),
        ("d_o", C.c_void_p), ("lddo", C.c_longlong),
        ("delta", C.c_void_p),
        ("dq", C.c_void_p), ("lddq", C.c_longlong),
        ("dk", C.c_void_p), ("lddk", C.c_longlong),
        ("dv", C.c_void_p), ("lddv", C.c_longlong),
        ("prep_done", C.c_int),
    ]


class MaskArgs(C.Structure):
    _fields_ = [
        ("n_mod", C.c_int), ("B", C.c_int), ("T", C.c_int),
        ("mask", C.c_void_p * MAX_MOD), ("mask_sb", C.c_longlong * MAX_MOD), ("mask_st", C.c_longlong * MAX_MOD),
        ("attn", C.c_void_p * MAX_MOD), ("attn_sb", C.c_longlong * MAX_MOD), ("attn_st", C.c_longlong * MAX_MOD),
        ("channels", C.c_int * MAX_MOD),
        ("sample_thresh", C.c_void_p), ("seed", C.c_void_p),
    ]


MAX_LN = 8


class LnMultiArgs(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("R", C.c_int), ("H", C.c_int), ("n", C.c_int), ("eps", C.c_float),
        ("gamma", C.c_void_p * MAX_LN), ("beta", C.c_void_p * MAX_LN), ("y", C.c_void_p * MAX_LN),
        ("mean", C.c_void_p), ("rstd", C.c_void_p),
        ("dy", C.c_void_p * MAX_LN), ("dgamma", C.c_void_p * MAX_LN), ("dbeta", C.c_void_p * MAX_LN),
        ("dx", C.c_void_p), ("dxb", C.c_void_p),
    ]


class CastItem(C.Structure):
    _fields_ = [
        ("src", C.c_void_p), ("ld_src", C.c_longlong),
        ("dst", C.c_void_p), ("ld_dst", C.c_longlong),
        ("dst_t", C.c_void_p), ("ld_dst_t", C.c_longlong),
        ("rows", C.c_int), ("cols", C.c_int),
        ("tile_start", C.c_int), ("pad_", C.c_int),
    ]


ADAMW_MAX_CLASSES = 64
ADAMW_CHUNK4 = 1024


class AdamwSeg(C.Structure):
    _fields_ = [("lo", C.c_longlong), ("hi", C.c_longlong), ("cls", C.c_int), ("chunk0", C.c_int)]


class AdamwClass(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("pad_", C.c_int), ("step", C.c_longlong)]


class DetWs(C.Structure):
    _fields_ = [("buf", C.c_void_p), ("bytes", C.c_longlong), ("tickets", C.c_void_p), ("n_tickets", C.c_int)]


ACT_NONE, ACT_GELU, ACT_SOFTSIGN, ACT_DGELU, ACT_DSOFTSIGN, ACT_GELU_DG, ACT_MULAUX, ACT_ROWDOT_DROP = 0, 1, 2, 3, 4, 5, 6, 7
MASK_KEY, MASK_KEY_OR_DIAG, MASK_CAUSAL = 0, 1, 2
LOSS_POISSON, LOSS_MSE, LOSS_CE = 0, 1, 2
(DET_WGRAD, DET_COLSUM, DET_LN_BWD, DET_LN_BWD_MULTI, DET_SCALENORM_BWD, DET_EMBED_ASM_BWD, DET_SMALLC_EMBED_BWD,
 DET_SMALLC_HEAD_BWD, DET_COLUMN_STATS) = range(9)

_vp, _i, _ll, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_float
_DP = C.POINTER(Dropout)
_WS = C.POINTER(DetWs)

# name -> argtypes; every function returns int except the three listed in _SPECIAL
SIGNATURES = {
    "mmfm_gemm_tn": [C.POINTER(GemmArgs), _vp],
    "mmfm_gemm_wgrad": [_vp, _ll, _vp, _ll, _i, _i, _i, _vp, _ll, _vp, _vp],
    "mmfm_colsum_bf16": [_vp, _ll, _i, _i, _vp, _vp],
    "mmfm_cast_bf16": [_vp, _ll, _vp, _ll, _vp, _ll, _i, _i, _vp],
    "mmfm_cast_bf16_multi": [_vp, _i, _i, _vp],
    "mmfm_scale_inplace": [_vp, _ll, _vp, _vp],
    "mmfm_session_grad_combine": [_vp, _vp, _i, _ll, _vp, _vp, _i, _f, _vp],
    "mmfm_csr_to_dense_u8": [_vp, _vp, _vp, _ll, _i, _vp, _vp],
    "mmfm_u8_expand": [_vp, _ll, _i, _vp, _ll, _vp, _ll, _vp],
    "mmfm_column_stats": [_vp, _vp, _ll, _i, _i, _vp, _vp],
    "mmfm_adamw_step": [_vp, _vp, _vp, _vp, _ll, _f, _f, _f, _f, _f, _ll, _vp],
    "mmfm_adamw_multi": [_vp, _vp, _vp, _vp, _ll, _vp, _i, _i, C.POINTER(AdamwClass), _i, _vp],
    "mmfm_layernorm_fwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _i, _i, _vp],
    "mmfm_layernorm_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _DP, _vp, _vp, _i, _i, _i, _i, _vp],
    "mmfm_layernorm_fwd_multi": [C.POINTER(LnMultiArgs), _vp],
    "mmfm_layernorm_bwd_multi": [C.POINTER(LnMultiArgs), _vp],
    "mmfm_scalenorm_fwd": [_vp, _vp, _vp, _vp, _i, _i, _f, _vp],
    "mmfm_scalenorm_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _DP, _vp, _i, _i, _f, _vp],
    "mmfm_attention_fwd": [C.POINTER(AttnArgs), _vp],
    "mmfm_attention_bwd": [C.POINTER(AttnArgs), _vp],
    "mmfm_mask_prep": [C.POINTER(MaskArgs), _vp, _vp, _vp, _vp, _vp, _vp],
    "mmfm_embed_assemble": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "mmfm_embed_assemble_bwd": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "mmfm_embed_grad_prep": [_vp, _vp, _vp, _DP, _i, _i, _i, _i, _i, _vp],
    "mmfm_smallc_embed_fwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _DP, _f, _i, _i, _i, _i, _i, _i, _i, _vp],
    "mmfm_smallc_embed_bwd": [_vp, _vp, _vp, _vp, _vp, _DP, _f, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "mmfm_smallc_head_fwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "mmfm_smallc_head_bwd": [_vp, _vp, _vp, _ll, _vp, _vp, _vp, _i, _i, _i, _vp],
    "mmfm_loss_fwd_bwd": [_vp, _vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _vp, _i, _vp, _ll, _vp],
    "mmfm_loss_finalize": [_vp, _i, _i, _vp, _vp, _vp, _vp],
    "mmfm_loss_grad": [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _ll, _ll, _ll, _i, _i, _i, _i, _vp, _ll, _vp],
    "mmfm_smallc_embed_dx": [_vp, _vp, _vp, _vp, _vp, _DP, _f, _i, _vp, _ll, _i, _i, _i, _i, _i, _i, _i, _vp],
    # deterministic mode: the same arguments plus the workspace (include/mmfm_b200.h)
    "mmfm_det_ws_bytes": [_i, _ll, _ll, _ll, C.POINTER(C.c_longlong), C.POINTER(C.c_int)],
    "mmfm_gemm_wgrad_det": [_vp, _ll, _vp, _ll, _i, _i, _i, _vp, _ll, _vp, _WS, _vp],
    "mmfm_colsum_bf16_det": [_vp, _ll, _i, _i, _vp, _WS, _vp],
    "mmfm_layernorm_bwd_det": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _DP, _vp, _vp, _i, _i, _i, _i, _WS, _vp],
    "mmfm_layernorm_bwd_multi_det": [C.POINTER(LnMultiArgs), _WS, _vp],
    "mmfm_scalenorm_bwd_det": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _DP, _vp, _i, _i, _f, _WS, _vp],
    "mmfm_embed_assemble_bwd_det": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _WS, _vp],
    "mmfm_smallc_embed_bwd_det": [_vp, _vp, _vp, _vp, _vp, _DP, _f, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _WS,
                                  _vp],
    "mmfm_smallc_head_bwd_det": [_vp, _vp, _vp, _ll, _vp, _vp, _vp, _i, _i, _i, _WS, _vp],
    "mmfm_column_stats_det": [_vp, _vp, _ll, _i, _i, _vp, _WS, _vp],
}
_SPECIAL = {
    "mmfm_last_error": ([], C.c_char_p),
    "mmfm_abi_version": ([], C.c_int),
    "mmfm_sm_count": ([], C.c_int),
}
EXPORTED_SYMBOLS = sorted(list(SIGNATURES) + list(_SPECIAL))

_LIB: Optional[C.CDLL] = None


class MmfmError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load (once) and return the library; raises when it is absent -- there is no fallback path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise MmfmError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  The B200 path has no CPU / PyTorch fallback.")
    L = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(L, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    for name, (argtypes, restype) in _SPECIAL.items():
        fn = getattr(L, name)
        fn.argtypes = argtypes
        fn.restype = restype
    if L.mmfm_abi_version() != ABI_VERSION:
        raise MmfmError("libmmfm_b200.so ABI version mismatch")
    _LIB = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().mmfm_last_error()
        raise MmfmError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
