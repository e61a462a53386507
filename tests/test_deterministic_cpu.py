"""Deterministic mode without a GPU: the SASS of the built library (no float atomics in any deterministic kernel, the
deterministic wgrad still on the tensor cores), the workspace sizing against a restatement of the launchers' grid
arithmetic, and the rejection of a workspace that is too small."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from multi_modal_foundation_model_b200 import _lib

FLOAT_ATOMIC = re.compile(r"\b(RED|REDG|ATOM|ATOMG)\.[A-Z0-9.]*ADD\.F(32|64)")


def _sass_by_kernel():
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool) and shutil.which(tool) is None:
        pytest.skip("cuobjdump not available")
    _lib.build()
    out = subprocess.run([tool, "-sass", _lib.LIB_PATH], stdout=subprocess.PIPE, text=True, check=True).stdout
    kernels, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            kernels[cur] = []
        elif cur is not None:
            kernels[cur].append(line)
    return kernels


def _is_det(name: str) -> bool:
    # the deterministic instantiations carry `true` as their last template argument (mangled "Lb1E")
    return "Lb1E" in name or "embed_pos_bwd_det" in name


def test_deterministic_kernels_have_no_float_atomics():
    kernels = _sass_by_kernel()
    det = {k: v for k, v in kernels.items() if _is_det(k)}
    families = ["gemm_wgrad", "colsum_bf16", "layernorm_bwd_kernel", "layernorm_bwd_multi", "scalenorm_bwd",
                "embed_assemble_bwd", "embed_pos_bwd_det", "smallc_embed_bwd_kernel", "smallc_embed_bwd16",
                "smallc_head_bwd", "column_stats"]
    for fam in families:
        assert any(fam in k for k in det), f"no deterministic instantiation of {fam}"
    for k, lines in det.items():
        bad = [l.strip() for l in lines if FLOAT_ATOMIC.search(l)]
        assert not bad, f"{k}: {bad[:3]}"
    # the pattern does find the atomics of the default instantiations
    assert any(FLOAT_ATOMIC.search(l) for k, v in kernels.items() if "gemm_wgrad" in k and not _is_det(k) for l in v)
    wgrad_det = [v for k, v in det.items() if "gemm_wgrad" in k]
    assert wgrad_det and all(any("UTCHMMA" in l for l in v) for v in wgrad_det)


def _sm():
    n = _lib.lib().mmfm_sm_count()
    return n if n > 0 else 148


def _need(kind, d0, d1, d2=0):
    nb, nt = ctypes.c_longlong(0), ctypes.c_int(0)
    assert _lib.lib().mmfm_det_ws_bytes(kind, d0, d1, d2, ctypes.byref(nb), ctypes.byref(nt)) == 0
    return nb.value, nt.value


def _wgrad_restated(R, NO, KI, sm):
    kBM, kBK, BN = 128, 64, 128
    tiles = -(-NO // kBM) * -(-KI // BN)
    kblocks = -(-R // kBK)
    splits = max(1, min((4 * sm // 2) // tiles, kblocks))
    rows = -(-kblocks // splits) * kBK
    splits = -(-R // rows)
    return tiles * splits * (kBM * BN + kBM) * 4, tiles * splits


@pytest.mark.skipif("MMFM_WGRAD_CTAS_X2" in os.environ, reason="restatement assumes the default split target")
@pytest.mark.parametrize("R,NO,KI", [
    (51200, 768, 256), (51200, 256, 256), (51200, 512, 256), (51200, 256, 512), (51200, 668, 256), (25600, 256, 1336),
    (25600, 1336, 668), (25600, 256, 4), (3200, 256, 256), (130, 200, 72), (64, 8, 8),
])
def test_wgrad_workspace_matches_split_arithmetic(R, NO, KI):
    assert _need(_lib.DET_WGRAD, R, NO, KI) == _wgrad_restated(R, NO, KI, _sm())


def test_column_sum_workspaces_match_grids():
    sm = _sm()
    R, H = 51200, 256
    g = min(max(1, -(-R // 32)), 2 * sm)
    assert _need(_lib.DET_LN_BWD, R, H) == (g * 2 * H * 4, g)
    g = min(sm * (2 if (H // 128) * 5 <= 4 else 1), -(-R // 8))
    assert _need(_lib.DET_LN_BWD_MULTI, R, H, 5) == (g * 2 * 5 * H * 4, g)
    assert _need(_lib.DET_COLSUM, 3000, 700) == (2 * 12 * 512 * 4, 24)
    B, T = 256, 100
    chunks = min(B, -(-4 * sm // T))
    chunks = -(-B // -(-B // chunks))
    assert _need(_lib.DET_EMBED_ASM_BWD, B, T, H) == (T * chunks * H * 4, T * chunks)
    gx = min(-(-25600 // 64), 2 * sm)
    assert _need(_lib.DET_SMALLC_HEAD_BWD, 25600, H, 2) == (gx * (8 * 256 + 8) * 4, gx)


def test_bad_kind_and_small_workspace_rejected_on_host():
    L = _lib.lib()
    nb, nt = ctypes.c_longlong(0), ctypes.c_int(0)
    assert L.mmfm_det_ws_bytes(99, 1, 1, 1, ctypes.byref(nb), ctypes.byref(nt)) == -1
    assert b"unknown kind" in L.mmfm_last_error()
    ws = _lib.DetWs(None, 1024, None, 1)
    rc = L.mmfm_gemm_wgrad_det(1, 256, 1, 256, 1000, 256, 256, 1, 256, None, ctypes.byref(ws), None)
    assert rc == -1 and b"workspace too small" in L.mmfm_last_error()
