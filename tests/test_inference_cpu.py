"""The GELU-only epilogue of the TMA-store GEMM (TS_GELU, the MLP-up projection of forward-only plans) without a GPU:
it is built for both tile widths, stores through TMA only, and stores one output where TS_GELU_DG stores two."""
import os
import re
import shutil
import subprocess

import pytest

from multi_modal_foundation_model_b200 import _lib


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


def _ts(kernels, epi, bn):
    (name,) = [k for k in kernels if f"gemm_tn_ts_kernelILi{epi}ELi{bn}E" in k]
    return kernels[name]


@pytest.mark.parametrize("bn", [128, 256])
def test_ts_gelu_stores_one_tensor_map_through_tma(bn):
    kernels = _sass_by_kernel()
    gelu, gelu_dg, plain = _ts(kernels, 3, bn), _ts(kernels, 4, bn), _ts(kernels, 0, bn)
    count = lambda lines, pat: sum(1 for l in lines if re.search(pat, l))
    assert not count(gelu, r"\bSTG\."), "TS_GELU issues global stores"
    n = count(gelu, r"\bUTMASTG\b")
    assert n > 0
    assert n == count(plain, r"\bUTMASTG\b")               # one [128 x 32] box store per slice, like TS_BF16
    assert 2 * n == count(gelu_dg, r"\bUTMASTG\b")         # TS_GELU_DG also stores the derivative
    assert count(gelu, r"\bUTMALDG\b") == count(plain, r"\bUTMALDG\b")     # A / B loads only: no saved-tensor input
