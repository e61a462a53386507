"""Autograd of every step output without a GPU: the two entry points behind it reject null or malformed arguments on
the host with a message, and their kernels carry no float atomics (they are deterministic as they are)."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from multi_modal_foundation_model_b200 import _lib

P = 256          # any non-null address: every call below must be rejected before it touches the device


def _loss_grad(**kw):
    a = dict(preds=P, targets=P, tok_mask=P, S=100, off=0, inv_n=P, g_loss=None, g_mod=None, g_preds=None, sb=0,
             st=0, sc=0, kind=_lib.LOSS_MSE, B=2, T=100, C=4, dpreds=P, lddp=8)
    a.update(kw)
    return _lib.lib().mmfm_loss_grad(*a.values(), None)


def _embed_dx(**kw):
    a = dict(hid=P, W1=P, W2=P, dx=P, row_zero=None, drop=None, act_scale=1.0, act=_lib.ACT_SOFTSIGN, dX=P, lddx=2,
             accumulate=0, B=2, T=100, S=200, off=100, C=2, H=128)
    a.update(kw)
    return _lib.lib().mmfm_smallc_embed_dx(*a.values(), None)


@pytest.mark.parametrize("kw,msg", [
    (dict(preds=None), b"null pointer"),
    (dict(inv_n=None), b"null pointer"),
    (dict(dpreds=None), b"null pointer"),
    (dict(kind=7), b"bad loss kind"),
    (dict(lddp=3), b"bad shape"),
    (dict(off=50), b"bad shape"),
    (dict(B=0), b"bad shape"),
    (dict(sc=-1), b"negative g_preds stride"),
    (dict(kind=_lib.LOSS_CE, C=65, lddp=72), b"up to 64 classes"),
])
def test_loss_grad_rejects_bad_arguments(kw, msg):
    assert _loss_grad(**kw) == -1
    assert msg in _lib.lib().mmfm_last_error()


@pytest.mark.parametrize("kw,msg", [
    (dict(hid=None), b"null pointer"),
    (dict(W1=None), b"null pointer"),
    (dict(dX=None), b"null pointer"),
    (dict(C=9, lddx=9), b"outside [1,8]"),
    (dict(act=_lib.ACT_GELU), b"bad act"),
    (dict(lddx=1), b"bad shape"),
    (dict(off=150), b"bad shape"),
    (dict(drop=ctypes.pointer(_lib.Dropout(None, 0, 10, 1.0))), b"dropout without seed"),
])
def test_smallc_embed_dx_rejects_bad_arguments(kw, msg):
    assert _embed_dx(**kw) == -1
    assert msg in _lib.lib().mmfm_last_error()


def test_new_kernels_have_no_float_atomics():
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
    new = [k for k in kernels if "loss_grad" in k or "smallc_embed_dx" in k]
    assert len(new) == 4, new
    for k in new:
        bad = [l for l in kernels[k] if re.search(r"\b(RED|REDG|ATOM|ATOMG)\.", l)]
        assert not bad, (k, bad[:2])
