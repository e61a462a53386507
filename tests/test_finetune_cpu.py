"""Fine-tuning support without a GPU: the fused AdamW's segment table (coalescing, exact coverage of the parameters it
updates, the class cap), host-side argument rejection of mmfm_adamw_multi, the AdamW kernel's SASS (no float atomics),
and the filtered backward call lists of frozen parameters (call indices of the gradient marks and of the
data-parallel buckets)."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from multi_modal_foundation_model_b200 import _lib
from multi_modal_foundation_model_b200._lib import ADAMW_CHUNK4, ADAMW_MAX_CLASSES, MmfmError
from multi_modal_foundation_model_b200.optim import segment_table


def _layout(sizes):
    offs, o = [], 0
    for n in sizes:
        offs.append(o)
        o += (n + 63) // 64 * 64
    return offs, o


def _covered(segs, total):
    mask = np.zeros(total, dtype=bool)
    for lo, hi, _, _ in segs:
        assert not mask[lo:hi].any(), "segments overlap"
        mask[lo:hi] = True
    return mask


def test_segment_table_coalesces_and_covers_exactly():
    rng = np.random.default_rng(0)
    sizes = [int(x) for x in rng.integers(1, 5000, size=60)] + [64, 128, 1, 3, 4096 * 3 + 5]
    offs, total = _layout(sizes)
    for trial in range(20):
        cls = [None if rng.random() < 0.3 else int(rng.integers(0, 3)) for _ in sizes]
        segs, n_chunks = segment_table(offs, sizes, cls)
        mask = _covered(segs, total)
        for o, n, c in zip(offs, sizes, cls):
            pad = slice(o + n, o + (n + 63) // 64 * 64)
            if c is None:      # not updated: neither the parameter nor its pad is touched
                assert not mask[o:o + n].any() and not mask[pad].any()
            else:
                assert mask[o:o + n].all()
                seg = next(s for s in segs if s[0] <= o < s[1])
                assert seg[2] == c and seg[1] >= o + n
        # a pad is covered only between two consecutive parameters of one class
        for i in range(len(sizes) - 1):
            pad = slice(offs[i] + sizes[i], offs[i + 1])
            inside = cls[i] is not None and cls[i] == cls[i + 1]
            assert mask[pad].all() == inside or offs[i] + sizes[i] == offs[i + 1]
        # maximal coalescing: consecutive segments never join two consecutive parameters of one class
        for a, b in zip(segs, segs[1:]):
            assert a[0] < a[1] <= b[0]
            i = offs.index(b[0])
            assert not (cls[i - 1] == b[2] and offs[i - 1] + sizes[i - 1] == a[1] and a[2] == b[2])
        # the kernel's chunk layout
        chunk = 0
        for lo, hi, _, c0 in segs:
            assert lo % 4 == 0 and c0 == chunk
            chunk += max(1, -(-((hi >> 2) - (lo >> 2)) // ADAMW_CHUNK4))
        assert n_chunks == chunk


def test_segment_table_one_class_is_one_segment():
    sizes = [100, 64, 7, 300000]
    offs, total = _layout(sizes)
    segs, n_chunks = segment_table(offs, sizes, [0] * 4)
    assert segs == [(0, offs[-1] + sizes[-1], 0, 0)]
    assert n_chunks == -(-((offs[-1] + sizes[-1]) // 4) // ADAMW_CHUNK4)
    assert segment_table(offs, sizes, [None] * 4) == ([], 0)


def test_segment_table_alternating_classes():
    sizes = [256, 64] * 5
    offs, _ = _layout(sizes)
    segs, _ = segment_table(offs, sizes, [0, 1] * 5)
    assert [(s[0], s[1], s[2]) for s in segs] == [(o, o + n, i % 2) for i, (o, n) in enumerate(zip(offs, sizes))]


def test_segment_table_class_cap():
    sizes = [64] * (ADAMW_MAX_CLASSES + 1)
    offs, _ = _layout(sizes)
    segment_table(offs[:-1], sizes[:-1], list(range(ADAMW_MAX_CLASSES)))
    with pytest.raises(MmfmError, match="at most 64"):
        segment_table(offs, sizes, list(range(ADAMW_MAX_CLASSES + 1)))


def test_segment_table_rejects_misaligned_offsets():
    with pytest.raises(MmfmError, match="aligned"):
        segment_table([2], [8], [0])


P = 256          # any non-null, 16-byte aligned address: every call below must be rejected before it touches the device


def _multi(**kw):
    cls = (_lib.AdamwClass * 2)(_lib.AdamwClass(1e-3, 0.9, 0.999, 1e-8, 0.01, 0, 1),
                                _lib.AdamwClass(1e-3, 0.9, 0.999, 1e-8, 0.01, 0, 1))
    a = dict(p=P, g=P, m=P, v=P, n=1024, segs=P, n_segs=1, n_chunks=1, classes=cls, n_classes=1)
    a.update(kw)
    return _lib.lib().mmfm_adamw_multi(*a.values(), None)


@pytest.mark.parametrize("kw,msg", [
    (dict(segs=None), b"null pointer"),
    (dict(classes=None), b"null pointer"),
    (dict(p=None), b"bad arguments"),
    (dict(n=0), b"bad arguments"),
    (dict(m=P + 4), b"16-byte aligned"),
    (dict(n_segs=0), b"bad segment count"),
    (dict(n_segs=3, n_chunks=2), b"bad segment count"),
    (dict(n_classes=0), b"n_classes must be in"),
    (dict(n_classes=ADAMW_MAX_CLASSES + 1), b"n_classes must be in"),
    (dict(classes=(_lib.AdamwClass * 1)(_lib.AdamwClass(1e-3, 0.9, 0.999, 1e-8, 0.0, 0, 0))), b"step must be >= 1"),
])
def test_adamw_multi_rejects_bad_arguments(kw, msg):
    assert _multi(**kw) == -1
    assert msg in _lib.lib().mmfm_last_error()


def test_adamw_struct_layout_matches_header():
    assert ctypes.sizeof(_lib.AdamwSeg) == 24 and ctypes.sizeof(_lib.AdamwClass) == 32
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                            "mmfm_b200.h")).read()
    assert f"#define MMFM_ADAMW_MAX_CLASSES {ADAMW_MAX_CLASSES}" in hdr
    assert f"#define MMFM_ADAMW_CHUNK4 {ADAMW_CHUNK4}" in hdr


def test_adamw_kernel_has_no_float_atomics():
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
    new = [k for k in kernels if "adamw_kernel" in k]
    assert len(new) == 1, new
    body = kernels[new[0]]
    assert not [l for l in body if re.search(r"\b(RED|REDG|ATOM|ATOMG)\.", l)]
    assert any(re.search(r"\bLDG\.E\.128\b", l) for l in body), "float4 loads of the vector path"


# ---- frozen parameters: filtered backward call lists -------------------------------------------------------------
class _P:
    def __init__(self, rg):
        self.requires_grad = rg


def _fake_plan(n_calls=12):
    """A Plan with a synthetic recorded backward: wgrad calls at 1, 3, 4, 7, 9, marks after 5 and 10 calls, then the
    gradient scale and one input-gradient call."""
    from multi_modal_foundation_model_b200.engine import Plan
    names = ["a", "b", "c", "d", "e", "f"]
    params = {n: _P(True) for n in names}
    pl = Plan.__new__(Plan)

    class _Store:
        pass

    class _Eng:
        pass

    pl.eng = _Eng()
    pl.eng.store = _Store()
    pl.eng.store.params = params
    pl.eng.store.total = 6000
    calls = [(None, (), "k%d" % i, {}) for i in range(n_calls - 2)]
    calls += [(None, (), "mmfm_scale_inplace", {}), (None, (), "input_grad", {})]
    pl.bwd_calls = calls
    pl.grad_marks = [(5, 2000), (10, 6000)]
    pl.wgrad_writes = [(1, ("a",)), (3, ("b", "c")), (4, ("d",)), (7, ("e",)), (9, ("f",))]
    pl._wgrad_params = [(ci, tuple(params[n] for n in ns)) for ci, ns in pl.wgrad_writes]
    pl._skip_of, pl._variants = {}, {}
    return pl, params


def test_backward_schedule_filters_frozen_wgrad_and_remaps_marks():
    pl, params = _fake_plan()
    skip, calls, marks = pl.backward_schedule()
    assert skip == () and calls is pl.bwd_calls and marks is pl.grad_marks
    params["a"].requires_grad = False
    params["b"].requires_grad = False            # c is trainable: the fused call 3 stays
    params["e"].requires_grad = False
    skip, calls, marks = pl.backward_schedule()
    assert skip == (1, 7)
    assert [c[2] for c in calls] == [c[2] for i, c in enumerate(pl.bwd_calls) if i not in (1, 7)]
    assert marks == [(4, 2000), (8, 6000)]
    assert calls[marks[-1][0]][2] == "mmfm_scale_inplace"
    assert pl.backward_schedule()[1] is calls           # cached per frozen set
    for p in params.values():                           # unfreezing switches back to the recorded list
        p.requires_grad = True
    assert pl.backward_schedule()[1] is pl.bwd_calls


def test_data_parallel_buckets_follow_the_filtered_list():
    from multi_modal_foundation_model_b200.parallel import DataParallel
    pl, params = _fake_plan()
    dp = DataParallel.__new__(DataParallel)
    dp.eng = pl.eng
    dp.bucket_elems = 1000
    params["b"].requires_grad = params["c"].requires_grad = False
    skip, (calls, n_calls, buckets, tail) = dp._segments(pl)
    assert skip == (3,) and n_calls == 9 and tail == 10 and calls[tail][2] == "input_grad"
    assert buckets == [(4, 0, 2000), (9, 2000, 6000)]
    for p in params.values():
        p.requires_grad = True
    skip, (calls, n_calls, buckets, tail) = dp._segments(pl)
    assert skip == () and calls is pl.bwd_calls and buckets == [(5, 0, 2000), (10, 2000, 6000)]
