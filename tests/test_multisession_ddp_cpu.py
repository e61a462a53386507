"""CPU: the data-parallel multi-session exchange without a GPU -- session ranges of the flat buffers, core-only
gradient buckets, a gloo (world 2) restatement of the exchange, and mmfm_session_grad_combine's host-side argument
checks and SASS (no float atomics)."""
import os
import re
import shutil
import socket
import subprocess

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from multi_modal_foundation_model_b200 import _lib, engine
from multi_modal_foundation_model_b200.config import default_model_config
from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
from multi_modal_foundation_model_b200.parallel import all_reduce_mean, core_buckets, plan_buckets

CHANS = {"sess-a": {"ap": 40, "behavior": 2}, "sess-b": {"ap": 88, "behavior": 2}, "sess-c": {"ap": 56, "behavior": 2}}


def _layout(n_layers=3):
    torch.manual_seed(0)
    m = MultiSessionMultiModal(CHANS, ["ap", "behavior"],
                               default_model_config(n_layers=n_layers, hidden_size=128, n_heads=4, inter_size=256))
    named = dict(m.named_parameters(remove_duplicate=False))
    order = engine.ParamStore._execution_reverse_order(m, named)
    alias, offset, shape, total = engine.flat_layout(order, named)
    prefixes = [p for p, _, _ in engine.embedding_groups(m)]
    core, ranges = engine.session_ranges(offset, shape, prefixes)
    return m, named, alias, offset, shape, total, prefixes, core, ranges


def _padded(shape, n):
    return (shape[n].numel() + 63) // 64 * 64


def test_session_ranges_contiguous_aligned_disjoint_and_complete():
    m, named, alias, offset, shape, total, prefixes, core, ranges = _layout()
    assert len(ranges) == len(CHANS) == len(prefixes)
    owner = torch.full((total,), -2, dtype=torch.int64)        # -1 = core, s = session s
    spans = [(core[0], core[1], -1)] + [(lo, hi, s) for s, r in enumerate(ranges) for lo, hi in (r[:2], r[2:])]
    for lo, hi, s in spans:
        assert lo % 64 == 0 and hi % 64 == 0 and lo < hi
        assert (owner[lo:hi] == -2).all(), "ranges overlap"
        owner[lo:hi] = s
    assert (owner != -2).all(), "the ranges and the core tile the whole buffer"
    # every parameter (aliases through their canonical name) lies in its own session's ranges or in the core, once
    seen = torch.zeros(total, dtype=torch.int64)
    for n, p in named.items():
        c = alias[n]
        s = next((k for k, pre in enumerate(prefixes) if n.startswith(pre)), -1)
        o = offset[c]
        assert (owner[o:o + _padded(shape, c)] == s).all(), n
        is_head = s >= 0 and n[len(prefixes[s]):].startswith("decoder_embeddings.") and ".out." in n
        h0, h1, e0, e1 = ranges[s] if s >= 0 else (0, 0, 0, 0)
        if s >= 0:
            assert (h0 <= o < h1) if is_head else (e0 <= o < e1), n
        if c == n:
            seen[o:o + _padded(shape, c)] += 1
    assert (seen == 1).all()
    # the shared mod_emb of a session is one parameter under two names, inside that session's embedder range
    pre = prefixes[1]
    enc, dec = pre + "encoder_embeddings.ap.embedder.mod_emb.weight", pre + "decoder_embeddings.ap.embedder.mod_emb.weight"
    assert named[enc] is named[dec] and alias[enc] == alias[dec]
    # the widest session has the widest ranges
    widths = [r[1] - r[0] + r[3] - r[2] for r in ranges]
    assert widths.index(max(widths)) == 1


def test_session_ranges_reject_a_gap_and_an_overlap():
    _, _, _, offset, shape, _, prefixes, _, _ = _layout(n_layers=1)
    name = next(n for n in offset if n.startswith(prefixes[0]) and n.endswith("projection.weight"))
    bad = dict(offset)
    bad[name] += 64
    with pytest.raises(_lib.MmfmError, match="not contiguous"):
        engine.session_ranges(bad, shape, prefixes)
    bad = {n: o - 64 if n.startswith(prefixes[1]) and ".out." in n else o for n, o in offset.items()}
    with pytest.raises(_lib.MmfmError, match="overlap"):      # session 1's heads, still contiguous, moved onto a neighbour
        engine.session_ranges(bad, shape, prefixes)


def _engine_marks(offset, total, s, n_dec, n_enc, fused, shift):
    """The gradient marks engine.Plan._build_backward records for session s (offsets by parameter name; call indices
    made session dependent, as a different number of embedder / head launches would)."""
    names = []
    for i in reversed(range(n_dec)):
        if i > 0:
            names.append(f"decoder.{i - 1}.mlp.down_proj.weight")
        elif fused:
            names.append(f"decoder.{n_dec - 1}.context_norm.weight")
    names.append("decoder_proj_context.weight")
    names += [f"encoder.{i - 1}.mlp.down_proj.weight" for i in reversed(range(1, n_enc))]
    offs = [offset[n] for n in names] + [total]
    return [(5 + s * shift + 10 * k, o) for k, o in enumerate(offs)]


@pytest.mark.parametrize("target", [1, 20000, 10 ** 9])
def test_core_buckets_are_the_same_for_every_session_and_touch_no_session_range(target):
    m, named, alias, offset, shape, total, prefixes, core, ranges = _layout()
    fused = engine.fuse_context_norms(named, m.n_dec_layers)
    got = []
    for s in range(len(ranges)):
        marks = _engine_marks(offset, total, s, m.n_dec_layers, m.n_enc_layers, fused, shift=3)
        b = core_buckets(marks, core, target)
        assert b[0][1] == core[0] and b[-1][2] == core[1] and b[-1][0] == marks[-1][0]
        for (_, _, hi0), (_, lo1, _) in zip(b, b[1:]):
            assert hi0 == lo1
        for ci, lo, hi in b:
            assert any(mc <= ci and off >= hi for mc, off in marks), "reduced before its mark"
            for h0, h1, e0, e1 in ranges:
                assert hi <= h0 or lo >= h1
                assert hi <= e0 or lo >= e1
        got.append([(lo, hi) for _, lo, hi in b])
    assert all(g == got[0] for g in got)
    if target == 1:
        assert len(got[0]) == len(marks)          # one bucket per mark: every core mark splits it


def test_core_buckets_match_plan_buckets_on_the_core_span():
    marks = [(3, 50), (6, 300), (9, 500), (12, 900), (15, 1000)]
    assert core_buckets(marks, (100, 800), 150) == [(6, 100, 300), (9, 300, 500), (15, 500, 800)]
    assert core_buckets(marks, (0, 1000), 150) == plan_buckets(marks, 1000, 150)


# ---- gloo, world 2: the exchange restated in torch -----------------------------------------------------------------
def _rank_grad(total, core, ranges, s, rank, step):
    """What a rank's backward leaves in the flat gradient: the core and its own session's ranges, zeros elsewhere."""
    g = torch.zeros(total)
    gen = torch.Generator().manual_seed(1000 * step + rank)
    h0, h1, e0, e1 = ranges[s]
    for lo, hi in (core, (h0, h1), (e0, e1)):
        g[lo:hi] = torch.randn(hi - lo, generator=gen)
    return g


def _exchange(g, core, ranges, s, world):
    """Core buckets all-reduced (mean); ids and padded head / embedder slabs all-gathered; every gathered session
    combined in ascending rank order as inv_world * (0 + sum), as mmfm_session_grad_combine does."""
    for _, lo, hi in core_buckets([(1, (core[0] + core[1]) // 2), (2, g.numel())], core, 1):
        all_reduce_mean(g[lo:hi])
    ids = [torch.zeros(1, dtype=torch.int32) for _ in range(world)]
    dist.all_gather(ids, torch.tensor([s], dtype=torch.int32))
    ids = [int(t) for t in ids]
    for part in ((0, 1), (2, 3)):
        L = max(r[part[1]] - r[part[0]] for r in ranges)
        lo, hi = ranges[s][part[0]], ranges[s][part[1]]
        send = torch.full((L,), float("nan"))               # the pad is never read
        send[:hi - lo] = g[lo:hi]
        slabs = [torch.empty(L) for _ in range(world)]
        dist.all_gather(slabs, send)
        for r0, t in enumerate(ids):
            if t in ids[:r0]:
                continue
            lo, hi = ranges[t][part[0]], ranges[t][part[1]]
            acc = torch.zeros(hi - lo)
            for r in range(r0, world):
                if ids[r] == t:
                    acc += slabs[r][:hi - lo]
            g[lo:hi] = acc * (1.0 / world)
    return ids


def _worker(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        *_, total, _, core, ranges = _layout(n_layers=1)
        for step, sess in enumerate([(0, 2), (2, 0), (1, 1)]):       # distinct, swapped, the same session
            g = _rank_grad(total, core, ranges, sess[rank], rank, step)
            ids = _exchange(g, core, ranges, sess[rank], world)
            assert ids == list(sess)
            want = sum(_rank_grad(total, core, ranges, sess[r], r, step) for r in range(world)) * (1.0 / world)
            for s, (h0, h1, e0, e1) in enumerate(ranges):
                for lo, hi in ((h0, h1), (e0, e1)):
                    if s in sess:
                        assert torch.equal(g[lo:hi], want[lo:hi]), (step, s)
                    else:
                        assert (g[lo:hi] == 0).all(), "a session no rank ran stays zero"
            assert torch.allclose(g[core[0]:core[1]], want[core[0]:core[1]], rtol=1e-6, atol=1e-7)
    finally:
        dist.destroy_process_group()


def test_gloo_world2_session_exchange_gives_each_session_its_rank_mean():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(2, port), nprocs=2, join=True)


# ---- the C entry point ------------------------------------------------------------------------------------------
P = 256          # any non-null, aligned address: every call below must be rejected before it touches the device


@pytest.mark.parametrize("kw,msg", [
    (dict(grad=None), b"null pointer"),
    (dict(gathered=None), b"null pointer"),
    (dict(ids=None), b"null pointer"),
    (dict(ranges=None), b"null pointer"),
    (dict(world=0), b"outside [1, 65535]"),
    (dict(world=70000), b"outside [1, 65535]"),
    (dict(stride=0), b"bad slab stride or session count"),
    (dict(n_sessions=0), b"bad slab stride or session count"),
    (dict(inv_world=float("inf")), b"inv_world must be finite"),
])
def test_session_grad_combine_rejects_bad_arguments(kw, msg):
    a = dict(grad=P, gathered=P, world=2, stride=1024, ids=P, ranges=P, n_sessions=3, inv_world=0.5)
    a.update(kw)
    assert _lib.lib().mmfm_session_grad_combine(*a.values(), None) == -1
    assert msg in _lib.lib().mmfm_last_error()


def test_session_grad_combine_has_no_float_atomics():
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
    new = [k for k in kernels if "session_grad_combine" in k]
    assert len(new) == 1, new
    body = kernels[new[0]]
    assert not [l for l in body if re.search(r"\b(RED|REDG|ATOM|ATOMG)\.", l)]
    assert any(re.search(r"\bLDG\.E\.128\b", l) for l in body), "float4 loads of the vector path"
    assert any(re.search(r"\bSTG\.E\.128\b", l) for l in body), "float4 stores of the vector path"
