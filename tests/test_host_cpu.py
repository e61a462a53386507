"""CPU: host-side logic -- Masker bit-exactness against the reference's masks, initial-weight parity of the module
classes, state_dict key parity, pickling, the C ABI export list, config restatement."""
import ctypes
import io
import os
import pickle
import re

import numpy as np
import pytest
import torch

import _reference as ref
from _util import GOLDEN, load_small, small_config
from multi_modal_foundation_model_b200 import _lib
from multi_modal_foundation_model_b200.config import default_model_config
from multi_modal_foundation_model_b200.masker import Masker
from multi_modal_foundation_model_b200.model import build_model


def test_masker_bit_exact_against_reference_masks():
    z = np.load(os.path.join(GOLDEN, "masker.npz"))
    n = len([k for k in z.files if k.endswith("/meta")])
    for i in range(n):
        seed, B, T, C, r1000 = [int(v) for v in z[f"case{i}/meta"]]
        cfg = default_model_config(mask_ratio=r1000 / 1000.0)
        mk = Masker(cfg["masker"], stream="reference")
        torch.manual_seed(seed)
        regions = np.array([["CA1"] * C] * B)
        for call in range(3):
            torch.poisson(torch.full((B, T, C), 0.3))            # the fixture generator drew its inputs in between
            m = mk.sample_token_mask((B, T, C), "cpu", regions)
            assert m.dtype == torch.int64 and m.shape == (B, T)
            assert np.array_equal(m.numpy().astype(np.int8), z[f"case{i}/masks"][call]), (i, call)


def test_masker_early_outs_and_forward_shape():
    cfg = default_model_config(mask_ratio=0.0)
    mk = Masker(cfg["masker"])
    x = torch.ones(2, 10, 3)
    y, m = mk(x, None)
    assert m.shape == (2, 10, 3) and m.sum() == 0 and y is x
    cfg = default_model_config(mask_ratio=0.3)
    mk = Masker(cfg["masker"])
    mk.force_active = False
    mk.eval()
    assert mk.sample_token_mask((2, 10, 3), "cpu").sum() == 0
    mk.mode = "no-such-mode"
    mk.train()
    with pytest.raises(Exception):                      # masker.py:129
        mk.sample_token_mask((2, 10, 3), "cpu", np.array([["CA1"] * 3] * 2))


def test_initial_weights_match_reference_seed42():
    z = np.load(os.path.join(GOLDEN, "init_default.npz"))
    torch.manual_seed(42)
    model = build_model(64, 2, default_model_config())
    sd = model.state_dict()
    assert sorted(sd.keys()) == sorted(z.files)
    for k, v in sd.items():
        got = np.array([v.double().sum().item(), v.double().abs().sum().item(), float(v.flatten()[0])])
        assert np.allclose(got, z[k], rtol=1e-12, atol=1e-12), k


def test_state_dict_keys_match_reference_golden():
    """The reference's state_dict keys, in its order, as stored by tests/golden/make_golden.py: the default model
    (init_default.npz) and the small fixture model, whose reference weights load into ours unchanged (mm_small.npz)."""
    ours = build_model(32, 2, default_model_config())
    assert list(ours.state_dict().keys()) == list(np.load(os.path.join(GOLDEN, "init_default.npz")).files)
    _, weights = load_small()
    small = build_model(40, 2, small_config())
    assert list(small.state_dict().keys()) == list(weights)
    small.load_state_dict(weights)
    assert small.decoder_embeddings["ap"].embedder.mod_emb is small.encoder_embeddings["ap"].embedder.mod_emb


def test_model_pickles_without_engine_handles():
    model = build_model(16, 2, small_config())
    buf = io.BytesIO()
    torch.save({"model": model, "epoch": 3}, buf)          # trainer/base.py:302-308
    buf.seek(0)
    m2 = torch.load(buf, weights_only=False)["model"]
    assert m2._engine is None and m2.masker.ratio == model.masker.ratio
    assert m2.mod_to_indx == {"ap": 0, "behavior": 1}


def test_cpu_model_refuses_to_run():
    from multi_modal_foundation_model_b200._lib import MmfmError
    model = build_model(16, 2, small_config())
    with pytest.raises(MmfmError):
        model({"ap": {}, "behavior": {}})


def test_library_exports_every_declared_symbol():
    _lib.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    hdr = open(os.path.join(os.path.dirname(GOLDEN), "..", "include", "mmfm_b200.h")).read()
    declared = set(re.findall(r"\b(mmfm_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(L, name), name
    assert _lib.lib().mmfm_abi_version() == _lib.ABI_VERSION
    # no compute call without a GPU: bad arguments are rejected on the host with a message
    assert _lib.lib().mmfm_gemm_tn(None, None) == -1
    assert b"null args" in _lib.lib().mmfm_last_error()


@pytest.mark.skipif(not ref.available(), reason="reference tree not mounted")
def test_default_config_restates_mm_yaml():
    cfg = ref.load_config()["model"]
    ours = default_model_config()

    def walk(a, b, path=""):
        for k, v in a.items():
            assert k in b, path + k
            if isinstance(v, dict):
                walk(v, b[k], path + k + ".")
            else:
                assert b[k] == v, (path + k, b[k], v)
    walk(dict(cfg), ours)


def test_multi_session_model_keys_and_pickle():
    """configs[3] container: shared layers keep the reference's names, per-session embedders sit under a prefix that,
    once stripped, gives the reference's single-session keys."""
    import pickle
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal, build_model
    cfg = default_model_config(n_layers=1, hidden_size=64, n_heads=2, inter_size=128)
    m = MultiSessionMultiModal({"e1": {"ap": 24, "behavior": 2}, "e2": {"ap": 40, "behavior": 2}}, ["ap", "behavior"], cfg)
    single = set(build_model(40, 2, cfg).state_dict().keys())
    pre = m.session_prefix("e2")
    keys = set(m.state_dict().keys())
    stripped = {k[len(pre):] if k.startswith(pre) else k for k in keys if not k.startswith("session_embeddings.") or k.startswith(pre)}
    assert stripped == single
    assert m.state_dict()[pre + "encoder_embeddings.ap.embedder.token_embed.weight"].shape == (80, 40)
    m2 = pickle.loads(pickle.dumps(m))
    assert m2.session_key("e1") == "s000" and m2.session_key("nope") is None


def test_activation_arena_bump_allocation():
    """engine.Arena: plans of different sessions alias one buffer; allocations are 256-byte aligned and bounded."""
    import torch
    from multi_modal_foundation_model_b200._lib import MmfmError
    from multi_modal_foundation_model_b200.engine import Arena
    a = Arena(4096, "cpu")
    t1 = a.take(100)
    t2 = a.take(300)
    assert t1.numel() == 100 and t2.numel() == 300
    assert (t2.data_ptr() - t1.data_ptr()) == 256 and a.off == 256 + 512
    a.reset()
    assert a.take(8).data_ptr() == t1.data_ptr()          # the next plan starts over on the same memory
    with pytest.raises(MmfmError):
        a.take(1 << 20)


def test_torch_philox_restatement_matches_numpy():
    """tests/_util.py's torch version of the dropout stream (used by the bench-size GPU tests) == oracle/philox_ref.py."""
    from _util import philox_bytes_torch, philox_prob_bytes_torch
    from oracle import philox_ref as px
    for seed in (0x0BADC0DE12345FF, 0xFBADC0DE12345FF1, 7):
        a = px.random_bytes(seed, 4101, 10, 50)
        assert (a == philox_bytes_torch(seed, 4101, 10, 50, "cpu").numpy()).all()
        assert (a[4:] == philox_bytes_torch(seed, 4101, 6, 50, "cpu", row0=4).numpy()).all()
        b = px.prob_random_bytes(seed, 33, 12, 200)
        assert (b == philox_prob_bytes_torch(seed, 33, 12, 200, "cpu").numpy()).all()
        assert (b[7:] == philox_prob_bytes_torch(seed, 33, 5, 200, "cpu", row0=7).numpy()).all()


def test_masker_every_mode_bit_exact_vs_reference_golden():
    """SURVEY 8f rank 3: the column-0 mask of EVERY reference masking mode (models/masker.py:79-168), three consecutive
    calls each, equals the unmodified reference's (tests/golden/make_masker_modes.py) -- torch CPU stream and python
    `random` consumption included."""
    import os
    import random
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_masker_modes as gm
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.masker import Masker
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "masker_modes.npz"))
    for i, (mode, seed, shape, over) in enumerate(gm.CASES):
        cfg = default_model_config()["masker"]
        cfg["mode"] = mode
        cfg.update(over)
        mk = Masker(cfg, stream="reference")
        torch.manual_seed(seed)
        random.seed(seed)
        regions = gm.regions_for(shape[0], shape[2])
        for call in range(3):
            got = mk.sample_token_mask(shape, "cpu", regions).numpy()
            assert (got == z[f"case{i}"][call]).all(), (mode, i, call)


def test_heldout_mask_compact_form_equals_reference():
    """SURVEY 8f rank 3: eval_masks.heldout_mask == the reference's heldout_mask (eval_utils.py:988-1045, golden from the
    unmodified function) in every mode: masked spikes, held-out indices, the dense eval mask and the (B,T) column the
    model reads (mm.py:269-270)."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_heldout_golden as gh
    from multi_modal_foundation_model_b200.eval_masks import heldout_mask
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "heldout.npz"))
    spikes, regions = gh.inputs()
    for i, (mode, kw) in enumerate(gh.CASES):
        r = heldout_mask(spikes.clone(), mode=mode, neuron_regions=regions, **kw)
        assert np.array_equal(r["spikes"].numpy(), z[f"case{i}/spikes"]), (mode, i)
        assert np.array_equal(np.asarray(r["heldout_idxs"]).astype(np.int64), z[f"case{i}/hd"]), (mode, i)
        dense = r["dense_eval_mask"]().numpy()
        assert np.array_equal(dense, z[f"case{i}/eval_mask"]), (mode, i)
        assert r["eval_mask"].dtype == torch.int64 and np.array_equal(r["eval_mask"].numpy(), dense[:, :, 0]), (mode, i)


def test_flat_gradient_order_with_fused_context_norms(monkeypatch):
    """The decoder layers' context_norm gradients come out of ONE launch after the last decoder layer of the backward
    (engine.fuse_context_norms), so in the flat gradient order -- reverse execution order, the data-parallel bucket
    order -- they sit behind every decoder-layer parameter and in front of decoder_proj_context; with the fusion off they
    stay inside their layers.  Either way the order is a permutation of all parameters."""
    from multi_modal_foundation_model_b200 import engine
    from multi_modal_foundation_model_b200.model import build_model
    m = build_model(40, 2, default_model_config(n_layers=3))
    named = dict(m.named_parameters(remove_duplicate=False))
    for fused in (True, False):
        monkeypatch.setenv("MMFM_FUSE_CTX_LN", "1" if fused else "0")
        assert engine.fuse_context_norms(named, 3) is fused
        order = engine.ParamStore._execution_reverse_order(m, named)
        assert sorted(order) == sorted(named)
        ctx = [order.index(f"decoder.{i}.context_norm.weight") for i in range(3)]
        last_layer_param = max(order.index(n) for n in order if n.startswith("decoder.") and ".context_norm." not in n)
        if fused:
            assert min(ctx) > last_layer_param and max(ctx) < order.index("decoder_proj_context.weight")
            assert ctx == sorted(ctx, reverse=True)          # layer 2 first: the order of the backward's dY list
        else:
            assert min(ctx) < last_layer_param
    assert not engine.fuse_context_norms(named, 1)           # a single decoder layer has nothing to share
