"""Forward-only plans: a step with gradients disabled (torch.no_grad / torch.inference_mode) runs the forward schedule
alone on buffers allocated by liveness.  It computes bit for bit what the grad-enabled forward computes, eager and
graph-replayed; its buffers do not grow with depth; it runs the scaled model at batches the training plan cannot hold;
back-to-back steps that change the masking mode without a sync each get their own masks; and a first step under
inference_mode leaves the engine fit for training."""
import contextlib

import numpy as np
import pytest
import torch

from _util import small_config

pytestmark = pytest.mark.gpu

INC = 0x632BE59BD9B4E019          # seed advance per forward (engine.Plan._fwd_body)
MASK64 = (1 << 64) - 1


@contextlib.contextmanager
def deterministic(on: bool = True):
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _batch_md(model, B, N, mods, T=100, n_beh=2, masks=None, eid=None, u8=False, step=1, pad=10):
    """mod_dict of a synthetic batch.  masks: None = token masking on the model's (device) sampler, else {mod: (B,T)}."""
    from multi_modal_foundation_model_b200.synthetic import make_batch
    batch = make_batch(B, N, n_beh, T, step=step, pad_bins=pad)
    attn, ts = batch["time_attn_mask"], batch["spikes_timestamps"]
    beh = [m for m in mods if m != "ap"]
    xs = {"ap": batch["spikes_data"]}
    for k, m in enumerate(beh):
        xs[m] = batch["target"] if len(beh) == 1 and n_beh > 1 else batch["target"][:, :, k:k + 1].contiguous()
    md = {}
    for m in mods:
        x = xs[m].cuda()
        if u8 and m == "ap":
            x = x.to(torch.uint8)
        d = dict(inputs=x, targets=x, inputs_attn_mask=attn.cuda(), inputs_timestamp=ts.cuda(),
                 inputs_modality=torch.tensor(model.mod_to_indx[m], device="cuda"), masking_mode=None,
                 eval_mask=None if masks is None else masks[m].cuda()[:, :, None].contiguous(),
                 inputs_regions=np.array([["CA1"] * x.shape[2]] * B))
        if eid is not None:
            d["eid"] = eid
        md[m] = d
    return md


def _snap(out, md):
    return dict(loss=out.loss.detach().clone(),
                mod_loss={m: v.detach().clone() for m, v in out.mod_loss.items()},
                preds={m: v.detach().clone() for m, v in out.mod_preds.items()},
                n={m: v.clone() for m, v in out.mod_n_examples.items()},
                mask={m: d["inputs_mask"].clone() for m, d in md.items()})


def _assert_equal(a, b, what):
    assert torch.equal(a["loss"], b["loss"]), f"{what}: loss {a['loss'].item()} vs {b['loss'].item()}"
    for m in a["preds"]:
        assert torch.equal(a["mod_loss"][m], b["mod_loss"][m]), f"{what}: mod_loss {m}"
        assert torch.equal(a["preds"][m], b["preds"][m]), f"{what}: preds {m}"
        assert torch.equal(a["n"][m], b["n"][m]), f"{what}: mod_n_examples {m}"
        assert torch.equal(a["mask"][m], b["mask"][m]), f"{what}: inputs_mask {m}"


def _parity(model, make_md, seed=4242):
    """reseed(s) + grad-enabled forward (no backward) against reseed(s) + no_grad forward; twice each, so the second
    forward of either plan replays its CUDA graph."""
    eng = model.engine()
    res = {}
    for grad in (True, False):
        res[grad] = []
        for rep in range(2):
            eng.reseed(seed + rep)
            md = make_md()
            with torch.set_grad_enabled(grad):
                out = model(md)
            assert out.loss.requires_grad == grad
            res[grad].append(_snap(out, md))
    torch.cuda.synchronize()
    for rep in range(2):
        _assert_equal(res[True][rep], res[False][rep], f"forward {rep}")
    from multi_modal_foundation_model_b200.engine import ForwardPlan
    assert isinstance(eng.last_plan, ForwardPlan) and eng.last_plan in eng.fwd_plans.values()
    assert all(not pl.bwd_calls for pl in eng.fwd_plans.values())
    return res


def _model(N, mods=("ap", "behavior"), extra=None, n_beh=2, **cfg_kw):
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import build_model
    torch.manual_seed(11)
    cfg = default_model_config(**cfg_kw)
    return build_model(N, n_beh, cfg, avail_mod=tuple(mods), extra_channels=extra).cuda()


@pytest.mark.parametrize("train", [False, True])
def test_default_b256_token_masking_bitwise(train):
    model = _model(668).train(train)
    _parity(model, lambda: _batch_md(model, 256, 668, ("ap", "behavior")))


@pytest.mark.parametrize("kw", [dict(decoder_causal_mask=True), dict(decoder_sep_mask=True),
                                dict(use_scalenorm=True)])
def test_decoder_masks_and_scalenorm_bitwise(kw):
    model = _model(96, n_layers=2, **kw).train()
    _parity(model, lambda: _batch_md(model, 8, 96, ("ap", "behavior")))


def test_five_modalities_dhead64_s500_bitwise():
    mods = ("ap", "beh0", "beh1", "beh2", "beh3")
    model = _model(128, mods, extra={m: 1 for m in mods[1:]}, n_beh=4, n_layers=2, n_heads=4, n_modality=5).eval()
    _parity(model, lambda: _batch_md(model, 6, 128, mods, n_beh=4))


def test_uint8_wire_format_bitwise():
    model = _model(72, n_layers=2).eval()
    _parity(model, lambda: _batch_md(model, 6, 72, ("ap", "behavior"), u8=True))


def test_multi_session_bitwise():
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
    chans = {"sess-a": {"ap": 40, "behavior": 2}, "sess-b": {"ap": 88, "behavior": 2}, "sess-c": {"ap": 56, "behavior": 2}}
    torch.manual_seed(21)
    model = MultiSessionMultiModal(chans, ["ap", "behavior"], small_config()).cuda().train()
    for k, (eid, ch) in enumerate(chans.items()):
        _parity(model, lambda: _batch_md(model, 4, ch["ap"], ("ap", "behavior"), eid=eid, step=k), seed=100 + k)
    eng = model.engine()
    assert len(eng.fwd_plans) == 3 and len(eng.fwd_arenas) == 1 and len(eng.arenas) == 1
    arena = next(iter(eng.fwd_arenas.values())).buf
    lo, hi = arena.data_ptr(), arena.data_ptr() + arena.numel()
    assert all(lo <= pl.xs[0].data_ptr() < hi for pl in eng.fwd_plans.values())


def test_deterministic_mode_bitwise():
    model = _model(668, n_layers=2).train()
    with deterministic():
        _parity(model, lambda: _batch_md(model, 32, 668, ("ap", "behavior")))


def _fwd_plan_bytes(n_layers, B=16, N=96):
    model = _model(N, n_layers=n_layers).eval()
    with torch.no_grad():
        model(_batch_md(model, B, N, ("ap", "behavior")))
    eng = model.engine()
    (pl,) = eng.fwd_plans.values()
    n_multi = eng.Ld if eng.fuse_ctx else 0
    return pl.arena_bytes, n_multi, pl.R, eng.H


def test_buffers_independent_of_depth():
    """2+2 and 8+8 layers of the same width: the forward-only plan's buffers differ by the multi-LN outputs at most
    (the fused context_norm kernel writes one [R, H] bf16 buffer per decoder layer, up to 8)."""
    b2, n2, R, H = _fwd_plan_bytes(2)
    b8, n8, _, _ = _fwd_plan_bytes(8)
    one = -(-R * H * 2 // 256) * 256
    assert abs(b8 - b2) <= max(n2, n8) * one, (b2, b8, n2, n8)


def test_default_model_peak_memory_bound():
    """B = 256, N = 668: the peak-memory increase of the first no-grad forward stays below the bytes of the buffers a
    forward-only plan needs, computed here from the shapes."""
    B, N, T = 256, 668, 100
    model = _model(N).eval()
    md = _batch_md(model, B, N, ("ap", "behavior"))
    eng = model.engine()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    with torch.no_grad():
        model(md)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    H, I, S, n_ctx = eng.H, eng.enc_inter, T * 2, eng.Ld
    R, BT, C = B * S, B * T, N + 2
    f32_stream = 5 * R * H * 4                                   # two residual buffers, two embedding sums, context
    bf16_acts = R * 2 * (H * (4 + n_ctx) + 3 * H + 2 * H + I)    # ln, ao, xq, decoder_norm, context_norms, qkv, kv, gelu
    per_mod = BT * C * (3 * 4 + 2 + 2 * 2 * 2 + 2 + 4)          # inp / tgt / preds, inputs bf16, hidden x2, dpreds, out
    bound = int(1.1 * (f32_stream + bf16_acts + per_mod)) + (64 << 20)
    assert grown < bound, (grown, bound)


def test_scaled_model_beyond_training_plan():
    """configs[4] (24+24 layers, H 1024, S 1000) at B = 128: its training plan needs about 1.8 MB per token row (~230 GB)
    and does not fit; the forward-only plan does.  Rows and attention items are computed independently, so the first
    16 trials equal a B = 16 forward of the same trials bit for bit."""
    from multi_modal_foundation_model_b200.config import scaled_model_config
    from multi_modal_foundation_model_b200.model import build_model
    mods = ("ap", "beh0", "beh1", "beh2", "beh3")
    torch.manual_seed(3)
    model = build_model(1024, 4, scaled_model_config(), avail_mod=mods, extra_channels={m: 1 for m in mods[1:]})
    model = model.cuda().eval()
    B = 128
    g = torch.Generator().manual_seed(9)
    masks = {m: (torch.rand(B, 200, generator=g) < 0.3).long() for m in mods}
    md = _batch_md(model, B, 1024, mods, T=200, n_beh=4, masks=masks, pad=20)
    with torch.no_grad():
        big = model(md)
        small = model({m: {k: (v[:16] if getattr(v, "ndim", 0) > 0 else v) for k, v in d.items()}
                       for m, d in md.items()})
    torch.cuda.synchronize()
    for m in mods:
        assert torch.equal(big.mod_preds[m][:16], small.mod_preds[m]), m
    assert torch.isfinite(big.loss)


def test_back_to_back_mode_changes_without_sync():
    """Encoding, decoding and token-masking steps enqueued while the device is still busy: every step's tmask is the
    mask that step asked for (the pinned threshold staging may not be rewritten before its copy has executed)."""
    from oracle import philox_ref as px
    B, N, T = 64, 96, 100
    model = _model(N, n_layers=2).eval()
    eng = model.engine()
    mods = ("ap", "behavior")
    full = lambda v: {m: torch.full((B, T), int(v[m]), dtype=torch.int64) for m in mods}
    modes = [None, full(dict(ap=1, behavior=0)), None, full(dict(ap=0, behavior=1)), None, full(dict(ap=1, behavior=0))]
    mds = [_batch_md(model, B, N, mods, masks=mk) for mk in modes]
    attn = mds[0]["ap"]["inputs_attn_mask"].cpu()
    with torch.no_grad():
        model(mds[0])                       # plan, module load and graph capture out of the way
        model(mds[0])
        torch.cuda.synchronize()
        eng.reseed(777)
        torch.cuda._sleep(200_000_000)      # keep the device busy while the host enqueues every step
        for md in mds:
            model(md)
    torch.cuda.synchronize()
    ratio = float(model.masker.ratio)
    for i, (md, mk) in enumerate(zip(mds, modes)):
        seed = (777 + (i + 1) * INC) & MASK64
        for m in mods:
            if mk is None:
                want = torch.from_numpy(px.mask_bernoulli(seed, model.mod_to_indx[m], B, T, ratio)) & attn
            else:
                want = mk[m] & attn
            assert torch.equal(md[m]["inputs_mask"].cpu(), want), (i, m)


def test_inference_mode_first_then_training():
    """The first call ever under torch.inference_mode(), then training steps with backward and AdamW: the same
    gradients and parameters as the same training steps on a fresh copy that never ran under inference_mode."""
    from multi_modal_foundation_model_b200.optim import AdamW
    B, N = 16, 96
    g = torch.Generator().manual_seed(2)
    masks = {m: (torch.rand(B, 100, generator=g) < 0.3).long() for m in ("ap", "behavior")}
    runs = []
    for first_inference in (True, False):
        model = _model(N, n_layers=2).eval()
        if first_inference:
            with torch.inference_mode():
                out = model(_batch_md(model, B, N, ("ap", "behavior"), masks=masks))
            assert out.loss.is_inference()
        opt = AdamW(model.parameters(), lr=1e-3)
        grads = []
        with deterministic():
            for step in range(3):
                opt.zero_grad(set_to_none=True)
                out = model(_batch_md(model, B, N, ("ap", "behavior"), masks=masks, step=step))
                out.loss.backward()
                grads.append(torch.cat([p.grad.reshape(-1) for p in model.parameters()]).clone())
                opt.step()
        torch.cuda.synchronize()
        assert not model.engine().store.flat.is_inference()
        runs.append((grads, [p.detach().clone() for p in model.parameters()]))
    for a, b in zip(runs[0][0], runs[1][0]):
        assert torch.equal(a, b)
    for a, b in zip(runs[0][1], runs[1][1]):
        assert torch.equal(a, b)
