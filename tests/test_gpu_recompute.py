"""Per-layer activation recomputation: a training plan that does not fit in device memory is replaced by one that saves
only the residual stream at the layer boundaries and records each layer's forward again before its backward.

Recomputation is forced by lowering torch's per-process memory fraction below the size of the plan that saves
everything while the engine chooses; the plan it is compared with is built first, in the same process, without a
limit.  The forward kernels are order-fixed, so in
deterministic mode outputs, gradients and AdamW states are bitwise those of the plan that saves everything."""
import contextlib
import gc
import json
import os
import socket
import warnings

import pytest
import torch

from test_gpu_inference import _batch_md, _model, deterministic

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MODS = ("ap", "behavior")


def _margin(eng, B, session, grad_inputs):
    from multi_modal_foundation_model_b200 import engine as E
    return E.step_margin(eng._step_transient_bytes(B, session, grad_inputs), E._round_alloc(4 * eng.store.total),
                         len(eng.store.moments) > 0)


def _set_fraction_for(eng, room, B, session, grad_inputs):
    """A per-process memory fraction under which the engine finds exactly `room` bytes for a new plan."""
    total = torch.cuda.mem_get_info()[1]
    torch.cuda.set_per_process_memory_fraction(
        (torch.cuda.memory_allocated() + _margin(eng, B, session, grad_inputs) + room) / total)


@contextlib.contextmanager
def forced_recompute():
    """Every training plan created inside is chosen under a per-process memory fraction that leaves one byte less than
    the plan saving every activation needs.  The fraction is back at 1.0 before the plan allocates, so the caching
    allocator's cached blocks never decide whether the smaller plan fits."""
    from multi_modal_foundation_model_b200.engine import Engine
    choose = Engine._choose_recompute

    def limited(self, B, training, session, u8_mods, grad_inputs):
        _set_fraction_for(self, self._plan_need(B, training, session, u8_mods, grad_inputs, False) - 1, B, session,
                          grad_inputs)
        try:
            return choose(self, B, training, session, u8_mods, grad_inputs)
        finally:
            torch.cuda.set_per_process_memory_fraction(1.0)
    Engine._choose_recompute = limited
    try:
        yield
    finally:
        Engine._choose_recompute = choose


@pytest.fixture
def restore_fraction():
    yield
    torch.cuda.set_per_process_memory_fraction(1.0)


def _grads(model):
    return {n: (None if p.grad is None else p.grad.detach().cpu()) for n, p in model.named_parameters()}


def _run(model, make_md, steps, back=None, opt=None, accumulate=False, seed=4242, grad_inputs=()):
    """`steps` training steps (the first eager, the second captured, later ones replayed); per step the outputs, the
    inputs_mask, every parameter gradient and the input gradients."""
    eng = model.engine()
    res = []
    model.zero_grad(set_to_none=True)
    for s in range(steps):
        if not accumulate:
            (opt or model).zero_grad(set_to_none=True)
        eng.reseed(seed + s)
        md = make_md(s)
        for m in grad_inputs:
            md[m]["inputs"] = md[m]["inputs"].clone().requires_grad_()
        out = model(md)
        (back or (lambda o, d: o.loss.backward()))(out, md)
        if opt is not None:
            opt.step()
        torch.cuda.synchronize()
        # snapshots on the host: under a memory limit the device holds the step's own allocations only
        res.append(dict(loss=out.loss.detach().cpu(), mod_loss={m: v.detach().cpu() for m, v in out.mod_loss.items()},
                        preds={m: v.detach().cpu() for m, v in out.mod_preds.items()},
                        mask={m: d["inputs_mask"].cpu() for m, d in md.items()}, grads=_grads(model),
                        dinp={m: md[m]["inputs"].grad.cpu() for m in grad_inputs}))
    return res


def _assert_same(a, b):
    for step, (x, y) in enumerate(zip(a, b)):
        assert torch.equal(x["loss"], y["loss"]), (step, x["loss"].item(), y["loss"].item())
        for m in x["preds"]:
            for k in ("mod_loss", "preds", "mask"):
                assert torch.equal(x[k][m], y[k][m]), (step, k, m)
        for n, g in x["grads"].items():
            if g is None:
                assert y["grads"][n] is None, (step, n)
            else:
                assert torch.equal(g, y["grads"][n]), (step, n, (g - y["grads"][n]).abs().max().item())
        for m, g in x["dinp"].items():
            assert torch.equal(g, y["dinp"][m]), (step, "input grad", m)


def _parity(build, make_md, B, steps=3, grad_inputs=(), prep=None, with_opt=False, **run_kw):
    """Full plan (no limit) against the recompute plan (limit between the two), same weights, seeds and batches;
    returns both models."""
    from multi_modal_foundation_model_b200.optim import AdamW
    runs, models = [], []
    for force in (False, True):
        model = build()
        if prep is not None:
            prep(model)
        models.append(model)
        opt = AdamW([p for p in model.parameters() if p.requires_grad], lr=1e-3, weight_decay=0.01) if with_opt else None
        if force:
            eng = model.engine()
            with forced_recompute(), warnings.catch_warnings(record=True) as caught:
                warnings.simplefilter("always")
                runs.append(_run(model, make_md, steps, opt=opt, grad_inputs=grad_inputs, **run_kw))
            said = [w for w in caught if "recomputing" in str(w.message)]
            assert len(said) == len(eng.plans) and all(f"batch size {B}:" in str(w.message) for w in said)
            assert eng.plans and all(pl.recompute for pl in eng.plans.values())
        else:
            runs.append(_run(model, make_md, steps, opt=opt, grad_inputs=grad_inputs, **run_kw))
            assert not any(pl.recompute for pl in model.engine().plans.values())
        if with_opt:
            runs[-1].append(dict(weights=[p.detach().cpu() for p in model.parameters()], m=opt._m.cpu(), v=opt._v.cpu()))
    if with_opt:
        w0, w1 = runs[0].pop(), runs[1].pop()
        assert all(torch.equal(a, b) for a, b in zip(w0["weights"], w1["weights"]))
        assert torch.equal(w0["m"], w1["m"]) and torch.equal(w0["v"], w1["v"])
    _assert_same(runs[0], runs[1])
    return models


# ---- bitwise parity in deterministic mode -----------------------------------------------------------------------
def test_default_b256_token_masking_bitwise():
    """Default model, B 256, N 668, train(): token masking on the device sampler, every dropout site on; eager step,
    two graph replays and three AdamW steps."""
    holder, build = _builder(lambda: _model(668).train())
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 256, 668, MODS, step=s), 256, with_opt=True)


def _builder(make):
    """(holder, build): build() makes a fresh model and leaves it in holder["m"] for the batch maker."""
    holder = {}

    def build():
        holder.pop("m", None)          # the previous model's memory is free before the next limit is computed
        gc.collect()
        holder["m"] = make()
        return holder["m"]
    return holder, build


def _small(**kw):
    # four layers: the two plans differ by far more than the caching allocator's segment granularity
    return _builder(lambda: _model(96, n_layers=4, **kw).train())


@pytest.mark.parametrize("kw", [dict(decoder_causal_mask=True), dict(decoder_sep_mask=True), dict(use_scalenorm=True)],
                         ids=["causal", "sep", "scalenorm"])
def test_decoder_masks_and_scalenorm_bitwise(kw):
    holder, build = _small(**kw)
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48)


def test_five_modalities_dhead64_bitwise():
    mods = ("ap", "beh0", "beh1", "beh2", "beh3")
    holder, build = _builder(lambda: _model(128, mods, extra={m: 1 for m in mods[1:]}, n_beh=4, n_layers=2, n_heads=4,
                                            n_modality=5).train())
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 32, 128, mods, n_beh=4, step=s), 32)


def test_uint8_wire_format_and_eval_bitwise():
    holder, build = _small()
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, u8=True, step=s), 48)
        _parity(lambda: build().eval(), lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48)


def test_input_gradients_bitwise():
    holder, build = _small()
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48, grad_inputs=MODS)


def test_weighted_mod_loss_and_preds_loss_bitwise():
    holder, build = _small()

    def back(out, md):
        (out.mod_loss["ap"] * 0.7 + out.mod_loss["behavior"] * 1.9 + out.mod_preds["behavior"].square().mean()).backward()
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48, back=back)


def test_frozen_core_bitwise():
    holder, build = _small()

    def prep(model):
        for n, p in model.named_parameters():
            p.requires_grad_(not n.startswith(("encoder.", "decoder.")))
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48, prep=prep, with_opt=True)


def test_retain_graph_and_accumulation_bitwise():
    holder, build = _small()

    def twice(out, md):
        out.loss.backward(retain_graph=True)
        out.loss.backward()
    with deterministic():
        _parity(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48, back=twice)
        _parity(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48, steps=2, accumulate=True)


def test_multi_session_bitwise():
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
    chans = {"sess-a": {"ap": 40, "behavior": 2}, "sess-b": {"ap": 88, "behavior": 2}, "sess-c": {"ap": 56, "behavior": 2}}
    eids = list(chans) * 2

    def make():
        torch.manual_seed(21)
        cfg = default_model_config(n_layers=4, hidden_size=128, n_heads=4, inter_size=256)
        return MultiSessionMultiModal(chans, list(MODS), cfg).cuda().train()
    holder, build = _builder(make)
    with deterministic():
        full, rec = _parity(build, lambda s: _batch_md(holder["m"], 64, chans[eids[s]]["ap"], MODS, eid=eids[s], step=s),
                            64, steps=6)
    eng = rec.engine()
    assert len(eng.plans) == 3 and list(eng.arenas) == [(64, True, False, True)]
    arena = eng.arenas[(64, True, False, True)].buf
    lo, hi = arena.data_ptr(), arena.data_ptr() + arena.numel()
    assert all(lo <= pl.xs[0].data_ptr() < hi for pl in eng.plans.values())


# ---- default (non-deterministic) mode --------------------------------------------------------------------------
def _within_run_to_run_spread(build, make_md, B, steps=3):
    """Forward outputs bitwise; gradients as close to the full plan's as a second full-plan run is."""
    full = build()
    a, b = _run(full, make_md, steps), _run(full, make_md, steps)
    rec = build()
    with forced_recompute(), pytest.warns(UserWarning, match="recomputing"):
        c = _run(rec, make_md, steps)
    assert rec.engine().last_plan.recompute
    flat = lambda r: torch.cat([g.reshape(-1) for g in r["grads"].values()])
    for x, y, z in zip(a, b, c):
        assert torch.equal(x["loss"], z["loss"])
        for m in x["preds"]:
            assert torch.equal(x["preds"][m], z["preds"][m]) and torch.equal(x["mask"][m], z["mask"][m])
        ref = flat(x)
        spread = (flat(y) - ref).norm() / ref.norm()
        got = (flat(z) - ref).norm() / ref.norm()
        assert got <= 2 * spread + 1e-6, (got.item(), spread.item())


def test_default_mode_within_run_to_run_spread():
    holder, build = _small()
    _within_run_to_run_spread(build, lambda s: _batch_md(holder["m"], 48, 96, MODS, step=s), 48)


# ---- data parallel: one rank recomputes, the other does not ----------------------------------------------------
def _ddp_md(rank, step):
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    return make_mod_dict(make_batch(128, 40, 2, 100, step=10 * step + rank, pad_bins=5), list(MODS),
                         "encoding" if step == 0 else "decoding", device="cuda")


def _ddp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from _util import small_config
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.parallel import DataParallel
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), MMFM_DDP_GRAPH="0")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(100 + rank)
        model = build_model(40, 2, small_config()).cuda().eval()
        ddp = DataParallel(model, bucket_mb=0.25)
        grads = []
        for step in range(3):
            model.zero_grad(set_to_none=True)
            with forced_recompute() if rank == 0 else contextlib.nullcontext():
                out = model(_ddp_md(rank, step))
            out.loss.backward()
            torch.cuda.synchronize()
            grads.append({n: p.grad.detach().cpu().clone() for n, p in model.named_parameters()})
        kinds = [pl.recompute for pl in model.engine().plans.values()]
        torch.save({"grads": grads, "recompute": kinds}, os.path.join(out_dir, f"rank{rank}.pt"))
        ddp.close()
    finally:
        dist.destroy_process_group()


def test_ddp_mixed_plan_kinds(tmp_path):
    import torch.multiprocessing as mp
    from _util import small_config
    from multi_modal_foundation_model_b200.model import build_model
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_ddp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r = [torch.load(tmp_path / f"rank{i}.pt") for i in range(2)]
    assert r[0]["recompute"] == [True] and r[1]["recompute"] == [False]
    torch.manual_seed(100)
    model = build_model(40, 2, small_config()).cuda().eval()
    for step in range(3):
        acc = None
        for rank in range(2):
            model.zero_grad(set_to_none=True)
            model(_ddp_md(rank, step)).loss.backward()
            g = {n: p.grad.detach().cpu().clone() for n, p in model.named_parameters()}
            acc = g if acc is None else {n: acc[n] + g[n] for n in g}
        for n, gref in acc.items():
            assert torch.equal(r[0]["grads"][step][n], r[1]["grads"][step][n]), (step, n)
            gref = gref / 2
            scale = gref.abs().max().item() + 1e-8
            assert (r[0]["grads"][step][n] - gref).abs().max().item() <= 2e-3 * scale + 1e-7, (step, n)


# ---- sizing and selection --------------------------------------------------------------------------------------
def _scaled_model():
    from multi_modal_foundation_model_b200.config import scaled_model_config
    from multi_modal_foundation_model_b200.model import build_model
    mods = ("ap", "beh0", "beh1", "beh2", "beh3")
    torch.manual_seed(3)
    model = build_model(1024, 4, scaled_model_config(), avail_mod=mods, extra_channels={m: 1 for m in mods[1:]})
    return model.cuda().train(), mods


def _scaled_md(model, mods, B, step=0):
    g = torch.Generator().manual_seed(9 + step)
    masks = {m: (torch.rand(B, 200, generator=g) < 0.3).long() for m in mods}
    return _batch_md(model, B, 1024, mods, T=200, n_beh=4, masks=masks, pad=20, step=step)


def _sized_equals_built(eng, B):
    from multi_modal_foundation_model_b200.engine import Plan
    for recompute in (False, True):
        dry = Plan(eng, B, True, recompute=recompute, dry=True)
        built = Plan(eng, B, True, recompute=recompute)
        assert built.recompute == recompute
        assert (dry.arena_bytes, dry.nbytes) == (built.arena_bytes, built.nbytes), recompute
        assert dry.nbytes == eng._plan_need(B, True, None, (), (), recompute)
        del built
        torch.cuda.empty_cache()


@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
def test_sizing_default_and_scaled(det):
    with deterministic(det):
        model = _model(668)
        with torch.no_grad():
            model(_batch_md(model, 8, 668, MODS))
        _sized_equals_built(model.engine(), 256)
        del model
        smodel, mods = _scaled_model()
        with torch.no_grad():
            smodel(_scaled_md(smodel, mods, 2))
        _sized_equals_built(smodel.engine(), 16)


def test_sizing_multi_session_arena():
    from _util import small_config
    from multi_modal_foundation_model_b200.engine import Plan
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
    chans = {"sess-a": {"ap": 40, "behavior": 2}, "sess-b": {"ap": 88, "behavior": 2}}
    model = MultiSessionMultiModal(chans, list(MODS), small_config()).cuda().train()
    model(_batch_md(model, 4, 40, MODS, eid="sess-a")).loss.backward()
    eng = model.engine()
    arena = eng.arenas[(4, True, False, False)]
    widest = Plan(eng, 4, True, model.session_key("sess-b"))
    assert arena.buf.numel() == widest.arena_bytes + (1 << 20)
    for recompute in (False, True):
        assert eng._arena_bytes(Plan, 4, True, (), recompute) == \
            Plan(eng, 4, True, model.session_key("sess-b"), recompute=recompute).arena_bytes + (1 << 20)


def test_recompute_plan_growth_per_layer():
    """Between 2+2 and 3+3 layers the recompute plan grows by one fp32 [R, H] checkpoint per layer, and per decoder
    layer by the fused context_norm output and its gradient (bf16 [R, H] each)."""
    from multi_modal_foundation_model_b200.engine import Plan
    sizes = []
    for n in (2, 3):
        model = _model(96, n_layers=n).train()
        with torch.no_grad():
            model(_batch_md(model, 8, 96, MODS))
        eng = model.engine()
        assert eng.fuse_ctx
        sizes.append(Plan(eng, 8, True, recompute=True, dry=True).nbytes)
    R, H = 8 * 200, eng.H
    al = lambda n: -(-n // 256) * 256
    assert sizes[1] - sizes[0] == 2 * al(4 * R * H) + 2 * al(2 * R * H)


def test_default_b256_is_the_full_plan():
    with open(os.path.join(GOLDEN, "default_b256_plan_calls.json")) as f:
        want = json.load(f)
    model = _model(668).train()
    model(_batch_md(model, 256, 668, MODS)).loss.backward()
    pl = model.engine().last_plan
    assert not pl.recompute
    assert [c[2] for c in pl.fwd_calls] == want["fwd"]
    assert [c[2] for c in pl.bwd_calls] == want["bwd"]


def test_out_of_memory_below_the_recompute_plan(restore_fraction):
    holder, build = _small()
    model = build()
    md = _batch_md(model, 48, 96, MODS)
    with torch.no_grad():
        model(md)                      # the engine learns T
    gc.collect()
    torch.cuda.empty_cache()
    eng = model.engine()
    _set_fraction_for(eng, eng._plan_need(48, True, None, (), (), True) // 2, 48, None, ())
    with pytest.warns(UserWarning, match="recomputing"), pytest.raises(torch.cuda.OutOfMemoryError):
        model(md)


def test_scaled_model_b256_trains():
    """configs[4] at B 256 with default memory settings: the engine picks the recompute plan by itself."""
    from multi_modal_foundation_model_b200.optim import AdamW
    model, mods = _scaled_model()
    with torch.no_grad():
        model(_scaled_md(model, mods, 2))
    eng = model.engine()
    need = eng._plan_need(256, True, None, (), (), True)
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info()[0] + torch.cuda.memory_reserved() - torch.cuda.memory_allocated()
    if need + 3 * 4 * eng.store.total > free:
        pytest.skip(f"the device is shared: the recompute plan needs {need} bytes, {free} are free")
    opt = AdamW(model.parameters(), lr=1e-4)
    with pytest.warns(UserWarning, match="recomputing"):
        out = model(_scaled_md(model, mods, 256))
    out.loss.backward()
    opt.step()
    torch.cuda.synchronize()
    assert eng.last_plan.recompute and torch.isfinite(out.loss)
    assert all(torch.isfinite(p).all() for p in model.parameters())


def test_scaled_model_b16():
    """configs[4] at B 16, full plan against recompute plan in default mode (deterministic mode does not run at
    H 1024: the deterministic embedding backward exceeds the launch's register budget there, with either plan)."""
    mods = ("ap", "beh0", "beh1", "beh2", "beh3")
    holder, build = _builder(lambda: _scaled_model()[0])
    _within_run_to_run_spread(build, lambda s: _scaled_md(holder["m"], mods, 16, step=s), 16, steps=2)
