"""GPU: every floating-point output of the step (loss, mod_loss, mod_preds) and every floating-point input is
differentiable as in the reference.  Each case runs a loss functional of the outputs through the B200 step and through
``oracle.mm_oracle.forward`` under fp64 autograd on the same inputs, masks and Philox stream, and compares parameter
and input gradients."""
import os
import socket

import numpy as np
import pytest
import torch

from _util import cosine, oracle_params, rel_l2, small_config

pytestmark = pytest.mark.gpu

LOSS_RTOL, GRAD_RL2, GRAD_COS = 2e-3, 2e-2, 0.999


class Case:
    pass


def _case(N=96, B=8, mods=("ap", "behavior"), train=False, mode="token_masking", pad=10, n_beh=2, cfg=None,
          extra=None, loss_kinds=None, seed=11):
    from multi_modal_foundation_model_b200.losses import one_hot_stream
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.synthetic import make_batch
    c = Case()
    c.cfg = cfg or small_config()
    c.mods = list(mods)
    torch.manual_seed(seed)
    kw = {} if not extra else dict(extra_channels=extra, loss_kinds=loss_kinds)
    model = build_model(N, n_beh, c.cfg, avail_mod=tuple(mods), **kw)
    c.W = {k: v.detach().clone() for k, v in model.state_dict().items()}
    c.model = model.cuda().train(train)
    batch = make_batch(B, N, n_beh, 100, step=2, pad_bins=pad)
    c.attn, c.ts = batch["time_attn_mask"], batch["spikes_timestamps"]
    g = torch.Generator().manual_seed(5)
    c.xs = {"ap": batch["spikes_data"], "behavior": batch["target"]}
    for m, k in (extra or {}).items():
        c.xs[m] = one_hot_stream(torch.randint(0, k, (B, 1), generator=g).expand(B, 100), k)
    if mode == "token_masking":
        c.masks = {m: (torch.rand(B, 100, generator=g) < 0.3).long() for m in mods}
    else:
        c.masks = {m: torch.full((B, 100), int((m == "ap") == (mode == "encoding")), dtype=torch.int64) for m in mods}
    return c


def _md(c, grad_inputs=(), two_d=()):
    md, leaves = {}, {}
    for i, m in enumerate(c.mods):
        x = c.xs[m].cuda()
        if m in two_d:
            x = x[:, :, 0].contiguous()
        if m in grad_inputs:
            x = x.clone().requires_grad_(True)
            leaves[m] = x
        md[m] = dict(inputs=x, targets=c.xs[m].cuda() if m not in two_d else c.xs[m][:, :, 0].cuda(),
                     inputs_attn_mask=c.attn.cuda(), inputs_timestamp=c.ts.cuda(),
                     inputs_modality=torch.tensor(c.model.mod_to_indx[m], device="cuda"), masking_mode=None,
                     eval_mask=c.masks[m].cuda()[:, :, None].contiguous(),
                     inputs_regions=np.array([["CA1"] * c.xs[m].shape[2]] * x.shape[0]))
    return md, leaves


def _step(c, fn, grad_inputs=(), two_d=(), n=2, zero=True):
    """n steps on one plan (the second replays the captured graphs); returns the last output and input leaves."""
    for _ in range(n):
        if zero:
            c.model.zero_grad(set_to_none=True)
        md, leaves = _md(c, grad_inputs, two_d)
        out = c.model(md)
        fn(out).backward()
    torch.cuda.synchronize()
    return out, leaves


def _oracle(c, fn, grad_inputs=(), two_d=(), train=False, prefix_params=None):
    from oracle import mm_oracle as orc
    seed = int(c.model.engine().last_plan.seed.item()) & 0xFFFFFFFFFFFFFFFF if train else None
    P = oracle_params(prefix_params if prefix_params is not None else c.W)
    uniq, Q = {}, {}
    for k, v in P.items():
        if v.data_ptr() not in uniq:
            uniq[v.data_ptr()] = v.detach().double().clone().requires_grad_(True)
        Q[k] = uniq[v.data_ptr()]
    spec = orc.OracleSpec.from_config(c.cfg, c.mods)
    for m in c.mods:
        if c.xs[m].shape[2] > 2 and m != "ap":
            spec.loss_kind[m] = "ce"
    ob, leaves = {}, {}
    for m in c.mods:
        x = c.xs[m].double()
        t = x
        if m in two_d:
            x, t = x[:, :, 0].contiguous(), t[:, :, 0].contiguous()
        if m in grad_inputs:
            x = x.clone().requires_grad_(True)
            leaves[m] = x
        ob[m] = dict(inputs=x, targets=t, attn_mask=c.attn, timestamp=c.ts, mask=c.masks[m] & c.attn)
    out = orc.forward(Q, spec, ob, dropout_seed=seed)
    fn(out).backward()
    grads = {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in Q.items()}
    return out, grads, {m: x.grad for m, x in leaves.items()}


def _close(got, ref, what, tol=GRAD_RL2, scale=1.0):
    """scale: norm of the whole reference gradient -- a gradient that is zero in exact arithmetic (e.g. of a key bias
    under softmax) carries rounding noise proportional to it (mod_loss is an unnormalised sum)"""
    got = got.detach().cpu().double()
    assert torch.isfinite(got).all(), f"{what}: non-finite gradient"
    if ref.norm() < 1e-6 * max(1.0, scale):
        assert got.norm().item() < 1e-4 * max(1.0, scale), f"{what}: {got.norm().item()} where the reference is zero"
        return
    r, cs = rel_l2(got, ref), cosine(got, ref)
    assert r < tol and cs > GRAD_COS, f"{what}: rel-L2 {r:.4g} cosine {cs:.6f}"


def _check_params(model, grads, tol=GRAD_RL2):
    scale = torch.cat([g.flatten() for g in grads.values()]).norm().item()
    for n, p in model.named_parameters():
        g = p.grad if p.grad is not None else torch.zeros_like(p)
        _close(g, grads[n], n, tol * (2.0 if p.numel() < 16 else 1.0), scale)


def _check_outputs(out, ref):
    assert abs(out.loss.item() - ref.loss.item()) <= LOSS_RTOL * abs(ref.loss.item()) + 1e-6
    for m in ref.mod_loss:
        assert abs(out.mod_loss[m].item() - ref.mod_loss[m].item()) <= 3e-3 * abs(ref.mod_loss[m].item()) + 1e-3, m


# ---- 1-2: weighted mod_loss ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("train", [False, True])
def test_weighted_mod_loss(train):
    c = _case(train=train)
    fn = lambda o: 0.3 * o.mod_loss["ap"] + 2.5 * o.mod_loss["behavior"]      # noqa: E731  (out.loss unused)
    out, _ = _step(c, fn)
    ref, grads, _ = _oracle(c, fn, train=train)
    _check_outputs(out, ref)
    _check_params(c.model, grads, tol=3e-2 if train else GRAD_RL2)


def test_weighted_mod_loss_cross_entropy():
    K = {"choice": 3}
    c = _case(N=72, B=6, mods=("ap", "behavior", "choice"), extra=K, loss_kinds={"choice": "ce"},
              cfg=small_config(n_modality=3))
    fn = lambda o: 0.5 * o.mod_loss["ap"] + 1.5 * o.mod_loss["behavior"] + 4.0 * o.mod_loss["choice"]  # noqa: E731
    out, _ = _step(c, fn)
    ref, grads, _ = _oracle(c, fn)
    _check_outputs(out, ref)
    _check_params(c.model, grads)


def test_loss_plus_weighted_behavior():
    c = _case()
    fn = lambda o: o.loss + 0.7 * o.mod_loss["behavior"]                      # noqa: E731
    out, _ = _step(c, fn)
    ref, grads, _ = _oracle(c, fn)
    _check_outputs(out, ref)
    _check_params(c.model, grads)


# ---- 3: losses on predictions (incl. stride-0 upstream gradients from sum() / mean()) -------------------------------
def test_losses_on_predictions():
    c = _case()
    R = torch.randn(8, 100, 2, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    fn = lambda o: (o.mod_preds["behavior"] * R.to(o.mod_preds["behavior"])).sum() + \
        o.mod_preds["ap"].square().mean() + o.mod_preds["behavior"].sum()   # noqa: E731
    out, _ = _step(c, fn)
    ref, grads, _ = _oracle(c, fn)
    for m in c.mods:
        assert (out.mod_preds[m].detach().cpu().double() - ref.mod_preds[m].detach()).abs().max().item() < 3e-2
    _check_params(c.model, grads)


# ---- 4: degenerate masks ------------------------------------------------------------------------------------------
def test_encoding_mode_weighted():
    c = _case(mode="encoding")           # behaviour mask all zero
    fn = lambda o: 2.0 * o.mod_loss["ap"] + 5.0 * o.mod_loss["behavior"]      # noqa: E731
    out, _ = _step(c, fn)
    ref, grads, _ = _oracle(c, fn)
    _check_params(c.model, grads)


def test_no_masked_token_preds_only():
    c = _case()
    c.masks = {m: torch.zeros_like(v) for m, v in c.masks.items()}      # sum n = 0: inv_n is inf, loss is NaN
    fn = lambda o: o.mod_preds["ap"].square().mean() + o.mod_preds["behavior"].sum()  # noqa: E731
    out, _ = _step(c, fn)
    ref, grads, _ = _oracle(c, fn)
    _check_params(c.model, grads)


# ---- 5: input gradients ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,train", [(96, False), (50, False), (96, True)])
def test_input_gradients(N, train):
    c = _case(N=N, train=train)
    fn = lambda o: o.loss + 0.5 * o.mod_loss["behavior"]                      # noqa: E731
    out, leaves = _step(c, fn, grad_inputs=("ap", "behavior"))
    ref, grads, dref = _oracle(c, fn, grad_inputs=("ap", "behavior"), train=train)
    tol = 3e-2 if train else GRAD_RL2
    for m in ("ap", "behavior"):
        assert leaves[m].grad is not None and leaves[m].grad.dtype == leaves[m].dtype
        assert leaves[m].grad.shape == leaves[m].shape
        _close(leaves[m].grad, dref[m], f"d inputs[{m}]", tol)
    _check_params(c.model, grads, tol=tol)
    # tokens zeroed by sample 0's mask (mm.py:147-149) get exactly zero input gradient
    zero_t = torch.nonzero((c.masks["ap"] & c.attn)[0] == 1).flatten()
    assert zero_t.numel() > 0
    assert torch.count_nonzero(leaves["ap"].grad[:, zero_t.cuda()]).item() == 0


def test_input_gradient_2d_behavior_and_plain_loss():
    c = _case(n_beh=1)
    fn = lambda o: o.loss                                                      # noqa: E731
    out, leaves = _step(c, fn, grad_inputs=("behavior",), two_d=("behavior",))
    ref, grads, dref = _oracle(c, fn, grad_inputs=("behavior",), two_d=("behavior",))
    assert leaves["behavior"].grad.shape == leaves["behavior"].shape == (8, 100)
    _close(leaves["behavior"].grad, dref["behavior"], "d inputs[behavior] (2-D)")
    _check_params(c.model, grads)


def test_input_gradients_frozen_model():
    c = _case()
    for p in c.model.parameters():
        p.requires_grad_(False)
    fn = lambda o: o.mod_preds["behavior"][:, :, 0].sum()                     # noqa: E731  saliency of one output
    out, leaves = _step(c, fn, grad_inputs=("ap", "behavior"))
    _, _, dref = _oracle(c, fn, grad_inputs=("ap", "behavior"))
    for m in ("ap", "behavior"):
        _close(leaves[m].grad, dref[m], f"d inputs[{m}] (frozen)")
    assert all(p.grad is None for p in c.model.parameters())


# ---- 6: graph replay, alternating plain and weighted backward -------------------------------------------------------
def test_alternating_plain_and_weighted_replay(monkeypatch):
    from multi_modal_foundation_model_b200 import ops
    c = _case()
    ce = _case()
    ce.model.engine().use_graphs = False
    plain = lambda o: o.loss                                                   # noqa: E731
    weighted = lambda o: 0.2 * o.mod_loss["ap"] + 3.0 * o.mod_loss["behavior"]  # noqa: E731
    calls = {"n": 0}
    real = ops.loss_grad

    def counting(*a, **k):
        calls["n"] += 1
        return real(*a, **k)

    monkeypatch.setattr(ops, "loss_grad", counting)
    graph = None
    for k in range(5):
        fn = plain if k % 2 == 0 else weighted
        for cc in (c, ce):
            cc.model.engine().reseed(99 + k)
        before = calls["n"]
        _step(c, fn, n=1)
        if k % 2 == 0:
            assert calls["n"] == before, "plain backward must not launch loss_grad"
        _step(ce, fn, n=1)
        pl = c.model.engine().last_plan
        if pl._g_bwd is not None:
            graph = pl._g_bwd if graph is None else graph
            assert pl._g_bwd is graph, "the plan's captured backward graph must be reused"
        for (n, p), q in zip(c.model.named_parameters(), ce.model.parameters()):
            _close(p.grad, q.grad.detach().cpu().double(), f"step {k} {n}", 1e-3)
    assert graph is not None


# ---- 7: deterministic mode --------------------------------------------------------------------------------------------
def test_deterministic_bitwise():
    torch.use_deterministic_algorithms(True)
    try:
        c = _case()
        res = []
        for fn in (lambda o: o.loss, lambda o: 1.0 * o.loss + 0.0 * o.mod_loss["ap"]):
            c.model.engine().reseed(5)
            _step(c, fn, n=1)
            res.append(c.model.engine().store.grad.clone())
        assert torch.equal(res[0], res[1])
        dx = []
        for _ in range(2):
            c.model.engine().reseed(5)
            _, leaves = _step(c, lambda o: o.loss, grad_inputs=("ap", "behavior"), n=1)
            dx.append({m: x.grad.clone() for m, x in leaves.items()})
        for m in dx[0]:
            assert torch.equal(dx[0][m], dx[1][m]), m
    finally:
        torch.use_deterministic_algorithms(False)


# ---- 8: accumulation --------------------------------------------------------------------------------------------------
def test_weighted_accumulates_on_plain():
    c = _case()
    c.model.zero_grad(set_to_none=True)
    _step(c, lambda o: o.loss, n=1, zero=False)
    _step(c, lambda o: 0.4 * o.mod_loss["ap"] + 2.0 * o.mod_loss["behavior"], n=1, zero=False)
    _, grads, _ = _oracle(c, lambda o: o.loss + 0.4 * o.mod_loss["ap"] + 2.0 * o.mod_loss["behavior"])
    _check_params(c.model, grads)


# ---- 9: multi-session ---------------------------------------------------------------------------------------------------
def test_multi_session_weighted():
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
    from multi_modal_foundation_model_b200.synthetic import make_batch
    cfg = small_config()
    chans = {"sess-a": {"ap": 40, "behavior": 2}, "sess-b": {"ap": 88, "behavior": 2}}
    torch.manual_seed(21)
    model = MultiSessionMultiModal(chans, ["ap", "behavior"], cfg)
    W = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.cuda().eval()
    c = _case()
    c.model, c.cfg = model, cfg
    batch = make_batch(4, 88, 2, 100, step=1, pad_bins=5)
    c.xs = {"ap": batch["spikes_data"], "behavior": batch["target"]}
    c.attn, c.ts = batch["time_attn_mask"], batch["spikes_timestamps"]
    c.masks = {m: (torch.rand(4, 100, generator=torch.Generator().manual_seed(1)) < 0.3).long() for m in c.mods}
    fn = lambda o: 0.5 * o.mod_loss["ap"] + 3.0 * o.mod_loss["behavior"]      # noqa: E731
    model.zero_grad(set_to_none=True)
    md, leaves = _md(c, ("ap",))
    for d in md.values():
        d["eid"] = "sess-b"
    fn(model(md)).backward()
    torch.cuda.synchronize()
    prefix = model.session_prefix("sess-b")
    P = {k[len(prefix):] if k.startswith(prefix) else k: v for k, v in W.items()
         if not k.startswith("session_embeddings.") or k.startswith(prefix)}
    _, grads, dref = _oracle(c, fn, grad_inputs=("ap",), prefix_params=P)
    scale = torch.cat([g.flatten() for g in grads.values()]).norm().item()
    for n, p in model.named_parameters():
        if n.startswith("session_embeddings.") and not n.startswith(prefix):
            assert p.grad is None or torch.count_nonzero(p.grad).item() == 0, n
        else:
            key = n[len(prefix):] if n.startswith(prefix) else n
            _close(p.grad if p.grad is not None else torch.zeros_like(p), grads[key], n,
                   GRAD_RL2 * (2.0 if p.numel() < 16 else 1.0), scale)
    _close(leaves["ap"].grad, dref["ap"], "d inputs[ap] (session b)")


# ---- 10: linear baselines ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["decoder", "encoder"])
def test_baseline_preds_and_input_gradients(kind):
    from multi_modal_foundation_model_b200.baselines import BaselineDecoder, BaselineEncoder
    from oracle import mm_oracle as orc
    torch.manual_seed(3)
    B, T, N, nb = 16, 20, 48, 2
    g = torch.Generator().manual_seed(2)
    if kind == "decoder":
        model = BaselineDecoder(N, nb)
        x, y = torch.randn(B, T, N, generator=g), torch.randn(B, T, nb, generator=g)
        ref_fn = orc.baseline_decoder
    else:
        model = BaselineEncoder(nb, N, seq_len=T)
        x, y = torch.randn(B, T, nb, generator=g), torch.poisson(torch.full((B, T, N), 0.5), generator=g)
        ref_fn = orc.baseline_encoder
    P = {k: v.detach().double().clone().requires_grad_(True) for k, v in model.state_dict().items()}
    model = model.cuda()
    xg = x.cuda().requires_grad_(True)
    out = model({"inputs": xg, "targets": y.cuda()})
    (0.5 * out.loss + out.preds.square().mean()).backward()
    xr = x.double().requires_grad_(True)
    loss_r, preds_r = ref_fn(P, xr, y.double())
    (0.5 * loss_r + preds_r.square().mean()).backward()
    _close(xg.grad, xr.grad, "d inputs")
    _close(model.layer.weight.grad, P["layer.weight"].grad, "d weight")
    _close(model.layer.bias.grad, P["layer.bias"].grad, "d bias")


# ---- 11: errors ---------------------------------------------------------------------------------------------------------
def test_errors():
    c = _case()
    md, _ = _md(c)
    md["behavior"]["targets"] = md["behavior"]["targets"].clone().requires_grad_(True)
    with pytest.raises(NotImplementedError):
        c.model(md)
    md, leaves = _md(c, ("ap",))
    out = c.model(md)
    (g,) = torch.autograd.grad(out.loss, [leaves["ap"]], create_graph=True)
    with pytest.raises(RuntimeError):
        g.sum().backward()


# ---- 12: data parallel ---------------------------------------------------------------------------------------------------
def _ddp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.parallel import DataParallel
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        torch.manual_seed(100)
        model = build_model(40, 2, small_config()).cuda().eval()
        ddp = DataParallel(model, bucket_mb=0.25)
        for _ in range(3):                     # eager, graph capture, graph replay
            batch = make_batch(4, 40, 2, 100, step=10 + rank, pad_bins=5)
            md = make_mod_dict(batch, ["ap", "behavior"], "decoding", device="cuda")
            model.zero_grad(set_to_none=True)
            out = model(md)
            (0.3 * out.mod_loss["ap"] + 2.0 * out.mod_loss["behavior"]).backward()
        torch.cuda.synchronize()
        torch.save({n: p.grad.detach().cpu().clone() for n, p in model.named_parameters()},
                   os.path.join(out_dir, f"rank{rank}.pt"))
        ddp.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_ddp_weighted_loss(tmp_path):
    import torch.multiprocessing as mp
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_ddp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r = [torch.load(tmp_path / f"rank{i}.pt") for i in range(2)]
    torch.manual_seed(100)
    model = build_model(40, 2, small_config()).cuda().eval()
    acc = None
    for rank in range(2):
        batch = make_batch(4, 40, 2, 100, step=10 + rank, pad_bins=5)
        md = make_mod_dict(batch, ["ap", "behavior"], "decoding", device="cuda")
        model.zero_grad(set_to_none=True)
        out = model(md)
        (0.3 * out.mod_loss["ap"] + 2.0 * out.mod_loss["behavior"]).backward()
        g = {n: p.grad.detach().cpu().clone() for n, p in model.named_parameters()}
        acc = g if acc is None else {n: acc[n] + g[n] for n in g}
    for n, gref in acc.items():
        assert torch.equal(r[0][n], r[1][n]), f"ranks disagree on {n}"
        gref = gref / 2
        scale = gref.abs().max().item() + 1e-8
        assert (r[0][n] - gref).abs().max().item() <= 2e-3 * scale + 1e-7, n
