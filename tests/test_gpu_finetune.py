"""Fine-tuning on the B200 path: the fused AdamW with parameter groups, subsets, skipped parameters, add_param_group and
torch-compatible state_dict, each against torch.optim.AdamW on fp32 shadow parameters fed the engine's gradients; and
the backward without the weight-gradient launches of frozen parameters."""
import copy
import os
import socket
from contextlib import contextmanager

import pytest
import torch

from _util import small_config

pytestmark = pytest.mark.gpu

RTOL, ATOL = 2e-6, 2e-8
MODES = ("encoding", "decoding", "token_masking")


def _is_core(name):
    return "embeddings." not in name


def _model(seed=1, N=40):
    from multi_modal_foundation_model_b200.model import build_model
    torch.manual_seed(seed)
    return build_model(N, 2, small_config()).cuda().eval()


def _md(step, N=40, B=3):
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    return make_mod_dict(make_batch(B, N, 2, 100, step=step), ["ap", "behavior"], MODES[step % 3], device="cuda")


class Shadow:
    """fp32 copies of the optimised parameters, driven by torch.optim.AdamW with the same group layout."""

    def __init__(self, groups, **kw):
        self.src = [list(g["params"]) for g in groups]
        self.ref = [[torch.nn.Parameter(p.detach().clone()) for p in ps] for ps in self.src]
        rg = []
        for g, rps in zip(groups, self.ref):
            d = {k: v for k, v in g.items() if k != "params"}
            d["params"] = rps
            rg.append(d)
        self.opt = torch.optim.AdamW(rg, **kw)

    def add(self, group):
        ps = list(group["params"])
        self.src.append(ps)
        self.ref.append([torch.nn.Parameter(p.detach().clone()) for p in ps])
        self.opt.add_param_group({**{k: v for k, v in group.items() if k != "params"}, "params": self.ref[-1]})

    def feed(self):
        for ps, rps in zip(self.src, self.ref):
            for p, rp in zip(ps, rps):
                rp.grad = None if p.grad is None else p.grad.detach().clone()

    def check(self, what=""):
        for ps, rps in zip(self.src, self.ref):
            for p, rp in zip(ps, rps):
                assert torch.allclose(p.detach(), rp.detach(), rtol=RTOL, atol=ATOL), (what, (p - rp).abs().max().item())


def _decay_groups(model, lr=(1e-3, 3e-3), wd=(0.05, 0.0)):
    decay = [p for n, p in model.named_parameters() if p.ndim >= 2]
    no_decay = [p for n, p in model.named_parameters() if p.ndim < 2]
    return [{"params": decay, "lr": lr[0], "weight_decay": wd[0]},
            {"params": no_decay, "lr": lr[1], "weight_decay": wd[1]}]


def _pads_are_zero(st, *bufs):
    mask = torch.ones(st.total, dtype=torch.bool, device=st.flat.device)
    for n in st.params:
        o = st.offset[n]
        mask[o:o + st.shape[n].numel()] = False
    for b in bufs:
        assert not b[mask].any()


def test_two_groups_under_onecycle():
    from multi_modal_foundation_model_b200.optim import AdamW
    model = _model()
    model(_md(0))          # the engine (and its flat buffers) exists before the optimizer binds
    groups = _decay_groups(model)
    opt = AdamW(groups, eps=1e-8)
    sh = Shadow(groups, eps=1e-8)
    kw = dict(total_steps=10, max_lr=[1e-3, 3e-3], pct_start=0.3, div_factor=10)      # cycle_momentum drives betas
    sched = torch.optim.lr_scheduler.OneCycleLR(opt, **kw)
    rsched = torch.optim.lr_scheduler.OneCycleLR(sh.opt, **kw)
    for step in range(5):
        opt.zero_grad(set_to_none=True)
        model(_md(step)).loss.backward()
        sh.feed()
        opt.step()
        sh.opt.step()
        sched.step()
        rsched.step()
        sh.check(step)
    assert opt.param_groups[0]["betas"] != (0.9, 0.999)
    st = model.engine().store
    _pads_are_zero(st, st.flat, st.grad, opt._m, opt._v)


def test_subset_with_frozen_core():
    from multi_modal_foundation_model_b200.optim import AdamW
    model = _model(2)
    for n, p in model.named_parameters():
        p.requires_grad_(not _is_core(n))
    frozen = {n: p.detach().clone() for n, p in model.named_parameters() if _is_core(n)}
    model(_md(0))
    opt = AdamW((p for p in model.parameters() if p.requires_grad), lr=2e-3, weight_decay=0.1)
    sh = Shadow(opt.param_groups, lr=2e-3, weight_decay=0.1)
    for step in range(4):
        opt.zero_grad(set_to_none=True)
        model(_md(step)).loss.backward()
        sh.feed()
        opt.step()
        sh.opt.step()
        sh.check(step)
    for n, p in model.named_parameters():
        if _is_core(n):
            assert p.grad is None and torch.equal(p.detach(), frozen[n]), n
            assert p not in opt.state
    m = opt._m
    st = model.engine().store
    for n in frozen:
        assert not st.view(m, n).any()


def test_parameter_without_gradient_keeps_its_own_step_count():
    """torch.optim.AdamW counts steps per parameter: a parameter skipped once is one bias-correction step behind."""
    from multi_modal_foundation_model_b200.optim import AdamW
    model = _model(3)
    model(_md(0))
    opt = AdamW(model.parameters(), lr=1e-2, weight_decay=0.1)
    sh = Shadow(opt.param_groups, lr=1e-2, weight_decay=0.1)
    named = dict(model.named_parameters())
    skipped = [named["encoder.0.mlp.up_proj.weight"], named["decoder.0.ln1.bias"]]
    for step in range(4):
        opt.zero_grad(set_to_none=True)
        model(_md(step)).loss.backward()
        if step == 1:
            for p in skipped:
                p.grad = None
        sh.feed()
        opt.step()
        sh.opt.step()
        sh.check(step)
    assert float(opt.state[skipped[0]]["step"]) == 3.0 and float(opt.state[named["decoder_norm.weight"]]["step"]) == 4.0


def test_add_param_group_mid_run():
    from multi_modal_foundation_model_b200.optim import AdamW
    model = _model(4)
    model(_md(0))
    heads = [p for n, p in model.named_parameters() if not _is_core(n)]
    core = [p for n, p in model.named_parameters() if _is_core(n)]
    opt = AdamW(heads, lr=2e-3)
    sh = Shadow(opt.param_groups, lr=2e-3)
    for step in range(5):
        if step == 2:
            opt.add_param_group({"params": core, "lr": 5e-4, "weight_decay": 0.0})
            sh.add(opt.param_groups[-1])
        opt.zero_grad(set_to_none=True)
        model(_md(step)).loss.backward()
        sh.feed()
        opt.step()
        sh.opt.step()
        sh.check(step)


def test_state_dict_round_trips_with_torch():
    from multi_modal_foundation_model_b200.optim import AdamW
    model = _model(5)
    model(_md(0))
    # the reference's lr (1e-4).  The kernel takes betas as fp32 (as mmfm_adamw_step always has), so its moments are
    # normalised for 1 - float(beta2) and torch's for 1 - beta2 in double: continuing from the other's moments, the
    # first updates differ by ~1e-5 of an update, i.e. ~1e-8 absolute at lr 3e-3 -- at the size of the atol for the
    # small (zero-initialised) biases.  At lr 1e-4 that is ~1e-9; a wrong state (step count, moments) is ~lr.
    groups = _decay_groups(model, lr=(1e-4, 3e-4))
    opt = AdamW(groups)
    sh = Shadow(groups)

    def run(fused, ref, steps):
        for step in steps:
            fused.zero_grad(set_to_none=True)
            model(_md(step)).loss.backward()
            sh.feed()
            fused.step()
            ref.step()
            sh.check(step)

    run(opt, sh.opt, range(2))
    # fused -> torch and torch -> fused: each continues from the other's state
    ref2 = torch.optim.AdamW([{**{k: v for k, v in g.items() if k != "params"}, "params": rps}
                              for g, rps in zip(sh.opt.param_groups, sh.ref)])
    ref2.load_state_dict(copy.deepcopy(opt.state_dict()))
    opt2 = AdamW(_decay_groups(model, lr=(1e-4, 3e-4)))
    opt2.load_state_dict(copy.deepcopy(sh.opt.state_dict()))
    run(opt2, ref2, range(2, 5))
    for p in model.parameters():
        assert float(opt2.state[p]["step"]) == 5.0


def test_clip_grad_norm_before_step():
    from multi_modal_foundation_model_b200.optim import AdamW
    model = _model(6)
    model(_md(0))
    opt = AdamW(model.parameters(), lr=1e-3)
    sh = Shadow(opt.param_groups, lr=1e-3)
    for step in range(3):
        opt.zero_grad(set_to_none=True)
        model(_md(step)).loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 0.05)
        sh.feed()
        opt.step()
        sh.opt.step()
        sh.check(step)
    assert all(p.grad.data_ptr() == model.engine().store.g(n).data_ptr() for n, p in model.named_parameters())


def test_multi_session_trains_one_session_over_frozen_core():
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
    from multi_modal_foundation_model_b200.optim import AdamW
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    chans = {"sess-a": {"ap": 40, "behavior": 2}, "sess-b": {"ap": 88, "behavior": 2}}
    torch.manual_seed(21)
    model = MultiSessionMultiModal(chans, ["ap", "behavior"], small_config()).cuda().eval()
    prefix = model.session_prefix("sess-b")
    for n, p in model.named_parameters():
        p.requires_grad_(n.startswith(prefix))
    before = {n: p.detach().clone() for n, p in model.named_parameters()}

    def md(step):
        d = make_mod_dict(make_batch(3, 88, 2, 100, step=step), ["ap", "behavior"], MODES[step % 3], device="cuda")
        for v in d.values():
            v["eid"] = "sess-b"
        return d

    model(md(0))
    opt = AdamW([p for n, p in model.named_parameters() if n.startswith(prefix)], lr=3e-3)
    sh = Shadow(opt.param_groups, lr=3e-3)
    for step in range(4):
        opt.zero_grad(set_to_none=True)
        model(md(step)).loss.backward()
        sh.feed()
        opt.step()
        sh.opt.step()
        sh.check(step)
    for n, p in model.named_parameters():
        if not n.startswith(prefix):
            assert p.grad is None and torch.equal(p.detach(), before[n]), n


def test_optimizer_errors():
    from multi_modal_foundation_model_b200._lib import MmfmError
    from multi_modal_foundation_model_b200.optim import AdamW
    a, b = _model(7), _model(8)
    a(_md(0))
    b(_md(0))
    foreign = torch.nn.Parameter(torch.zeros(8, device="cuda"))
    opt = AdamW(list(a.parameters()) + [foreign])
    a(_md(1)).loss.backward()
    foreign.grad = torch.ones_like(foreign)
    with pytest.raises(MmfmError, match="ONE engine"):
        opt.step()
    opt = AdamW([{"params": list(a.parameters())}, {"params": list(b.parameters())}])
    with pytest.raises(MmfmError, match="ONE engine"):
        opt.step()
    with pytest.raises(NotImplementedError, match="tensor lr"):
        AdamW(a.parameters(), lr=torch.tensor(1e-3))
    with pytest.raises(NotImplementedError, match="tensor lr"):
        AdamW([{"params": list(a.parameters()), "lr": torch.tensor(1e-3)}])
    opt = AdamW(a.parameters())
    opt.param_groups[0]["lr"] = torch.tensor(1e-3)
    with pytest.raises(NotImplementedError, match="tensor lr"):
        opt.step()


# ---- frozen parameters skip their weight gradient -----------------------------------------------------------------
@contextmanager
def _deterministic():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _freeze_core(model, frozen=True):
    for n, p in model.named_parameters():
        p.requires_grad_(not (frozen and _is_core(n)))


def test_frozen_core_backward_has_no_frozen_wgrad():
    model = _model(9)
    _freeze_core(model)
    model(_md(0)).loss.backward()
    pl = model.engine().last_plan
    st = model.engine().store
    skip, calls, marks = pl.backward_schedule()
    assert skip and len(calls) == len(pl.bwd_calls) - len(skip)
    kept = {id(c) for c in calls}
    for ci, names in pl.wgrad_writes:
        all_frozen = not any(st.params[n].requires_grad for n in names)
        assert (id(pl.bwd_calls[ci]) in kept) != all_frozen, names
    assert [off for _, off in marks] == [off for _, off in pl.grad_marks]


def test_frozen_gradients_bitwise_and_unfreezing():
    """Deterministic mode: the trainable gradients of the frozen-core backward equal those of the full backward bit for
    bit (same forward, same seed); frozen .grad stays None; unfreezing switches back to the full list."""
    model = _model(10)
    model.train(True)
    md = _md(2)
    eng = model.engine

    def grads(frozen, n=2):
        _freeze_core(model, frozen)
        for _ in range(n):                      # eager, then the captured graph of this call list
            model.zero_grad(set_to_none=True)
            eng().reseed(7)
            model({m: dict(d) for m, d in md.items()}).loss.backward()
        torch.cuda.synchronize()
        return {n: (None if p.grad is None else p.grad.detach().clone()) for n, p in model.named_parameters()}

    with _deterministic():
        model({m: dict(d) for m, d in md.items()})
        full = grads(False)
        part = grads(True)
        pl = eng().last_plan
        assert pl.backward_schedule()[0]
        again = grads(False)
        assert pl.backward_schedule()[1] is pl.bwd_calls
        part2 = grads(True)
    for n in full:
        assert torch.equal(again[n], full[n]), n
        if _is_core(n):
            assert part[n] is None and part2[n] is None, n
        else:
            assert torch.equal(part[n], full[n]) and torch.equal(part2[n], full[n]), n


def test_all_frozen_input_gradients_match_oracle():
    from test_gpu_autograd_outputs import _case, _close, _oracle, _step
    c = _case()
    for p in c.model.parameters():
        p.requires_grad_(False)
    fn = lambda o: o.loss                                                      # noqa: E731
    out, leaves = _step(c, fn, grad_inputs=("ap", "behavior"))
    _, _, dref = _oracle(c, fn, grad_inputs=("ap", "behavior"))
    for m in ("ap", "behavior"):
        _close(leaves[m].grad, dref[m], f"d inputs[{m}] (frozen)")
    pl = c.model.engine().last_plan
    skip, calls, _ = pl.backward_schedule()
    assert len(skip) == len(pl.wgrad_writes) and not any(k[2].startswith("mmfm_gemm_wgrad") for k in calls)
    assert all(p.grad is None for p in c.model.parameters())


def _ddp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from multi_modal_foundation_model_b200.parallel import DataParallel
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        model = _model(100 + rank)
        _freeze_core(model)
        ddp = DataParallel(model, bucket_mb=0.25)
        for step in (0, 2, 1):                   # eager, graph capture, graph replay
            batch = make_batch(4, 40, 2, 100, step=10 * step + rank, pad_bins=5)
            md = make_mod_dict(batch, ["ap", "behavior"], "encoding" if step == 0 else "decoding", device="cuda")
            model.zero_grad(set_to_none=True)
            model(md).loss.backward()
        torch.cuda.synchronize()
        grads = {n: p.grad.detach().cpu().clone() for n, p in model.named_parameters() if p.grad is not None}
        torch.save(grads, os.path.join(out_dir, f"rank{rank}.pt"))
        ddp.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_ddp_frozen_core_is_rank_mean(tmp_path):
    import torch.multiprocessing as mp
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    world = 2
    mp.spawn(_ddp_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    r = [torch.load(tmp_path / f"rank{i}.pt") for i in range(world)]
    assert set(r[0]) == {n for n, _ in _model(100).named_parameters() if not _is_core(n)}
    model = _model(100)                          # rank 0's weights (broadcast)
    _freeze_core(model)
    acc = None
    for rank in range(world):
        batch = make_batch(4, 40, 2, 100, step=10 + rank, pad_bins=5)
        md = make_mod_dict(batch, ["ap", "behavior"], "decoding", device="cuda")
        model.zero_grad(set_to_none=True)
        model(md).loss.backward()
        g = {n: p.grad.detach().cpu().clone() for n, p in model.named_parameters() if p.grad is not None}
        acc = g if acc is None else {n: acc[n] + g[n] for n in g}
    for n, gref in acc.items():
        gref = gref / world
        assert torch.equal(r[0][n], r[1][n]), n
        scale = gref.abs().max().item() + 1e-8
        assert (r[0][n] - gref).abs().max().item() <= 2e-3 * scale + 1e-7, n
