"""Deterministic mode (torch.use_deterministic_algorithms(True)): the *_det kernels give bitwise-identical results run
to run, also while a GEMM loop on a second stream perturbs CTA scheduling, and stay within the tolerances of the
default kernels.  wgrad is checked against fp32 torch; the column-sum kernels against their default twins, which
tests/test_gpu_norm_glue.py checks against fp32 torch.  The whole training step is bitwise repeatable under the flag,
eager and graph-replayed, and the flag off leaves the recorded schedule as it was."""
import contextlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@contextlib.contextmanager
def deterministic(on: bool = True):
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _perturb():
    """Queue a GEMM loop on a side stream so that the next kernels share the GPU with it."""
    s = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device="cuda")
    with torch.cuda.stream(s):
        for _ in range(8):
            a = a @ a * 1e-3
    return s, a


def _three_runs(run, outs):
    """run(outs) three times on fresh copies of `outs` (the second with the side-stream perturbation); asserts bitwise
    equality and returns the first result."""
    res = []
    for k in range(3):
        o = [t.clone() for t in outs]
        keep = _perturb() if k == 1 else None
        with deterministic():
            run(o)
        torch.cuda.synchronize()
        del keep
        res.append(o)
    for k in (1, 2):
        for a, b in zip(res[0], res[k]):
            assert torch.equal(a, b), f"run {k} differs from run 0"
    return res[0]


def _close(out, ref, tol, what):
    out, ref = out.float(), ref.float()
    scale = ref.abs().max().item() + 1e-6
    err = (out - ref).abs().max().item()
    assert err <= tol * scale, f"{what}: max err {err:.4g} vs scale {scale:.4g} (tol {tol})"


def _mk(rows, cols, scale=1.0, seed=0):
    """bf16 [rows, cols] view with a row pitch padded to 8 elements (the 16-byte pitch the TMA maps need)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    ld = (cols + 7) // 8 * 8
    return (torch.randn(rows, ld, generator=g, device="cuda") * scale).to(torch.bfloat16)[:, :cols]


@pytest.mark.parametrize("R,NO,KI", [(51200, 768, 256), (51200, 256, 512), (51200, 1336, 668), (130, 200, 72)])
def test_wgrad_det(R, NO, KI):
    from multi_modal_foundation_model_b200 import ops
    dY, X = _mk(R, NO, 0.1, seed=9), _mk(R, KI, seed=10)
    dW0, db0 = torch.ones(NO, KI, device="cuda"), torch.full((NO,), 2.0, device="cuda")
    dW, db = _three_runs(lambda o: ops.gemm_wgrad(dY, X, o[0], dbias=o[1]), [dW0, db0])
    _close(dW, dY.float().T @ X.float() + 1.0, 3e-3, "wgrad")
    _close(db, dY.float().sum(0) + 2.0, 3e-3, "wgrad bias")


def test_colsum_det():
    from multi_modal_foundation_model_b200 import ops
    dY = _mk(3000, 700, seed=3)
    (out,) = _three_runs(lambda o: ops.colsum_bf16(dY, o[0]), [torch.zeros(700, device="cuda")])
    _close(out, dY.float().sum(0), 1e-4, "colsum")


@pytest.mark.parametrize("R,H,mm", [(51200, 256, False), (600, 256, True), (123, 128, False), (500, 1024, False)])
def test_layernorm_bwd_det(R, H, mm):
    from multi_modal_foundation_model_b200 import ops
    T, S = (100, 200) if mm else (0, 0)
    dy = torch.randn(R, H, device="cuda").to(torch.bfloat16)
    x = torch.randn(R, H, device="cuda") * 2 + 0.5
    mean, rstd = x.mean(1), (x.var(1, unbiased=False) + 1e-5).rsqrt()
    g, dres = torch.randn(H, device="cuda"), torch.randn(R, H, device="cuda")

    def run(o):
        ops.layernorm_bwd(dy, x, mean, rstd, g, dres, o[0], o[1], ops.NO_DROP, o[2], o[3], R=R, H=H, modmajor_T=T, S=S)

    outs = [torch.zeros(R, H, device="cuda"), torch.zeros(R, H, device="cuda", dtype=torch.bfloat16),
            torch.full((H,), 0.5, device="cuda"), torch.full((H,), -0.5, device="cuda")]
    det = _three_runs(run, outs)
    ref = [t.clone() for t in outs]
    run(ref)
    torch.cuda.synchronize()
    assert torch.equal(det[0], ref[0]) and torch.equal(det[1], ref[1])   # the row outputs do not reduce across CTAs
    _close(det[2], ref[2], 1e-5, "dgamma")
    _close(det[3], ref[3], 1e-5, "dbeta")


@pytest.mark.parametrize("R,H,n", [(51200, 256, 5), (77, 128, 8)])
def test_layernorm_bwd_multi_det(R, H, n):
    from multi_modal_foundation_model_b200 import ops
    dys = [torch.randn(R, H, device="cuda").to(torch.bfloat16) for _ in range(n)]
    x = torch.randn(R, H, device="cuda")
    mean, rstd = x.mean(1), (x.var(1, unbiased=False) + 1e-5).rsqrt()
    gs = [torch.randn(H, device="cuda") for _ in range(n)]

    def run(o):
        ops.layernorm_bwd_multi(dys, x, mean, rstd, gs, o[0], None, o[1:1 + n], o[1 + n:], R=R, H=H)

    outs = [torch.zeros(R, H, device="cuda")] + [torch.zeros(H, device="cuda") for _ in range(2 * n)]
    det = _three_runs(run, outs)
    ref = [t.clone() for t in outs]
    run(ref)
    torch.cuda.synchronize()
    assert torch.equal(det[0], ref[0])
    for a, b in zip(det[1:], ref[1:]):
        _close(a, b, 1e-5, "dgamma / dbeta")


def test_scalenorm_bwd_det():
    from multi_modal_foundation_model_b200 import ops
    R, H = 20000, 256
    dy = torch.randn(R, H, device="cuda").to(torch.bfloat16)
    x = torch.randn(R, H, device="cuda")
    rn = 1.0 / x.norm(dim=1).clamp_min(1e-5)
    g = torch.tensor([1.7], device="cuda")

    def run(o):
        ops.scalenorm_bwd(dy, x, rn, g, None, o[0], None, ops.NO_DROP, o[1], R=R, H=H)

    outs = [torch.zeros(R, H, device="cuda"), torch.zeros(1, device="cuda")]
    det = _three_runs(run, outs)
    ref = [t.clone() for t in outs]
    run(ref)
    torch.cuda.synchronize()
    _close(det[1], ref[1], 1e-5, "dg")


@pytest.mark.parametrize("order", ["repeated", "permuted"])
def test_embed_assemble_bwd_det(order):
    from multi_modal_foundation_model_b200 import ops
    B, T, M, H, P = 256, 100, 2, 256, 100
    S = T * M
    gen = torch.Generator().manual_seed(4)
    if order == "repeated":   # padded trials repeat their last timestamp
        ts = torch.arange(T).repeat(B, 1)
        ts[:, 90:] = 89
    else:
        ts = torch.stack([torch.randperm(T, generator=gen) for _ in range(B)])
    ts = ts.cuda()
    g, g2 = torch.randn(B * S, H, device="cuda"), torch.randn(B * S, H, device="cuda")

    def run(o):
        ops.embed_assemble_bwd(g, g2, ts, o[0], o[1], B=B, T=T, S=S, off=T, H=H)

    outs = [torch.zeros(P, H, device="cuda"), torch.zeros(H, device="cuda")]
    dpos, dmod = _three_runs(run, outs)
    rows = (g + g2).view(B, M, T, H)[:, 1].reshape(B * T, H)
    ref_pos = torch.zeros(P, H, device="cuda").index_add_(0, ts.reshape(-1), rows)
    _close(dpos, ref_pos, 1e-5, "dpos")
    _close(dmod, rows.sum(0), 1e-5, "dmod")


@pytest.mark.parametrize("C", [1, 2, 5])
def test_smallc_embed_head_bwd_det(C):
    from multi_modal_foundation_model_b200 import ops
    B, T, M, H = 64, 100, 2, 256
    S, BT = T * M, B * T
    inp = torch.randn(BT, C, device="cuda")
    hid = torch.randn(BT, 2 * C, device="cuda").clamp(-0.9, 0.9)
    W2 = torch.randn(H, 2 * C, device="cuda")
    dx = torch.randn(B * S, H, device="cuda")

    def run_embed(o):
        ops.smallc_embed_bwd(inp, hid, W2, dx, None, ops.NO_DROP, 1.0, 0, o[0], o[1], o[2], o[3], B=B, T=T, S=S, off=T,
                             Cc=C, H=H)

    outs = [torch.zeros(2 * C, C, device="cuda"), torch.zeros(2 * C, device="cuda"), torch.zeros(H, 2 * C, device="cuda"),
            torch.zeros(H, device="cuda")]
    det = _three_runs(run_embed, outs)
    ref = [t.clone() for t in outs]
    run_embed(ref)
    torch.cuda.synchronize()
    for a, b in zip(det, ref):
        _close(a, b, 1e-5, "smallc embed bwd")

    y = torch.randn(BT, H, device="cuda").to(torch.bfloat16)
    W = torch.randn(C, H, device="cuda")
    dp = (torch.randn(BT, C, device="cuda") * 0.1).to(torch.bfloat16)

    def run_head(o):
        ops.smallc_head_bwd(y, W, dp, o[0], o[1], o[2], R=BT, H=H, Cc=C)

    outs = [torch.zeros(BT, H, device="cuda", dtype=torch.bfloat16), torch.zeros(C, H, device="cuda"),
            torch.zeros(C, device="cuda")]
    det = _three_runs(run_head, outs)
    ref = [t.clone() for t in outs]
    run_head(ref)
    torch.cuda.synchronize()
    assert torch.equal(det[0], ref[0])
    _close(det[1], ref[1], 1e-5, "smallc head dW")
    _close(det[2], ref[2], 1e-5, "smallc head db")


def test_column_stats_det():
    from multi_modal_foundation_model_b200 import ops
    R, C = 25600, 668
    p, y = torch.randn(R, C, device="cuda") * 0.3, torch.poisson(torch.full((R, C), 0.5, device="cuda"))
    (out,) = _three_runs(lambda o: ops.column_stats(p, y, o[0], log_rate=True),
                         [torch.empty(4 * C, dtype=torch.float64, device="cuda")])
    ref = torch.empty(4 * C, dtype=torch.float64, device="cuda")
    ops.column_stats(p, y, ref, log_rate=True)
    torch.cuda.synchronize()
    assert ((out - ref).abs() <= 1e-9 * ref.abs().clamp_min(1.0)).all()


def test_too_small_workspace_is_rejected():
    from multi_modal_foundation_model_b200 import _lib, ops
    dY, X = _mk(1000, 256, seed=1), _mk(1000, 256, seed=2)
    dW = torch.zeros(256, 256, device="cuda")
    ws = ops.DetWorkspace()
    ws.require(1024, 1)
    ws.materialize(dW.device)
    with deterministic(), pytest.raises(_lib.MmfmError, match="workspace too small"):
        ops._launch("mmfm_gemm_wgrad_det", dY.data_ptr(), dY.stride(0), X.data_ptr(), X.stride(0), 1000, 256, 256,
                    dW.data_ptr(), 256, None, ops.C.byref(ws.c))


# ------------------------------------------------------------------------------------------------------------
# whole training step
# ------------------------------------------------------------------------------------------------------------
def _model_and_batch(N, B, mods=("ap", "behavior"), cfg_kw=None, pad=10):
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.synthetic import make_batch
    cfg = default_model_config(**(cfg_kw or {}))
    torch.manual_seed(11)
    model = build_model(N, 2, cfg, avail_mod=tuple(mods)).cuda()
    model.train(True)
    batch = make_batch(B, N, 2, 100, step=2, pad_bins=pad)
    attn, ts = batch["time_attn_mask"], batch["spikes_timestamps"]
    xs = {"ap": batch["spikes_data"], "behavior": batch["target"]}
    g = torch.Generator().manual_seed(5)
    md = {}
    for m in mods:
        x = xs[m]
        md[m] = dict(inputs=x.cuda(), targets=x.cuda(), inputs_attn_mask=attn.cuda(), inputs_timestamp=ts.cuda(),
                     inputs_modality=torch.tensor(model.mod_to_indx[m], device="cuda"), masking_mode=None,
                     eval_mask=(torch.rand(B, 100, generator=g) < 0.3).long().cuda()[:, :, None].contiguous(),
                     inputs_regions=np.array([["CA1"] * x.shape[2]] * B))
    return model, md


def _steps(model, md, n=3):
    eng = model.engine()
    res = []
    for k in range(n):
        eng.reseed(1234)
        model.zero_grad(set_to_none=True)
        out = model({m: dict(d) for m, d in md.items()})
        out.loss.backward()
        torch.cuda.synchronize()
        res.append((out.loss.detach().clone(), {m: p.detach().clone() for m, p in out.mod_preds.items()},
                    eng.store.grad.detach().clone()))
    return res


def _assert_bitwise(res):
    for k in range(1, len(res)):
        assert torch.equal(res[0][0], res[k][0]), f"loss of step {k} differs"
        for m in res[0][1]:
            assert torch.equal(res[0][1][m], res[k][1][m]), f"preds {m} of step {k} differ"
        assert torch.equal(res[0][2], res[k][2]), f"gradients of step {k} differ"


@pytest.mark.parametrize("N,B,mods,cfg_kw", [
    (668, 256, ("ap", "behavior"), None),                   # the benchmarked workload
    (512, 16, ("ap",), None),                               # spike-only
    (64, 8, ("ap", "behavior"), {"use_scalenorm": True}),
])
def test_step_bitwise_repeatable(N, B, mods, cfg_kw):
    model, md = _model_and_batch(N, B, mods, cfg_kw)
    with deterministic():
        res = _steps(model, md)      # eager, then two graph replays
        plan = model.engine().last_plan
        assert plan.det_ws is not None
        assert any(c[2].endswith("_det") for c in plan.bwd_calls)
    _assert_bitwise(res)


def test_step_deterministic_matches_oracle():
    from test_gpu_bench_shape import _step_vs_oracle
    with deterministic():
        _step_vs_oracle(668, 32, ("ap", "behavior"), True, "token_masking", grad_rl2=3e-2)


def test_flag_off_schedule_unchanged_and_toggle():
    model, md = _model_and_batch(64, 8)
    with deterministic(False):
        _steps(model, md, 2)
    eng = model.engine()
    off_plan = eng.last_plan
    names_off = [c[2] for c in off_plan.bwd_calls]
    assert off_plan.det_ws is None and not any(n.endswith("_det") for n in names_off)
    with deterministic():
        res_on = _steps(model, md, 2)
    on_plan = eng.last_plan
    assert on_plan is not off_plan and len(eng.plans) == 2
    assert [n[:-4] if n.endswith("_det") else n for n in (c[2] for c in on_plan.bwd_calls)] == names_off
    with deterministic(False):
        res_off = _steps(model, md, 2)
    assert eng.last_plan is off_plan
    # both modes compute the same step up to summation order
    assert abs(res_on[0][0].item() - res_off[0][0].item()) <= 1e-4 * abs(res_off[0][0].item())


def test_adamw_trajectory_bitwise():
    from multi_modal_foundation_model_b200.optim import AdamW
    model, md = _model_and_batch(64, 8)
    state = {k: v.clone() for k, v in model.state_dict().items()}
    runs = []
    for _ in range(2):
        model.load_state_dict(state)
        opt = AdamW(model.parameters(), lr=1e-3)
        with deterministic():
            for _ in range(3):
                model.engine().reseed(7)
                opt.zero_grad(set_to_none=True)
                model({m: dict(d) for m, d in md.items()}).loss.backward()
                opt.step()
        torch.cuda.synchronize()
        runs.append([p.detach().clone() for p in model.parameters()])
    for a, b in zip(*runs):
        assert torch.equal(a, b)
