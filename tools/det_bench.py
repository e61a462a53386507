"""Cost of the deterministic mode (torch.use_deterministic_algorithms(True)).

    python tools/det_bench.py [--out FILE] [--steps K] [--rounds N]

1. Graph-replayed training step (train(), all dropout sites on) with the flag off and on, alternating in one process
   (both plans built and warmed first), at the benchmarked workload (B = 256, N = 668) and at B = 16.
2. Per-launch times of the deterministic wgrad / LayerNorm backward against the default kernels at the bench shapes
   (CUDA events around 50 launches each, inputs resident in L2 after the first pass).
Prints one JSON document (with the device name and power limit) and writes it to --out when given.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def make(B, N):
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    torch.manual_seed(0)
    model = build_model(N, 2, default_model_config()).cuda().train()
    batch = make_batch(B, N, 2, 100, step=0, pad_bins=10)
    md = make_mod_dict(batch, ["ap", "behavior"], "token_masking", device="cuda")
    return model, md


def step(model, md):
    model.zero_grad(set_to_none=True)
    model({m: dict(d) for m, d in md.items()}).loss.backward()


def time_steps(model, md, det, k):
    torch.use_deterministic_algorithms(det)
    try:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(k):
            step(model, md)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k
    finally:
        torch.use_deterministic_algorithms(False)


def bench_step(B, N, steps, rounds):
    model, md = make(B, N)
    for det in (False, True):
        for _ in range(3):          # eager, capture, replay
            time_steps(model, md, det, 1)
    t = {False: [], True: []}
    for _ in range(rounds):
        for det in (False, True):
            t[det].append(time_steps(model, md, det, steps))
    off, on = sorted(t[False])[len(t[False]) // 2], sorted(t[True])[len(t[True]) // 2]
    return {"B": B, "N": N, "ms_per_step_default": off, "ms_per_step_deterministic": on,
            "overhead_pct": 100.0 * (on - off) / off, "samples_default": t[False], "samples_deterministic": t[True]}


def time_call(fn, det, n=50):
    torch.use_deterministic_algorithms(det)
    try:
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return 1000.0 * e0.elapsed_time(e1) / n
    finally:
        torch.use_deterministic_algorithms(False)


def bench_kernels():
    from multi_modal_foundation_model_b200 import ops
    R, H = 51200, 256
    out = []
    for NO, KI, what in ((768, 256, "qkv"), (256, 256, "out_proj"), (512, 256, "mlp_up"), (256, 512, "mlp_down")):
        dY = torch.randn(R, NO, device="cuda").to(torch.bfloat16)
        X = torch.randn(R, KI, device="cuda").to(torch.bfloat16)
        dW, db = torch.zeros(NO, KI, device="cuda"), torch.zeros(NO, device="cuda")
        ws = ops.DetWorkspace()
        f = lambda: ops.gemm_wgrad(dY, X, dW, dbias=db, ws=ws)   # noqa: E731
        out.append({"kernel": f"wgrad {what} {R}x{NO}x{KI}", "us_default": time_call(f, False),
                    "us_deterministic": time_call(f, True)})
    dy = torch.randn(R, H, device="cuda").to(torch.bfloat16)
    x = torch.randn(R, H, device="cuda")
    mean, rstd = x.mean(1), (x.var(1, unbiased=False) + 1e-5).rsqrt()
    g, dres, dx = torch.randn(H, device="cuda"), torch.randn(R, H, device="cuda"), torch.empty(R, H, device="cuda")
    dxb = torch.empty(R, H, device="cuda", dtype=torch.bfloat16)
    dg, dbt = torch.zeros(H, device="cuda"), torch.zeros(H, device="cuda")
    ws = ops.DetWorkspace()
    f = lambda: ops.layernorm_bwd(dy, x, mean, rstd, g, dres, dx, dxb, ops.NO_DROP, dg, dbt, R=R, H=H, ws=ws)  # noqa
    out.append({"kernel": f"layernorm_bwd {R}x{H}", "us_default": time_call(f, False), "us_deterministic": time_call(f, True)})
    dys = [torch.randn(R, H, device="cuda").to(torch.bfloat16) for _ in range(5)]
    gs = [torch.randn(H, device="cuda") for _ in range(5)]
    dgs = [torch.zeros(H, device="cuda") for _ in range(10)]
    ws2 = ops.DetWorkspace()
    f = lambda: ops.layernorm_bwd_multi(dys, x, mean, rstd, gs, dx, dxb, dgs[:5], dgs[5:], R=R, H=H, ws=ws2)  # noqa
    out.append({"kernel": f"layernorm_bwd_multi n=5 {R}x{H}", "us_default": time_call(f, False),
                "us_deterministic": time_call(f, True)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "det_bench needs a GPU"
    import __graft_entry__
    __graft_entry__.build()
    res = {"device": device_line(), "steps": [bench_step(256, 668, a.steps, a.rounds), bench_step(16, 668, a.steps, a.rounds)],
           "kernels": bench_kernels()}
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
