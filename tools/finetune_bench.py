"""Cost of the fine-tuning set-ups: parameter groups in the fused AdamW, and a frozen core.

    python tools/finetune_bench.py [--out FILE] [--steps K] [--rounds N] [--host-calls M] [--bench LABEL=FILE ...]

Times the graph-replayed training step (train(), token masking; forward + loss.backward() + opt.step()) of the default
model at the benchmarked workload (B = 256, N = 668) and at B = 16, with three variants alternating in one process
after every plan and optimizer is built and warmed:
  full         AdamW(model.parameters())                                   -- one group, every parameter
  two_groups   AdamW([{decay: weights}, {no decay: biases and norms}])     -- 1-D parameters without weight decay
  core_frozen  the shared transformer frozen (requires_grad=False), AdamW over the embedders and heads
For each: ms per step (median of --rounds windows of --steps steps), backward kernel launches, the optimizer's device
time (CUDA events around opt.step() while the GPU is held busy, so no host time is in it) and the host time of
opt.step() (median over --host-calls calls).  --bench LABEL=FILE adds `ms_per_step` and `with_optimizer.ms_per_step`
of a bench.py JSON line (e.g. `python bench.py --batch 16` of two builds run in the same session).  Prints one JSON
document (with the device name and power limit read in the same process) and writes it to --out when given.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

VARIANTS = ("full", "two_groups", "core_frozen")


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def is_core(name):
    return "embeddings." not in name


class Setup:
    def __init__(self, B, N):
        from multi_modal_foundation_model_b200.config import default_model_config
        from multi_modal_foundation_model_b200.model import build_model
        from multi_modal_foundation_model_b200.optim import AdamW
        from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
        torch.manual_seed(0)
        self.model = m = build_model(N, 2, default_model_config()).cuda().train()
        self.md = make_mod_dict(make_batch(B, N, 2, 100, step=0, pad_bins=10), ["ap", "behavior"], "token_masking",
                                device="cuda")
        m({k: dict(v) for k, v in self.md.items()})       # engine + flat buffers exist before the optimizers bind
        named = list(m.named_parameters())
        self.opt = {
            "full": AdamW(m.parameters(), lr=1e-5, weight_decay=0.01),
            "two_groups": AdamW([{"params": [p for _, p in named if p.ndim >= 2], "weight_decay": 0.01},
                                 {"params": [p for _, p in named if p.ndim < 2], "weight_decay": 0.0}], lr=1e-5),
            "core_frozen": AdamW([p for n, p in named if not is_core(n)], lr=1e-5, weight_decay=0.01),
        }

    def select(self, v):
        for n, p in self.model.named_parameters():
            p.requires_grad_(not (v == "core_frozen" and is_core(n)))

    def fwd_bwd(self, v):
        self.opt[v].zero_grad(set_to_none=True)
        self.model({k: dict(x) for k, x in self.md.items()}).loss.backward()

    def step(self, v):
        self.fwd_bwd(v)
        self.opt[v].step()


def time_steps(s, v, k):
    s.select(v)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(k):
        s.step(v)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k


def opt_times(s, v, n):
    """(device ms, host ms) medians of opt.step() after a fresh backward."""
    s.select(v)
    dev, host = [], []
    for _ in range(n):
        s.fwd_bwd(v)
        torch.cuda._sleep(20_000_000)          # keep the GPU busy: the events below bracket device work only
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        s.opt[v].step()
        t1 = time.perf_counter()
        e1.record()
        torch.cuda.synchronize()
        dev.append(e0.elapsed_time(e1))
        host.append((t1 - t0) * 1e3)
    return sorted(dev)[n // 2], sorted(host)[n // 2]


def bench(B, N, steps, rounds, host_calls):
    from multi_modal_foundation_model_b200 import ops
    s = Setup(B, N)
    launches = {}
    for v in VARIANTS:
        for _ in range(3):                      # eager, capture, replay of this variant's backward list
            time_steps(s, v, 1)
        _, calls, _ = s.model.engine().last_plan.backward_schedule()
        launches[v] = ops.count_kernels(calls)
    t = {v: [] for v in VARIANTS}
    for _ in range(rounds):
        for v in VARIANTS:
            t[v].append(time_steps(s, v, steps))
    med = {v: sorted(x)[len(x) // 2] for v, x in t.items()}
    out = {"B": B, "N": N, "variants": {}}
    for v in VARIANTS:
        dev, host = opt_times(s, v, host_calls)
        out["variants"][v] = {"ms_per_step_median": med[v], "backward_launches": launches[v],
                              "opt_step_device_ms": dev, "opt_step_host_ms": host, "samples_ms": t[v]}
    return out


def bench_line(path):
    with open(path) as f:
        line = [ln for ln in f if ln.strip().startswith("{")][-1]
    r = json.loads(line)
    return {"ms_per_step": r["ms_per_step"], "with_optimizer_ms_per_step": r["with_optimizer"]["ms_per_step"],
            "batch_per_gpu": r["config"].get("batch_per_gpu") if isinstance(r.get("config"), dict) else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--host-calls", type=int, default=60)
    ap.add_argument("--bench", action="append", default=[], help="LABEL=FILE: a bench.py JSON line to report")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "finetune_bench needs a GPU"
    import __graft_entry__
    __graft_entry__.build()
    res = {"device": device_line(), "steps": a.steps, "rounds": a.rounds, "host_calls": a.host_calls,
           "results": [bench(256, 668, a.steps, a.rounds, a.host_calls), bench(16, 668, a.steps, a.rounds, a.host_calls)]}
    if a.bench:
        res["bench_py"] = {lab: bench_line(path) for lab, path in (b.split("=", 1) for b in a.bench)}
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
