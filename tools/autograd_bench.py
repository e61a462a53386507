"""Cost of backward passes through outputs other than `loss`.

    python tools/autograd_bench.py [--out FILE] [--steps K] [--rounds N]

Times the graph-replayed training step (train(), all dropout sites on, token masking) with four backward variants,
alternating within one process after every plan is built and warmed (eager, capture, replay):
  plain     out.loss.backward()  -- the default schedule
  weighted  (0.3 * mod_loss['ap'] + 2.0 * mod_loss['behavior']).backward()
  preds     (out.loss + 1e-3 * mod_preds['behavior'].square().mean()).backward()
  inputs    out.loss.backward() with `ap` and `behavior` inputs requiring grad (input-gradient plan)
at the benchmarked workload (B = 256, N = 668) and at B = 16.  Prints one JSON document (with the device name and power
limit read in the same process) and writes it to --out when given.
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

VARIANTS = ("plain", "weighted", "preds", "inputs")


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
    leaves = {m: md[m]["inputs"].detach().clone().requires_grad_(True) for m in ("ap", "behavior")}
    return model, md, leaves


def step(model, md, leaves, variant):
    model.zero_grad(set_to_none=True)
    d = {m: dict(x) for m, x in md.items()}
    if variant == "inputs":
        for m, x in leaves.items():
            x.grad = None
            d[m]["inputs"] = x
    out = model(d)
    if variant == "weighted":
        (0.3 * out.mod_loss["ap"] + 2.0 * out.mod_loss["behavior"]).backward()
    elif variant == "preds":
        (out.loss + 1e-3 * out.mod_preds["behavior"].square().mean()).backward()
    else:
        out.loss.backward()


def time_steps(model, md, leaves, variant, k):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(k):
        step(model, md, leaves, variant)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k


def bench(B, N, steps, rounds):
    model, md, leaves = make(B, N)
    for v in VARIANTS:
        for _ in range(3):
            time_steps(model, md, leaves, v, 1)
    t = {v: [] for v in VARIANTS}
    for _ in range(rounds):
        for v in VARIANTS:
            t[v].append(time_steps(model, md, leaves, v, steps))
    med = {v: sorted(s)[len(s) // 2] for v, s in t.items()}
    return {"B": B, "N": N, "ms_per_step_median": med,
            "overhead_pct_vs_plain": {v: 100.0 * (med[v] - med["plain"]) / med["plain"] for v in VARIANTS},
            "samples_ms": t}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "autograd_bench needs a GPU"
    import __graft_entry__
    __graft_entry__.build()
    res = {"device": device_line(), "steps": a.steps, "rounds": a.rounds,
           "results": [bench(256, 668, a.steps, a.rounds), bench(16, 668, a.steps, a.rounds)]}
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
