"""No-grad forward on the forward-only plan against the same forward on the training plan (grad enabled, no backward:
the same kernels plus the gelu'(u) store), alternated in one process.

Workloads: the default model (N 668) at B 256 and 16, and the scaled configs[4] model at B 16 and at the largest batch
whose training plan fits.  Per workload and path: ms per forward (CUDA events, median of rounds, graph-replayed),
the peak-memory increase of the first forward (torch.cuda.max_memory_allocated after a reset) and the plan's buffer
bytes.  Also runs one no-grad forward of the scaled model at a batch the training plan cannot hold.  Writes one JSON
file (default profiles/r03_inference.json) with the GPU name, power limit and max SM clock read in the same run.

    python tools/inference_bench.py [--rounds 7] [--iters 10] [--out profiles/r03_inference.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from multi_modal_foundation_model_b200.config import default_model_config, scaled_model_config  # noqa: E402
from multi_modal_foundation_model_b200.model import build_model  # noqa: E402
from multi_modal_foundation_model_b200.synthetic import make_batch  # noqa: E402


def device_facts():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def mod_dict(model, mods, B, N, T, n_beh):
    batch = make_batch(B, N, n_beh, T, step=3, pad_bins=T // 10)
    xs = {"ap": batch["spikes_data"]}
    beh = [m for m in mods if m != "ap"]
    for k, m in enumerate(beh):
        xs[m] = batch["target"] if len(beh) == 1 else batch["target"][:, :, k:k + 1].contiguous()
    g = torch.Generator().manual_seed(7)
    md = {}
    for m in mods:
        x = xs[m].cuda()
        md[m] = dict(inputs=x, targets=x, inputs_attn_mask=batch["time_attn_mask"].cuda(),
                     inputs_timestamp=batch["spikes_timestamps"].cuda(),
                     inputs_modality=torch.tensor(model.mod_to_indx[m], device="cuda"), masking_mode=None,
                     eval_mask=(torch.rand(B, T, generator=g) < 0.3).long().cuda()[:, :, None].contiguous(),
                     inputs_regions=np.array([["CA1"] * x.shape[2]] * B))
    return md


def forward(model, md, grad):
    with torch.set_grad_enabled(grad):
        return model({m: dict(d) for m, d in md.items()})


def first_forward(model, md, grad):
    """Build the plan and run its eager forward; returns (peak-memory increase, plan buffer bytes).  The engine (flat
    parameters, gradients, bf16 weight shadows) exists before the baseline is read: the figure is the plan's."""
    model.engine()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    forward(model, md, grad)
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base, model.engine().last_plan.arena_bytes


def free_plans(model):
    eng = model.engine()
    for d in (eng.plans, eng.arenas, eng.fwd_plans, eng.fwd_arenas):
        d.clear()
    eng.last_plan = None
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def compare(model, mods, B, N, T, n_beh, rounds, iters):
    md = mod_dict(model, mods, B, N, T, n_beh)
    peak_new, bytes_new = first_forward(model, md, False)
    peak_old, bytes_old = first_forward(model, md, True)
    for grad in (False, True):          # graph capture of both plans
        forward(model, md, grad)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t = {False: [], True: []}
    for r in range(rounds):
        for grad in ((False, True) if r % 2 == 0 else (True, False)):
            ev[0].record()
            for _ in range(iters):
                forward(model, md, grad)
            ev[1].record()
            ev[1].synchronize()
            t[grad].append(ev[0].elapsed_time(ev[1]) / iters)
    out = dict(B=B, N=N, T=T, modalities=len(mods), rounds=rounds, iters_per_round=iters,
               forward_only=dict(ms=statistics.median(t[False]), ms_rounds=t[False], peak_bytes=peak_new,
                                 plan_buffer_bytes=bytes_new),
               training_plan=dict(ms=statistics.median(t[True]), ms_rounds=t[True], peak_bytes=peak_old,
                                  plan_buffer_bytes=bytes_old))
    out["speedup"] = out["training_plan"]["ms"] / out["forward_only"]["ms"]
    print(json.dumps({k: v for k, v in out.items() if k not in ("forward_only", "training_plan")}),
          {k: (out[k]["ms"], out[k]["peak_bytes"]) for k in ("forward_only", "training_plan")}, flush=True)
    free_plans(model)
    return out


def training_plan_fits(model, mods, B, N, T, n_beh):
    md = mod_dict(model, mods, B, N, T, n_beh)
    try:
        forward(model, md, True)
        torch.cuda.synchronize()
        ok = True
    except torch.OutOfMemoryError:
        ok = False
    free_plans(model)
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=os.path.join("profiles", "r03_inference.json"))
    ap.add_argument("--scaled-beyond", type=int, default=128,
                    help="batch of the scaled no-grad forward that the training plan cannot hold")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "tools/inference_bench.py measures on the GPU"
    res = dict(device=device_facts(), method="alternating rounds in one process, CUDA events around `iters` "
               "graph-replayed forwards, median over rounds; eval() mode, explicit eval masks", workloads=[])

    torch.manual_seed(0)
    model = build_model(668, 2, default_model_config()).cuda().eval()
    for B in (256, 16):
        res["workloads"].append(dict(model="default configs[1]", **compare(model, ("ap", "behavior"), B, 668, 100, 2,
                                                                           a.rounds, a.iters)))
    del model
    torch.cuda.empty_cache()

    mods = ("ap", "beh0", "beh1", "beh2", "beh3")
    torch.manual_seed(0)
    model = build_model(1024, 4, scaled_model_config(), avail_mod=mods, extra_channels={m: 1 for m in mods[1:]})
    model = model.cuda().eval()
    res["workloads"].append(dict(model="scaled configs[4]", **compare(model, mods, 16, 1024, 200, 4, a.rounds, a.iters)))
    b_train = None
    for B in (112, 104, 96, 88, 80, 72, 64, 56, 48, 32):
        if training_plan_fits(model, mods, B, 1024, 200, 4):
            b_train = B
            break
    res["scaled_largest_training_plan_batch"] = dict(B=b_train, batches_tried=[112, 104, 96, 88, 80, 72, 64, 56, 48, 32])
    if b_train is not None:
        res["workloads"].append(dict(model="scaled configs[4]", **compare(model, mods, b_train, 1024, 200, 4,
                                                                          a.rounds, max(2, a.iters * 16 // b_train))))
    B = a.scaled_beyond
    md = mod_dict(model, mods, B, 1024, 200, 4)
    peak, nbytes = first_forward(model, md, False)
    forward(model, md, False)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    forward(model, md, False)
    ev[1].record()
    ev[1].synchronize()
    res["scaled_no_grad_beyond_training_plan"] = dict(B=B, ms=ev[0].elapsed_time(ev[1]), peak_bytes=peak,
                                                      plan_buffer_bytes=nbytes,
                                                      training_plan_fits=training_plan_fits(model, mods, B, 1024, 200, 4))
    print(json.dumps(res["scaled_no_grad_beyond_training_plan"]), flush=True)
    res["device_after"] = device_facts()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
