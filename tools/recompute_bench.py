"""Training steps on the recompute plan (Plan.recompute: per-layer activation recomputation) against the plan that saves
every activation.

Workloads: the default model (N 668) at B 256 and the scaled configs[4] model at B 16, each with both plans held at
once and timed in alternating rounds; the scaled model at B 96 (the largest batch whose full plan fits), where the two
plans cannot be held together, timed one after the other.  Per workload and plan: ms per train() step (forward +
backward, CUDA events, median of rounds, graph-replayed), with and without AdamW.step(), the peak-memory increase of
the first step and the plan's buffer bytes.  Then the recompute plan alone, as the engine picks it without any limit,
at scaled B 128, 192, 256 and beyond until a batch does not fit: trials/s and peak memory.  The engine must pick the
full plan for the default B 256 and scaled B 16 workloads (bench.py's), and the tool asserts it.  Writes one JSON file
(default profiles/r03_recompute.json) with the GPU name, power limit and max SM clock read in the same run.

    python tools/recompute_bench.py [--rounds 5] [--iters 6] [--out profiles/r03_recompute.json]
"""
import argparse
import json
import os
import statistics
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from multi_modal_foundation_model_b200.config import default_model_config, scaled_model_config  # noqa: E402
from multi_modal_foundation_model_b200.engine import Plan  # noqa: E402
from multi_modal_foundation_model_b200.model import build_model  # noqa: E402
from multi_modal_foundation_model_b200.optim import AdamW  # noqa: E402
from tools.inference_bench import device_facts, free_plans, mod_dict  # noqa: E402

SCALED_MODS = ("ap", "beh0", "beh1", "beh2", "beh3")


def step(model, md, opt):
    model.zero_grad(set_to_none=True)
    model({m: dict(d) for m, d in md.items()}).loss.backward()
    if opt is not None:
        opt.step()


def timed(model, md, opt, iters):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(iters):
        step(model, md, opt)
    ev[1].record()
    ev[1].synchronize()
    return ev[0].elapsed_time(ev[1]) / iters


def first_step(model, md, opt, make=None):
    """Run the first step (plan creation when `make` is None, else on the plan `make` builds); returns (plan, peak
    memory increase)."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    eng = model.engine()
    if make is not None:
        pl = make()
        eng.plans[key(md)] = pl
    step(model, md, opt)
    torch.cuda.synchronize()
    return eng.last_plan, torch.cuda.max_memory_allocated() - base


def key(md):
    B = next(iter(md.values()))["inputs"].shape[0]
    return (B, True, None, (), False, ())


def use(model, md, pl):
    model.engine().plans[key(md)] = pl


def rounds_of(model, md, opt, plans, rounds, iters):
    """{name: [ms per step, one per round]} with the plans alternated (each round reverses the order)."""
    t = {n: [] for n in plans}
    names = list(plans)
    for r in range(rounds):
        for n in (names if r % 2 == 0 else names[::-1]):
            use(model, md, plans[n])
            t[n].append(timed(model, md, opt, iters))
    return t


def summary(t, peak, pl):
    return dict(ms=statistics.median(t), ms_rounds=t, peak_bytes=peak, plan_buffer_bytes=pl["nbytes"],
                recompute=pl["recompute"])


def facts(pl):
    return dict(nbytes=pl.nbytes, recompute=pl.recompute)


def compare(model, mods, B, N, T, n_beh, rounds, iters, together=True):
    md = mod_dict(model, mods, B, N, T, n_beh)
    opt = AdamW(model.parameters(), lr=1e-5)
    eng = model.engine()
    full, peak_full = first_step(model, md, opt)
    assert not full.recompute, f"B {B}: the engine picked the recompute plan without a memory limit"
    out = dict(B=B, N=N, T=T, modalities=len(mods), rounds=rounds, iters_per_round=iters, alternated=together)
    if together:
        rec, peak_rec = first_step(model, md, opt, lambda: Plan(eng, B, True, recompute=True))
        plans = dict(full=full, recompute=rec)
        for p in plans.values():                       # graph capture of every plan
            use(model, md, p)
            step(model, md, opt)
        for label, o in (("step", None), ("step_adamw", opt)):
            t = rounds_of(model, md, o, plans, rounds, iters)
            out[label] = dict(full=summary(t["full"], peak_full, facts(full)),
                              recompute=summary(t["recompute"], peak_rec, facts(rec)))
    else:
        step(model, md, opt)
        tf = {label: [timed(model, md, o, iters) for _ in range(rounds)] for label, o in (("step", None),
                                                                                        ("step_adamw", opt))}
        full = facts(full)          # the two plans do not fit together: the full one goes first
        free_plans(model)
        rec, peak_rec = first_step(model, md, opt, lambda: Plan(eng, B, True, recompute=True))
        step(model, md, opt)
        for label, o in (("step", None), ("step_adamw", opt)):
            tr = [timed(model, md, o, iters) for _ in range(rounds)]
            out[label] = dict(full=summary(tf[label], peak_full, full), recompute=summary(tr, peak_rec, facts(rec)))
    for label in ("step", "step_adamw"):
        out[label]["recompute_over_full"] = out[label]["recompute"]["ms"] / out[label]["full"]["ms"]
    print(json.dumps({k: v for k, v in out.items() if k not in ("step", "step_adamw")}),
          {label: (out[label]["full"]["ms"], out[label]["recompute"]["ms"]) for label in ("step", "step_adamw")},
          flush=True)
    del opt, full, rec
    free_plans(model)
    return out


def recompute_alone(model, B, rounds):
    md = mod_dict(model, SCALED_MODS, B, 1024, 200, 4)
    opt = AdamW(model.parameters(), lr=1e-5)
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            pl, peak = first_step(model, md, opt)
        assert pl.recompute
        step(model, md, opt)
        t = [timed(model, md, opt, 2) for _ in range(rounds)]
        ms = statistics.median(t)
        out = dict(B=B, ran=True, ms_step_adamw=ms, ms_rounds=t, trials_per_s=B * 1000.0 / ms, peak_bytes=peak,
                   plan_buffer_bytes=pl.nbytes)
        del pl
    except torch.OutOfMemoryError as e:
        out = dict(B=B, ran=False, error=str(e).splitlines()[0][:200])
    print(json.dumps(out), flush=True)
    del opt
    free_plans(model)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=6)
    ap.add_argument("--out", default=os.path.join("profiles", "r03_recompute.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "tools/recompute_bench.py measures on the GPU"
    res = dict(device=device_facts(), method="CUDA events around `iters` graph-replayed train() steps (forward + "
               "backward [+ AdamW.step()]), median over rounds; train() mode, explicit eval masks, dropout on",
               workloads=[])
    torch.manual_seed(0)
    model = build_model(668, 2, default_model_config()).cuda().train()
    res["workloads"].append(dict(model="default configs[1]", **compare(model, ("ap", "behavior"), 256, 668, 100, 2,
                                                                       a.rounds, a.iters)))
    del model
    torch.cuda.empty_cache()

    torch.manual_seed(0)
    model = build_model(1024, 4, scaled_model_config(), avail_mod=SCALED_MODS,
                        extra_channels={m: 1 for m in SCALED_MODS[1:]}).cuda().train()
    res["workloads"].append(dict(model="scaled configs[4]", **compare(model, SCALED_MODS, 16, 1024, 200, 4, a.rounds,
                                                                      a.iters)))
    eng = model.engine()
    with warnings.catch_warnings():       # the largest batch whose full plan fits (AdamW moments included)
        warnings.simplefilter("ignore")
        b_full = next(B for B in (96, 88, 80, 72, 64) if not eng._choose_recompute(B, True, None, (), ()))
    res["workloads"].append(dict(model="scaled configs[4]", **compare(model, SCALED_MODS, b_full, 1024, 200, 4, 3, 2,
                                                                      together=False)))
    res["scaled_recompute_alone"] = []
    for B in (128, 192, 256, 320, 384):
        r = recompute_alone(model, B, 3)
        res["scaled_recompute_alone"].append(r)
        if not r["ran"]:
            break
    ran = [r["B"] for r in res["scaled_recompute_alone"] if r["ran"]]
    res["scaled_largest_batch_ran"] = max(ran) if ran else None
    res["device_after"] = device_facts()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
