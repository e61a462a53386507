"""Data-parallel multi-session pre-training: the session exchange against the dense all-reduce it replaces.

    python tools/multisession_ddp_bench.py [--worlds 1,2,8] [--steps K] [--rounds N] [--out FILE]

Workload: BASELINE configs[3] -- 32 sessions of 256..1024 neurons (seeded exactly as `bench.py --workload
multisession`), the default transformer, B = 256 trials per GPU, train(), graph-replayed forward + loss.backward()
(no optimizer step).  Each world size runs under torch.distributed.run.  At timed step i, rank r runs session
(i * world + r) % 32, so the sessions of one step are distinct.  Every session's plan is warmed (eager, capture,
replay) on every rank before timing, for every variant.  Variants, alternated round by round in one process:
  exchange       parallel.DataParallel: core-only all-reduce buckets + the session exchange
  dense          the previous behaviour, kept here as the baseline: all-reduce buckets over the whole flat gradient
                 (every session's heads and embedders, zeros included), no exchange
  same_*         both of the above with every rank on the same session (i % 32) at step i
  local          the same sessions per rank without any communication (each rank's single-GPU step)
Per variant: ms per step (median over rounds of the max over ranks of a window of --steps steps), trials/s, weak-scaling
efficiency against world x the 1-GPU rate, bytes each rank sends and receives per step (payload, and what NCCL's ring
algorithms move), and the exposed communication time, step - local step.  The device name and power limit are read
in the same run.
"""
import argparse
import json
import os
import random
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_SESSIONS, B, T = 32, 256, 100


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()}


def session_neurons():
    rng = random.Random(2024)                      # bench.py Workload, --sessions 32
    return [rng.randint(256, 1024) for _ in range(N_SESSIONS)]


def build(neurons):
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
    torch.manual_seed(42)
    chans = {f"session-{k:02d}": {"ap": n, "behavior": 2} for k, n in enumerate(neurons)}
    return MultiSessionMultiModal(chans, ["ap", "behavior"], default_model_config()).cuda().train()


def batches(neurons, rank):
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    out = []
    for k, n in enumerate(neurons):
        b = make_batch(B, n, 2, T, step=1000 * rank + k)
        b["eid"] = [f"session-{k:02d}"] * B
        out.append(make_mod_dict(b, ["ap", "behavior"], ("encoding", "decoding", "token_masking")[k % 3], device="cuda"))
    return out


def bytes_per_step(store, xchg, world):
    """(payload sent, payload received, ring sent, ring received) bytes per rank per step."""
    if world == 1:
        return {"payload_sent": 0, "payload_recv": 0, "ring_sent": 0, "ring_recv": 0}
    if xchg is None:
        ar = 4 * store.total
        ring = 2 * (world - 1) / world * ar
        return {"payload_sent": ar, "payload_recv": ar, "ring_sent": ring, "ring_recv": ring}
    lo, hi = store.core_range
    ar = 4 * (hi - lo)
    sent, recv = xchg.bytes_per_step()
    chunk = sent                                       # each rank's all-gather contribution
    ring_ag = (world - 1) * chunk
    return {"payload_sent": ar + sent, "payload_recv": ar + recv,
            "ring_sent": 2 * (world - 1) / world * ar + ring_ag, "ring_recv": 2 * (world - 1) / world * ar + ring_ag,
            "all_reduce_bytes": ar, "all_gather_bytes_per_rank": chunk}


def worker(a):
    import torch.distributed as dist
    from multi_modal_foundation_model_b200.parallel import DataParallel
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    neurons = session_neurons()
    data = batches(neurons, rank)
    models = {}
    models["exchange"] = build(neurons)
    if world > 1:
        models["dense"] = build(neurons)
        ddp = {"exchange": DataParallel(models["exchange"]), "dense": DataParallel(models["dense"])}
        ddp["dense"].xchg = None                   # the previous behaviour: buckets over the whole flat gradient
        assert ddp["exchange"].xchg is not None

    def step(m, s):
        m.zero_grad(set_to_none=True)
        m({k: dict(v) for k, v in data[s].items()}).loss.backward()

    def run(variant, sessions):
        """Steps over `sessions` (this rank's session per step); the window's ms per step, max over ranks."""
        base = variant.replace("same_", "")
        m = models["exchange" if base == "local" else base]
        eng = m.engine()
        saved = eng.ddp
        if base == "local":
            eng.ddp = None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for s in sessions:
            step(m, s)
        e1.record()
        torch.cuda.synchronize()
        eng.ddp = saved
        ms = torch.tensor([e0.elapsed_time(e1) / len(sessions)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    variants = ["local"] if world == 1 else ["exchange", "dense", "same_exchange", "same_dense", "local"]
    # warm-up: every session's plan three times on every rank (eager, capture, replay), distinct sessions per step
    warm = [(i + rank) % N_SESSIONS for i in range(3 * N_SESSIONS)]
    for v in variants:
        if not v.startswith("same_"):
            run(v, warm)
    distinct = [(i * world + rank) % N_SESSIONS for i in range(a.steps)]
    same = [i % N_SESSIONS for i in range(a.steps)]
    t = {v: [] for v in variants}
    for _ in range(a.rounds):
        for v in variants:
            t[v].append(run(v, same if v.startswith("same_") else distinct))
    if rank == 0:
        res = {"world": world, "variants": {}}
        for v in variants:
            base = v.replace("same_", "")
            ms = sorted(t[v])[len(t[v]) // 2]
            x = ddp[base].xchg if world > 1 and base != "local" else None
            store = models["exchange"].engine().store
            res["variants"][v] = {"ms_per_step": ms, "trials_per_s": B * world / (ms / 1e3), "samples_ms": t[v],
                                  "bytes_per_rank": bytes_per_step(store, x, 1 if base == "local" else world)}
        for v in variants:
            if v != "local":
                res["variants"][v]["exposed_comm_ms"] = (res["variants"][v]["ms_per_step"]
                                                         - res["variants"]["local"]["ms_per_step"])
        st = models["exchange"].engine().store
        res["flat_gradient_elems"] = st.total
        res["core_elems"] = st.core_range[1] - st.core_range[0]
        res["session_slab_elems"] = [h1 - h0 + e1 - e0 for h0, h1, e0, e1 in st.session_ranges]
        res["device"] = device_line()
        with open(a.part, "w") as f:
            json.dump(res, f)
    if world > 1:
        for d in ddp.values():
            d.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", default="1,2,8")
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--part", default=None, help=argparse.SUPPRESS)     # worker mode: rank 0 writes its result here
    a = ap.parse_args()
    assert torch.cuda.is_available(), "multisession_ddp_bench needs a GPU"
    if a.part is not None:
        worker(a)
        return
    import __graft_entry__
    __graft_entry__.build()
    res = {"workload": f"configs[3]: {N_SESSIONS} sessions (neurons {min(session_neurons())}..{max(session_neurons())}, "
                       f"seeded as bench.py), B = {B} per GPU, T = {T}, train(), graph-replayed fwd + loss.backward()",
           "steps": a.steps, "rounds": a.rounds, "gpus_available": torch.cuda.device_count(), "runs": []}
    with tempfile.TemporaryDirectory() as tmp:
        for w in (int(x) for x in a.worlds.split(",")):
            if w > torch.cuda.device_count():
                res["runs"].append({"world": w, "not_measured": f"only {torch.cuda.device_count()} GPUs"})
                continue
            part = os.path.join(tmp, f"w{w}.json")
            cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc_per_node={w}",
                   os.path.abspath(__file__), "--part", part, "--steps", str(a.steps), "--rounds", str(a.rounds)]
            r = subprocess.run(cmd, cwd=ROOT)
            if r.returncode != 0 or not os.path.exists(part):
                res["runs"].append({"world": w, "not_measured": f"run failed (exit {r.returncode})"})
                continue
            with open(part) as f:
                res["runs"].append(json.load(f))
    one = next((r for r in res["runs"] if r["world"] == 1 and "variants" in r), None)
    if one is not None:
        rate1 = one["variants"]["local"]["trials_per_s"]
        for r in res["runs"]:
            for v in r.get("variants", {}).values():
                v["weak_scaling_efficiency"] = v["trials_per_s"] / (r["world"] * rate1)
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
