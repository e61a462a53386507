#!/usr/bin/env python
"""bench.py -- train trials/sec (forward + backward) of the masked multi-modal encoder/decoder on B200.

    python bench.py --gpus N --steps K --warmup W            our arm (hand-written sm_100a kernels via the C ABI)
    python bench.py --impl reference ...                     the reference algorithm's CPU path (oracle port) on the
                                                             box's host cores, same workload / metric / unit
    python bench.py ... --dump-outputs DIR                   also write the last timed step's loss, predictions and
                                                             gradients as DIR/<name>.npy (compare two builds)

Workload (BASELINE.json configs[1]): mm.yaml default MultiModal (5+5 layers, H 256, 8 heads, MLP 512), modalities
ap (N=668 spike channels, the yaml's n_channels) + behavior (wheel speed, whisker motion energy), T=100 bins,
B=256 trials per GPU, model.train() (all six dropout sites + masking active), training mode cycling through
encoding / decoding / token_masking as ``--mixed_training`` does (trainer/base.py:189-190), synthetic IBL-shaped
data (multi_modal_foundation_model_b200/synthetic.py), random-init weights at seed 42.  One step = one
``model(mod_dict)`` + ``loss.backward()`` (optimizer excluded, as in the metric's definition).

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how every field is produced.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODES = ("encoding", "decoding", "token_masking")
METRIC = "train trials/sec fwd+bwd"
UNIT = "trials/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="default", choices=["default", "scaled", "multisession"],
                    help="default = BASELINE configs[1] (the metric's config); scaled = configs[4] (24+24 layers, "
                         "H 1024, 200 bins, spikes + 4 behaviour streams); multisession = configs[3] (32 sessions with "
                         "256-1024 neurons, per-session embedders) -- extra profile lines, not the headline")
    ap.add_argument("--sessions", type=int, default=32)
    ap.add_argument("--batch", type=int, default=None, help="trials per GPU per step (256 default / 16 scaled)")
    ap.add_argument("--neurons", type=int, default=None, help="spike channels (668 default / 1024 scaled)")
    ap.add_argument("--cpu-batch", type=int, default=16, help="trials per step of the CPU sample")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eval-mode", action="store_true", help="dropout off (parity configuration)")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: --batch is the GLOBAL batch, split evenly over the ranks (SURVEY 8d config 3)")
    ap.add_argument("--no-library-bar", action="store_true",
                    help="skip timing the unmodified reference on the GPU through stock PyTorch")
    ap.add_argument("--sustained-seconds", type=float, default=2.0,
                    help="length of the extra back-to-back leg that reports throughput under sustained clocks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (loss, per-modality losses, "
                         "example counts and predictions, parameter gradients) as DIR/<name>.npy in float32 / float64, "
                         "at most 60 MiB in all: an array over its share is replaced by a fixed, seeded sample of its "
                         "elements (1-D, in flat-index order)")
    a = ap.parse_args()
    scaled = a.workload == "scaled"
    if a.batch is None:
        a.batch = 16 if scaled else 256
    if a.neurons is None:
        a.neurons = 1024 if scaled else 668
    if scaled:
        a.cpu_batch = 1
    return a


class Workload:
    """Model / data shape of a bench run (SURVEY.md section 8d)."""

    def __init__(self, a):
        from multi_modal_foundation_model_b200.config import default_model_config, scaled_model_config
        self.scaled = a.workload == "scaled"
        self.multi = a.workload == "multisession"
        self.neurons = a.neurons
        self.session_neurons = None
        if self.multi:
            import random
            rng = random.Random(2024)
            self.session_neurons = [rng.randint(256, 1024) for _ in range(a.sessions)]
            self.cfg = default_model_config()
            self.mods = ["ap", "behavior"]
            self.extra = None
            self.n_beh, self.T = 2, 100
            self.neurons = max(self.session_neurons)
            self.chan = [sum(self.session_neurons) / len(self.session_neurons), 2]
            self.desc = (f"configs[3]: multi-session pre-training, {a.sessions} synthetic sessions with "
                         f"{min(self.session_neurons)}-{max(self.session_neurons)} neurons (seeded), per-session embedders "
                         "and heads selected by eid, shared mm.yaml default transformer, one session per batch")
        elif self.scaled:
            self.cfg = scaled_model_config()
            self.mods = ["ap", "beh0", "beh1", "beh2", "beh3"]
            self.extra = {m: 1 for m in self.mods[1:]}
            self.n_beh, self.T = 4, 200
            self.chan = [a.neurons, 1, 1, 1, 1]
            self.desc = ("configs[4]: scaled variant, 24+24 layers, d_model 1024, 16 heads (d_head 64), MLP 2048, 200 "
                         "time bins, ap spikes + 4 single-channel behaviour streams (S = 1000 tokens per trial)")
        else:
            self.cfg = default_model_config()
            self.mods = ["ap", "behavior"]
            self.extra = None
            self.n_beh, self.T = 2, 100
            self.chan = [a.neurons, 2]
            self.desc = ("configs[1]: multi-modal encoder/decoder (ap spikes + wheel speed + whisker motion energy), "
                         "mm.yaml default model 5+5 layers H256 8 heads MLP512, single synthetic IBL-shaped session")
        tr = self.cfg["encoder"]["transformer"]
        self.H, self.I, self.Le = tr["hidden_size"], tr["inter_size"], tr["n_layers"]
        self.Ld = self.cfg["decoder"]["transformer"]["n_layers"]
        self.S = self.T * len(self.mods)

    def session_of(self, step):
        return step % len(self.session_neurons)

    def build(self):
        from multi_modal_foundation_model_b200.model import MultiSessionMultiModal, build_model
        if self.multi:
            chans = {f"session-{k:02d}": {"ap": n, "behavior": 2} for k, n in enumerate(self.session_neurons)}
            return MultiSessionMultiModal(chans, self.mods, self.cfg)
        return build_model(self.neurons, self.n_beh, self.cfg, avail_mod=tuple(self.mods), extra_channels=self.extra)

    def batch(self, B, step, pin=False):
        from multi_modal_foundation_model_b200.synthetic import make_batch
        if self.multi:
            k = self.session_of(step)
            out = make_batch(B, self.session_neurons[k], self.n_beh, self.T, step=step, pin=pin)
            out["eid"] = [f"session-{k:02d}"] * B
            return out
        return make_batch(B, self.neurons, self.n_beh, self.T, step=step, pin=pin)

    def inputs_of(self, batch):
        out = []
        for k, m in enumerate(self.mods):
            if m == "ap":
                out.append((m, batch["spikes_data"]))
            elif m == "behavior":
                out.append((m, batch["target"]))
            else:
                out.append((m, batch["target"][:, :, k - 1:k].contiguous()))
        return out

    def flops_fwd_per_trial(self) -> float:
        """SURVEY.md section 8d 'Algorithmic work per trial' (dense attention, 2 FLOPs per multiply-add)."""
        T, S, H, I = self.T, self.S, self.H, self.I
        if self.multi:   # mean over the sessions
            f = sum(2 * (2 * T * C * 2 * C + 2 * T * 2 * C * H) + 2 * T * H * C for C in self.session_neurons) / len(self.session_neurons)
            f += 2 * (2 * T * 2 * 4 + 2 * T * 4 * H) + 2 * T * H * 2
        else:
            f = sum(2 * (2 * T * C * 2 * C + 2 * T * 2 * C * H) + 2 * T * H * C for C in self.chan)
        f += self.Le * (8 * S * H * H + 4 * S * S * H + 4 * S * H * I)
        f += self.Ld * (16 * S * H * H + 8 * S * S * H + 4 * S * H * I)
        return float(f + 2 * S * H * H)


def workload_config(a, n_gpus):
    w = Workload(a)
    return {
        "workload": w.desc,
        "neurons": a.neurons, "behaviors": w.n_beh, "time_bins": w.T, "tokens_per_trial": w.S,
        "batch_per_gpu": per_gpu_batch(a, n_gpus), "global_batch": per_gpu_batch(a, n_gpus) * n_gpus,
        "mode": "eval() (dropout off)" if a.eval_mode else "train() (dropout 0.2/0.4 + masker active)",
        "training_modes": "encoding/decoding/token_masking cycled",
        "parallelism": f"dp{n_gpus}",
        "l2_policy": "per-step working set (activations + saved tensors, several GB at B=256) >> 126 MB L2",
    }


def per_gpu_batch(a, n_gpus):
    if a.strong:
        assert a.batch % n_gpus == 0, "--strong needs a global batch divisible by the number of GPUs"
        return a.batch // n_gpus
    return a.batch


# ------------------------------------------------------------------------------------------------------------
def reference_available(a) -> bool:
    """The unmodified reference (baseline/_ref) covers the default workload; configs[3] / configs[4] (per-session
    embedders, 5 modalities) are extensions it cannot build, so those lines fall back to the oracle port."""
    from baseline import ref_loader
    return a.workload == "default" and ref_loader.available()


def cpu_reference(a, seconds: float, fixed_steps: int = 0, warmup: int = 1, threads=None, train=None):
    """cpu_baseline dict: the reference's own CPU implementation of the path on the host cores."""
    train = (not a.eval_mode) if train is None else train
    if reference_available(a):
        from baseline import ref_bench
        w = Workload(a)
        r = ref_bench.cpu_rate(a.neurons, w.n_beh, w.T, a.cpu_batch, steps=fixed_steps, warmup=warmup, seconds=seconds,
                               train=train, threads=threads)
        return {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "reference",
                "sample": f"{r['steps']} fwd+bwd steps (+{r['warmup']} warm-up) of {a.cpu_batch} trials each -- a bounded "
                          f"sample of the {a.batch}-trial workload step -- through the UNMODIFIED reference MultiModal "
                          f"(baseline/_ref, built as train_multi_modal.py:160-189), {r['mode']}, torch fp32, "
                          f"{r['threads']} threads of {r['cores']} cores, {r['s_per_step']:.2f} s/step",
                "s_per_step": r["s_per_step"], "steps": r["steps"], "warmup": r["warmup"]}
    rate, cores, n, per = cpu_reference_rate(a, seconds, fixed_steps=fixed_steps, warmup=warmup)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} fwd+bwd steps of {a.cpu_batch} trials (same model / N / T), oracle/mm_oracle.py (the reference "
                      f"classes cannot build this extension workload), torch fp32, {cores} threads, {per:.2f} s/step",
            "s_per_step": per, "steps": n, "warmup": warmup}


def cpu_reference_rate(a, seconds: float, min_steps: int = 2, fixed_steps: int = 0, warmup: int = 1):
    """The reference algorithm on the host CPU: oracle/mm_oracle.py (PyTorch fp32 restatement pinned to the
    reference by tests/golden) forward + backward, all host threads.  Returns (trials/s, cores, steps, s/step)."""
    import torch
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.synthetic import make_batch
    from oracle import mm_oracle as orc

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    wl = Workload(a)
    cfg = wl.cfg
    torch.manual_seed(42)
    model = wl.build()
    SD = {k: v.detach() for k, v in model.state_dict().items()}

    def params_for(step):
        if wl.multi:   # the batch's session: its embedders under the reference's single-session names
            pre = model.session_prefix(f"session-{wl.session_of(step):02d}")
            P = {(k[len(pre):] if k.startswith(pre) else k): v for k, v in SD.items()
                 if k.startswith(pre) or not k.startswith("session_embeddings.")}
        else:
            P = dict(SD)
        for k in list(P):
            if k.startswith("decoder_embeddings.") and k.endswith("mod_emb.weight"):
                P[k] = P[k.replace("decoder_embeddings.", "encoder_embeddings.")]
        return P

    spec = orc.OracleSpec.from_config(cfg, wl.mods)
    B = a.cpu_batch

    def one(step):
        P = params_for(step)
        batch = wl.batch(B, step)
        attn = batch["time_attn_mask"]
        mode = MODES[step % 3]
        g = torch.Generator().manual_seed(step)
        ob = {}
        for m, x in wl.inputs_of(batch):
            if mode == "token_masking":
                mk = torch.bernoulli(torch.full((B, wl.T), 0.3), generator=g).long()
            else:
                mk = torch.full((B, wl.T), 1 if (m == "ap") == (mode == "encoding") else 0, dtype=torch.int64)
            ob[m] = dict(inputs=x, targets=x, attn_mask=attn, timestamp=batch["spikes_timestamps"], mask=mk & attn)
        t0 = time.perf_counter()
        # dropout_seed set: train() mode like the GPU arm (masks from the documented Philox stream)
        orc.forward_backward(P, spec, ob, dropout_seed=None if a.eval_mode else 1000 + step)
        return time.perf_counter() - t0

    for s in range(warmup):
        one(s)
    times = []
    t_start = time.perf_counter()
    s = warmup
    while True:
        times.append(one(s))
        s += 1
        if fixed_steps and len(times) >= fixed_steps:
            break
        if not fixed_steps and len(times) >= min_steps and time.perf_counter() - t_start >= seconds:
            break
    per = sum(times) / len(times)
    return B / per, cores, len(times), per


def run_reference(a):
    """--impl reference: the reference's own CPU implementation, K timed steps after W warm-up steps exactly as asked,
    every step a bounded sample (--cpu-batch trials) of the workload step; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps, warmup = max(1, a.steps), max(0, a.warmup)
    cpu = cpu_reference(a, 0.0, fixed_steps=steps, warmup=warmup)
    extras = {}
    if reference_available(a):
        # BASELINE.md section 3 also asks for eval() mode and single-thread numbers (bounded: 3 / 2 steps)
        ev = cpu_reference(a, 0.0, fixed_steps=3, warmup=1, train=False)
        one = cpu_reference(a, 0.0, fixed_steps=2, warmup=1, threads=1)
        extras = {"eval_mode": {"value": ev["value"], "unit": UNIT, "sample": ev["sample"]},
                  "one_thread": {"value": one["value"], "unit": UNIT, "sample": one["sample"]}}
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": a.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": cpu["s_per_step"] * 1e3, "higher_is_better": True,
        "scaling": "strong" if a.strong else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(a, a.gpus),
        "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "extras": extras,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "25"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 60 << 20       # --dump-outputs: all arrays together
DUMP_SAMPLE_SEED = 20240601


def dump_outputs(path, out, model, store):
    """Write one step's results (``MultiModalOutput`` + the gradients in the engine's flat buffer) as .npy files, so two
    builds can be compared output for output.  Smallest arrays first, each keeps at most an equal share of the bytes
    still left; a larger array is replaced by that many elements at seeded positions (the same positions in every run
    with the same shapes)."""
    import numpy as np
    import torch
    arrays = {"loss": out.loss}
    for m in out.mod_loss:
        arrays[f"mod_loss.{m}"] = out.mod_loss[m]
        arrays[f"mod_n_examples.{m}"] = out.mod_n_examples[m]
        arrays[f"mod_preds.{m}"] = out.mod_preds[m]
    for n, _ in model.named_parameters():
        arrays[f"grad.{n}"] = store.g(n)
    host = {k: v.detach().to("cpu", torch.float32 if v.is_floating_point() else torch.float64) for k, v in arrays.items()}
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES - 256 * len(host)          # .npy headers
    items = sorted(host.items(), key=lambda kv: kv[1].numel())
    for i, (name, v) in enumerate(items):
        keep = min(v.numel(), left // (len(items) - i) // v.element_size())
        if keep < v.numel():
            g = torch.Generator().manual_seed(DUMP_SAMPLE_SEED)
            idx = torch.randperm(v.numel(), generator=g)[:keep].sort().values
            v = v.flatten()[idx]
        left -= keep * v.element_size()
        np.save(os.path.join(path, f"{name}.npy"), v.numpy())


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)

    import torch
    import torch.distributed as dist
    from multi_modal_foundation_model_b200 import ops
    from multi_modal_foundation_model_b200.config import default_model_config
    from multi_modal_foundation_model_b200.model import build_model
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world

    wl = Workload(a)
    torch.manual_seed(42)
    model = wl.build().to(dev)
    model.train(not a.eval_mode)
    # token-masking steps use the model's DEFAULT mask stream ('device': Bernoulli field sampled inside mmfm_mask_prep)
    eng = model.engine()
    ddp = None
    if world > 1:
        from multi_modal_foundation_model_b200.parallel import DataParallel
        ddp = DataParallel(model)
    B = per_gpu_batch(a, world)

    # rank r's shard of every global batch: its own seeded trials (weak scaling: B per GPU)
    NB = len(wl.session_neurons) if wl.multi else 3    # multi-session: one batch per session, visited round-robin
    first = (rank * (NB // max(world, 1))) if wl.multi else 1000 * rank
    host_batches = [wl.batch(B, first + i, pin=True) for i in range(NB)]
    dev_batches = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in hb.items()} for hb in host_batches]
    dev_dicts = [make_mod_dict(dev_batches[i], wl.mods, MODES[i % 3], device=dev) for i in range(NB)]

    last_out = [None]

    def step_resident(i):
        md = {k: dict(v) for k, v in dev_dicts[i % NB].items()}
        out = model(md)
        out.loss.backward()
        model.zero_grad(set_to_none=True)
        last_out[0] = out
        return out

    from multi_modal_foundation_model_b200.synthetic import DevicePrefetcher
    pf = DevicePrefetcher(dev)

    e2e_compact = [False]     # trainer-form dense int64 eval masks (False) or the compact scalar / (B,T) forms (True)
    host_loss = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_losses = []

    def step_e2e(i):
        # every step copies one batch host -> device (pinned memory, side stream: batch i+1 moves while step i computes)
        # and reads its loss back (asynchronous D2H into pinned memory, consumed one step later -- the way a trainer
        # logs without stalling the launch queue; the last one is consumed right after the timed loop's barrier)
        if pf._next is None:
            pf.put(host_batches[i % NB])
        db = pf.get()                                                                                  # H2D of batch i
        pf.put(host_batches[(i + 1) % NB])                                                             # H2D of batch i+1
        md = make_mod_dict(db, wl.mods, MODES[i % 3], device=dev, compact_masks=e2e_compact[0])
        out = model(md)
        out.loss.backward()
        model.zero_grad(set_to_none=True)
        slot = i & 1
        host_loss[slot].copy_(out.loss.detach().reshape(1), non_blocking=True)                         # D2H of step i
        loss_ev[slot].record()
        if i > 0:
            loss_ev[slot ^ 1].synchronize()
            e2e_losses.append(float(host_loss[slot ^ 1][0]))                                            # loss of step i-1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    for i in range(max(a.warmup, 3, 3 * NB if wl.multi else 0)):   # every session's plan built, run and graph-captured
        step_resident(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms = timed(step_resident, a.steps)
    clocks = sampler.stop() if rank == 0 else None
    value = B * n_gpus * a.steps / (ms / 1e3)
    if a.dump_outputs and rank == 0:
        # zero_grad(set_to_none) only drops the .grad views: the flat buffer still holds the last timed step's gradients
        dump_outputs(a.dump_outputs, last_out[0], model, eng.store)

    # the same loop held for >= --sustained-seconds back to back: throughput under the clocks a long job really sees
    sustained = None
    if a.sustained_seconds > 0:
        n_sus = max(a.steps, int(a.sustained_seconds / (ms / a.steps / 1e3)) + 1)
        sampler2 = ClockSampler(local)
        if rank == 0:
            sampler2.start()
        ms_sus = timed(step_resident, n_sus)
        clk2 = sampler2.stop() if rank == 0 else None
        sustained = {"value": B * n_gpus * n_sus / (ms_sus / 1e3), "unit": UNIT, "steps": n_sus,
                     "seconds": ms_sus / 1e3, "ms_per_step": ms_sus / n_sus, "clocks": clk2}

    # second number of SURVEY section 8d: the same step with the optimizer (fused AdamW over the flat buffers) included
    from multi_modal_foundation_model_b200.optim import AdamW
    opt = AdamW(model.parameters(), lr=1e-4, weight_decay=0.01, eps=1e-8)

    def step_optim(i):
        md = {k: dict(v) for k, v in dev_dicts[i % NB].items()}
        out = model(md)
        out.loss.backward()
        opt.step()
        model.zero_grad(set_to_none=True)
        return out

    for i in range(3):
        step_optim(i)
    ms_opt = timed(step_optim, a.steps)
    value_opt = B * n_gpus * a.steps / (ms_opt / 1e3)

    for i in range(3):
        step_e2e(i)
    ms_e2e = timed(step_e2e, a.steps)
    pl = eng.last_plan            # the fp32-batch plan: the per-kernel table and the launch count below describe it
    ms_e2e_u8 = None
    if not wl.scaled:
        # the same leg with the spike counts shipped as bytes (uint8 wire format, expanded by mmfm_u8_expand on the device)
        fp32_batches = host_batches
        host_batches = [dict(hb, spikes_data=hb["spikes_data"].to(torch.uint8).pin_memory()) for hb in fp32_batches]
        pf._next = None
        e2e_compact[0] = True          # the wire format of this path: byte counts + compact masks (SURVEY 8f rank 2 / 3)
        for i in range(6 if not wl.multi else 3 * NB):   # (multi-session: every session's byte-input plan built, run, captured)
            step_e2e(i)
        ms_e2e_u8 = timed(step_e2e, a.steps)
        e2e_compact[0] = False
        h2d_u8 = sum(sum(v.numel() * v.element_size() for v in hb.values() if torch.is_tensor(v)) for hb in host_batches) // NB
        host_batches = fp32_batches
        pf._next = None
    e2e_losses.append(float(host_loss[(a.steps - 1) & 1][0]))
    assert all(v == v for v in e2e_losses[-a.steps:]), "non-finite loss in the end-to-end leg"
    e2e_value = B * n_gpus * a.steps / (ms_e2e / 1e3)
    h2d = sum(sum(v.numel() * v.element_size() for v in hb.values() if torch.is_tensor(v)) for hb in host_batches) // NB

    launches = (ops.count_kernels(pl.fwd_calls) + ops.count_kernels(pl.bwd_calls)) * a.steps

    # ---- per-kernel timing (events around every launch, separate pass) -> roofline of the dominant kernel ----
    roofline = None
    kernel_table = {}
    if rank == 0:
        agg = {}
        reps = 3
        for _ in range(reps):
            pl.seed.add_(1)
            for name, meta, t in ops.run_recorded_timed(pl.fwd_calls + pl.bwd_calls):
                d = agg.setdefault(name, {"ms": 0.0, "n": 0, "flops": 0.0, "bytes": 0.0})
                d["ms"] += t
                d["n"] += 1
                d["flops"] += meta.get("flops", 0.0)
                d["bytes"] += meta.get("bytes", 0.0)
        # The eager pass pays a launch gap + event cost at every boundary that the graph-replayed step does not
        # (LayerNorm forward: 19.3 us between events, 15.1 us per launch inside a graph).  Calibrate it out: the average
        # per-launch overhead is (eager pass - graph-replayed step) / launches, subtracted from every launch.
        n_calls = sum(d["n"] for d in agg.values()) / reps
        eager_ms = sum(d["ms"] for d in agg.values()) / reps
        graph_ms = ms / a.steps
        gap_ms = max(0.0, (eager_ms - graph_ms) / max(n_calls, 1))
        for d in agg.values():
            d["ms"] = max(d["ms"] - gap_ms * d["n"], 0.25 * d["ms"])
        total = sum(d["ms"] for d in agg.values())
        for name, d in sorted(agg.items(), key=lambda kv: -kv[1]["ms"]):
            kernel_table[name] = {"ms_per_step": round(d["ms"] / reps, 4), "launches_per_step": d["n"] // reps,
                                  "share": round(d["ms"] / total, 4),
                                  "tflops": round(d["flops"] / (d["ms"] * 1e-3) / 1e12, 2) if d["flops"] else None,
                                  "gbs": round(d["bytes"] / (d["ms"] * 1e-3) / 1e9, 1) if d["bytes"] else None}
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        traffic, traffic_src = {}, None
        try:   # per-launch DRAM bytes of the same command under ncu (tools/launch_summary.py), default workload only
            if a.workload == "default":
                tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
                traffic = tj["kernels"]
                traffic_src = ("static: dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu "
                               "capture profiles/ncu_traffic.json (" + str(tj.get("captured", "round 1")) + "), not re-measured by this run")
        except Exception:
            pass
        top = next(iter(kernel_table))
        d = agg[top]
        peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
        peak_bw = float(peaks.get("hbm_gbs", 6650.0))
        src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
        sec = d["ms"] * 1e-3
        ach_tf = d["flops"] / sec / 1e12 if d["flops"] else 0.0
        ach_bw = d["bytes"] / sec / 1e9 if d["bytes"] else 0.0
        # the binding roofline of the family: the larger of (algorithmic flops / tensor peak) and (algorithmic bytes /
        # HBM peak); the skinny-K GEMMs of the default model (K 256-768, fp32 residual in/out) are HBM-bound
        if ach_bw / peak_bw >= ach_tf / peak_tf:
            roofline = {"kernel": top, "bound": "hbm", "achieved": ach_bw, "peak": peak_bw, "unit": "GB/s",
                        "frac": ach_bw / peak_bw, "traffic": traffic.get(top, {}).get("dram_bytes_per_launch"),
                        "algorithmic_bytes_per_launch": d["bytes"] / d["n"], "tensor_tflops": ach_tf,
                        "tensor_frac": ach_tf / peak_tf, "peak_source": f"{src} hbm_gbs (copy: read + write)", "traffic_source": traffic_src}
        else:
            roofline = {"kernel": top, "bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s",
                        "frac": ach_tf / peak_tf, "traffic": traffic.get(top, {}).get("dram_bytes_per_launch"),
                        "algorithmic_bytes_per_launch": (d["bytes"] / d["n"]) if d["bytes"] else None,
                        "hbm_gbs": ach_bw, "hbm_frac": ach_bw / peak_bw,
                        "peak_source": f"{src} bf16_tflops_sustained", "traffic_source": traffic_src}

    cpu = None
    if rank == 0 and n_gpus == 1 and not a.no_cpu_baseline:
        c = cpu_reference(a, a.cpu_seconds)
        cpu = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}

    # the "library bar" (SURVEY 2.2 / 8d): the unmodified reference model on this GPU through stock PyTorch kernels
    libbar = None
    if rank == 0 and n_gpus == 1 and not a.no_library_bar and reference_available(a):
        from baseline import ref_bench
        del dev_dicts, dev_batches
        torch.cuda.empty_cache()
        try:
            libbar = ref_bench.library_bar(a.neurons, wl.n_beh, wl.T, B, dev, train=not a.eval_mode)
            for k in ("fp32_cycled", "bf16_autocast_cycled", "fp32_no_masker", "bf16_autocast_no_masker"):
                libbar[k]["ours_over_this"] = value / libbar[k]["value"]
        except Exception as e:                                   # the bar is a side measurement: never lose the line
            libbar = {"unavailable": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        cfgj = workload_config(a, n_gpus)
        flops_step = 3 * wl.flops_fwd_per_trial() * B
        e2e_trainer = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                       "ms_per_step": ms_e2e / a.steps,
                       "what": "model(mod_dict) + loss.backward() on pinned HOST batches in the reference trainer's own form "
                               "(fp32 spikes; mod_dict with dense int64 eval masks built as trainer/base.py:51-103 builds it), "
                               "H2D of every batch and D2H of every loss inside the timed region"}
        e2e_wire = (None if ms_e2e_u8 is None else
                    {"value": B * n_gpus * a.steps / (ms_e2e_u8 / 1e3), "unit": UNIT,
                     "h2d_bytes_per_step": h2d_u8, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e_u8 / a.steps,
                     "what": "model(mod_dict) + loss.backward() on pinned HOST batches in this path's wire format: spike counts "
                             "shipped as uint8 and expanded on the device (bit-identical to the fp32 batch), compact eval masks "
                             "(scalar / (B,T)) instead of dense (B,T,N) int64 tensors (SURVEY 8f rank 2 / 3); H2D of every batch "
                             "and D2H of every loss inside the timed region"})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": a.steps,
            "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "strong" if a.strong else "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfgj, "clocks": clocks,
            # `e2e`: the public call on pinned HOST batches in this path's wire format (uint8 spike counts, compact eval
            # masks) -- the leg VERDICT r01 #7 asked for; `e2e_trainer_form`: the same call on batches exactly as the
            # reference trainer hands them over (fp32 spikes, dense int64 masks).  Workloads without a byte leg (scaled)
            # report the trainer form under `e2e`.
            "e2e": e2e_wire if e2e_wire is not None else e2e_trainer,
            "gpu_launches": launches,
            "e2e_trainer_form": e2e_trainer,
            "with_optimizer": {"value": value_opt, "unit": UNIT, "ms_per_step": ms_opt / a.steps,
                               "what": "fwd + bwd + fused AdamW step (mmfm_adamw_step over the flat fp32 buffers)"},
            "sustained": sustained, "library_bar": libbar,
            "roofline": roofline, "cpu_baseline": cpu, "kernels": kernel_table,
            "kernels_note": "per-kernel times: one CUDA event at every launch boundary of an eager pass, minus the average "
                            "per-launch gap of that pass ((eager pass - graph-replayed step) / launches), so the table sums to "
                            "the graph-replayed step that `value` times; tools/gemm_bench.py / ln_bench.py time single kernels "
                            "inside a graph for comparison",
            "flops_per_trial_fwd_bwd": 3 * wl.flops_fwd_per_trial(),
            "step_tensor_frac": flops_step / (ms / a.steps * 1e-3) / 1e12 / 1370.0,
        }
        print(json.dumps(line))
    if world > 1:
        if ddp is not None:
            ddp.close()
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
