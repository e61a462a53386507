"""GPU: data-parallel multi-session training, where every rank may run another session.

mmfm_session_grad_combine against a torch restatement doing the same fp32 operations in the same order (bitwise), and
a three-session model on two ranks with different sessions per rank: gradients equal across ranks, equal to the mean
of the two single-GPU gradients, idle sessions exactly zero, three AdamW steps leaving equal weights.  Over NCCL on two
GPUs (eager runs, capture and replay of every plan, also with a frozen core), and over gloo with both ranks on one GPU."""
import os
import random
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _combine_ref(grad, gathered, ids, ranges, inv_world):
    out = grad.clone()
    ids = ids.tolist()
    for r0, s in enumerate(ids):
        if not 0 <= s < ranges.shape[0] or s in ids[:r0]:
            continue
        lo0, hi0, lo1, hi1 = ranges[s].tolist()
        n = (hi0 - lo0) + (hi1 - lo1)
        if min(lo0, lo1) < 0 or hi0 < lo0 or hi1 < lo1 or n > gathered.stride(0):      # skipped: malformed entry
            continue
        acc = torch.zeros(n, device=grad.device)
        for r in range(r0, len(ids)):
            if ids[r] == s:
                acc = acc + gathered[r, :n]
        acc = acc * inv_world
        out[lo0:hi0] = acc[:hi0 - lo0]
        out[lo1:hi1] = acc[hi0 - lo0:]
    return out


def _check_combine(grad, gathered, ids, ranges, inv_world):
    from multi_modal_foundation_model_b200 import ops
    want = _combine_ref(grad, gathered, ids, ranges, inv_world)
    ops.session_grad_combine(grad, gathered, ids, ranges, inv_world)
    torch.cuda.synchronize()
    assert torch.equal(grad, want)


def test_combine_at_multisession_sizes():
    """configs[3] sizes: 8 ranks, H 256, sessions of 256..1024 neurons; each session's head range and embedder range
    (the first laid out before the shared core, the second after it), in one table and as two one-range tables."""
    rng = random.Random(3)
    H, n_sess = 256, 6
    neurons = [rng.randint(256, 1024) for _ in range(n_sess)]
    pad = lambda n: (n + 63) // 64 * 64
    head = [pad(H * N + N) + pad(2 * H + 2) for N in neurons]
    emb = [2 * (pad(2 * N * N) + pad(2 * N) + pad(H * 2 * N) + pad(H) + pad(100 * H)) for N in neurons]
    core = 6_700_000
    off, hr = 0, []
    for n in head:
        hr.append((off, off + n))
        off += n
    off += core
    er = []
    for n in emb:
        er.append((off, off + n))
        off += n
    total = off
    ids = torch.tensor([3, 1, 3, 0, 5, 5, 5, 2], dtype=torch.int32, device="cuda")       # session 4 idle
    L = max(h1 - h0 + e1 - e0 for (h0, h1), (e0, e1) in zip(hr, er))
    g = torch.Generator(device="cuda").manual_seed(0)
    gathered = torch.randn(8, L, device="cuda", generator=g)
    both = torch.tensor([[h0, h1, e0, e1] for (h0, h1), (e0, e1) in zip(hr, er)], dtype=torch.int64, device="cuda")
    sentinel = 7.25
    grad = torch.full((total,), sentinel, device="cuda")
    _check_combine(grad, gathered, ids, both, 1.0 / 8)
    h4, e4 = hr[4], er[4]
    assert (grad[h4[0]:h4[1]] == sentinel).all() and (grad[e4[0]:e4[1]] == sentinel).all(), "idle session touched"
    assert (grad[hr[-1][1]:er[0][0]] == sentinel).all(), "shared core touched"
    # the data-parallel path's two one-range tables
    for tab in ([[h0, h1, 0, 0] for h0, h1 in hr], [[e0, e1, 0, 0] for e0, e1 in er]):
        grad = torch.full((total,), sentinel, device="cuda")
        _check_combine(grad, gathered, ids, torch.tensor(tab, dtype=torch.int64, device="cuda"), 1.0 / 8)


def test_combine_ragged_ranges_and_bad_entries():
    """Scalar path: ranges at odd offsets and lengths, an odd slab stride; ids out of range and a malformed range
    entry are skipped."""
    g = torch.Generator(device="cuda").manual_seed(1)
    ranges = torch.tensor([[3, 10, 41, 42], [11, 11, 20, 37], [50, 51, 60, 60], [70, 90, 95, 60]],
                          dtype=torch.int64, device="cuda")          # session 3: hi1 < lo1, malformed
    full = torch.randn(5, 33, device="cuda", generator=g)
    gathered = full[:, :31]                                          # row stride 33, slab width 31 >= 17
    for ids in ([1, 0, 1, 2, 0], [2, 2, 2, 2, 2], [0, 9, -1, 3, 1]):
        grad = torch.full((100,), -3.5, device="cuda")
        _check_combine(grad, gathered, torch.tensor(ids, dtype=torch.int32, device="cuda"), ranges, 0.2)
        if 3 in ids:
            assert (grad[70:] == -3.5).all()
    # float4 path with a scalar tail: aligned ranges whose lengths are not multiples of 4
    ranges = torch.tensor([[0, 1030, 2048, 2051], [1032, 2040, 2052, 2400]], dtype=torch.int64, device="cuda")
    gathered = torch.randn(3, 1400, device="cuda", generator=g)
    grad = torch.zeros(2400, device="cuda")
    _check_combine(grad, gathered, torch.tensor([1, 0, 1], dtype=torch.int32, device="cuda"), ranges, 1.0 / 3)


# ---- two GPUs ------------------------------------------------------------------------------------------------------
CHANS = {"sess-a": {"ap": 40, "behavior": 2}, "sess-b": {"ap": 88, "behavior": 2}, "sess-c": {"ap": 56, "behavior": 2}}
PHASES = [("sess-a", "sess-b"), ("sess-b", "sess-a"), ("sess-c", "sess-c")]     # rank 0's and rank 1's session
OPT_STEPS = [("sess-a", "sess-c"), ("sess-c", "sess-c"), ("sess-b", "sess-a")]


def _md(sess, seed, mode):
    from multi_modal_foundation_model_b200.synthetic import make_batch, make_mod_dict
    d = make_mod_dict(make_batch(4, CHANS[sess]["ap"], 2, 100, step=seed, pad_bins=5), ["ap", "behavior"], mode,
                      device="cuda")
    for v in d.values():
        v["eid"] = sess
    return d


def _model(seed, frozen):
    from _util import small_config
    from multi_modal_foundation_model_b200.model import MultiSessionMultiModal
    torch.manual_seed(seed)
    model = MultiSessionMultiModal(CHANS, ["ap", "behavior"], small_config()).cuda().eval()
    if frozen:
        for n, p in model.named_parameters():
            p.requires_grad_(n.startswith("session_embeddings."))
    return model


def _grads(model):
    st = model.engine().store
    return {n: st.g(n).detach().cpu().clone() for n in st.params}


def _worker(rank, world, port, out_dir, frozen, backend):
    import torch.distributed as dist
    from multi_modal_foundation_model_b200.optim import AdamW
    from multi_modal_foundation_model_b200.parallel import DataParallel
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    if backend == "nccl":
        torch.cuda.set_device(rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    else:       # both ranks on one GPU: gloo collectives cannot be captured, so the backward stays eager
        os.environ["MMFM_DDP_GRAPH"] = "0"
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        model = _model(100 + rank, frozen)                # different init per rank: rank 0's is broadcast
        ddp = DataParallel(model, bucket_mb=0.25)
        assert ddp.xchg is not None
        grads = []
        for ph, sess in enumerate(PHASES):
            for k in range(3):                             # eager, graph capture, graph replay of this plan
                model.zero_grad(set_to_none=True)
                model(_md(sess[rank], 100 * ph + 10 * k + rank, "encoding" if k == 0 else "decoding")).loss.backward()
                grads.append(_grads(model))
        weights0 = {n: p.detach().cpu().clone() for n, p in model.named_parameters()}
        opt = AdamW([p for p in model.parameters() if p.requires_grad], lr=1e-3, weight_decay=0.01)
        for k, sess in enumerate(OPT_STEPS):
            opt.zero_grad(set_to_none=True)
            model(_md(sess[rank], 1000 + 10 * k + rank, "decoding")).loss.backward()
            opt.step()
        torch.cuda.synchronize()
        weights = {n: p.detach().cpu().clone() for n, p in model.named_parameters()}
        torch.save({"grads": grads, "weights0": weights0, "weights": weights},
                   os.path.join(out_dir, f"rank{rank}.pt"))
        ddp.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("frozen", [False, True], ids=["full", "frozen_core"])
def test_two_gpus_different_sessions_per_rank(tmp_path, frozen):
    _two_ranks(tmp_path, frozen, "nccl")


def test_two_ranks_on_one_gpu_over_gloo(tmp_path):
    """The same exchange, eager, with both ranks on one device (runs where only one GPU is present)."""
    _two_ranks(tmp_path, False, "gloo")


def _two_ranks(tmp_path, frozen, backend):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    world = 2
    mp.spawn(_worker, args=(world, port, str(tmp_path), frozen, backend), nprocs=world, join=True)
    r = [torch.load(tmp_path / f"rank{i}.pt") for i in range(world)]
    for step, (g0, g1) in enumerate(zip(r[0]["grads"], r[1]["grads"])):
        for n in g0:
            assert torch.equal(g0[n], g1[n]), f"ranks disagree on {n} at step {step}"
    for n in r[0]["weights"]:
        assert torch.equal(r[0]["weights0"][n], r[1]["weights0"][n]), f"weights not broadcast: {n}"
        assert torch.equal(r[0]["weights"][n], r[1]["weights"][n]), f"AdamW steps diverged on {n}"
        if frozen and not n.startswith("session_embeddings."):
            assert torch.equal(r[0]["weights"][n], r[0]["weights0"][n]), n
    # single-GPU reference: rank 0's weights, each rank's batch in turn, mean of the two gradients
    model = _model(100, frozen)
    prefix = {k: model.session_prefix(k) for k in CHANS}
    step = 0
    for ph, sess in enumerate(PHASES):
        for k in range(3):
            acc = None
            for rank in range(world):
                model.zero_grad(set_to_none=True)
                model(_md(sess[rank], 100 * ph + 10 * k + rank, "encoding" if k == 0 else "decoding")).loss.backward()
                g = _grads(model)
                acc = g if acc is None else {n: acc[n] + g[n] for n in g}
            got = r[0]["grads"][step]
            for n, gref in acc.items():
                owner = next((s for s, p in prefix.items() if n.startswith(p)), None)
                if owner is not None and owner not in sess:
                    assert (got[n] == 0).all(), f"idle session {owner}: {n} not zero"
                    continue
                gref = gref / world
                scale = gref.abs().max().item() + 1e-8
                assert (got[n] - gref).abs().max().item() <= 2e-3 * scale + 1e-7, (step, n)
            step += 1
