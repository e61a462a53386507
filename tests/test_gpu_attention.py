"""GPU parity of the masked attention kernels (csrc/attention.cu) against a plain fp32 torch restatement of
F.scaled_dot_product_attention with the reference's boolean masks (mm.py:152-158,178-194; mm_utils.py:105-112)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _allowed(mode, key_valid, Sq, Sk, mod_q=None, mod_k=None):
    B = key_valid.shape[0]
    if mode == 2:
        a = torch.ones(Sq, Sk, device="cuda").tril().bool()[None].expand(B, Sq, Sk)
    else:
        a = key_valid.bool()[:, None, :].expand(B, Sq, Sk)
    if mode == 1:
        a = a | torch.eye(Sq, Sk, device="cuda").bool()[None]
    if mod_q is not None:
        a = a | (mod_q[None, :, None] != mod_k[None, None, :])
    return a


def _ref(q, k, v, allowed, nh, d, keep_p=None, keep_o=None):
    B, Sq, H = q.shape
    Sk = k.shape[1]
    qh = q.view(B, Sq, nh, d).transpose(1, 2)
    kh = k.view(B, Sk, nh, d).transpose(1, 2)
    vh = v.view(B, Sk, nh, d).transpose(1, 2)
    s = (qh @ kh.transpose(-1, -2)) / math.sqrt(d)
    s = s.masked_fill(~allowed[:, None], float("-inf"))
    lse = torch.logsumexp(s, dim=-1)
    p = torch.softmax(s, dim=-1)
    if keep_p is not None:
        p = p * keep_p
    o = (p @ vh).transpose(1, 2).reshape(B, Sq, H)
    if keep_o is not None:
        o = o * keep_o
    return o, lse


@pytest.mark.parametrize("B,nh,d,Sq,Sk,mode,sep,pad", [
    (3, 8, 32, 200, 200, 1, False, 0),
    (3, 8, 32, 200, 200, 0, False, 30),
    (2, 8, 32, 200, 200, 1, False, 30),
    (2, 4, 64, 130, 130, 2, False, 0),
    (2, 4, 64, 257, 257, 0, True, 20),
    (1, 16, 64, 1000, 1000, 1, False, 100),
    (2, 8, 32, 64, 200, 0, False, 72),
    (2, 4, 32, 300, 300, 2, False, 0),        # long sequence, causal, d_head 32: streaming kernels
    (1, 8, 32, 520, 520, 1, False, 40),
    (2, 4, 64, 130, 330, 0, False, 50),       # Sq != Sk across several key blocks
    (1, 4, 64, 330, 130, 1, False, 0),
    (2, 4, 32, 100, 100, 1, False, 10),       # one key half, one query tile (persistent fused backward, smallest form)
    (1, 4, 32, 256, 256, 0, False, 0),        # the largest shape the fused kernels take: two full halves / tiles
    (2, 4, 32, 200, 120, 2, False, 0),        # two query tiles over a single key half, causal
    (2, 4, 32, 150, 150, 1, False, 10),       # Sq % 4 != 0: the fused backward refuses it, the streamed pair takes it
])
@pytest.mark.parametrize("dropout", [False, True])
def test_attention_fwd_bwd(B, nh, d, Sq, Sk, mode, sep, pad, dropout):
    from multi_modal_foundation_model_b200 import ops
    from oracle import philox_ref as px
    H = nh * d
    g = torch.Generator(device="cuda").manual_seed(5)
    qkv = (torch.randn(B * Sq, 3 * H, generator=g, device="cuda")).to(torch.bfloat16)
    if Sq == Sk:
        q, k, v = qkv[:, :H], qkv[:, H:2 * H], qkv[:, 2 * H:]
    else:
        q = qkv[:, :H]
        kv = torch.randn(B * Sk, 2 * H, generator=g, device="cuda").to(torch.bfloat16)
        k, v = kv[:, :H], kv[:, H:]
    key_valid = torch.ones(B, Sk, dtype=torch.uint8, device="cuda")
    if pad:
        key_valid[:, Sk - pad:] = 0
        key_valid[0, : Sk // 3] = 0
    mod_q = mod_k = None
    if sep:
        mod_q = (torch.arange(Sq, device="cuda") // 100).to(torch.int16)
        mod_k = (torch.arange(Sk, device="cuda") // 100).to(torch.int16)
    o = torch.zeros(B * Sq, H, device="cuda", dtype=torch.bfloat16)
    lse = torch.zeros(B, nh, Sq, device="cuda")
    nkb = (Sk + 63) // 64
    p_keep = torch.zeros(B * nh * Sq * nkb * 4, dtype=torch.int16, device="cuda")
    seed_val = 0x0BADC0DE12345
    seed = torch.tensor([seed_val], dtype=torch.int64, device="cuda")
    dp = ops.DropSpec(seed, 33, 0.4) if dropout else ops.NO_DROP
    do_ = ops.DropSpec(seed, 34, 0.4) if dropout else ops.NO_DROP
    kw = dict(B=B, n_heads=nh, Sq=Sq, Sk=Sk, d_head=d, mask_mode=mode, mod_q=mod_q, mod_k=mod_k, drop_p=dp, drop_o=do_,
              p_keep=p_keep)
    ops.attention_fwd(q, k, v, o, lse, key_valid, **kw)
    torch.cuda.synchronize()

    keep_p = keep_o = None
    if dropout:
        keep_p = torch.from_numpy(px.prob_keep_mask(seed_val, 33, B * nh * Sq, Sk, 0.4)).cuda().view(B, nh, Sq, Sk)
        keep_o = torch.from_numpy(px.keep_mask(seed_val, 34, B * Sq, H, 0.4)).cuda().view(B, Sq, H)
    qf = q.float().reshape(B, Sq, H).requires_grad_(True)
    kf = k.float().reshape(B, Sk, H).requires_grad_(True)
    vf = v.float().reshape(B, Sk, H).requires_grad_(True)
    allowed = _allowed(mode, key_valid, Sq, Sk, mod_q, mod_k)
    o_ref, lse_ref = _ref(qf, kf, vf, allowed, nh, d, keep_p, keep_o)
    err_o = (o.float().view(B, Sq, H) - o_ref).abs().max().item()
    assert err_o < 3e-2, f"attention fwd max err {err_o}"
    fin = torch.isfinite(lse_ref)
    err_l = (lse[fin] - lse_ref[fin]).abs().max().item()
    assert err_l < 2e-3, f"lse max err {err_l}"

    # backward: upstream gradient wrt the (post output-dropout) attention output
    d_o = (torch.randn(B * Sq, H, generator=g, device="cuda") * 0.1).to(torch.bfloat16)
    o_ref.backward(d_o.float().view(B, Sq, H))
    dq = torch.zeros(B * Sq, H, device="cuda", dtype=torch.bfloat16)
    dk = torch.zeros(B * Sk, H, device="cuda", dtype=torch.bfloat16)
    dv = torch.zeros(B * Sk, H, device="cuda", dtype=torch.bfloat16)
    delta = torch.zeros(B, nh, Sq, device="cuda")
    d_o_work = d_o.clone()
    ops.attention_bwd(q, k, v, o, lse, key_valid, d_o=d_o_work, delta=delta, dq=dq, dk=dk, dv=dv, **kw)
    torch.cuda.synchronize()
    for name, got, ref in (("dq", dq, qf.grad), ("dk", dk, kf.grad), ("dv", dv, vf.grad)):
        ref = ref.reshape(got.shape)
        scale = ref.abs().max().item() + 1e-6
        err = (got.float() - ref).abs().max().item()
        assert err <= 3e-2 * scale + 1e-3, f"{name}: max err {err:.4g} (scale {scale:.4g})"
