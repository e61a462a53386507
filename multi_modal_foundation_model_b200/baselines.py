"""Linear baselines of ``train_baseline.py`` on the same kernels (SURVEY.md section 8a, row a18).

``BaselineDecoder`` (reference ``src/models/baseline_decoder.py:18-49``): ``Linear(N -> n_beh)`` per time bin,
``MSE.sum() / B``.  ``BaselineEncoder`` (``src/models/baseline_encoder.py:18-53``): ``Linear(T*n_beh -> T*N)`` on the
flattened trial, ``PoissonNLL(log_input).sum() / B``.  Same constructor arguments, attribute names (``layer``),
``state_dict`` keys and output dataclasses; forward = tcgen05 GEMM + fused loss/gradient kernel, backward = tcgen05
wgrad (weight + bias).  No PyTorch fallback.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable

from . import ops
from ._lib import LOSS_MSE, LOSS_POISSON, MmfmError
from .model import ModelOutput

bf16 = torch.bfloat16


@dataclass
class DecoderOutput(ModelOutput):
    loss: Optional[torch.Tensor] = None
    n_examples: Optional[int] = None
    preds: Optional[torch.Tensor] = None
    targets: Optional[torch.Tensor] = None


@dataclass
class EncoderOutput(DecoderOutput):
    pass


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


class _LinearLossFn(torch.autograd.Function):
    """loss = sum(ell(x W^T + b, targets)) / n_examples, with d loss / d preds produced by the fused loss kernel.
    loss and preds are both differentiable, and so is x: a gradient of loss alone scales the forward's dpreds; any
    other combination rebuilds dpreds with mmfm_loss_grad (mask of ones, T = S = 1)."""

    @staticmethod
    def forward(ctx, x2d, weight, bias, targets2d, kind, n_examples):
        if not x2d.is_cuda:
            raise MmfmError("the B200 path runs on a CUDA device only; there is no CPU fallback")
        R, K = x2d.shape
        N = weight.shape[0]
        dev = x2d.device
        xb = torch.empty(R, _pad8(K), device=dev, dtype=bf16)[:, :K]
        wb = torch.empty(N, _pad8(K), device=dev, dtype=bf16)[:, :K]
        ops.cast_bf16(x2d.detach().float().contiguous(), xb)
        ops.cast_bf16(weight.detach().contiguous(), wb)
        preds = torch.empty(R, N, device=dev, dtype=torch.float32)
        ops.gemm_tn(xb, wb, preds, bias=bias.detach() if bias is not None else None)
        # every element counts: a one-row "token mask" of ones, S = T = 1
        ones = torch.ones(R, 1, device=dev, dtype=torch.uint8)
        inv_n = torch.full((1,), 1.0 / float(n_examples), device=dev)
        npart = 296
        partials = torch.zeros(npart, device=dev)
        dpreds = torch.empty(R, _pad8(N), device=dev, dtype=bf16)[:, :N]
        targets = targets2d.detach().float().contiguous()
        ops.loss_fwd_bwd(preds, targets, ones, inv_n, kind, partials, dpreds, B=R, T=1, Cc=N, S=1, off=0)
        mod_loss, loss = torch.empty(1, device=dev), torch.empty(1, device=dev)
        ops.loss_finalize(partials, npart, 1, inv_n, mod_loss, loss)
        ctx.save_for_backward(xb, dpreds, preds, targets, ones, inv_n)
        ctx.weight = weight.detach()
        ctx.shape = (N, K, bias is not None, kind, x2d.dtype)
        ctx.set_materialize_grads(False)
        return loss.reshape(()), preds

    @staticmethod
    @once_differentiable
    def backward(ctx, g_loss, g_preds):
        xb, dpreds, preds, targets, ones, inv_n = ctx.saved_tensors
        N, K, has_bias, kind, x_dtype = ctx.shape
        R = xb.shape[0]
        dev = xb.device
        want_x = ctx.needs_input_grad[0]
        plain = g_preds is None and not want_x
        if plain:
            scale = g_loss.reshape(1).float()
        else:
            scale = None
            ops.loss_grad(preds, targets, ones, inv_n, kind, dpreds,
                          g_loss=g_loss.reshape(1).float() if g_loss is not None else None,
                          g_preds=g_preds.float().unsqueeze(1) if g_preds is not None else None, B=R, T=1, Cc=N, S=1,
                          off=0)
        dW = db = dx = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dW = torch.zeros(N, K, device=dev)
            db = torch.zeros(N, device=dev) if has_bias else None
            ops.gemm_wgrad(dpreds, xb, dW, dbias=db)
            if scale is not None:
                ops.scale_inplace(dW, scale)
                if db is not None:
                    ops.scale_inplace(db, scale)
        if want_x:       # dX = dpreds . W on a transposed bf16 copy of W
            wt = torch.empty(K, _pad8(N), device=dev, dtype=bf16)[:, :N]
            ops.cast_bf16(ctx.weight.contiguous(), None, wt)
            dx32 = torch.empty(R, K, device=dev, dtype=torch.float32)
            ops.gemm_tn(dpreds, wt, dx32)
            dx = dx32.to(x_dtype)
        return dx, dW, db, None, None, None


class BaselineDecoder(nn.Module):
    """models/baseline_decoder.py:18-49"""

    def __init__(self, in_channel, out_channel, **kwargs):
        super().__init__()
        self.in_channel = in_channel
        self.out_channel = out_channel
        self.layer = nn.Linear(self.in_channel, self.out_channel)

    def forward(self, data_dict: Dict[str, torch.Tensor]) -> DecoderOutput:
        inputs, targets = data_dict["inputs"], data_dict["targets"]
        B, T, _ = targets.shape
        loss, preds = _LinearLossFn.apply(inputs.reshape(B * T, self.in_channel), self.layer.weight, self.layer.bias,
                                          targets.reshape(B * T, self.out_channel), LOSS_MSE, B)
        return DecoderOutput(loss=loss, n_examples=B, preds=preds.view(B, T, self.out_channel), targets=targets)


class BaselineEncoder(nn.Module):
    """models/baseline_encoder.py:18-53"""

    def __init__(self, in_channel, out_channel, seq_len=100, **kwargs):
        super().__init__()
        self.seq_len = seq_len
        self.in_channel = in_channel
        self.out_channel = out_channel
        self.layer = nn.Linear(self.seq_len * self.in_channel, self.seq_len * self.out_channel)

    def forward(self, data_dict: Dict[str, torch.Tensor]) -> EncoderOutput:
        inputs, targets = data_dict["inputs"], data_dict["targets"]
        B, T, N = targets.shape
        loss, preds = _LinearLossFn.apply(inputs.flatten(1), self.layer.weight, self.layer.bias, targets.flatten(1),
                                          LOSS_POISSON, B)
        return EncoderOutput(loss=loss, n_examples=B, preds=preds.view(B, T, N), targets=targets)
