"""Training objectives beyond the reference's sampled BCE, as autograd functions for the drop-in models.

``catalogue_cross_entropy(hidden, item_table, target, weight=None)`` -- full-catalogue softmax cross-entropy over the
logits ``predict`` computes (SRFR_model.py:144-152 with label = arange(1, N+1)): for every position with a target,
``w (logsumexp_j <h, E_j> - <h, E_target>)`` over items j = 1..N (row 0, the pad item, is never a candidate), summed and
divided by the sum of the weights.  The (positions, N) logits are never materialised: the loss and both gradients come
from the tcgen05 kernels of csrc/catalogue_ce.cu.  ``FusedTrainer(loss="ce")`` runs the same kernels inside its step.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import ops

__all__ = ["catalogue_cross_entropy"]

bf16 = torch.bfloat16


def _padded(D: int) -> int:
    return (D + 15) // 16 * 16


def check_ce_width(D: int) -> int:
    """Padded width Dp of a D-wide table, or ValueError when the kernels cannot serve it (Dp > 256)."""
    Dp = _padded(D)
    try:
        ops.catalogue_ce_plan(Dp)
    except RuntimeError as ex:
        raise ValueError(f"catalogue cross-entropy: item table width {D} is not supported ({ex})") from None
    return Dp


def _bf16_rows(src: torch.Tensor, Dp: int) -> torch.Tensor:
    """(R, D) fp32 -> (R, Dp) bf16, zero padding columns."""
    out = torch.zeros(src.shape[0], Dp, dtype=bf16, device=src.device)
    if src.shape[0]:
        ops.f32_to_bf16_split(src, out[:, :src.shape[1]])
    return out


class _CatalogueCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, hidden, item_table, target, weight):
        D = item_table.shape[1]
        N = item_table.shape[0] - 1
        Dp = check_ce_width(D)
        dev = hidden.device
        h = hidden.detach().reshape(-1, D).float().contiguous()
        t = target.reshape(-1).to(torch.int64).contiguous()
        w = None if weight is None else (weight.detach().reshape(-1).float() * (t != 0)).contiguous()
        hb = _bf16_rows(h, Dp)
        tb = _bf16_rows(item_table.detach().float().contiguous(), Dp)
        norm = torch.zeros(2, dtype=torch.float32, device=dev)
        acc = torch.zeros(2, dtype=torch.float32, device=dev)
        lse = torch.empty(h.shape[0], dtype=torch.float32, device=dev)
        if h.shape[0]:
            ops.weight_sums(t, w, None, norm)
            ops.catalogue_ce_fwd(hb, tb, t, w, lse, acc)
        ctx.save_for_backward(hb, tb, t, w if w is not None else torch.empty(0, device=dev), norm, lse)
        ctx.has_w, ctx.D, ctx.shape = w is not None, D, hidden.shape
        return torch.where(norm[0] > 0, acc[0] / norm[0], torch.zeros_like(acc[0]))

    @staticmethod
    def backward(ctx, g):
        hb, tb, t, w, norm, lse = ctx.saved_tensors
        w = w if ctx.has_w else None
        D = ctx.D
        dh = dE = None
        if ctx.needs_input_grad[0]:
            dh = torch.zeros(hb.shape[0], D, dtype=torch.float32, device=hb.device)
        if ctx.needs_input_grad[1]:
            dE = torch.zeros(tb.shape[0], D, dtype=torch.float32, device=hb.device)
        if hb.shape[0] and (dh is not None or dE is not None):
            ops.catalogue_ce_bwd(hb, tb, t, w, norm, lse, dh, dE, D)
        if dh is not None:
            dh = (dh * g).view(ctx.shape)
        if dE is not None:
            dE = dE * g
        return dh, dE, None, None


def catalogue_cross_entropy(hidden: torch.Tensor, item_table: torch.Tensor, target: torch.Tensor,
                            weight: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Full-catalogue softmax cross-entropy (scalar): hidden (..., D) fp32, item_table (N + 1, D) fp32 (row 0 = pad),
    target (...) int64 with 0 = no loss term and 1..N = the positive item, weight (...) fp32 or None (= 1[target != 0]).
    loss = sum w (logsumexp_j z_j - z_target) / sum w over the logits z_j = <hidden, E_j>, j = 1..N; 0 when every weight
    is 0.  Gradients flow to hidden and to item_table (row 0 gets none).  Operands are rounded to bf16, accumulation and
    the log-sum-exp are fp32.  Targets outside 0..N raise ValueError (one host sync)."""
    if item_table.dim() != 2 or hidden.shape[-1] != item_table.shape[1]:
        raise ValueError(f"catalogue cross-entropy: hidden (..., {hidden.shape[-1]}) does not match item_table "
                         f"{tuple(item_table.shape)}")
    if target.shape != hidden.shape[:-1] or (weight is not None and weight.shape != target.shape):
        raise ValueError("catalogue cross-entropy: target / weight must have hidden's leading shape")
    N = item_table.shape[0] - 1
    if target.numel() and bool(((target < 0) | (target > N)).any()):
        raise ValueError(f"catalogue cross-entropy: targets must lie in 0..{N} (0 = no loss term)")
    return _CatalogueCE.apply(hidden, item_table, target, weight)
