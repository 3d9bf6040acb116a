"""Training objectives beyond the reference's sampled BCE, as autograd functions for the drop-in models.

``catalogue_cross_entropy(hidden, item_table, target, weight=None)`` -- full-catalogue softmax cross-entropy over the
logits ``predict`` computes (SRFR_model.py:144-152 with label = arange(1, N+1)): for every position with a target,
``w (logsumexp_j <h, E_j> - <h, E_target>)`` over items j = 1..N (row 0, the pad item, is never a candidate), summed and
divided by the sum of the weights.  The (positions, N) logits are never materialised: the loss and both gradients come
from the tcgen05 kernels of csrc/catalogue_ce.cu.  ``FusedTrainer(loss="ce")`` runs the same kernels inside its step.

``sampled_gbce(hidden, item_table, target, negatives, weight=None, t=0.75, exclude=None)`` -- gSASRec's gBCE
(Petrov & Macdonald, RecSys 2023) over k negatives shared by every position: with alpha = k / (N - 1) and
beta = 1 - t (1 - alpha), ``(sum w beta softplus(-z_pos) + sum w sum_j m_j softplus(z_j)) / sum w``, where m_j = 0 when
negative j occurs in the position's sequence (``exclude``).  gSASRec divides by (k + 1) sum w; this loss is (k + 1) times
theirs, on the scale of the reference's BCE.  Kernels: csrc/gbce.cu; ``FusedTrainer(loss="gbce")`` draws the negatives on
the device and runs the same kernels inside its step.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import ops

__all__ = ["catalogue_cross_entropy", "sampled_gbce"]

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


def gbce_beta(k: int, N: int, t: float) -> float:
    """gSASRec's calibration exponent: beta = 1 - t (1 - alpha) with alpha = k / (N - 1), the sampling rate of the
    negatives among the N - 1 items that are not the positive."""
    return 1.0 - float(t) * (1.0 - k / (N - 1))


def check_gbce(k: int, t: float, N: int, D: int) -> int:
    """Padded width Dp, or ValueError for a setting the gBCE kernels do not serve: k outside 1..256, t outside [0, 1],
    fewer than 2 items, or a table wider than 256 columns after padding."""
    if not (1 <= int(k) <= 256) or int(k) != k:
        raise ValueError(f"gbce: num_negatives = {k} must be an integer in 1..256")
    if not (0.0 <= float(t) <= 1.0):
        raise ValueError(f"gbce: t = {t} must lie in [0, 1]")
    if N < 2:
        raise ValueError(f"gbce: needs at least 2 items (N = {N})")
    Dp = _padded(D)
    if Dp > 256:
        raise ValueError(f"gbce: item table width {D} is not supported (padded width {Dp} > 256)")
    return Dp


class _SampledGBCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, hidden, item_table, target, negatives, weight, t, exclude):
        D = item_table.shape[1]
        N = item_table.shape[0] - 1
        k = negatives.numel()
        Dp = check_gbce(k, t, N, D)
        dev = hidden.device
        h = hidden.detach().reshape(-1, D).float().contiguous()
        R = h.shape[0]
        tg = target.reshape(-1).to(torch.int64).contiguous()
        w = None if weight is None else (weight.detach().reshape(-1).float() * (tg != 0)).contiguous()
        E = item_table.detach().float().contiguous()
        Kp, n_split, _, _ = ops.gbce_plan(k, Dp, R)
        ids = negatives.reshape(-1).to(torch.int64).contiguous()
        nb = torch.empty(Kp, Dp, dtype=bf16, device=dev)
        n_seq = exclude.shape[0] if exclude is not None else 0
        excl = torch.zeros(max(n_seq, 1), (k + 31) // 32, dtype=torch.int32, device=dev) if exclude is not None else None
        ops.gbce_draw(E, ids, nb, excl, ex_a=exclude, draw=False)
        hb = _bf16_rows(h, Dp)
        norm = torch.zeros(2, dtype=torch.float32, device=dev)
        acc = torch.zeros(2, dtype=torch.float32, device=dev)
        dh = torch.zeros(R, D, dtype=torch.float32, device=dev)
        dE = torch.zeros(N + 1, D, dtype=torch.float32, device=dev)
        part = torch.empty(n_split * Kp * Dp, dtype=torch.float32, device=dev)
        if R:
            L = R // n_seq if exclude is not None else 1
            ops.weight_sums(tg, w, None, norm)
            ops.gbce_loss(hb, nb, ids, E, tg, w, norm, excl, L, gbce_beta(k, N, t), acc, dh, dE, part)
        ctx.save_for_backward(dh, dE)
        ctx.shape = hidden.shape
        return torch.where(norm[0] > 0, (acc[0] + acc[1]) / norm[0], torch.zeros_like(acc[0]))

    @staticmethod
    def backward(ctx, g):
        dh, dE = ctx.saved_tensors
        return (dh * g).view(ctx.shape), dE * g, None, None, None, None, None


def sampled_gbce(hidden: torch.Tensor, item_table: torch.Tensor, target: torch.Tensor, negatives: torch.Tensor,
                 weight: Optional[torch.Tensor] = None, t: float = 0.75, exclude: Optional[torch.Tensor] = None
                 ) -> torch.Tensor:
    """gSASRec's gBCE (scalar) over negatives shared by every position: hidden (..., D) fp32, item_table (N + 1, D) fp32
    (row 0 = pad), target (...) int64 with 0 = no loss term, negatives (k,) int64 in 1..N (duplicates count once per
    draw), weight (...) fp32 or None (= 1[target != 0]), t in [0, 1].  exclude (B, M) int64 (ids per sequence, 0 = none)
    or None: position p belongs to sequence p // (positions / B) in hidden's flattened order, and a negative that occurs
    in its sequence's row of exclude is left out of its loss.  The loss and both gradients are computed together in the
    forward (bf16 operands, fp32 accumulation); gradients flow to hidden and item_table (row 0 gets none).  Ids out of
    range and settings the kernels do not serve raise ValueError (one host sync for the id checks)."""
    if item_table.dim() != 2 or hidden.shape[-1] != item_table.shape[1]:
        raise ValueError(f"gbce: hidden (..., {hidden.shape[-1]}) does not match item_table {tuple(item_table.shape)}")
    if target.shape != hidden.shape[:-1] or (weight is not None and weight.shape != target.shape):
        raise ValueError("gbce: target / weight must have hidden's leading shape")
    N = item_table.shape[0] - 1
    if negatives.dim() != 1:
        raise ValueError("gbce: negatives must be a (k,) tensor of item ids")
    check_gbce(negatives.numel(), t, N, item_table.shape[1])
    if exclude is not None:
        if exclude.dim() != 2 or exclude.shape[0] < 1 or target.numel() % exclude.shape[0] != 0:
            raise ValueError("gbce: exclude must be (B, M) with B dividing the number of positions")
    if target.numel() and bool(((target < 0) | (target > N)).any()):
        raise ValueError(f"gbce: targets must lie in 0..{N} (0 = no loss term)")
    if bool(((negatives < 1) | (negatives > N)).any()):
        raise ValueError(f"gbce: negatives must lie in 1..{N}")
    return _SampledGBCE.apply(hidden, item_table, target, negatives, weight, float(t),
                              None if exclude is None else exclude.to(torch.int64).contiguous())
