"""Thin tensor-level wrappers over the C ABI (include/srfrd_b200.h).

Every function takes CUDA torch tensors, passes raw device pointers plus the caller's current
stream, and returns nothing (outputs are pre-allocated by the caller).  PyTorch is used only for
device memory and streams.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from contextlib import contextmanager

from ._lib import CastDesc, GemmEpilogue, Mlp2Epilogue, PackDesc, RepackPart, call

bf16 = torch.bfloat16


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _chk(t: torch.Tensor, dtype, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"srfrd_b200: {name} must be a CUDA tensor (there is no CPU fallback)")
    if t.dtype != dtype:
        raise RuntimeError(f"srfrd_b200: {name} must be {dtype}, got {t.dtype}")
    if t.stride(-1) != 1:
        raise RuntimeError(f"srfrd_b200: {name} must be contiguous in its last dimension")


def embed_ln_fwd(item_table, pos_table, aux_table, mode, seq, aux_ids, item_scale, ln_w, ln_b, eps,
                 x0_bf16=None, x0_f32=None, q_bf16=None, stats=None, drop_p=0.0, drop_seed=0, drop_stream=0,
                 drop_step=None):
    _lib.require_device()
    B, L = seq.shape
    D = item_table.shape[1]
    F = aux_table.shape[1] if (aux_table is not None and mode == 1) else 0
    _chk(item_table, torch.float32, "item_table"); _chk(seq, torch.int64, "seq")
    ldx = (x0_bf16 if x0_bf16 is not None else q_bf16).stride(0) if (x0_bf16 is not None or q_bf16 is not None) else D + F
    call("srfrd_embed_ln_fwd", _p(item_table), item_table.shape[0], D, _p(pos_table), _p(aux_table),
         0 if aux_table is None else aux_table.shape[0], F, mode, _p(seq), _p(aux_ids), B, L, float(item_scale),
         _p(ln_w), _p(ln_b), float(eps), _p(x0_bf16), _p(x0_f32), _p(q_bf16), _p(stats), ldx, float(drop_p),
         int(drop_seed), int(drop_stream), _p(drop_step), _stream())


def srfu_labels(fake_ids, kind: int, labels):
    _lib.require_device()
    B, L = fake_ids.shape
    call("srfrd_srfu_labels", _p(fake_ids), B, L, kind, _p(labels), _stream())


def embed_bwd(dx0, seq, aux_ids, D, F, mode, item_scale, d_item, d_aux):
    B, L = seq.shape
    call("srfrd_embed_bwd", _p(dx0), dx0.stride(0), _p(seq), _p(aux_ids), B, L, D, F, mode, float(item_scale),
         _p(d_item), _p(d_aux), _stream())


def layernorm_fwd(x, w, b, eps, y_bf16=None, y_f32=None, stats=None, T=None, H=None, row_stride=1, row_offset=0):
    _lib.require_device()
    T = x.shape[0] if T is None else T
    H = x.shape[1] if H is None else H
    y = y_bf16 if y_bf16 is not None else y_f32
    call("srfrd_layernorm_fwd", _p(x), x.stride(0), _p(w), _p(b), float(eps), _p(y_bf16), _p(y_f32), y.stride(0),
         _p(stats), T, H, row_stride, row_offset, _stream())


def layernorm_bwd(dy, x, stats, w, dx, dw, db, add=None, row_ids=None, H=None):
    T = x.shape[0]
    H = x.shape[1] if H is None else H          # valid (LayerNorm) width; the row pitch may be padded
    dyb = dy if dy.dtype == bf16 else None
    dyf = dy if dy.dtype == torch.float32 else None
    call("srfrd_layernorm_bwd", _p(dyb), _p(dyf), dy.stride(0), _p(x), x.stride(0), _p(stats), _p(w), _p(add),
         0 if add is None else add.stride(0), _p(row_ids), _p(dx), dx.stride(0), _p(dw), _p(db), T, H, _stream())


def gemm_tn(A, B, out_bf16=None, out_f32=None, bias=None, residual=None, gate=None, row_ids=None, relu=False,
            drop_p=0.0, drop_seed=0, drop_stream=0, drop_step=None, M=None, ln_out=None, ln_w=None, ln_b=None, ln_eps=0.0,
            ln_stats=None):
    """out[M,N] = epilogue(A[M,K] @ B[N,K]^T); with ln_out also ln_out = LayerNorm(out) * ln_w + ln_b (+ ln_stats)."""
    _lib.require_device()
    M = A.shape[0] if M is None else M
    K = A.shape[1]
    N = B.shape[0]
    out = out_bf16 if out_bf16 is not None else out_f32
    ep = GemmEpilogue(_p(bias), _p(residual), _p(gate), _p(row_ids), _p(out_bf16), _p(out_f32),
                      0 if residual is None else residual.stride(0), 0 if gate is None else gate.stride(0),
                      out.stride(0), int(relu), float(drop_p), int(drop_stream), int(drop_seed), _p(drop_step),
                      _p(ln_out), _p(ln_w), _p(ln_b), _p(ln_stats), 0 if ln_out is None else ln_out.stride(0), float(ln_eps))
    call("srfrd_gemm_tn", _p(A), A.stride(0), _p(B), B.stride(0), M, N, K, C.byref(ep), _stream())


def gemm_wgrad(dY, X, dW, dbias=None, Mo=None, No=None):
    """dW[Mo,No] += dY[T,Mo]^T @ X[T,No]  (dW fp32, atomically accumulated); dbias[Mo] += column sums of dY.
    Mo / No default to the operand widths; pass the true widths when the operands carry zero padding columns."""
    T = dY.shape[0]
    Mo = dY.shape[1] if Mo is None else Mo
    No = X.shape[1] if No is None else No
    call("srfrd_gemm_wgrad", _p(dY), dY.stride(0), _p(X), X.stride(0), T, Mo, No, _p(dW), dW.stride(0), _p(dbias),
         _stream())


def gemm_ref(A, B, Cout, a_mn_major=False, b_mn_major=False):
    _lib.require_device()
    M, N = Cout.shape
    K = A.shape[0] if a_mn_major else A.shape[1]
    call("srfrd_gemm_ref", _p(A), A.stride(0), _p(B), B.stride(0), _p(Cout), Cout.stride(0), M, N, K,
         int(a_mn_major), int(b_mn_major), _stream())


def colsum(X, out, M=None, N=None, ld=None):
    M = X.shape[0] if M is None else M
    N = X.shape[1] if N is None else N
    ld = X.stride(0) if ld is None else ld
    call("srfrd_colsum", _p(X), M, N, ld, _p(out), _stream())


def add_segments(src, n, seg_in, seg_out, out):
    call("srfrd_add_segments", _p(src), n, seg_in, seg_out, _p(out), _stream())


def dropout_apply(x, out, N, drop_p, seed, stream_id, drop_step=None):
    call("srfrd_dropout_apply", _p(x), x.stride(0), _p(out), out.stride(0), x.shape[0], N, float(drop_p), int(seed),
         int(stream_id), _p(drop_step), _stream())


def cast_weights(descs_dev, n):
    call("srfrd_cast_weights", _p(descs_dev), n, _stream())


def make_cast_table(entries, device):
    """entries: list of (src fp32 2-D view, dst bf16 or None, dst_t bf16 or None) -> uint8 device tensor.
    A fp32 ``dst`` makes the entry a plain fp32 copy (zero-padded shadows of bias / LayerNorm vectors)."""
    arr = (CastDesc * len(entries))()
    for i, (src, dst, dst_t) in enumerate(entries):
        is_f32 = int(dst is not None and dst.dtype == torch.float32)
        arr[i] = CastDesc(src.data_ptr(), src.stride(0), _p(dst), 0 if dst is None else dst.stride(0), _p(dst_t),
                          0 if dst_t is None else dst_t.stride(0), src.shape[0], src.shape[1], is_f32)
    raw = bytes(arr)
    host = torch.frombuffer(bytearray(raw), dtype=torch.uint8)
    return host.to(device), len(entries)


def f32_to_bf16_split(src, hi, lo=None, row_index=None):
    _lib.require_device()
    rows = src.shape[0] if row_index is None else row_index.numel()
    cols = src.shape[1]
    call("srfrd_f32_to_bf16_split", _p(src), src.stride(0), _p(row_index), _p(hi), _p(lo), rows, cols, hi.stride(0),
         _stream())


def attention_fwd(q, k, v, o, B, L, H, heads, drop_p=0.0, seed=0, stream_id=0, drop_step=None, stats=None):
    """stats: optional fp32 (B*L*heads, 4) row statistics, required later by attention_bwd when L > 128."""
    _lib.require_device()
    call("srfrd_attention_fwd", _p(q), q.stride(0), _p(k), _p(v), k.stride(0), _p(o), o.stride(0), _p(stats), B, L, H, heads,
         float(drop_p), int(seed), int(stream_id), _p(drop_step), _stream())


def attention_bwd(dout, q, k, v, dq, dk, dv, B, L, H, heads, drop_p=0.0, seed=0, stream_id=0, drop_step=None, o=None,
                  stats=None):
    call("srfrd_attention_bwd", _p(dout), dout.stride(0), _p(q), q.stride(0), _p(k), _p(v), k.stride(0), _p(o),
         0 if o is None else o.stride(0), _p(stats), _p(dq), dq.stride(0), _p(dk), _p(dv), dk.stride(0), B, L, H, heads,
         float(drop_p), int(seed), int(stream_id), _p(drop_step), _stream())


def score_fwd(h, item_table, fake_table, pos, neg, prs, nrs, zp, zn):
    _lib.require_device()
    T = pos.numel()
    D = item_table.shape[1]
    F = 0 if fake_table is None else fake_table.shape[1]
    call("srfrd_score_fwd", _p(h), h.stride(0), _p(item_table), _p(fake_table), _p(pos), _p(neg), _p(prs), _p(nrs), T,
         D, F, _p(zp), _p(zn), _stream())


def score_bwd(h, item_table, fake_table, pos, neg, prs, nrs, dzp, dzn, dh, d_item, d_fake):
    T = pos.numel()
    D = item_table.shape[1]
    F = 0 if fake_table is None else fake_table.shape[1]
    call("srfrd_score_bwd", _p(h), h.stride(0), _p(item_table), _p(fake_table), _p(pos), _p(neg), _p(prs), _p(nrs),
         _p(dzp), _p(dzn), T, D, F, _p(dh), dh.stride(0), _p(d_item), _p(d_fake), _stream())


def score_loss_fused(h, item_table, fake_table, pos, neg, prs, nrs, w_pos, w_neg, norm, loss_acc, dh, d_item, d_fake,
                     zp=None, zn=None):
    T = pos.numel()
    D = item_table.shape[1]
    F = 0 if fake_table is None else fake_table.shape[1]
    call("srfrd_score_loss_fused", _p(h), h.stride(0), _p(item_table), _p(fake_table), _p(pos), _p(neg), _p(prs),
         _p(nrs), _p(w_pos), _p(w_neg), _p(norm), T, D, F, _p(zp), _p(zn), _p(loss_acc), _p(dh),
         0 if dh is None else dh.stride(0), _p(d_item), _p(d_fake), _stream())


def weight_sums(pos, w_pos, w_neg, out2):
    _lib.require_device()
    call("srfrd_weight_sums", _p(pos), _p(w_pos), _p(w_neg), pos.numel(), _p(out2), _stream())


def loss_finalize(acc2, norm2, loss):
    call("srfrd_loss_finalize", _p(acc2), _p(norm2), _p(loss), _stream())


def adam_tick(state3, beta1, beta2):
    call("srfrd_adam_tick", _p(state3), float(beta1), float(beta2), _stream())


def adam_step(p, g, m, v, lr, beta1, beta2, eps, state3, zero_grad=True):
    _lib.require_device()
    call("srfrd_adam_step", _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2), float(eps),
         _p(state3), int(zero_grad), _stream())


def adam_step_fused(p, g, m, v, lr, beta1, beta2, eps, state8, zero_grad=True, acc2=None, norm2=None, loss=None,
                    l2: Optional["ParamL2"] = None):
    """adam_tick + adam_step + loss_finalize in one launch (state8: 8 floats, see the header).  With ``l2`` (after its
    ``launch``) the gradient gains the l2_emb term and the loss its value."""
    _lib.require_device()
    call("srfrd_adam_step_fused", _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2), float(eps),
         _p(state8), int(zero_grad), _p(acc2), _p(norm2), _p(loss), _stream(), *_l2_args(l2))


class ParamL2:
    """The l2_emb regulariser's per-tensor norms over a flat parameter buffer (srfrd_param_l2): ``segments`` = the
    (offset, numel) of every parameter tensor in the buffer.  ``launch(p)`` writes ``coef[t] = l2 / ||p_t||`` (0 for a
    zero tensor) and ``reg[0] = l2 * sum_t ||p_t||``, deterministically; the Adam entry points take the object to add
    ``coef[t] * p`` to the gradient and ``reg`` to the loss."""

    def __init__(self, segments, l2: float, device):
        host = (C.c_int64 * (2 * len(segments)))(*[int(x) for s in segments for x in s])
        n_chunks = C.c_int64(0)
        call("srfrd_param_l2_plan", host, len(segments), C.byref(n_chunks))
        self.n_seg, self.n_chunks, self.l2 = len(segments), int(n_chunks.value), float(l2)
        self.seg = torch.tensor([int(x) for s in segments for x in s], dtype=torch.int64).to(device)
        self.coef = torch.zeros(self.n_seg, dtype=torch.float32, device=device)
        self.reg = torch.zeros(1, dtype=torch.float32, device=device)
        self.ws = torch.zeros(self.n_chunks + 1, dtype=torch.float64, device=device)

    def launch(self, p: torch.Tensor):
        _lib.require_device()
        _chk(p, torch.float32, "p")
        call("srfrd_param_l2", _p(p), _p(self.seg), self.n_seg, self.n_chunks, self.l2, _p(self.coef), _p(self.reg),
             _p(self.ws), _stream())


def _l2_args(l2: Optional[ParamL2]):
    return (None, 0, None, None) if l2 is None else (_p(l2.seg), l2.n_seg, _p(l2.coef), _p(l2.reg))


def catalogue_topk_plan(U, n_rows, row_lo, D, n_split, k=10) -> int:
    """Chunk count of the (U, chunks, max(k, 10)) list buffers; raises if k is outside 1..catalogue_topk_kmax(D, n_split)."""
    out = C.c_int(0)
    call("srfrd_catalogue_topk_plan", U, n_rows, row_lo, D, n_split, C.byref(out), int(k))
    return out.value


def catalogue_topk_kmax(D, n_split) -> int:
    """Largest k catalogue_topk serves for this table width and split (host arithmetic, no launch)."""
    out = C.c_int(0)
    call("srfrd_catalogue_topk_kmax", D, n_split, C.byref(out))
    return out.value


def catalogue_topk(feats, U, u_pad, n_split, table, row_lo, id_base, chunks, part_scores, part_ids, packed=None, k=10):
    """part_scores / part_ids: (U, chunks, L) with L = max(k, 10).  packed: optional (U, 2L) fp32 -- each user's final
    local list as L scores + L int32 ids (all-gather send buffer)."""
    _lib.require_device()
    D = table.shape[1]
    call("srfrd_catalogue_topk", _p(feats), U, u_pad, n_split, _p(table), table.shape[0], row_lo, id_base, D,
         feats.stride(0), table.stride(0), chunks, _p(part_scores), _p(part_ids), _p(packed), _stream(), int(k))


def catalogue_rank(feats, U, u_pad, n_split, table, row_lo, id_base, target_rows, target_ids, rank_out,
                   target_scores=None):
    """rank_out (U,) int32 <- items of table rows [row_lo, n_rows) (global id id_base + row) ahead of each user's target
    under (score desc, id asc).  target_rows: (U, D) bf16 rows of the targets; target_ids: (U,) int64 global ids;
    target_scores: optional (U,) fp32 output of the targets' own scores."""
    _lib.require_device()
    D = table.shape[1]
    call("srfrd_catalogue_rank", _p(feats), U, u_pad, n_split, _p(table), table.shape[0], row_lo, id_base, D,
         feats.stride(0), table.stride(0), _p(target_rows), target_rows.stride(0), _p(target_ids), _p(target_scores),
         _p(rank_out), _stream())


def merge_topk_packed(packed, U, nlists, k, out_scores, out_ids):
    _lib.require_device()
    call("srfrd_merge_topk_packed", _p(packed), U, nlists, k, _p(out_scores), _p(out_ids), _stream())


def merge_topk(scores, ids, U, nlists, k, out_scores, out_ids):
    _lib.require_device()
    call("srfrd_merge_topk", _p(scores), _p(ids), U, nlists, k, _p(out_scores), _p(out_ids), _stream())


def sample_batch(offsets, items, labels, p_fake, eligible, itemnum, B, L, policy, seed, step, out, w_pos=None):
    """out: dict with int64 (B, L) tensors seq, rsq, pos, prs, neg, nrs and int64 (B,) users."""
    _lib.require_device()
    call("srfrd_sample_batch", _p(offsets), _p(items), _p(labels), _p(p_fake), _p(eligible), eligible.numel(), int(itemnum),
         B, L, int(policy), int(seed), _p(step), _p(out.get("users")), _p(out["seq"]), _p(out["rsq"]), _p(out["pos"]),
         _p(out["prs"]), _p(out["neg"]), _p(out["nrs"]), _p(w_pos), _stream())


def sample_candidates(offsets, items, users0, target, itemnum, C, seed, cand):
    """cand (U, C) int64: column 0 = the held-out item, the rest uniform ids outside the user's train row."""
    _lib.require_device()
    call("srfrd_sample_candidates", _p(offsets), _p(items), _p(users0), _p(target), users0.numel(), int(itemnum), int(C),
         int(seed), _p(cand), _stream())


def candidate_rank(feats, item_table, cand, D, fake_table=None, user_label=None, logits=None, rank=None, err_flag=None):
    _lib.require_device()
    _chk(feats, torch.float32, "feats"); _chk(item_table, torch.float32, "item_table"); _chk(cand, torch.int64, "cand")
    U, Cn = cand.shape
    F = 0 if fake_table is None else fake_table.shape[1]
    call("srfrd_candidate_rank", _p(feats), feats.stride(0), _p(item_table), item_table.shape[0], int(D), _p(cand), U, Cn,
         _p(fake_table), F, _p(user_label), _p(logits), 0 if logits is None else logits.stride(0), _p(rank), _p(err_flag),
         _stream())


def add_user_term(logits, feats_tail, fake_table, label):
    _lib.require_device()
    U, I = logits.shape
    call("srfrd_add_user_term", _p(logits), logits.stride(0), U, I, _p(feats_tail), feats_tail.stride(0), _p(fake_table),
         _p(label), fake_table.shape[1], _stream())


# ---------------------------------------------------------------------------------------------------- packed token layout
class PackedPlan:
    """Device buffers of the packed token layout for up to B sequences of length L (srfrd_pack_t).  `build` runs the
    three plan kernels; afterwards `rows[0]` holds the dynamic row count every packed / row-limited kernel reads."""

    def __init__(self, B: int, L: int, device):
        self.B, self.L = B, L
        self.cap = (B * (L + 1) + 127) // 128 * 128
        i32 = lambda n: torch.zeros(n, dtype=torch.int32, device=device)
        self.rows, self.cnt, self.seq_first = i32(4), i32(B), i32(B + 1)
        self.tok_row, self.row_tok = i32(B * L), i32(self.cap)
        self.row_ids = torch.zeros(self.cap, dtype=torch.int64, device=device)
        self.row_info = i32(4 * self.cap)
        self.tile_row0, self.last_row = i32(B + 130), i32(B)
        self.desc = PackDesc(_p(self.rows), _p(self.cnt), _p(self.seq_first), _p(self.tok_row), _p(self.row_tok),
                             _p(self.row_ids), _p(self.row_info), _p(self.tile_row0), _p(self.last_row), self.cap)

    def build(self, seq, keep=None):
        _lib.require_device()
        B, L = seq.shape
        assert (B, L) == (self.B, self.L)
        _chk(seq, torch.int64, "seq")
        call("srfrd_pack_plan", _p(seq), _p(keep), B, L, C.byref(self.desc), _stream())


@contextmanager
def row_limit(rows_dev):
    """Within the block, gemm_tn / gemm_wgrad / layernorm_fwd / layernorm_bwd / dropout_apply process
    min(their row argument, rows_dev[0]) rows (rows_dev: int32 device tensor, read when the kernel runs)."""
    call("srfrd_set_row_limit", _p(rows_dev))
    try:
        yield
    finally:
        call("srfrd_set_row_limit", None)


class LiveTiles:
    """Live query tiles of the hybrid packed layout (srfrd_attention_live_items): which 128-position query tiles of the dense
    (B, L) attention tensors hold a kept token.  `build(plan, heads)` after the pack plan; `with live.active():` around the
    maxlen > 128 attention calls makes them skip the dead tiles."""

    def __init__(self, B: int, L: int, heads: int, device):
        nq = (L + 127) // 128
        self.B, self.L, self.heads = B, L, heads
        self.q_lo = torch.zeros(B, dtype=torch.int32, device=device)
        self.items = torch.zeros(B * heads * nq, dtype=torch.int32, device=device)
        self.n_live = torch.zeros(1, dtype=torch.int32, device=device)

    def build(self, plan: "PackedPlan"):
        _lib.require_device()
        assert (plan.B, plan.L) == (self.B, self.L)
        self.tok_row = plan.tok_row
        call("srfrd_attention_live_items", _p(plan.tok_row), self.B, self.L, self.heads, _p(self.q_lo), _p(self.items),
             _p(self.n_live), _stream())

    @contextmanager
    def active(self):
        call("srfrd_set_attention_live", _p(self.q_lo), _p(self.items), _p(self.n_live), _p(self.tok_row))
        try:
            yield
        finally:
            call("srfrd_set_attention_live", None, None, None, None)


def attention_packed_supported(L: int, H: int, heads: int) -> bool:
    return bool(_lib.load().srfrd_attention_packed_supported(int(L), int(H), int(heads)))


def embed_ln_fwd_packed(item_table, pos_table, aux_table, mode, seq, aux_ids, item_scale, ln_w, ln_b, eps, x0_bf16, q_bf16,
                        stats, plan: PackedPlan, drop_p=0.0, drop_seed=0, drop_stream=0, drop_step=None):
    _lib.require_device()
    B, L = seq.shape
    D = item_table.shape[1]
    F = aux_table.shape[1] if (aux_table is not None and mode == 1) else 0
    call("srfrd_embed_ln_fwd_packed", _p(item_table), item_table.shape[0], D, _p(pos_table), _p(aux_table),
         0 if aux_table is None else aux_table.shape[0], F, mode, _p(seq), _p(aux_ids), B, L, float(item_scale), _p(ln_w),
         _p(ln_b), float(eps), _p(x0_bf16), _p(q_bf16), _p(stats), x0_bf16.stride(0), float(drop_p), int(drop_seed),
         int(drop_stream), _p(drop_step), _p(plan.row_tok), _p(plan.rows), plan.cap, _stream())


def layernorm_fwd_rows(x, w, b, eps, y_f32, row_index, n, H):
    _lib.require_device()
    call("srfrd_layernorm_fwd_rows", _p(x), x.stride(0), _p(w), _p(b), float(eps), _p(y_f32), y_f32.stride(0), _p(row_index),
         n, H, _stream())


def attention_packed_oproj_supported(L: int, H: int, heads: int) -> int:
    """Bit 0: attention_fwd_packed can take the out-projection (wo=...); bit 1: attention_bwd_packed can (dr=...)."""
    return int(_lib.load().srfrd_attention_packed_oproj_supported(int(L), int(H), int(heads)))


def attention_fwd_packed(q, k, v, o, plan: PackedPlan, L, H, heads, drop_p=0.0, seed=0, stream_id=0, drop_step=None,
                         wo=None, bias=None, residual=None, r=None, y=None, ln_w=None, ln_b=None, ln_eps=0.0, ln_stats=None):
    """With wo: also r = o @ wo^T + bias + residual, y = LayerNorm(r) (ln_w, ln_b, ln_eps; (mean, rstd) -> ln_stats),
    the rows gemm_tn(o, wo, out_bf16=r, bias=bias, residual=residual, ln_out=y, ...) would write."""
    _lib.require_device()
    st = lambda t: 0 if t is None else t.stride(0)
    call("srfrd_attention_fwd_packed", _p(q), q.stride(0), _p(k), _p(v), k.stride(0), _p(o), o.stride(0), C.byref(plan.desc),
         L, H, heads, float(drop_p), int(seed), int(stream_id), _p(drop_step), _stream(), _p(wo), st(wo), _p(bias),
         _p(residual), st(residual), _p(ln_w), _p(ln_b), float(ln_eps), _p(ln_stats), _p(r), st(r), _p(y), st(y))


def attention_bwd_packed(dout, q, k, v, dq, dk, dv, plan: PackedPlan, L, H, heads, drop_p=0.0, seed=0, stream_id=0,
                         drop_step=None, dr=None, woT=None):
    """With dr (dout None): dout = dr @ woT^T is computed inside the kernel (what gemm_tn(dr, woT) would write)."""
    st = lambda t: 0 if t is None else t.stride(0)
    call("srfrd_attention_bwd_packed", _p(dout), st(dout), _p(q), q.stride(0), _p(k), _p(v), k.stride(0), _p(dq),
         dq.stride(0), _p(dk), _p(dv), dk.stride(0), C.byref(plan.desc), L, H, heads, float(drop_p), int(seed),
         int(stream_id), _p(drop_step), _stream(), _p(dr), st(dr), _p(woT), st(woT))


def score_loss_fused_packed(h, item_table, fake_table, pos, neg, prs, nrs, w_pos, w_neg, norm, loss_acc, dh, d_item, d_fake,
                            plan: PackedPlan):
    D = item_table.shape[1]
    F = 0 if fake_table is None else fake_table.shape[1]
    call("srfrd_score_loss_fused_packed", _p(h), h.stride(0), _p(item_table), _p(fake_table), _p(pos), _p(neg), _p(prs),
         _p(nrs), _p(w_pos), _p(w_neg), _p(norm), D, F, _p(loss_acc), _p(dh), dh.stride(0), _p(d_item), _p(d_fake),
         _p(plan.row_tok), _p(plan.rows), plan.cap, _stream())


def embed_bwd_packed(dx0, seq, aux_ids, plan: PackedPlan, D, F, mode, item_scale, d_item, d_aux, d_pos):
    B, L = seq.shape
    call("srfrd_embed_bwd_packed", _p(dx0), dx0.stride(0), _p(seq), _p(aux_ids), _p(plan.row_tok), _p(plan.rows), plan.cap,
         L, D, F, mode, float(item_scale), _p(d_item), _p(d_aux), _p(d_pos), _stream())


def dp_adam_step(grad_ptrs_dev: int, param_ptrs_dev: int, signal_ptrs_dev: int, rank, world, n, m, v, lr, beta1, beta2, eps,
                 state8, norm2, local4, l2: Optional[ParamL2] = None):
    """Reduce-scatter + Adam + all-gather over peer memory in one launch (csrc/dp_adam.cu); the *_ptrs_dev arguments are
    device addresses of arrays of `world` peer-mapped pointers (symmetric memory handles' buffer_ptrs_dev).  ``l2``: the
    l2_emb term of adam_step_fused, added once to the reduced gradient."""
    _lib.require_device()
    call("srfrd_dp_adam_step", grad_ptrs_dev, param_ptrs_dev, signal_ptrs_dev, int(rank), int(world), int(n), _p(m), _p(v),
         float(lr), float(beta1), float(beta2), float(eps), _p(state8), _p(norm2), _p(local4), _stream(), *_l2_args(l2))


def _parts(parts):
    arr = (RepackPart * len(parts))()
    for i, (src, dst, W, mode) in enumerate(parts):
        arr[i] = RepackPart(_p(src), src.stride(0), _p(dst), dst.stride(0), int(W), int(mode))
    return arr


def unpack_rows(parts, plan: PackedPlan):
    """parts: [(packed src, dense dst, columns, mode)]; mode 0: pad slots take the representative row, 1: zeros."""
    _lib.require_device()
    arr = _parts(parts)
    call("srfrd_unpack_rows", arr, len(parts), C.byref(plan.desc), plan.B, plan.L, _stream())


def pack_rows(parts, plan: PackedPlan):
    """parts: [(dense src, packed dst, columns, mode)]; mode 0: representative rows zero, 1: sum of the dropped pad slots."""
    _lib.require_device()
    arr = _parts(parts)
    call("srfrd_pack_rows", arr, len(parts), C.byref(plan.desc), plan.B, plan.L, _stream())


def mlp2_tn(A, W1, W2, mid_out, out, bias1=None, bias2=None, gate=None, relu1=False, drop1_p=0.0, drop2_p=0.0, drop1_stream=0,
            drop2_stream=0, drop_seed=0, drop_step=None, residual=None, residual_is_a=False, row_ids=None, ln_out=None,
            ln_w=None, ln_b=None, ln_stats=None, ln_eps=0.0, M=None):
    """out = stage2(stage1(A W1^T) W2^T) in one launch (csrc/ffn.cu); W1, W2 square (N, N) bf16, N <= 128."""
    _lib.require_device()
    M = A.shape[0] if M is None else M
    N = W1.shape[0]
    ep = Mlp2Epilogue(_p(bias1), _p(bias2), _p(gate), 0 if gate is None else gate.stride(0), int(relu1), float(drop1_p),
                      float(drop2_p), int(drop1_stream), int(drop2_stream), int(drop_seed), _p(drop_step), _p(residual),
                      0 if residual is None else residual.stride(0), int(residual_is_a), _p(row_ids), _p(mid_out),
                      mid_out.stride(0), _p(out), out.stride(0), _p(ln_out), 0 if ln_out is None else ln_out.stride(0),
                      _p(ln_w), _p(ln_b), _p(ln_stats), float(ln_eps))
    call("srfrd_mlp2_tn", _p(A), A.stride(0), _p(W1), W1.stride(0), _p(W2), W2.stride(0), M, N, C.byref(ep), _stream())


def catalogue_ce_plan(Dp: int):
    """(shared-memory bytes, ring stages, TMEM columns) of the cross-entropy kernels for padded width Dp (host only);
    raises for a Dp they cannot serve (not a multiple of 16, or above 256)."""
    smem, stages, tmem = C.c_int64(0), C.c_int(0), C.c_int(0)
    call("srfrd_catalogue_ce_plan", int(Dp), C.byref(smem), C.byref(stages), C.byref(tmem))
    return int(smem.value), int(stages.value), int(tmem.value)


def _ce_rows(h, plan):
    return (None, None, h.shape[0]) if plan is None else (plan.row_tok, plan.rows, plan.cap)


def catalogue_ce_fwd(h, table, pos, w_pos, lse, loss_acc, plan: Optional[PackedPlan] = None):
    """Pass 1 of the full-catalogue cross-entropy: lse (fp32, one per h row) and loss_acc[0] += sum w (lse - z_pos).
    h: (rows, Dp) bf16; table: (N + 1, Dp) bf16; pos / w_pos indexed by dense token (plan: packed h rows)."""
    _lib.require_device()
    _chk(h, bf16, "h"); _chk(table, bf16, "table"); _chk(pos, torch.int64, "pos")
    row_tok, rows, cap = _ce_rows(h, plan)
    call("srfrd_catalogue_ce_fwd", _p(h), h.stride(0), _p(table), table.stride(0), table.shape[0] - 1, table.shape[1],
         _p(pos), _p(w_pos), _p(row_tok), _p(rows), cap, _p(lse), _p(loss_acc), _stream())


def catalogue_ce_bwd(h, table, pos, w_pos, norm, lse, dh, d_item, D, plan: Optional[PackedPlan] = None):
    """Passes 2 and 3: dh (fp32 rows, first D columns written) and d_item ((N + 1, D) fp32, added to); either may be
    None.  norm[0] is the loss normaliser (sum of the weights), read on the device."""
    _lib.require_device()
    _chk(h, bf16, "h"); _chk(table, bf16, "table"); _chk(pos, torch.int64, "pos")
    row_tok, rows, cap = _ce_rows(h, plan)
    call("srfrd_catalogue_ce_bwd", _p(h), h.stride(0), _p(table), table.stride(0), table.shape[0] - 1, table.shape[1],
         int(D), _p(pos), _p(w_pos), _p(norm), _p(row_tok), _p(rows), cap, _p(lse), _p(dh),
         0 if dh is None else dh.stride(0), _p(d_item), 0 if d_item is None else d_item.stride(0), _stream())
