"""Evaluation on the hot path: full-catalogue top-k, 1 <= k <= 64 (tcgen05 scoring fused with a streaming top-k), the
exact full-catalogue rank of each user's held-out item (HR@k / NDCG@k at any cutoff, MRR) and the reference's sampled-101
protocol (utils.py:544-602), all batched and all on the library's own kernels.

Full-catalogue scoring is the reference's ``predict(user_ids, seq, rsq, label)`` called with
``label = arange(1, itemnum + 1)`` followed by ``(-logits).argsort().argsort()`` (utils.py:589-591),
i.e. a ranking by (score desc, item id asc) -- except that the (U, N) logits are never written to HBM.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import ops

bf16 = torch.bfloat16
TK = 10          # list length of the top-10 kernels; a smaller k is the prefix of their lists
KMAX = 64        # longest top-k (the per-row lists of the k-list kernels live in shared memory)


def list_len(k: int) -> int:
    """Length of every candidate list for a top-k: max(k, 10).  k outside 1..KMAX is refused before any launch."""
    if not 1 <= int(k) <= KMAX:
        raise RuntimeError(f"catalogue_topk: k must be in 1..{KMAX} (got {k})")
    return max(int(k), TK)


class CatalogueIndex:
    """bf16 copy of (a row shard of) the item table, resident on the device for scoring.

    table_f32 : (n_rows_local, D) fp32 rows of the item table owned by this rank
    id_base   : global item id of local row 0 (0 on the rank that owns the pad row)
    Item id 0 is the pad row and is never a candidate (utils.py:575-583 draws candidates from 1..itemnum).
    """

    def __init__(self, table_f32: torch.Tensor, id_base: int = 0):
        self.id_base = int(id_base)
        self.n_rows, self.D = table_f32.shape
        self.Dp = (self.D + 15) // 16 * 16          # zero-padded K (tcgen05 K step / 16-byte rows)
        self.row_lo = 1 if self.id_base == 0 else 0
        self.table = torch.zeros(self.n_rows, self.Dp, dtype=bf16, device=table_f32.device)
        if self.n_rows > 0:                           # (more ranks than table rows: an empty shard is legal)
            ops.f32_to_bf16_split(table_f32.contiguous(), self.table[:, :self.D], None)

    @staticmethod
    def shard_bounds(n_rows_total: int, rank: int, world: int) -> Tuple[int, int]:
        """Row-sharding of the (N+1)-row table: rank g owns rows [g*S, min((g+1)*S, N+1)), S = ceil((N+1)/G)."""
        S = (n_rows_total + world - 1) // world
        return min(rank * S, n_rows_total), min((rank + 1) * S, n_rows_total)


def _split_feats(feats_f32: torch.Tensor, Dp: int, n_split: int):
    U, D = feats_f32.shape
    dev = feats_f32.device
    u_pad = (U + 255) // 256 * 256          # whole user groups (2 tiles of 128) per split
    fb = torch.zeros(n_split * u_pad, Dp, dtype=bf16, device=dev)
    f = feats_f32.contiguous()
    if n_split == 1:
        ops.f32_to_bf16_split(f, fb[:U, :D], None)
    elif n_split == 2:
        ops.f32_to_bf16_split(f, fb[:U, :D], fb[u_pad:u_pad + U, :D])
    else:
        # three-way split: hi, mid, lo  (f = hi + mid + lo to ~24 mantissa bits)
        hi, mid = fb[:U, :D], fb[u_pad:u_pad + U, :D]
        ops.f32_to_bf16_split(f, hi, mid)
        rest = f - hi.float() - mid.float()
        ops.f32_to_bf16_split(rest.contiguous(), fb[2 * u_pad:2 * u_pad + U, :D], None)
    return fb, u_pad


def _local_lists(feats_f32: torch.Tensor, index: CatalogueIndex, n_split: int, packed: Optional[torch.Tensor],
                 k: int = TK):
    """Run K8 on the local shard; returns the (U, chunks, L) list buffers (L = max(k, 10)) whose slot 0 holds each
    user's exact local top-L (sorted, global ids) and, when `packed` is given, the same list in the all-gather wire
    format."""
    U = feats_f32.shape[0]
    dev = feats_f32.device
    L = list_len(k)
    chunks = ops.catalogue_topk_plan(U, index.n_rows, index.row_lo, index.Dp, n_split, k)   # refuses k above the limit
    fb, u_pad = _split_feats(feats_f32, index.Dp, n_split)
    ps = torch.empty(U, chunks, L, dtype=torch.float32, device=dev)
    pi = torch.empty(U, chunks, L, dtype=torch.int32, device=dev)
    ops.catalogue_topk(fb, U, u_pad, n_split, index.table, index.row_lo, index.id_base, chunks, ps, pi, packed, k=k)
    return ps, pi, chunks


def local_topk(feats_f32: torch.Tensor, index: CatalogueIndex, n_split: int = 1, k: int = TK):
    """Per-user top-k of feats (U, D) against the local shard -> (scores (U,k) fp32, ids (U,k) int64); (-inf, -1) past
    the last candidate."""
    U = feats_f32.shape[0]
    dev = feats_f32.device
    list_len(k)
    if index.n_rows <= index.row_lo:                      # empty shard
        return (torch.full((U, k), float("-inf"), device=dev), torch.full((U, k), -1, dtype=torch.int64, device=dev))
    ps, pi, chunks = _local_lists(feats_f32, index, n_split, None, k)
    out_s = torch.empty(U, k, dtype=torch.float32, device=dev)
    out_i = torch.empty(U, k, dtype=torch.int64, device=dev)
    ops.merge_topk(ps, pi, U, chunks, k, out_s, out_i)
    return out_s, out_i


def merge_shards(scores: torch.Tensor, ids: torch.Tensor, k: int = TK):
    """scores/ids: (U, G, L) candidate lists gathered from G shards, L = max(k, 10), each sorted as local_topk returns
    them -> global (U, k)."""
    U, G, W = scores.shape
    if W != list_len(k):
        raise ValueError(f"merge_shards: top-{k} needs lists of {list_len(k)} entries, got {W}")
    out_s = torch.empty(U, k, dtype=torch.float32, device=scores.device)
    out_i = torch.empty(U, k, dtype=torch.int64, device=scores.device)
    ops.merge_topk(scores.contiguous(), ids.to(torch.int32).contiguous(), U, G, k, out_s, out_i)
    return out_s, out_i


def sharded_topk(feats_f32: torch.Tensor, index: CatalogueIndex, process_group=None, n_split: int = 1, k: int = TK):
    """Row-sharded catalogue scoring: local top-k, ONE all-gather of the packed lists (L fp32 scores + L int32 global
    ids, L = max(k, 10): 8L B / user / rank, written in wire format by the scoring kernel itself), merge straight out of
    the gathered buffer -> identical (U, k) on every rank.  No int64 on the wire, no permute / contiguous copies."""
    from . import parallel
    if process_group is None or torch.distributed.get_world_size(process_group) == 1:
        return local_topk(feats_f32, index, n_split, k)
    G = torch.distributed.get_world_size(process_group)
    U = feats_f32.shape[0]
    dev = feats_f32.device
    L = list_len(k)
    packed = torch.empty(U, 2 * L, dtype=torch.float32, device=dev)
    if index.n_rows <= index.row_lo:                      # empty shard: ids -1 (bit pattern of int32 -1 in every id word)
        packed.view(torch.int32).fill_(-1)
    else:
        _local_lists(feats_f32, index, n_split, packed, k)
    gathered = parallel.allgather_packed_topk(packed, process_group)        # (G, U, 2L)
    out_s = torch.empty(U, k, dtype=torch.float32, device=dev)
    out_i = torch.empty(U, k, dtype=torch.int64, device=dev)
    ops.merge_topk_packed(gathered, U, G, k, out_s, out_i)
    return out_s, out_i


UNIT_FORM_MAX = 256   # largest n_split * D the unit-form scoring kernel serves; only that form computes ranks


def _targets(target, U: int, N: int, device) -> torch.Tensor:
    """(U,) int64 item ids on `device`; ValueError unless there are U of them, each in 1..N."""
    t = torch.as_tensor(target).reshape(-1)
    if t.numel() != U:
        raise ValueError(f"catalogue_ranks: {t.numel()} targets for {U} users")
    t = t.to(device=device, dtype=torch.int64)
    if U and (int(t.min()) < 1 or int(t.max()) > N):
        raise ValueError(f"catalogue_ranks: targets must be item ids in 1..{N} (got {int(t.min())}..{int(t.max())})")
    return t


def catalogue_ranks(feats_f32: torch.Tensor, index: CatalogueIndex, table_f32: torch.Tensor, target,
                    process_group=None, n_split: int = 1) -> torch.Tensor:
    """Exact full-catalogue rank of each user's held-out item -> int64 (U,): the number of items 1..N ahead of target[u]
    under (score desc, id asc), i.e. the reference's (-logits).argsort().argsort()[0] (utils.py:589-591) with every item
    a candidate.  Scores as local_topk ranks them (bf16 operands, fp32 accumulation, n_split feature splits).

    index     : the local (shard of the) table the count runs over; an empty shard contributes 0 without a launch
    table_f32 : the full (N+1, D) fp32 item table, replicated like the model parameters: the targets' rows are gathered
                from it with the conversion CatalogueIndex uses, so every rank scores the target with the same bits
    With a process group the per-shard counts are summed by ONE int32 all-reduce (4 B per user)."""
    from . import parallel
    U = feats_f32.shape[0]
    dev = feats_f32.device
    if table_f32.shape[1] != index.D:
        raise ValueError(f"catalogue_ranks: table width {table_f32.shape[1]} != index width {index.D}")
    tgt = _targets(target, U, table_f32.shape[0] - 1, dev)
    if n_split * index.Dp > UNIT_FORM_MAX:
        raise RuntimeError(f"catalogue_rank: needs the unit form (n_split * D <= {UNIT_FORM_MAX}); D={index.Dp} with "
                           f"n_split={n_split} runs the tile form")
    rank = torch.zeros(U, dtype=torch.int32, device=dev)
    if U and index.n_rows > index.row_lo:
        rows = torch.zeros(U, index.Dp, dtype=bf16, device=dev)
        ops.f32_to_bf16_split(table_f32.contiguous(), rows[:, :index.D], None, row_index=tgt)
        fb, u_pad = _split_feats(feats_f32, index.Dp, n_split)
        ops.catalogue_rank(fb, U, u_pad, n_split, index.table, index.row_lo, index.id_base, rows, tgt, rank)
    parallel.allreduce_sum_(rank, process_group)
    return rank.to(torch.int64)


def metrics_from_ranks(ranks, ks=(10,)) -> dict:
    """HR@k = mean(rank < k), NDCG@k = mean(1 / log2(rank + 2) where rank < k) for every k in ks, and MRR =
    mean(1 / (rank + 1)), from 0-based ranks (utils.py:595-597 generalised to any cutoff)."""
    r = np.asarray(ranks.cpu() if torch.is_tensor(ranks) else ranks, dtype=np.int64).reshape(-1)
    n = max(len(r), 1)
    out = {}
    for k in ks:
        hit = r < k
        out[f"HR@{k}"] = float(hit.sum() / n)
        out[f"NDCG@{k}"] = float(np.where(hit, 1.0 / np.log2(r + 2.0), 0.0).sum() / n)
    out["MRR"] = float((1.0 / (r + 1.0)).sum() / n)
    return out


@torch.no_grad()
def encode_users(model, seq, rsq, process_group=None) -> torch.Tensor:
    """hidden[:, -1, :] for every user (U, Dout) fp32.  With a process group the USERS are split over the ranks (a sequence's
    encoding does not depend on the rest of the batch) and ONE all-gather of the representations (Dout fp32 per user)
    gives every rank all of them -- the item table is sharded by rows, so every rank needs every user, but nobody needs to
    encode them G times (at 8 ranks the replicated encode was 40 % of a catalogue pass)."""
    from . import parallel
    if process_group is None or torch.distributed.get_world_size(process_group) == 1:
        return model.encode_last(seq, rsq)
    G, r = torch.distributed.get_world_size(process_group), torch.distributed.get_rank(process_group)
    U = seq.shape[0]
    per = (U + G - 1) // G
    lo, hi = min(r * per, U), min((r + 1) * per, U)
    if hi > lo:
        mine = model.encode_last(seq[lo:hi], None if rsq is None else rsq[lo:hi])
        width = mine.shape[1]
    else:                                                 # more ranks than users: an empty slice still joins the all-gather
        width = model.encode_last(seq[:1], None if rsq is None else rsq[:1]).shape[1]
        mine = torch.empty(0, width, dtype=torch.float32, device=seq.device if torch.is_tensor(seq) else None)
    buf = torch.zeros(per, width, dtype=torch.float32, device=mine.device)
    buf[:hi - lo] = mine
    return parallel.allgather_rows(buf, process_group)[:U]


def hr_ndcg_from_topk(topk_ids: torch.Tensor, target: torch.Tensor, k: int = 10) -> Tuple[float, float]:
    """(NDCG@k, HR@k) in the reference's return order (utils.py:595-602): a hit at 0-based rank r < k adds
    1 to HT and 1/log2(r+2) to NDCG; means over users.  Reads k ids per user back to the host.  k may not exceed the
    width of topk_ids (a narrower list cannot tell a miss from a hit at a rank it does not hold)."""
    if k > topk_ids.shape[1]:
        raise ValueError(f"hr_ndcg_from_topk: k={k} exceeds the {topk_ids.shape[1]} ids per user given")
    ids = topk_ids[:, :k].cpu().numpy()
    tgt = np.asarray(target.cpu() if torch.is_tensor(target) else target).reshape(-1, 1)
    hit = ids == tgt
    rank = hit.argmax(1)
    has = hit.any(1)
    ndcg = np.where(has, 1.0 / np.log2(rank + 2.0), 0.0)
    n = max(len(tgt), 1)
    return float(ndcg.sum() / n), float(has.sum() / n)


@torch.no_grad()
def evaluate_full_catalogue(model, seq, rsq, target, batch_users: int = 16384, n_split: int = 1, process_group=None,
                            index: Optional[CatalogueIndex] = None, k: int = TK):
    """Encode users, score the whole catalogue, return (NDCG@k, HR@k, topk_ids (U, k)); 1 <= k <= KMAX."""
    list_len(k)
    eng = model._sync_flat()
    if index is None:
        index = CatalogueIndex(eng.P.view(model.spec.item_key), 0)
    outs = []
    for s in range(0, seq.shape[0], batch_users):
        feats = encode_users(model, seq[s:s + batch_users], None if rsq is None else rsq[s:s + batch_users], process_group)
        _, ids = sharded_topk(feats[:, :model.spec.D], index, process_group, n_split, k)
        outs.append(ids)
    ids = torch.cat(outs)
    ndcg, hr = hr_ndcg_from_topk(ids, target, k)
    return ndcg, hr, ids


@torch.no_grad()
def evaluate_full_catalogue_ranks(model, seq, rsq, target, ks=(10,), batch_users: int = 16384, n_split: int = 1,
                                  process_group=None, index: Optional[CatalogueIndex] = None):
    """Encode users, rank each held-out item among the whole catalogue -> (metrics_from_ranks(ranks, ks), ranks int64
    (U,)).  Any cutoff and MRR.  Without `index`, the rank's row shard of the item table (the whole table on one GPU)."""
    eng = model._sync_flat()
    table = eng.P.view(model.spec.item_key)
    U = seq.shape[0]
    tgt = _targets(target, U, table.shape[0] - 1, "cpu")
    if index is None:
        G = 1 if process_group is None else torch.distributed.get_world_size(process_group)
        r = 0 if G == 1 else torch.distributed.get_rank(process_group)
        lo, hi = CatalogueIndex.shard_bounds(table.shape[0], r, G)
        index = CatalogueIndex(table[lo:hi], lo)
    outs = []
    for s in range(0, U, batch_users):
        feats = encode_users(model, seq[s:s + batch_users], None if rsq is None else rsq[s:s + batch_users], process_group)
        outs.append(catalogue_ranks(feats[:, :model.spec.D], index, table, tgt[s:s + batch_users], process_group, n_split))
    ranks = torch.cat(outs) if outs else torch.zeros(0, dtype=torch.int64)
    return metrics_from_ranks(ranks, ks), ranks


def dataset_to_csr(dataset):
    """The reference's [user_train, user_test, usernum, itemnum] dicts (utils.py:92-139) -> CSR arrays over user rows
    0..usernum-1 (row u-1 = user u): offsets int64, items int32, labels int8, first held-out item (0 = none)."""
    train, test, usernum, itemnum = dataset
    lens = np.fromiter((len(train["item_ids"].get(u, ())) for u in range(1, usernum + 1)), np.int64, usernum)
    offsets = np.zeros(usernum + 1, np.int64)
    np.cumsum(lens, out=offsets[1:])
    items = np.fromiter((i for u in range(1, usernum + 1) for i in train["item_ids"].get(u, ())), np.int32, int(offsets[-1]))
    labels = np.fromiter((r for u in range(1, usernum + 1) for r in train["review_ids"].get(u, ())), np.int8, int(offsets[-1]))
    target = np.fromiter((test["item_ids"][u][0] if len(test["item_ids"].get(u, ())) >= 1 else 0
                          for u in range(1, usernum + 1)), np.int32, usernum)
    return offsets, items, labels, target, int(usernum), int(itemnum)


def eval_users(csr, max_users: int = 10000, rng: Optional[np.random.Generator] = None) -> np.ndarray:
    """User rows the reference would evaluate (utils.py:551-559): at most ``max_users`` sampled without replacement,
    then those with at least one train and one held-out interaction."""
    offsets, _, _, target, usernum, _ = csr
    rows = np.arange(usernum)
    if usernum > max_users:
        rng = rng or np.random.default_rng()
        rows = np.sort(rng.choice(usernum, max_users, replace=False))
    ok = (np.diff(offsets)[rows] >= 1) & (target[rows] != 0)
    return rows[ok].astype(np.int32)


def right_aligned(csr, rows: np.ndarray, maxlen: int):
    """seq / rsq as evaluation() builds them (utils.py:561-574): the last ``maxlen`` train items, right-aligned."""
    offsets, items, labels = csr[0], csr[1], csr[2]
    a, b = offsets[rows], offsets[rows + 1]
    t = np.arange(maxlen)[None, :]
    src = (b - a)[:, None] - (maxlen - t)
    valid = src >= 0
    gi = np.where(valid, a[:, None] + src, 0)
    if len(items) == 0:
        z = np.zeros((len(rows), maxlen), np.int64)
        return z, z.copy()
    return (np.where(valid, items[gi], 0).astype(np.int64), np.where(valid, labels[gi], 0).astype(np.int64))


@torch.no_grad()
def sampled_ranks(model, csr, rows: np.ndarray, maxlen: int, device, seed: int = 0, n_neg: int = 100,
                  candidates: Optional[np.ndarray] = None, chunk: int = 8192, return_logits: bool = False):
    """0-based rank of each user's held-out item among itself + ``n_neg`` sampled negatives (utils.py:576-591), on the
    device: candidate draw (srfrd_sample_candidates, rejection against the user's train row), encoder on the hot-path
    kernels, candidate scoring + rank (srfrd_candidate_rank).  ``candidates`` (len(rows), 1 + n_neg) overrides the
    draw (parity tests feed the reference's own sets).  Returns ranks (numpy int64)[, logits (numpy)]."""
    offsets, items, labels, target, usernum, itemnum = csr
    dev = torch.device(device)
    eng = model._sync_flat()
    spec = model.spec
    d_off = torch.from_numpy(offsets).to(dev)
    d_items = torch.from_numpy(items if len(items) else np.zeros(1, np.int32)).to(dev)
    d_target = torch.from_numpy(target).to(dev)
    C = 1 + n_neg if candidates is None else candidates.shape[1]
    ranks, logits_out = [], []
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    for s in range(0, len(rows), chunk):
        r = rows[s:s + chunk]
        seq, rsq = right_aligned(csr, r, maxlen)
        seq_d, rsq_d = torch.from_numpy(seq).to(dev), torch.from_numpy(rsq).to(dev)
        if candidates is None:
            cand = torch.empty(len(r), C, dtype=torch.int64, device=dev)
            ops.sample_candidates(d_off, d_items, torch.from_numpy(np.ascontiguousarray(r, np.int32)).to(dev), d_target,
                                  itemnum, C, seed + s, cand)
        else:
            cand = torch.from_numpy(np.ascontiguousarray(candidates[s:s + chunk], np.int64)).to(dev)
        feats = model.encode_last(seq_d, rsq_d)                          # (u, Dout) fp32
        rank = torch.empty(len(r), dtype=torch.int32, device=dev)
        lg = torch.empty(len(r), C, dtype=torch.float32, device=dev) if return_logits else None
        ft = lab = None
        if spec.kind == "SRFRN":                                         # rows E[id] || Fe[user label], SRFR_model.py:244-257
            ft = eng.P.view("embedding_layer.fake_embed.weight")
            lab = torch.empty(len(r), dtype=torch.int64, device=dev)
            ops.srfu_labels(rsq_d.contiguous(), 3, lab)
        ops.candidate_rank(feats, eng.P.view(spec.item_key), cand, spec.D, ft, lab, lg, rank, err)
        ranks.append(rank)
        if return_logits:
            logits_out.append(lg)
    if not ranks:
        return (np.zeros(0, np.int64), np.zeros((0, C), np.float32)) if return_logits else np.zeros(0, np.int64)
    out = torch.cat(ranks).cpu().numpy().astype(np.int64)                # one D2H read for all users
    if int(err.item()):
        raise IndexError("index out of range in self: a candidate item id is outside the item table")
    if return_logits:
        return out, torch.cat(logits_out).cpu().numpy()
    return out


@torch.no_grad()
def evaluation(model, dataset, maxlen, device, max_users: int = 10000, seed: Optional[int] = None, chunk: int = 8192,
               candidates: Optional[np.ndarray] = None, users: Optional[np.ndarray] = None):
    """The reference's evaluation() (utils.py:544-602), batched on the device: per user 1 held-out target + 100 uniform
    negatives not in the user's train set, rank of the target among the 101, HR@10 / NDCG@10.  Returns
    (NDCG@10, HR@10).  Candidate draw, encoder and candidate scoring / ranking all run on the library's kernels
    (sampled_ranks); ``users`` (1-based ids) / ``candidates`` pin the user order and candidate sets for parity tests."""
    csr = dataset_to_csr(dataset)
    rng = np.random.default_rng(seed)
    rows = eval_users(csr, max_users, rng) if users is None else (np.asarray(users, np.int64) - 1).astype(np.int32)
    rank = sampled_ranks(model, csr, rows, maxlen, device, seed=int(rng.integers(1 << 31)), candidates=candidates, chunk=chunk)
    hit = rank < 10
    n = max(len(rows), 1)
    return float(np.where(hit, 1.0 / np.log2(rank + 2.0), 0.0).sum() / n), float(hit.sum() / n)
