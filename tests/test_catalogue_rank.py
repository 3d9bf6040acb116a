"""Exact full-catalogue rank of each user's held-out item: the rank variant of the unit-form scoring kernel
(srfrd_catalogue_rank, srfrd_b200/csrc/topk.cu), evaluation.catalogue_ranks, metrics_from_ranks and
evaluate_full_catalogue_ranks.

GPU tests: bit-exact against O.full_catalogue_rank on dyadic inputs (widths, splits, ragged last tiles, user groups cut
into pieces, forced ties at ids on both sides of the target), agreement with the top-k, Gaussian precision, row shards
summed on one GPU, the benchmark size, the metrics and the refusals.  CPU tests: metrics_from_ranks against the oracle's
HR / NDCG and a gloo all-reduce of per-shard counts."""
import numpy as np
import pytest
import torch
import torch.distributed as dist

from oracle import srfrd_oracle as O
from tests.test_dp_protocol import _run

bf16 = torch.bfloat16
gpu = pytest.mark.gpu


def _dyadic(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(-16, 17, shape, generator=g).float() / 8.0


def _targets(U, N, seed):
    return np.random.default_rng(seed).integers(1, N + 1, U).astype(np.int64)


def _rank64(feats, table, target, operand_dtype=None, near=1e-5):
    """Oracle rank with fp64 accumulation (operands optionally rounded to `operand_dtype` first) and, per user, the
    number of other items whose score is within `near` of the target's -- the only items a rounding can move."""
    f, t = feats.float(), table[1:].float()
    if operand_dtype is not None:
        f, t = f.to(operand_dtype), t.to(operand_dtype)
    sc = (f.double() @ t.double().T).numpy()
    U = len(target)
    tsc = sc[np.arange(U), target - 1][:, None]
    ids = np.arange(1, sc.shape[1] + 1)[None, :]
    rank = (sc > tsc).sum(1) + ((sc == tsc) & (ids < target[:, None])).sum(1)
    close = ((np.abs(sc - tsc) <= near) & (ids != target[:, None])).sum(1)
    return rank, close


def _ranks(feats, table, target, n_split=1, lo=0, hi=None):
    """catalogue_ranks over table rows [lo, hi) (a shard; the whole table by default)"""
    from srfrd_b200 import evaluation as EV
    hi = table.shape[0] if hi is None else hi
    tab = table.cuda()
    index = EV.CatalogueIndex(tab[lo:hi].contiguous(), lo)
    return EV.catalogue_ranks(feats.cuda(), index, tab, torch.from_numpy(target), None, n_split)


def _shards(n_rows, G):
    """G - 1 ceil-split row ranges followed by one empty shard"""
    from srfrd_b200.evaluation import CatalogueIndex
    return [CatalogueIndex.shard_bounds(n_rows, r, G - 1) for r in range(G - 1)] + [(n_rows, n_rows)]


# ------------------------------------------------------------------------------------------------------------ GPU
@gpu
@pytest.mark.parametrize("U,N,D,n_split", [(5, 300, 16, 1), (40, 2000, 16, 2), (40, 2000, 16, 3), (200, 5000, 64, 1),
                                           (300, 20000, 64, 2), (150, 9000, 64, 3), (100, 3000, 128, 1),
                                           (100, 3000, 128, 2), (64, 1000, 256, 1), (130, 70000, 64, 1),
                                           (260, 9000, 64, 1), (7, 30, 64, 1)])
def test_rank_bit_exact_on_dyadic_inputs(U, N, D, n_split):
    """Entries j/8 with |j| <= 16: every score is exact in fp32 and in bf16 splits, so the rank must equal the oracle's.
    5000 / 9000 / 20000 items leave ragged last tiles; 130 users x 70 000 items cut the user group into many pieces;
    260 and 300 users fill two user groups.  Targets 1, N and one in the last tile; rows forced equal to a target's row
    at lower and higher ids (only the lower ones count); the dyadic data holds many more exact ties of its own."""
    from srfrd_b200 import evaluation as EV, ops
    feats, table = _dyadic((U, D), 300 + D + n_split), _dyadic((N + 1, D), 301 + N)
    target = _targets(U, N, U + N)
    target[0], target[1], target[2] = 1, N, max(1, N - 3)
    t3 = max(8, N // 2)
    if U > 4 and N > 20:
        table[t3 - 5] = table[t3]
        table[t3 - 1] = table[t3]
        table[t3 + 7] = table[t3]
        target[3], target[4] = t3, t3 + 7
    ref = O.full_catalogue_rank(feats, table, target)
    if (U, N) == (130, 70000):
        idx = EV.CatalogueIndex(table.cuda(), 0)
        assert ops.catalogue_topk_plan(U, idx.n_rows, idx.row_lo, idx.Dp, 1, 10) > 2
    got = _ranks(feats, table, target, n_split)
    assert got.dtype == torch.int64 and got.shape == (U,)
    assert np.array_equal(got.cpu().numpy(), ref)


@gpu
def test_target_scores_output_is_the_simt_score():
    """ops.catalogue_rank's optional output: the target's own score, exact on dyadic inputs; rank_out is zeroed by the
    call (pre-filled with garbage here)."""
    from srfrd_b200 import evaluation as EV, ops
    U, N, D = 300, 7000, 64
    feats, table = _dyadic((U, D), 11), _dyadic((N + 1, D), 12)
    target = _targets(U, N, 13)
    idx = EV.CatalogueIndex(table.cuda(), 0)
    tgt = torch.from_numpy(target).cuda()
    rows = torch.zeros(U, idx.Dp, dtype=bf16, device="cuda")
    ops.f32_to_bf16_split(table.cuda(), rows[:, :D], None, row_index=tgt)
    fb, u_pad = EV._split_feats(feats.cuda(), idx.Dp, 1)
    rank = torch.full((U,), 12345, dtype=torch.int32, device="cuda")
    tsc = torch.full((U,), float("nan"), device="cuda")
    ops.catalogue_rank(fb, U, u_pad, 1, idx.table, idx.row_lo, idx.id_base, rows, tgt, rank, tsc)
    want = (feats * table[target]).sum(1).numpy()
    assert np.array_equal(tsc.cpu().numpy(), want.astype(np.float32))
    assert np.array_equal(rank.cpu().numpy(), O.full_catalogue_rank(feats, table, target))


@gpu
@pytest.mark.parametrize("k", [10, 64])
def test_rank_agrees_with_the_topk(k):
    """rank < k exactly when the target is among local_topk's ids, and then the rank is its column."""
    from srfrd_b200 import evaluation as EV
    U, N, D = 400, 30000, 64
    feats, table = _dyadic((U, D), 20 + k), _dyadic((N + 1, D), 21 + k)
    _, ids = EV.local_topk(feats.cuda(), EV.CatalogueIndex(table.cuda(), 0), 1, k)
    ids = ids.cpu().numpy()
    target = _targets(U, N, k)
    target[: U // 2] = ids[np.arange(U // 2), np.arange(U // 2) % k]       # half the users: a target inside the top-k
    rank = _ranks(feats, table, target).cpu().numpy()
    hit = ids == target[:, None]
    assert np.array_equal(rank < k, hit.any(1))
    assert np.array_equal(rank[hit.any(1)], hit.argmax(1)[hit.any(1)])
    assert (rank < k).sum() >= U // 2


@gpu
def test_rank_gaussian_precision():
    """Tensor-core item scores against a SIMT target score: a rank may differ from the exact one only by items whose
    score is within rounding (1e-5) of the target's.  bf16 operands vs an fp64 oracle on bf16-rounded operands, and
    n_split = 3 vs fp32 features."""
    g = torch.Generator().manual_seed(92)
    U, N, D = 300, 40000, 64
    feats = torch.randn(U, D, generator=g)
    table = (torch.randn(N + 1, D, generator=g) * 0.05).to(bf16).float()
    target = _targets(U, N, 92)
    target[:100] = np.argsort(-(feats[:100].to(bf16).float() @ table[1:].T).numpy(), 1)[:, 0] + 1   # rank 0 users
    for n_split, dtype in ((1, bf16), (3, None)):
        ref, close = _rank64(feats, table, target, dtype)
        got = _ranks(feats, table, target, n_split).cpu().numpy()
        assert np.all(np.abs(got - ref) <= close), (n_split, np.abs(got - ref).max())
        assert np.mean(got == ref) > 0.9


@gpu
@pytest.mark.parametrize("data", ["dyadic", "gaussian"])
def test_row_shards_sum_to_the_unsharded_rank(data):
    """8 row shards, the last one empty, counted one after another on one GPU: the sum equals the unsharded rank.  On
    Gaussian data this holds because a tensor-core score does not depend on the item's column within a tile (shards move
    the tile boundaries) and the target's SIMT score uses the same bits on every shard."""
    U, N, D = 150, 9000, 64
    if data == "dyadic":
        feats, table = _dyadic((U, D), 93), _dyadic((N + 1, D), 94)
    else:
        g = torch.Generator().manual_seed(95)
        feats, table = torch.randn(U, D, generator=g), torch.randn(N + 1, D, generator=g) * 0.05
    target = _targets(U, N, 96)
    full = _ranks(feats, table, target)
    total = torch.zeros_like(full)
    for lo, hi in _shards(N + 1, 8):
        total += _ranks(feats, table, target, 1, lo, hi)
    assert torch.equal(total, full)
    if data == "dyadic":
        assert np.array_equal(full.cpu().numpy(), O.full_catalogue_rank(feats, table, target))


@gpu
def test_benchmark_size_rank():
    """1 M items x D = 64 x 768 users, dyadic, uniformly random targets (ranks around 500 k: nearly every unit reaches
    the target's score and is counted): bit-exact against the oracle on a user subset."""
    U, N, D = 768, 1_000_000, 64
    feats, table = _dyadic((U, D), 97), _dyadic((N + 1, D), 98)
    target = _targets(U, N, 99)
    got = _ranks(feats, table, target).cpu().numpy()
    sub = np.arange(0, U, 12)
    ref = O.full_catalogue_rank(feats[sub], table, target[sub])
    assert np.array_equal(got[sub], ref)
    assert np.median(got) > 100_000


@gpu
def test_full_catalogue_rank_metrics_match_oracle():
    """evaluate_full_catalogue_ranks on a synthetic SRFR: HR / NDCG @10 and @20 agree with evaluate_full_catalogue and
    with the oracle's exact ranking; HR@100, HR@1000 and MRR with the oracle (1e-3, the bound of the top-k tests)."""
    from srfrd_b200 import SRFR_model as M, evaluation as EV, synth
    data = synth.make_interactions(21, 3000, 5000, 5, 4.0, 50)
    torch.manual_seed(1)
    m = M.SRFR(data.itemnum, 50, 64, 16, 0.0, 2, 1, "cuda")
    for _, p in m.named_parameters():
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    m = m.to("cuda").eval()
    users0 = np.nonzero(data.test_item > 0)[0][:2000]
    seq, rsq, tgt = synth.eval_sequences(data, 50, users0)
    seq_d, rsq_d = torch.from_numpy(seq).cuda(), torch.from_numpy(rsq).cuda()
    met, ranks = EV.evaluate_full_catalogue_ranks(m, seq_d, rsq_d, torch.from_numpy(tgt), ks=(10, 20, 100, 1000),
                                                  n_split=3, batch_users=768)
    assert ranks.shape == (len(users0),) and ranks.dtype == torch.int64
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items()}
    table = sd["embedding_layer.item_embed.weight"]
    # the kernel alone: exact ranks of the device's own user representations, up to items within rounding of the target
    feats = EV.encode_users(m, seq_d, rsq_d)[:, :64].cpu()
    exact, close = _rank64(feats, table.to(bf16).float(), tgt)        # n_split = 3: ~fp32 features x the bf16 table
    assert np.all(np.abs(ranks.cpu().numpy() - exact) <= close)
    # end to end against the oracle's fp32 encoder: the device encoder's rounding moves a target by a few places, which
    # decides HR@1000 for about 1 user in 1000 (1e-3 = 2 of these 2000 users; the epsilon absorbs its fp64 spelling)
    h = O.encode(sd, "SRFR", torch.from_numpy(seq), torch.from_numpy(rsq), 1)[:, -1, :]
    ref = O.full_catalogue_rank(h, table, tgt)
    for k in (10, 20, 100, 1000):
        ndcg_ref, hr_ref = O.hr_ndcg_from_rank(ref, k)
        assert abs(met[f"HR@{k}"] - hr_ref) <= 1e-3 + 1e-12 and abs(met[f"NDCG@{k}"] - ndcg_ref) <= 1e-3, (k, met, hr_ref)
    assert abs(met["MRR"] - float(np.mean(1.0 / (ref + 1.0)))) <= 1e-3
    for k in (10, 20):
        ndcg, hr, _ = EV.evaluate_full_catalogue(m, seq_d, rsq_d, torch.from_numpy(tgt), n_split=3, k=k)
        assert abs(met[f"HR@{k}"] - hr) <= 1e-3 and abs(met[f"NDCG@{k}"] - ndcg) <= 1e-3, (k, met, hr, ndcg)


@gpu
def test_rank_refusals_before_any_launch():
    from srfrd_b200 import _lib, evaluation as EV
    U, N = 10, 100
    feats, table = _dyadic((U, 128), 1).cuda(), _dyadic((N + 1, 128), 2).cuda()
    idx64, idx128 = EV.CatalogueIndex(table[:, :64], 0), EV.CatalogueIndex(table, 0)
    empty = EV.CatalogueIndex(table[N + 1:, :64], N + 1)
    good = _targets(U, N, 3)
    bad = {"target 0": np.where(np.arange(U) == 4, 0, good), "target > N": np.where(np.arange(U) == 4, N + 1, good),
           "length": good[:-1]}
    n0 = _lib.launch_count
    for name, t in bad.items():
        with pytest.raises(ValueError):
            EV.catalogue_ranks(feats[:, :64], idx64, table[:, :64], torch.from_numpy(t))
    with pytest.raises(RuntimeError, match="tile form"):                 # n_split * D = 384 > 256
        EV.catalogue_ranks(feats, idx128, table, torch.from_numpy(good), None, 3)
    assert _lib.launch_count == n0                                      # no library call got through
    # an empty shard contributes 0 without a launch
    r = EV.catalogue_ranks(feats[:, :64], empty, table[:, :64], torch.from_numpy(good))
    assert torch.equal(r, torch.zeros(U, dtype=torch.int64, device="cuda")) and _lib.launch_count == n0
    r = EV.catalogue_ranks(feats[:, :64], idx64, table[:, :64], torch.from_numpy(good))
    assert np.array_equal(r.cpu().numpy(), O.full_catalogue_rank(feats[:, :64].cpu(), table[:, :64].cpu(), good))


# ------------------------------------------------------------------------------------------------------------ CPU
def test_metrics_from_ranks_match_the_oracle():
    from srfrd_b200 import evaluation as EV
    rank = np.random.default_rng(0).integers(0, 3000, 5000)
    rank[:50] = 0
    met = EV.metrics_from_ranks(torch.from_numpy(rank), ks=(1, 10, 20, 100, 1000))
    for k in (1, 10, 20, 100, 1000):
        ndcg, hr = O.hr_ndcg_from_rank(rank, k)
        assert met[f"HR@{k}"] == pytest.approx(hr, abs=1e-12) and met[f"NDCG@{k}"] == pytest.approx(ndcg, abs=1e-12)
    assert met["MRR"] == pytest.approx(np.mean(1.0 / (rank + 1.0)), abs=1e-12)
    assert set(EV.metrics_from_ranks(rank)) == {"HR@10", "NDCG@10", "MRR"}
    assert EV.metrics_from_ranks(np.array([0, 1, 3]), ks=(2,)) == pytest.approx(
        {"HR@2": 2 / 3, "NDCG@2": (1 + 1 / np.log2(3)) / 3, "MRR": (1 + 1 / 2 + 1 / 4) / 3})


def _host_count(feats, table, target, lo, hi):
    """items with ids in [max(lo, 1), hi) ahead of the target (whose score comes from the whole table)"""
    sc = (feats @ table.T).numpy()
    tsc = sc[np.arange(len(target)), target][:, None]
    ids = np.arange(table.shape[0])[None, :]
    inside = (ids >= max(lo, 1)) & (ids < hi) & (ids != target[:, None])
    return (inside & ((sc > tsc) | ((sc == tsc) & (ids < target[:, None])))).sum(1)


def _rank_sum_job(rank, world):
    from srfrd_b200 import parallel as P
    g = torch.Generator().manual_seed(23)
    feats = torch.randint(-16, 17, (37, 32), generator=g).float() / 8
    table = torch.randint(-16, 17, (1001, 32), generator=g).float() / 8
    target = np.random.default_rng(23).integers(1, 1001, 37)
    lo, hi = P.shard_rows(table.shape[0], rank, world)
    cnt = torch.from_numpy(_host_count(feats, table, target, lo, hi).astype(np.int32))
    return P.allreduce_sum_(cnt, dist.group.WORLD).numpy()


def test_gloo_allreduce_of_shard_counts_gives_the_full_rank():
    g = torch.Generator().manual_seed(23)
    feats = torch.randint(-16, 17, (37, 32), generator=g).float() / 8
    table = torch.randint(-16, 17, (1001, 32), generator=g).float() / 8
    target = np.random.default_rng(23).integers(1, 1001, 37)
    ref = O.full_catalogue_rank(feats, table, target)
    assert np.array_equal(_host_count(feats, table, target, 0, 1001), ref)
    for got in _run(_rank_sum_job, port=29641):
        np.testing.assert_array_equal(got, ref)
