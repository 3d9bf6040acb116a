"""gSASRec's gBCE over k negatives shared by every row of a step (csrc/gbce.cu, losses.sampled_gbce,
FusedTrainer(loss="gbce")).

With alpha = k / (N - 1), beta = 1 - t (1 - alpha), z_r = <h_r, E[pos_r]>, s_rj = <h_r, E[n_j]> and m_rj = 0 when n_j
occurs in row r's sequence:  loss = (sum_r w_r beta softplus(-z_r) + sum_r w_r sum_j m_rj softplus(s_rj)) / sum_r w_r.

CPU: the fp64 oracle below against gSASRec's own form (BCEWithLogits on logit(sigmoid(z)^beta)), the plan and its
refusals, and the model check of the kernels' mbarrier protocol (the CE kernels' pipeline at the gBCE stream lengths).
GPU: the kernels against the oracle on the same bf16 operands (dense, packed, 16 384 sequences), exact properties, the
device draw and exclusion mask, FusedTrainer(loss="gbce") against autograd + Adam over losses.sampled_gbce, the BCE
equivalence at t = 0 and k = 1, refusals and launch counts.
"""
import math

import numpy as np
import pytest
import torch


# ------------------------------------------------------------------------------------------------------------ oracle
def gbce_oracle(h, E, pos, negs, w=None, t=0.75, mask=None):
    """float64 gBCE on bf16-rounded operands, on h's device.  h (R, D), E (N + 1, D), pos (R,) in 0..N (0 = no term),
    negs (k,) in 1..N, w (R,) or None (= 1[pos != 0]), mask (R, k) m_rj or None (all ones).
    Returns (loss, dh (R, D), dE (N + 1, D))."""
    hb, Eb = h.to(torch.bfloat16).double(), E.to(torch.bfloat16).double()
    N, k = Eb.shape[0] - 1, negs.numel()
    pos, negs = pos.long(), negs.long()
    valid = pos != 0
    wv = valid.double() if w is None else w.double() * valid
    W = float(wv.sum())
    inv = 1.0 / W if W > 0 else 0.0
    beta = 1.0 - t * (1.0 - k / (N - 1))
    m = torch.ones(hb.shape[0], k, dtype=torch.float64, device=h.device) if mask is None else mask.double()
    z = (hb * Eb[pos]).sum(1)
    s = hb @ Eb[negs].T
    sp = torch.nn.functional.softplus
    loss = float((wv * beta * sp(-z)).sum() + (wv[:, None] * m * sp(s)).sum()) * inv
    dz = wv * beta * (torch.sigmoid(z) - 1) * inv
    ds = wv[:, None] * m * torch.sigmoid(s) * inv
    dh = dz[:, None] * Eb[pos] + ds @ Eb[negs]
    dE = torch.zeros_like(Eb)
    dE.index_add_(0, pos, dz[:, None] * hb)
    dE.index_add_(0, negs, ds.T @ hb)
    dE[0] = 0
    return loss, dh, dE


def exclusion_mask(seqs, negs):
    """numpy: (n_seq, ceil(k / 32)) uint32, bit j % 32 of word j // 32 set when negs[j] occurs in seqs[b]."""
    seqs, negs = np.asarray(seqs), np.asarray(negs)
    k = len(negs)
    hit = (seqs[:, :, None] == negs[None, None, :]).any(1)               # (n_seq, k)
    words = np.zeros((seqs.shape[0], (k + 31) // 32), dtype=np.uint64)
    for j in range(k):
        words[:, j // 32] |= hit[:, j].astype(np.uint64) << np.uint64(j % 32)
    return words.astype(np.uint32)


def test_oracle_matches_gsasrec_form():
    g = torch.Generator().manual_seed(0)
    R, N, D, k = 41, 300, 24, 17
    h = torch.randn(R, D, generator=g, dtype=torch.float64).bfloat16().double().requires_grad_(True)
    E = torch.randn(N + 1, D, generator=g, dtype=torch.float64).bfloat16().double().requires_grad_(True)
    pos = torch.randint(1, N + 1, (R,), generator=g)
    pos[::6] = 0
    negs = torch.randint(1, N + 1, (k,), generator=g)
    negs[3] = negs[5]                                              # a duplicate draw counts twice
    mask = (torch.rand(R, k, generator=g) > 0.2).double()
    w = torch.rand(R, generator=g, dtype=torch.float64)
    bce = torch.nn.BCEWithLogitsLoss(reduction="none")
    for t in (0.0, 0.75, 1.0):
        for weights in (None, w):
            beta = 1.0 - t * (1.0 - k / (N - 1))
            wv = (pos != 0).double() if weights is None else weights * (pos != 0)
            z = (h * E[pos]).sum(1)
            s = h @ E[negs].T
            p = torch.sigmoid(z) ** beta                             # gSASRec: the positive's probability to the beta
            zt = torch.log(p) - torch.log1p(-p)                      # logit(sigmoid(z)^beta)
            per = bce(zt, torch.ones_like(zt)) + (mask * bce(s, torch.zeros_like(s))).sum(1)
            ref = (wv * per).sum() / wv.sum()
            gh, gE = torch.autograd.grad(ref, (h, E))
            gE[0] = 0
            loss, dh, dE = gbce_oracle(h.detach(), E.detach(), pos, negs, weights, t, mask)
            assert abs(loss - float(ref)) < 1e-11
            assert torch.allclose(dh, gh, atol=1e-12) and torch.allclose(dE, gE, atol=1e-12)


def test_exclusion_mask_reference():
    seqs = np.array([[0, 5, 7, 9], [3, 3, 0, 0]])
    negs = [7, 3, 7, 1] + [9] * 30
    m = exclusion_mask(seqs, negs)
    assert m.shape == (2, 2)
    assert m[0, 0] == (1 << 0) | (1 << 2) | sum(1 << j for j in range(4, 32)) and m[0, 1] == 0b11
    assert m[1, 0] == (1 << 1) and m[1, 1] == 0


# ------------------------------------------------------------------------------------------------------------- plan
def test_plan_and_refusals():
    from srfrd_b200 import ops
    for k, Kp in ((1, 128), (128, 128), (129, 256), (256, 256)):
        for Dp in (16, 64, 80, 256):
            kp, n_split, smem, stages = ops.gbce_plan(k, Dp, 209024)
            kb = (Dp + 63) // 64
            assert kp == Kp and stages >= 2 and smem == (kb + 2 + stages * kb) * 16384 + 1280 and smem <= 227 * 1024
            assert 1 <= n_split <= 1633
    assert ops.gbce_plan(64, 64, 100)[1] == 1                      # one row tile: one split
    for k, Dp in ((0, 64), (257, 64), (64, 8), (64, 272)):
        with pytest.raises(RuntimeError, match="gbce"):
            ops.gbce_plan(k, Dp, 1000)
    from srfrd_b200.losses import check_gbce, gbce_beta
    assert check_gbce(256, 0.75, 12101, 250) == 256
    for args in ((0, 0.5, 100, 64), (257, 0.5, 100, 64), (8, -0.1, 100, 64), (8, 1.5, 100, 64), (8, 0.5, 1, 64),
                 (8, 0.5, 100, 257)):
        with pytest.raises(ValueError, match="gbce"):
            check_gbce(*args)
    assert gbce_beta(256, 12101, 0.0) == 1.0
    assert abs(gbce_beta(256, 12101, 0.75) - (1 - 0.75 * (1 - 256 / 12100))) < 1e-15
    # gSASRec's own form of beta
    a = 256 / 12100
    assert abs(gbce_beta(256, 12101, 0.75) - a * (0.75 * (1 - 1 / a) + 1 / a)) < 1e-12


# --------------------------------------------------------------------------------------------------- protocol model
@pytest.mark.parametrize("mode", ["dh", "de"])
@pytest.mark.parametrize("stages", [2, 3, 5, 8])
def test_pipeline_protocol_model(mode, stages):
    """The gBCE kernel keeps catalogue_ce_kernel's barriers and warp roles for its DH / DN passes (the loss pass of CE
    has no gBCE counterpart): the DH pass streams Kp / 128 = 1 or 2 negative blocks, the DN pass a split's row tiles."""
    from tests.test_catalogue_ce import _ce_protocol
    lengths = (1, 2) if mode == "dh" else (1, 2, 3, 7, 12)
    for seed in range(6):
        for nstream in lengths:
            _ce_protocol(mode, nstream, stages, seed * 100 + nstream + 7)


# ------------------------------------------------------------------------------------------------------------- GPU
class _RowMap:
    def __init__(self, row_tok, rows):
        self.row_tok = torch.tensor(row_tok, dtype=torch.int32, device="cuda")
        self.rows = torch.tensor([rows, 0, 0, 0], dtype=torch.int32, device="cuda")
        self.cap = len(row_tok)


def _run(h, E, pos, negs, w=None, t=0.75, seqs=None, L=1, plan=None, want_dE=True):
    """h (cap, D) fp32, E (N + 1, D) fp32, pos / w per dense token, negs (k,) given ids, seqs (n_seq, M) exclusion ids
    (the sequence of dense token i is i // L) -> (loss, dh, dE, acc) from the kernels."""
    from srfrd_b200 import ops
    from srfrd_b200.losses import _bf16_rows, gbce_beta
    D, N, k = E.shape[1], E.shape[0] - 1, negs.numel()
    Dp = (D + 15) // 16 * 16
    Kp, n_split, _, _ = ops.gbce_plan(k, Dp, h.shape[0])
    nb = torch.full((Kp, Dp), float("nan"), dtype=torch.bfloat16, device="cuda")
    excl = None if seqs is None else torch.full((seqs.shape[0], (k + 31) // 32), -1, dtype=torch.int32, device="cuda")
    ids = negs.clone()
    ops.gbce_draw(E, ids, nb, excl, ex_a=seqs, draw=False)
    hb = _bf16_rows(h.contiguous(), Dp)
    norm = torch.zeros(2, device="cuda")
    ops.weight_sums(pos, w, None, norm)
    acc = torch.zeros(2, device="cuda")
    dh = torch.full((h.shape[0], D), float("nan"), device="cuda")
    dE = torch.zeros(N + 1, D, device="cuda") if want_dE else None
    part = torch.full((n_split * Kp * Dp,), float("nan"), device="cuda")
    ops.gbce_loss(hb, nb, ids, E, pos, w, norm, excl, L, gbce_beta(k, N, t), acc, dh, dE, part, plan)
    torch.cuda.synchronize()
    n = float(norm[0])
    return (float(acc[0] + acc[1]) / n if n > 0 else 0.0), dh, dE, acc, excl


def _mask(seqs, negs, L, R, row_seq=None):
    """m (R, k) on cuda from the numpy exclusion reference; row r's sequence is r // L (or row_seq[r])."""
    bits = exclusion_mask(seqs.cpu().numpy(), negs.cpu().numpy())
    k = negs.numel()
    ex = (bits[:, np.arange(k) // 32] >> (np.arange(k) % 32).astype(np.uint32)) & 1          # (n_seq, k)
    rs = np.arange(R) // L if row_seq is None else row_seq
    return torch.from_numpy(1.0 - ex[rs].astype(np.float64)).cuda()


def _rel_cos(got, ref):
    got, ref = got.double().flatten(), ref.double().flatten()
    rel = float((got - ref).norm() / ref.norm().clamp_min(1e-300))
    cos = float(torch.dot(got, ref) / (got.norm() * ref.norm()).clamp_min(1e-300))
    return rel, cos


# dh / dE against the fp64 oracle on the same bf16 operands: sigmoid(S) enters the second products as bf16
REL, COS = 1e-2, 0.9999


def _close(got, ref, what):
    rel, cos = _rel_cos(got, ref)
    assert rel <= REL and cos >= COS, (what, rel, cos)


def _case(R, N, D, k, seed, L=50):
    """hidden rows of R // L sequences, negatives with duplicates, negatives equal to some positives and some history
    ids, weight-0 rows."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    h = torch.randn(R, D, device="cuda", generator=g) * (2.0 / math.sqrt(D))
    E = torch.randn(N + 1, D, device="cuda", generator=g) * 0.5
    E[0] = 0
    pos = torch.randint(1, N + 1, (R,), device="cuda", generator=g)
    pos[::7] = 0
    negs = torch.randint(1, N + 1, (k,), device="cuda", generator=g)
    if k >= 4:
        negs[1] = negs[0]                                           # duplicate draw
        negs[2] = pos[1]                                            # a row's positive
    seqs = torch.randint(0, N + 1, (R // L, L), device="cuda", generator=g)
    if k >= 4:
        seqs[0, 3] = negs[3]                                        # in one sequence's history
    w = torch.rand(R, device="cuda", generator=g) * (pos != 0)
    w[5::11] = 0
    return h, E, pos, negs, seqs, w


def _check(res, ref):
    loss, dh, dE, _, _ = res
    rloss, rdh, rdE = ref
    assert abs(loss - rloss) <= 1e-4 + 1e-4 * abs(rloss), (loss, rloss)
    _close(dh, rdh, "dh")
    if dE is not None:
        _close(dE, rdE, "dE")
        assert torch.equal(dE[0], torch.zeros_like(dE[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("N", [2, 129, 12101, 150000])
@pytest.mark.parametrize("D", [16, 64, 80, 128, 256])
@pytest.mark.parametrize("k", [1, 16, 127, 128, 129, 256])
def test_kernels_match_oracle_dense(N, D, k):
    if N == 150000 and D > 64:
        pytest.skip("the 150 k table is covered at D = 16 and 64")
    R, L = 300, 50
    h, E, pos, negs, seqs, w = _case(R, N, D, k, seed=N + D + k, L=L)
    m = _mask(seqs, negs, L, R)
    for weights, t in ((None, 0.75), (w, 0.0), (w, 1.0)):
        res = _run(h, E, pos, negs, weights, t, seqs, L)
        _check(res, gbce_oracle(h, E, pos, negs, weights, t, m))
    res = _run(h, E, pos, negs, w, 0.75)                           # no exclusion
    _check(res, gbce_oracle(h, E, pos, negs, w, 0.75))


@pytest.mark.gpu
@pytest.mark.parametrize("D,k", [(16, 5), (64, 256), (200, 129)])
def test_kernels_match_oracle_packed_row_map(D, k):
    """Packed rows: filler rows (-1), a device row count below the capacity (rows beyond it untouched), tokens in
    shuffled order; pos / w indexed by dense token, row r's sequence = row_tok[r] // L."""
    N, B, L = 3001, 14, 50
    T = B * L
    h, E, pos, negs, seqs, w = _case(T, N, D, k, seed=D + k, L=L)
    rng = np.random.default_rng(D)
    toks = rng.permutation(T)[:450].tolist()
    row_tok = []
    for i, tk in enumerate(toks):
        row_tok.append(tk)
        if i % 9 == 0:
            row_tok.append(-1)
    rows = len(row_tok)
    row_tok += [-1] * (640 - rows)
    hp = torch.randn(640, D, device="cuda") * (2.0 / math.sqrt(D))
    res = _run(hp, E, pos, negs, w, 0.75, seqs, L, _RowMap(row_tok, rows))
    rt = np.array(row_tok[:rows])
    rtt = torch.tensor(rt, device="cuda")
    tgt = torch.where(rtt >= 0, pos[rtt.clamp(min=0)], torch.zeros_like(rtt))
    wr = torch.where(rtt >= 0, w[rtt.clamp(min=0)], torch.zeros_like(w[:rows]))
    m = _mask(seqs, negs, L, rows, row_seq=np.maximum(rt, 0) // L)
    loss, dh, dE = gbce_oracle(hp[:rows], E, tgt, negs, wr, 0.75, m)
    scale = float(wr.sum()) / float(w.sum())                        # the kernel divides by the sum over ALL tokens
    _check((res[0], res[1][:rows], res[2], res[3], None), (loss * scale, dh * scale, dE * scale))
    assert torch.isnan(res[1][rows:]).all(), "rows beyond the device row count must stay untouched"
    assert torch.equal(res[1][:rows][rtt < 0], torch.zeros_like(res[1][:rows][rtt < 0]))


@pytest.mark.gpu
def test_sixteen_thousand_sequences():
    N, D, k, L, B = 12101, 64, 256, 4, 16384
    h, E, pos, negs, seqs, w = _case(B * L, N, D, k, seed=9, L=L)
    res = _run(h, E, pos, negs, w, 0.75, seqs, L)
    assert np.array_equal(res[4].cpu().numpy().view(np.uint32), exclusion_mask(seqs.cpu().numpy(), negs.cpu().numpy()))
    _check(res, gbce_oracle(h, E, pos, negs, w, 0.75, _mask(seqs, negs, L, B * L)))


@pytest.mark.gpu
def test_exact_properties():
    N, D, k, R, L = 5000, 64, 200, 1000, 50
    h, E, pos, negs, seqs, w = _case(R, N, D, k, seed=11, L=L)
    a = _run(h, E, pos, negs, w, 0.75, seqs, L)
    b = _run(h, E, pos, negs, w, 0.75, seqs, L)
    assert torch.equal(a[1], b[1]), "dh differs between two launches"
    # the negatives' part of dE is summed in a fixed order; the positives' part uses red.add
    only_neg = torch.zeros(N + 1, dtype=torch.bool, device="cuda")
    only_neg[negs] = True
    only_neg[pos] = False
    assert int(only_neg.sum()) > 100
    assert torch.equal(a[2][only_neg], b[2][only_neg]), "the negatives' dE differs between two launches"
    assert torch.equal(a[2][0], torch.zeros(D, device="cuda"))
    # every weight zero: loss 0, zero gradients, no NaN
    d = _run(h, E, pos, negs, torch.zeros(R, device="cuda"), 0.75, seqs, L)
    assert d[0] == 0.0 and float(d[3].abs().sum()) == 0.0
    assert torch.equal(d[1], torch.zeros_like(d[1])) and torch.equal(d[2], torch.zeros_like(d[2]))


@pytest.mark.gpu
def test_draw_range_determinism_uniformity_and_mask():
    from srfrd_b200 import ops
    dev = "cuda"
    N, D, k = 16, 32, 256
    E = torch.randn(N + 1, D, device=dev)
    seqs = torch.randint(0, N + 1, (37, 9), device=dev)
    posr = torch.randint(0, N + 1, (37, 9), device=dev)
    step = torch.zeros(1, device=dev)

    def draw(seed, s):
        step.copy_(torch.tensor([s], dtype=torch.int32).view(torch.float32))
        ids = torch.zeros(k, dtype=torch.int64, device=dev)
        nb = torch.zeros(256, 32, dtype=torch.bfloat16, device=dev)
        excl = torch.zeros(37, 8, dtype=torch.int32, device=dev)
        ops.gbce_draw(E, ids, nb, excl, seqs, posr, seed=seed, step=step)
        torch.cuda.synchronize()
        return ids, nb, excl

    counts = np.zeros(N + 1)
    prev = None
    for s in range(64):
        ids, nb, excl = draw(123, s)
        assert int(ids.min()) >= 1 and int(ids.max()) <= N
        assert torch.equal(nb.float(), E[ids].bfloat16().float())
        ref = exclusion_mask(torch.cat([seqs, posr], 1).cpu().numpy(), ids.cpu().numpy())
        assert np.array_equal(excl.cpu().numpy().view(np.uint32), ref)
        again = draw(123, s)[0]
        assert torch.equal(ids, again), "the draw is not a function of (seed, step)"
        if prev is not None:
            assert not torch.equal(ids, prev)
        prev = ids
        counts += np.bincount(ids.cpu().numpy(), minlength=N + 1)
    assert not torch.equal(draw(124, 0)[0], draw(123, 0)[0])
    exp = counts[1:].sum() / N
    chi2 = float(((counts[1:] - exp) ** 2 / exp).sum())
    assert counts[0] == 0 and chi2 < 60.0, chi2                  # 15 degrees of freedom
    # zero-padded rows past k and columns past D
    ids = torch.zeros(5, dtype=torch.int64, device=dev)
    nb = torch.full((128, 48), float("nan"), dtype=torch.bfloat16, device=dev)
    ops.gbce_draw(E, ids, nb, None, seed=1, step=step)
    torch.cuda.synchronize()
    assert torch.equal(nb[:5, :32].float(), E[ids].bfloat16().float())
    assert torch.equal(nb[5:].float(), torch.zeros(123, 48, device=dev)) and float(nb[:, 32:].float().abs().sum()) == 0


@pytest.mark.gpu
def test_draw_differs_across_graph_replays():
    from srfrd_b200 import ops
    E = torch.randn(1001, 64, device="cuda")
    step = torch.zeros(1, device="cuda")
    ids = torch.zeros(64, dtype=torch.int64, device="cuda")
    nb = torch.zeros(128, 64, dtype=torch.bfloat16, device="cuda")
    ops.gbce_draw(E, ids, nb, None, seed=5, step=step)
    g = torch.cuda.CUDAGraph()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        ops.gbce_draw(E, ids, nb, None, seed=5, step=step)
    seen = []
    for s in range(3):
        step.copy_(torch.tensor([s + 1], dtype=torch.int32).view(torch.float32))
        g.replay()
        torch.cuda.synchronize()
        seen.append(ids.clone())
        assert torch.equal(nb[:64].float(), E[ids].bfloat16().float())
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])


# ------------------------------------------------------------------------------------------------------- training
def _oracle_gbce(O, tr, k, t, l2=0.0):
    class OracleGBCE(O.OracleTrainer):
        """The oracle step (fp32 autograd encoder + torch Adam) with losses.sampled_gbce as the objective, fed the
        negatives the fused step drew."""

        def step(self, batch, w_pos=None):
            from srfrd_b200.losses import sampled_gbce
            self.opt.zero_grad(set_to_none=True)
            h = O.encode(self.sd, self.kind, batch["seq"], batch["rsq"], self.num_heads)
            E = self.sd[O._emb_keys(self.kind)[0]]
            ex = torch.cat([batch["seq"], batch["pos"]], 1).cuda()
            negs = tr._gbce_ws["ids"].clone()
            w = None if w_pos is None else w_pos.cuda()
            loss = sampled_gbce(h.cuda(), E.cuda(), batch["pos"].cuda(), negs, w, t, ex).cpu()
            loss.backward()
            self._zero_pad_rows()
            reg = 0.0
            if l2:
                params = list(self.sd.values())
                reg = l2 * sum(torch.linalg.vector_norm(p) for p in params)
                for p, g in zip(params, torch.autograd.grad(reg, params)):
                    p.grad = g if p.grad is None else p.grad + g
                reg = float(reg.detach())
            self.opt.step()
            return float(loss.detach()) + reg
    return OracleGBCE


CASES = [("SRFR", True, True), ("SRFR", False, False), ("SASRec", True, False), ("SASRec", False, True),
         ("SRFU_F", True, True), ("SRFU_F", False, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,packed,graph", CASES)
def test_fused_trainer_gbce_matches_oracle(kind, packed, graph):
    from oracle import srfrd_oracle as O
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, smp = _c2_like()
    m = _model(kind, data.itemnum)
    heads = 2 if kind == "SASRec" else 1
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    tr = FusedTrainer(m, use_graph=graph, packed=packed, loss="gbce", num_negatives=128, gbce_t=0.75)
    orc = _oracle_gbce(O, tr, 128, 0.75)(sd0, kind, heads)
    drawn = []
    for step in range(5):
        tb = {k: torch.from_numpy(v) for k, v in smp.next_batch(256).items()}
        loss = float(tr.step({k: v.cuda() for k, v in tb.items()}))
        drawn.append(tr._gbce_ws["ids"].clone())
        ref = orc.step(tb)
        assert math.isfinite(loss) and abs(loss - ref) < 5e-3 * max(1.0, abs(ref)), f"{kind} step {step}: {loss} vs {ref}"
    assert not torch.equal(drawn[0], drawn[1]) and not torch.equal(drawn[3], drawn[4]), "negatives must change per step"
    _check_tensors(m.state_dict(), orc.state_dict(), sd0, 2 * 5 * 1e-3 + 5e-4)


@pytest.mark.gpu
def test_fused_trainer_gbce_step_sampled_soft_weights_l2():
    from oracle import srfrd_oracle as O
    from srfrd_b200.trainer import DeviceSampler, FusedTrainer
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, _ = _c2_like()
    smp = DeviceSampler(data, 50, "cuda", seed=5)
    m = _model("SRFR", data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    tr = FusedTrainer(m, use_graph=True, loss="gbce", l2_emb=1e-4)
    orc = _oracle_gbce(O, tr, 256, 0.75, l2=1e-4)(sd0, "SRFR", 1)
    for step in range(5):
        loss = float(tr.step_sampled(smp, 256, policy="soft"))
        tb = {k: tr._static[k].cpu().clone() for k in FusedTrainer._KEYS}
        w = tr._static["w_pos"].cpu().clone()
        assert float(w.min()) >= 0 and 0 < float(w[tb["pos"] != 0].mean()) < 1
        ref = orc.step(tb, w)
        assert math.isfinite(loss) and abs(loss - ref) < 5e-3 * max(1.0, abs(ref)), f"step {step}: {loss} vs {ref}"
    _check_tensors(m.state_dict(), orc.state_dict(), sd0, 2 * 5 * 1e-3 + 5e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("packed", [True, False])
def test_t0_k1_equals_bce_step(packed):
    """t = 0 and k = 1 with a negative that occurs in no sequence (mask all ones) is the BCE with that id as every
    position's negative."""
    from srfrd_b200 import ops
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, smp = _c2_like()
    m_g, m_b = _model("SASRec", data.itemnum), _model("SASRec", data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m_g.state_dict().items()}
    tr_g = FusedTrainer(m_g, use_graph=False, packed=packed, loss="gbce", num_negatives=1, gbce_t=0.0)
    tr_b = FusedTrainer(m_b, use_graph=False, packed=packed)
    E = tr_g.P.view(tr_g.spec.item_key)
    for step in range(3):
        # the id this step will draw: same seed and device step counter as the step's own draw
        nid = torch.zeros(1, dtype=torch.int64, device="cuda")
        ops.gbce_draw(E, nid, torch.zeros(128, tr_g.spec.Dp, dtype=torch.bfloat16, device="cuda"), None,
                      seed=tr_g.eng.drop_seed, step=tr_g.eng.step_state[3:4])
        n = int(nid)
        cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
        other = n % data.itemnum + 1
        for key in ("seq", "pos"):
            cb[key] = torch.where(cb[key] == n, torch.full_like(cb[key], other), cb[key])
        cb["neg"] = torch.where(cb["pos"] != 0, torch.full_like(cb["neg"], n), torch.zeros_like(cb["neg"]))
        lg = float(tr_g.step(cb))
        assert int(tr_g._gbce_ws["ids"][0]) == n
        lb = float(tr_b.step(cb))
        assert abs(lg - lb) < 3e-3 * max(1.0, abs(lb)), (step, lg, lb)
    ref_sd = {k: v.detach().cpu() for k, v in m_b.state_dict().items()}
    _check_tensors(m_g.state_dict(), ref_sd, sd0, 6.5e-3)     # Adam turns bf16 noise in near-zero gradients into sign flips


@pytest.mark.gpu
def test_autograd_loss_matches_oracle():
    from srfrd_b200.losses import sampled_gbce
    R, N, D, k, L = 400, 2000, 48, 100, 50
    h, E, pos, negs, seqs, w = _case(R, N, D, k, seed=3, L=L)
    hh, EE = h.view(8, 50, 48).clone().requires_grad_(True), E.clone().requires_grad_(True)
    loss = sampled_gbce(hh, EE, pos.view(8, 50), negs, w.view(8, 50), 0.5, seqs)
    (2.0 * loss).backward()
    ref = gbce_oracle(h, E, pos, negs, w, 0.5, _mask(seqs, negs, L, R))
    assert abs(float(loss) - ref[0]) <= 1e-4 + 1e-4 * abs(ref[0])
    for got, want in ((hh.grad.view(R, D), 2 * ref[1]), (EE.grad, 2 * ref[2])):
        rel, cos = _rel_cos(got, want)
        assert rel <= REL and cos >= COS
    assert torch.equal(EE.grad[0], torch.zeros(48, device="cuda"))


@pytest.mark.gpu
def test_refusals_before_any_launch():
    from srfrd_b200 import _lib
    from srfrd_b200 import SRFR_model as M
    from srfrd_b200.losses import sampled_gbce
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, smp = _c2_like()
    c0 = _lib.launch_count
    with pytest.raises(ValueError, match="SRFRN"):
        FusedTrainer(_model("SRFRN", data.itemnum), loss="gbce")
    for kw in (dict(num_negatives=0), dict(num_negatives=257), dict(gbce_t=-0.5), dict(gbce_t=1.01)):
        with pytest.raises(ValueError, match="gbce"):
            FusedTrainer(_model("SRFR", data.itemnum), loss="gbce", **kw)
    with pytest.raises(ValueError, match="2 items"):
        FusedTrainer(M.SASRec(1, 50, 64, 0.0, 1, 1, "cuda").to("cuda"), loss="gbce")
    with pytest.raises(ValueError, match="width"):
        FusedTrainer(M.SASRec(data.itemnum, 50, 272, 0.0, 1, 1, "cuda").to("cuda"), loss="gbce")
    for loss in ("bce", "ce"):
        for kw in (dict(num_negatives=64), dict(gbce_t=0.5)):
            with pytest.raises(ValueError, match="num_negatives"):
                FusedTrainer(_model("SRFR", data.itemnum), loss=loss, **kw)
    E = torch.randn(101, 64, device="cuda")
    h = torch.randn(4, 5, 64, device="cuda")
    t = torch.ones(4, 5, dtype=torch.int64, device="cuda")
    negs = torch.arange(1, 9, device="cuda")
    for bad in (101, -1):
        tb = t.clone()
        tb[1, 2] = bad
        with pytest.raises(ValueError, match="targets"):
            sampled_gbce(h, E, tb, negs)
    for bad in (0, 101):
        nb = negs.clone()
        nb[3] = bad
        with pytest.raises(ValueError, match="negatives"):
            sampled_gbce(h, E, t, nb)
    with pytest.raises(ValueError, match="gbce"):
        sampled_gbce(h, E, t, torch.ones(257, dtype=torch.int64, device="cuda"))
    with pytest.raises(ValueError, match="gbce"):
        sampled_gbce(h, E, t, negs, t=2.0)
    assert _lib.launch_count == c0
    tr = FusedTrainer(_model("SRFR", data.itemnum), loss="gbce")
    cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(64).items()}
    c1 = _lib.launch_count
    with pytest.raises(ValueError, match="w_neg"):
        tr.step(cb, w_neg=torch.ones(64, 50, device="cuda"))
    assert _lib.launch_count == c1


@pytest.mark.gpu
def test_bce_step_launches_unchanged_and_gbce_adds_two_calls():
    from srfrd_b200 import _lib
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, smp = _c2_like()
    cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
    counts = []
    for loss in ("bce", "ce", "gbce"):
        tr = FusedTrainer(_model("SRFR", data.itemnum), use_graph=False, loss=loss)
        tr.step(cb)
        c0 = _lib.launch_count
        tr.step(cb)
        counts.append(_lib.launch_count - c0)
    assert counts[1] == counts[0] + 2, counts        # CE's own test: the BCE step is the same as before
    # score_loss_fused (1 kernel) -> f32_to_bf16_split + gbce_draw (1 kernel) + gbce_loss (DH, DN and scatter kernels)
    assert counts[2] == counts[0] + 2, counts
