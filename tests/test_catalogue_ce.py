"""Full-catalogue softmax cross-entropy (csrc/catalogue_ce.cu, losses.catalogue_cross_entropy, FusedTrainer(loss="ce")).

The logits are predict()'s (SRFR_model.py:144-152 with label = arange(1, N+1)) at every position with a target:
loss = sum_t w_t (logsumexp_j z_tj - z_t,pos) / sum_t w_t over items j = 1..N; there is no reference counterpart.

CPU: the fp64 oracle below against F.cross_entropy over predict logits, the plan's refusals, and a model check of the
kernel's mbarrier protocol.  GPU: the three kernels against the oracle on the same bf16-rounded operands, exact
properties, a 1 M-item scale run, FusedTrainer(loss="ce") against an autograd + Adam oracle, the drop-in loop, refusals.
"""
import math
import random

import numpy as np
import pytest
import torch
import torch.nn.functional as F


# ------------------------------------------------------------------------------------------------------------ oracle
def ce_oracle(h, E, target, w=None, rows=None, items=None, chunk=256):
    """float64 cross-entropy on bf16-rounded operands, on h's device.  h (R, D), E (N + 1, D), target (R,) in 0..N
    (0 = no term), w (R,) or None (= 1[target != 0]).  Returns (loss, lse (R,), dh (R, D), dE (N + 1, D)); `rows` /
    `items` restrict dh / dE to those indices (the loss, lse and normaliser always cover every row)."""
    hb, Eb = h.to(torch.bfloat16).double(), E.to(torch.bfloat16).double()
    R, D = hb.shape
    N = Eb.shape[0] - 1
    target = target.long()
    valid = target != 0
    wv = valid.double() if w is None else w.double() * valid
    norm = float(wv.sum())
    inv = 1.0 / norm if norm > 0 else 0.0
    lse = torch.empty(R, dtype=torch.float64, device=h.device)
    loss = 0.0
    for s in range(0, R, chunk):
        z = hb[s:s + chunk] @ Eb[1:].T
        lse[s:s + chunk] = torch.logsumexp(z, 1)
        zt = z.gather(1, (target[s:s + chunk].clamp(min=1) - 1)[:, None])[:, 0]
        loss += float((wv[s:s + chunk] * (lse[s:s + chunk] - zt)).sum())
    loss *= inv
    coef = wv * inv
    rsel = torch.arange(R, device=h.device) if rows is None else rows.to(h.device)
    dh = torch.zeros(len(rsel), D, dtype=torch.float64, device=h.device)
    for s in range(0, len(rsel), chunk):
        r = rsel[s:s + chunk]
        p = torch.exp(hb[r] @ Eb[1:].T - lse[r][:, None])
        p[torch.arange(len(r), device=h.device), target[r].clamp(min=1) - 1] -= valid[r].double()
        dh[s:s + chunk] = coef[r][:, None] * (p @ Eb[1:])
    isel = torch.arange(1, N + 1, device=h.device) if items is None else items.to(h.device)
    dE = torch.zeros(len(isel), D, dtype=torch.float64, device=h.device)
    Es = Eb[isel]
    for s in range(0, R, chunk):
        p = torch.exp(hb[s:s + chunk] @ Es.T - lse[s:s + chunk][:, None])
        p -= (target[s:s + chunk][:, None] == isel[None, :]).double() * valid[s:s + chunk, None].double()
        dE += (coef[s:s + chunk][:, None] * p).T @ hb[s:s + chunk]
    dE[isel == 0] = 0
    return loss, lse, dh, dE


def test_oracle_matches_cross_entropy_over_predict_logits():
    g = torch.Generator().manual_seed(0)
    R, N, D = 37, 211, 24
    h = torch.randn(R, D, generator=g, dtype=torch.float64).bfloat16().double().requires_grad_(True)
    E = torch.randn(N + 1, D, generator=g, dtype=torch.float64).bfloat16().double().requires_grad_(True)
    t = torch.randint(1, N + 1, (R,), generator=g)
    t[::5] = 0
    w = torch.rand(R, generator=g, dtype=torch.float64)
    for weights in (None, w):
        logits = h @ E[1:].T                                   # predict(..., label = arange(1, N + 1))
        keep = t != 0
        wk = torch.ones(int(keep.sum()), dtype=torch.float64) if weights is None else weights[keep]
        ce = F.cross_entropy(logits[keep], t[keep] - 1, reduction="none")
        ref = (wk * ce).sum() / wk.sum()
        gh, gE = torch.autograd.grad(ref, (h, E))
        loss, lse, dh, dE = ce_oracle(h.detach(), E.detach(), t, weights)
        assert abs(loss - float(ref.detach())) < 1e-12
        assert torch.allclose(lse, torch.logsumexp(logits.detach(), 1), atol=1e-12)
        assert torch.allclose(dh, gh, atol=1e-13) and torch.allclose(dE[:, :], gE[1:], atol=1e-13)
        assert float(gE[0].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------------------- plan
def test_plan_reports_and_refuses_before_any_launch():
    from srfrd_b200 import ops
    for Dp in (16, 64, 128, 192, 256):
        smem, stages, tmem = ops.catalogue_ce_plan(Dp)
        kb = (Dp + 63) // 64
        assert stages >= 2 and tmem == 512
        assert smem == (kb + 2 + stages * kb) * 16384 + 1280 and smem <= 227 * 1024
    for Dp in (0, 8, 24, 272, 512):
        with pytest.raises(RuntimeError, match="Dp"):
            ops.catalogue_ce_plan(Dp)
    from srfrd_b200.losses import check_ce_width
    assert check_ce_width(250) == 256
    with pytest.raises(ValueError):
        check_ce_width(257)


# --------------------------------------------------------------------------------------------------- protocol model
class _Bar:
    def __init__(self, count):
        self.count, self.arrived, self.tx, self.phase = count, 0, 0, 0

    def arrive(self):
        self.arrived += 1
        assert self.arrived <= self.count
        if self.arrived == self.count and self.tx == 0:
            self.arrived, self.phase = 0, self.phase + 1

    def passes(self, parity):            # try_wait.parity: the last completed phase has this parity (fresh: parity 1)
        return ((self.phase - 1) & 1) == parity


def _ce_protocol(mode, nstream, stages, seed):
    """The three warp roles of catalogue_ce_kernel as generators over simulated mbarriers; asynchronous completions
    (TMA, tcgen05.commit) land after random delays.  Checks that every wait passes on the phase it means, that no ring
    slot, S buffer or X is overwritten while it is still read, and that everything terminates."""
    rng = random.Random(seed)
    full, empty = [_Bar(1) for _ in range(stages)], [_Bar(1) for _ in range(stages)]
    s_full, s_free = [_Bar(1) for _ in range(2)], [_Bar(8) for _ in range(2)]
    x_full, x_free, acc_full = _Bar(8), _Bar(1), _Bar(1)
    pending = []
    slot_data = [None] * stages       # streamed block held by each ring slot
    s_data = [None] * 2               # block whose S each TMEM buffer holds
    x_data = [None]
    log = []

    def later(fn):
        pending.append([rng.randint(1, 5), fn])

    def wait(bar, parity, want_phase):
        while not bar.passes(parity):
            yield
        assert bar.phase == want_phase, (bar.phase, want_phase)

    def producer():
        slot, ph = 0, 0
        for n in range(nstream):
            yield from wait(empty[slot], ph ^ 1, n // stages)
            assert slot_data[slot] is None
            slot_data[slot] = n

            def land(s=slot):
                full[s].arrive()
            later(land)
            slot += 1
            if slot == stages:
                slot, ph = 0, ph ^ 1

    def commit(bar, before=None):
        def fire():
            if before:
                before()
            bar.arrive()
        later(fire)

    def mma():
        slot, prev, ph = 0, 0, 0

        def out(m, st):
            yield from wait(x_full, m & 1, m + 1)
            assert x_data[0] == m and slot_data[st] == m

            def release(s=st):
                slot_data[s] = None
            commit(empty[st], release)
            commit(x_free)
        for n in range(nstream):
            buf = n & 1
            yield from wait(s_free[buf], ((n >> 1) & 1) ^ 1, n >> 1)
            yield from wait(full[slot], ph, n // stages + 1)
            assert slot_data[slot] == n and s_data[buf] is None
            s_data[buf] = n
            commit(s_full[buf])
            if mode == "lse":
                def release(s=slot):
                    slot_data[s] = None
                commit(empty[slot], release)
            if mode != "lse" and n > 0:
                yield from out(n - 1, prev)
            prev = slot
            slot += 1
            if slot == stages:
                slot, ph = 0, ph ^ 1
        if mode != "lse":
            yield from out(nstream - 1, prev)
            commit(acc_full)

    def softmax(wid):
        for n in range(nstream):
            buf = n & 1
            yield from wait(s_full[buf], (n >> 1) & 1, (n >> 1) + 1)
            assert s_data[buf] == n
            yield
            s_free[buf].arrive()
            if s_free[buf].arrived == 0:
                s_data[buf] = None
            if mode != "lse":
                yield from wait(x_free, (n & 1) ^ 1, n)
                x_data[0] = n
                x_full.arrive()
        if mode != "lse":
            yield from wait(acc_full, 0, 1)
        log.append(wid)

    roles = [producer(), mma()] + [softmax(w) for w in range(8)]
    live = list(roles)
    for _ in range(200000):
        if not live and not pending:
            break
        for ev in list(pending):
            ev[0] -= 1
            if ev[0] <= 0:
                pending.remove(ev)
                ev[1]()
        if live:
            r = rng.choice(live)
            try:
                next(r)
            except StopIteration:
                live.remove(r)
    assert not live and not pending, "deadlock"
    assert sorted(log) == list(range(8))


@pytest.mark.parametrize("mode", ["lse", "dh", "de"])
@pytest.mark.parametrize("stages", [2, 3, 5, 8])
def test_pipeline_protocol_model(mode, stages):
    for seed in range(6):
        for nstream in (1, 2, 3, 7, 12):
            _ce_protocol(mode, nstream, stages, seed * 100 + nstream)


# ------------------------------------------------------------------------------------------------------------- GPU
class _RowMap:
    """A packed row map as ops.catalogue_ce_* read it (row_tok, rows, cap)."""

    def __init__(self, row_tok, rows):
        self.row_tok = torch.tensor(row_tok, dtype=torch.int32, device="cuda")
        self.rows = torch.tensor([rows, 0, 0, 0], dtype=torch.int32, device="cuda")
        self.cap = len(row_tok)


def _run(h, E, pos, w=None, plan=None, nan_dh=True, want_dh=True, want_dE=True):
    """h (cap, D) fp32, E (N + 1, D) fp32 on cuda -> (loss, lse, dh, dE) from the kernels."""
    from srfrd_b200 import ops
    from srfrd_b200.losses import _bf16_rows
    D = E.shape[1]
    Dp = (D + 15) // 16 * 16
    hb, tb = _bf16_rows(h.contiguous(), Dp), _bf16_rows(E.contiguous(), Dp)
    norm = torch.zeros(2, device="cuda")
    ops.weight_sums(pos, w, None, norm)
    acc = torch.zeros(2, device="cuda")
    lse = torch.full((h.shape[0],), float("nan"), device="cuda")
    ops.catalogue_ce_fwd(hb, tb, pos, w, lse, acc, plan)
    dh = torch.full((h.shape[0], D), float("nan") if nan_dh else 0.0, device="cuda") if want_dh else None
    dE = torch.zeros(E.shape[0], D, device="cuda") if want_dE else None
    ops.catalogue_ce_bwd(hb, tb, pos, w, norm, lse, dh, dE, D, plan)
    torch.cuda.synchronize()
    n = float(norm[0])
    return (float(acc[0]) / n if n > 0 else 0.0), lse, dh, dE, float(acc[1])


def _data(R, N, D, seed, zero_every=7):
    g = torch.Generator(device="cuda").manual_seed(seed)
    h = torch.randn(R, D, device="cuda", generator=g) * (3.0 / math.sqrt(D))
    E = torch.randn(N + 1, D, device="cuda", generator=g)
    E[0] = 0
    pos = torch.randint(1, N + 1, (R,), device="cuda", generator=g)
    pos[::zero_every] = 0
    return h, E, pos


def _rel_cos(got, ref):
    got, ref = got.double().flatten(), ref.double().flatten()
    rel = float((got - ref).norm() / ref.norm().clamp_min(1e-300))
    cos = float(torch.dot(got, ref) / (got.norm() * ref.norm()).clamp_min(1e-300))
    return rel, cos


# dh / dE bars against the fp64 oracle on the same bf16 operands (P enters the second product as bf16)
REL, COS = 1e-2, 0.999


def _close(got, ref, what):
    if float(ref.abs().max()) == 0.0:                  # N = 1: p = 1 at the target, every gradient is 0
        assert float(got.abs().max()) <= 1e-5, (what, float(got.abs().max()))
        return
    rel, cos = _rel_cos(got, ref)
    assert rel <= REL and cos >= COS, (what, rel, cos)


def _check(res, ref, rows_sel=None):
    loss, lse, dh, dE, acc1 = res
    rloss, rlse, rdh, rdE = ref
    assert acc1 == 0.0
    assert abs(loss - rloss) <= 1e-4 + 1e-4 * abs(rloss), (loss, rloss)
    sel = slice(None) if rows_sel is None else rows_sel
    assert torch.allclose(lse[sel].double(), rlse[sel], atol=1e-4, rtol=1e-4), float((lse[sel].double() - rlse[sel]).abs().max())
    if dh is not None:
        _close(dh[sel], rdh, "dh")
    if dE is not None:
        _close(dE[1:], rdE, "dE")
        assert torch.equal(dE[0], torch.zeros_like(dE[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 127, 128, 129, 12101, 150000])
@pytest.mark.parametrize("D", [16, 64, 128, 256])
def test_kernels_match_oracle_dense(N, D):
    if N == 150000 and D > 64:
        pytest.skip("the 150 k table is covered at D = 16 and 64")
    R = 300 if N < 150000 else 200
    h, E, pos = _data(R, N, D, seed=N + D)
    w = torch.rand(R, device="cuda") * (pos != 0)
    for weights in (None, w):
        res = _run(h, E, pos, weights)
        _check(res, ce_oracle(h, E, pos, weights))


@pytest.mark.gpu
@pytest.mark.parametrize("D", [16, 64, 200])
def test_kernels_match_oracle_packed_row_map(D):
    """Rows of a packed layout: filler rows (-1), a device row count below the capacity (rows beyond it untouched),
    tokens in shuffled order; pos / w indexed by the dense token."""
    N, T = 3001, 700
    g = torch.Generator(device="cuda").manual_seed(D)
    h, E, _ = _data(640, N, D, seed=D + 1)
    pos = torch.randint(0, N + 1, (T,), device="cuda", generator=g)
    w = torch.rand(T, device="cuda", generator=g) * (pos != 0)
    rng = np.random.default_rng(D)
    toks = rng.permutation(T)[:450].tolist()
    row_tok = []
    for i, tk in enumerate(toks):
        row_tok.append(tk)
        if i % 9 == 0:
            row_tok.append(-1)                     # filler / pad representative
    rows = len(row_tok)
    row_tok += [-1] * (640 - rows)
    plan = _RowMap(row_tok, rows)
    res = _run(h, E, pos, w, plan)
    rt = torch.tensor(row_tok[:rows], device="cuda")
    tgt = torch.where(rt >= 0, pos[rt.clamp(min=0)], torch.zeros_like(rt))
    wr = torch.where(rt >= 0, w[rt.clamp(min=0)], torch.zeros_like(w[:rows]))
    ref = list(ce_oracle(h[:rows], E, tgt, wr))
    # the kernel divides by sum(w) over ALL tokens (the trainer's normaliser); the oracle by the mapped rows' sum
    scale = float(wr.sum()) / float(w.sum())
    ref[0] *= scale; ref[2] = ref[2] * scale; ref[3] = ref[3] * scale
    _check(res, ref, rows_sel=slice(0, rows))
    assert torch.isnan(res[2][rows:]).all(), "rows beyond the device row count must stay untouched"
    assert torch.equal(res[2][:rows][rt < 0], torch.zeros_like(res[2][:rows][rt < 0]))


@pytest.mark.gpu
def test_exact_properties():
    N, D, R = 5000, 64, 513
    h, E, pos = _data(R, N, D, seed=11)
    w = torch.rand(R, device="cuda") * (pos != 0)
    w[::5] = 0                                         # zero weights on rows that do have a target
    a = _run(h, E, pos, w)
    b = _run(h, E, pos, w)
    assert torch.equal(a[2], b[2]) and torch.equal(a[3], b[3]), "dh / dE differ between two launches"
    assert torch.equal(a[3][0], torch.zeros(D, device="cuda"))
    # rows with w = 0 change nothing: give them other hidden states and targets
    z = (w == 0)
    h2, pos2 = h.clone(), pos.clone()
    h2[z] = torch.randn(int(z.sum()), D, device="cuda") * 10
    pos2[z & (pos != 0)] = 1
    c = _run(h2, E, pos2, w)
    assert torch.equal(c[3], a[3]) and torch.equal(c[2][~z], a[2][~z]) and torch.equal(c[2][z], torch.zeros_like(c[2][z]))
    assert abs(c[0] - a[0]) <= 1e-6 * abs(a[0])
    # every weight zero: loss 0, zero gradients, no NaN
    d = _run(h, E, pos, torch.zeros(R, device="cuda"))
    assert d[0] == 0.0 and torch.equal(d[2], torch.zeros_like(d[2])) and torch.equal(d[3], torch.zeros_like(d[3]))


@pytest.mark.gpu
def test_scale_one_million_items():
    N, D, R = 1_000_000, 64, 4096
    h, E, pos = _data(R, N, D, seed=5, zero_every=13)
    res = _run(h, E, pos)
    rows = torch.arange(0, R, 61, device="cuda")
    items = torch.cat([torch.arange(1, 300, device="cuda"), pos[pos != 0][:200], torch.arange(N - 100, N + 1, device="cuda")])
    ref = ce_oracle(h, E, pos, rows=rows, items=items)
    loss, lse, dh, dE, _ = res
    assert abs(loss - ref[0]) <= 1e-4 + 1e-4 * abs(ref[0])
    assert torch.allclose(lse.double(), ref[1], atol=1e-4, rtol=1e-4)
    for got, want in ((dh[rows], ref[2]), (dE[items], ref[3])):
        rel, cos = _rel_cos(got, want)
        assert rel <= REL and cos >= COS, (rel, cos)


# ------------------------------------------------------------------------------------------------------- training
def _oracle_ce(O, l2=0.0):
    class OracleCE(O.OracleTrainer):
        """The oracle step with the cross-entropy objective over predict's logits (fp32 autograd + torch Adam)."""

        def loss(self, batch, w_pos=None, w_neg=None):
            h = O.encode(self.sd, self.kind, batch["seq"], batch["rsq"], self.num_heads)
            E = self.sd[O._emb_keys(self.kind)[0]]
            t = batch["pos"]
            z = h @ E[1:].T
            zt = z.gather(-1, (t.clamp(min=1) - 1)[..., None])[..., 0]
            w = (t != 0).float() if w_pos is None else w_pos * (t != 0)
            return (w * (torch.logsumexp(z, -1) - zt)).sum() / w.sum()

        def step(self, batch, w_pos=None, w_neg=None):
            self.opt.zero_grad(set_to_none=True)
            loss = self.loss(batch, w_pos)
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
    return OracleCE


CASES = [("SRFR", True, True), ("SRFR", False, False), ("SASRec", True, False), ("SASRec", False, True),
         ("SRFU_F", True, True), ("SRFU_F", False, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,packed,graph", CASES)
def test_fused_trainer_ce_matches_oracle(kind, packed, graph):
    from oracle import srfrd_oracle as O
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, smp = _c2_like()
    m = _model(kind, data.itemnum)
    heads = 2 if kind == "SASRec" else 1
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    orc = _oracle_ce(O)(sd0, kind, heads)
    tr = FusedTrainer(m, use_graph=graph, packed=packed, loss="ce")
    for step in range(5):
        tb = {k: torch.from_numpy(v) for k, v in smp.next_batch(256).items()}
        ref = orc.step(tb)
        loss = float(tr.step({k: v.cuda() for k, v in tb.items()}))
        assert math.isfinite(loss) and abs(loss - ref) < 5e-3, f"{kind} step {step}: {loss} vs oracle {ref}"
    _check_tensors(m.state_dict(), orc.state_dict(), sd0, 2 * 5 * 1e-3 + 5e-4)


@pytest.mark.gpu
def test_fused_trainer_ce_step_sampled_soft_weights_l2():
    from oracle import srfrd_oracle as O
    from srfrd_b200.trainer import DeviceSampler, FusedTrainer
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, _ = _c2_like()
    smp = DeviceSampler(data, 50, "cuda", seed=5)
    m = _model("SRFR", data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    orc = _oracle_ce(O, l2=1e-4)(sd0, "SRFR", 1)
    tr = FusedTrainer(m, use_graph=True, loss="ce", l2_emb=1e-4)
    for step in range(5):
        loss = float(tr.step_sampled(smp, 256, policy="soft"))
        tb = {k: tr._static[k].cpu().clone() for k in FusedTrainer._KEYS}
        w = tr._static["w_pos"].cpu().clone()
        assert float(w.min()) >= 0 and 0 < float(w[tb["pos"] != 0].mean()) < 1
        ref = orc.step(tb, w)
        assert math.isfinite(loss) and abs(loss - ref) < 5e-3, f"step {step}: {loss} vs oracle {ref}"
    _check_tensors(m.state_dict(), orc.state_dict(), sd0, 2 * 5 * 1e-3 + 5e-4)


@pytest.mark.gpu
@pytest.mark.parametrize("packed", [True, False])
def test_drop_in_loop_agrees_with_fused_trainer(packed):
    from srfrd_b200.losses import catalogue_cross_entropy
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, smp = _c2_like()
    m, m_ref = _model("SRFR", data.itemnum), _model("SRFR", data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    tr = FusedTrainer(m, use_graph=True, packed=packed, loss="ce")
    opt = torch.optim.Adam(m_ref.parameters(), lr=1e-3, betas=(0.9, 0.98))
    table = dict(m_ref.named_parameters())[m_ref.spec.item_key]
    for step in range(3):
        cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
        loss = float(tr.step(cb))
        h, _, _ = m_ref(None, cb["seq"], cb["rsq"])
        opt.zero_grad()
        ref = catalogue_cross_entropy(h, table, cb["pos"])
        ref.backward()
        opt.step()
        assert abs(loss - float(ref.detach())) < 5e-3, f"step {step}: {loss} vs drop-in {float(ref.detach())}"
    ref_sd = {k: v.detach().cpu() for k, v in m_ref.state_dict().items()}
    _check_tensors(m.state_dict(), ref_sd, sd0, 6.5e-3)


@pytest.mark.gpu
def test_autograd_loss_matches_oracle_and_kernels():
    from srfrd_b200.losses import catalogue_cross_entropy
    h, E, pos = _data(400, 2000, 48, seed=3)
    w = torch.rand(400, device="cuda")
    hh, EE = h.view(8, 50, 48).clone().requires_grad_(True), E.clone().requires_grad_(True)
    loss = catalogue_cross_entropy(hh, EE, pos.view(8, 50), w.view(8, 50))
    (2.0 * loss).backward()
    ref = ce_oracle(h, E, pos, w * (pos != 0))
    assert abs(float(loss) - ref[0]) <= 1e-4 + 1e-4 * abs(ref[0])
    for got, want in ((hh.grad.view(400, 48), 2 * ref[2]), (EE.grad[1:], 2 * ref[3])):
        rel, cos = _rel_cos(got, want)
        assert rel <= REL and cos >= COS
    assert torch.equal(EE.grad[0], torch.zeros(48, device="cuda"))


@pytest.mark.gpu
def test_refusals_before_any_launch():
    from srfrd_b200 import _lib
    from srfrd_b200 import SRFR_model as M
    from srfrd_b200.losses import catalogue_cross_entropy
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, smp = _c2_like()
    c0 = _lib.launch_count
    with pytest.raises(ValueError, match="SRFRN"):
        FusedTrainer(_model("SRFRN", data.itemnum), loss="ce")
    with pytest.raises(ValueError, match="width"):
        FusedTrainer(M.SASRec(data.itemnum, 50, 272, 0.0, 1, 1, "cuda").to("cuda"), loss="ce")
    with pytest.raises(ValueError):
        FusedTrainer(_model("SRFR", data.itemnum), loss="softmax")
    E = torch.randn(101, 64, device="cuda")
    h = torch.randn(4, 5, 64, device="cuda")
    for bad in (101, -1):
        t = torch.ones(4, 5, dtype=torch.int64, device="cuda")
        t[1, 2] = bad
        with pytest.raises(ValueError, match="targets"):
            catalogue_cross_entropy(h, E, t)
    with pytest.raises(ValueError, match="width"):
        catalogue_cross_entropy(torch.randn(3, 272, device="cuda"), torch.randn(11, 272, device="cuda"),
                                torch.ones(3, dtype=torch.int64, device="cuda"))
    assert _lib.launch_count == c0
    tr = FusedTrainer(_model("SRFR", data.itemnum), loss="ce")
    cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(64).items()}
    c1 = _lib.launch_count
    with pytest.raises(ValueError, match="w_neg"):
        tr.step(cb, w_neg=torch.ones(64, 50, device="cuda"))
    assert _lib.launch_count == c1


@pytest.mark.gpu
def test_bce_step_launches_unchanged_and_ce_adds_its_three_calls():
    from srfrd_b200 import _lib
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, smp = _c2_like()
    cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
    counts = []
    for loss in ("bce", "ce"):
        tr = FusedTrainer(_model("SRFR", data.itemnum), use_graph=False, loss=loss)
        tr.step(cb)
        c0 = _lib.launch_count
        tr.step(cb)
        counts.append(_lib.launch_count - c0)
    assert counts[1] == counts[0] + 2, counts        # score_loss_fused -> cast + CE forward + CE backward
