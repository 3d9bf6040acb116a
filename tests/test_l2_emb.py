"""The reference's l2_emb regulariser in FusedTrainer (trainer.py:31-39): loss += l2 * sum_p ||p||_2 over every tensor of
model.parameters(), gradient l2 * p / ||p|| (0 for a zero tensor), applied before Adam -- including to the pad row and to
item rows no batch touches, which then drift at Adam speed.

Host tests: the segment table of the flat buffer and the chunk plan.  GPU tests: the norm kernel against float64 torch,
FusedTrainer against the oracle (autograd + torch Adam) and against the drop-in autograd loop on our own module."""
import math

import numpy as np
import pytest
import torch

from srfrd_b200.engine import FlatParams, ModelSpec

# (kind, D, F, n_labels, num_blocks): every model kind, plus the reference's ragged widths (45 + 5, 50 + 10)
SPECS = [("SRFR", 64, 16, 0, 2), ("SRFRN", 64, 16, 0, 2), ("SASRec", 64, 0, 0, 2), ("SRFU_B", 64, 0, 51, 2),
         ("SRFU_F", 64, 0, 51, 3), ("SRFU_R", 64, 0, 51, 2), ("SRFR", 45, 5, 0, 2), ("SRFR", 50, 10, 0, 4)]


@pytest.mark.parametrize("kind,D,F,nl,nb", SPECS)
def test_segments_cover_exactly_the_reference_state_dict(kind, D, F, nl, nb):
    from oracle import srfrd_oracle as O
    spec = ModelSpec(kind, 301, 50, D, F, nl, nb)
    P = FlatParams(spec, "cpu")
    segs = P.segments()
    sd = O.init_state_dict(kind, 301, 50, D, F, nl, nb)
    names = [n for n, _ in spec.param_shapes()]
    assert len(segs) == len(names) == len(sd)
    assert {n: s[1] for n, s in zip(names, segs)} == {k: v.numel() for k, v in sd.items()}
    end = 0
    for off, n in segs:                                 # 4-aligned, increasing; padding lies only between segments
        assert off % 4 == 0 and off >= end and off - end < 4
        end = off + n
    assert P.numel - end < 4 and P.numel % 4 == 0


def test_chunk_plan_counts_chunks_per_tensor_and_rejects_bad_tables():
    import ctypes as C
    from srfrd_b200 import _lib
    lib = _lib.load()
    seg = [0, 5, 8, 8192, 8200, 8193, 16396, 0]
    host = (C.c_int64 * len(seg))(*seg)
    out = C.c_int64(-1)
    assert lib.srfrd_param_l2_plan(host, 4, C.byref(out)) == 0 and out.value == 1 + 1 + 2 + 0
    bad = (C.c_int64 * 4)(0, 8, 6, 4)                    # second tensor unaligned and overlapping the first
    assert lib.srfrd_param_l2_plan(bad, 2, C.byref(out)) != 0
    assert lib.srfrd_param_l2_plan(host, 0, C.byref(out)) != 0


# ------------------------------------------------------------------------------------------------------------- GPU
def _seg_norms64(p, segs):
    return [float(torch.linalg.vector_norm(p[o:o + n].double())) for o, n in segs]


@pytest.mark.gpu
def test_norm_kernel_matches_float64_and_is_deterministic():
    from srfrd_b200 import ops
    numels = [7, 0 + 6, 1, 4 * 37 + 1, 4 * 11 + 2, 4 * 5 + 3, 64 << 20, 8192, 8193, 3]
    segs, off = [], 0
    for n in numels:
        segs.append((off, n))
        off += (n + 3) // 4 * 4
    g = torch.Generator(device="cuda").manual_seed(0)
    p = torch.randn(off, device="cuda", generator=g) * 0.05
    p[segs[1][0]:segs[1][0] + segs[1][1]] = 0.0                       # a zero tensor
    for (o, n), (o2, _) in zip(segs, segs[1:] + [(off, 0)]):
        p[o + n:o2] = float("nan")                                     # padding is never read as data
    l2 = 1e-4
    k = ops.ParamL2(segs, l2, "cuda")
    k.launch(p)
    torch.cuda.synchronize()
    coef1, reg1 = k.coef.clone(), k.reg.clone()
    ref = _seg_norms64(p, segs)
    for t, r in enumerate(ref):
        want = l2 / r if r > 0 else 0.0
        if want == 0.0:
            assert float(coef1[t]) == 0.0, t
        else:
            assert abs(float(coef1[t]) - want) <= 1e-6 * want, (t, float(coef1[t]), want)
    want_reg = l2 * math.fsum(ref)
    assert abs(float(reg1) - want_reg) <= 1e-6 * want_reg
    assert torch.isfinite(coef1).all()
    k.launch(p)
    torch.cuda.synchronize()
    assert torch.equal(k.coef, coef1) and torch.equal(k.reg, reg1)
    k.coef.zero_(); k.reg.zero_()
    gr = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        k.launch(p)                                                    # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    k.coef.zero_(); k.reg.zero_()
    with torch.cuda.graph(gr):
        k.launch(p)
    gr.replay()
    torch.cuda.synchronize()
    assert torch.equal(k.coef, coef1) and torch.equal(k.reg, reg1)


def _c2_like(B=256, N=3000, seed=7):
    from srfrd_b200 import synth
    data = synth.make_interactions(seed, 4000, N, 5, 4.0, 50)
    return data, synth.BatchSampler(data, 50, 3)


def _srfr_reference_init(N, seed=0):
    from srfrd_b200 import SRFR_model as M
    torch.manual_seed(seed)
    m = M.SRFR(N, 50, 64, 16, 0.0, 2, 1, "cuda")
    for _, p in m.named_parameters():                      # trainer.py:364-369: xavier_normal_, biases stay 0
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    return m.to("cuda")


def _oracle_l2(O):
    class OracleL2(O.OracleTrainer):
        """The oracle step with the regulariser: its gradient is added after the pad rows' data gradient is zeroed,
        because nn.Embedding(padding_idx=0) drops only the lookup gradient of row 0, not the norm's."""

        def __init__(self, sd, kind, heads, l2):
            super().__init__(sd, kind, heads)
            self.l2 = l2

        def step(self, batch, w_pos=None, w_neg=None):
            self.opt.zero_grad(set_to_none=True)
            loss = self.loss(batch, w_pos, w_neg)
            loss.backward()
            self._zero_pad_rows()
            params = list(self.sd.values())
            reg = self.l2 * sum(torch.linalg.vector_norm(p) for p in params)
            for p, g in zip(params, torch.autograd.grad(reg, params)):
                p.grad = g if p.grad is None else p.grad + g
            self.opt.step()
            return float(loss.detach()) + float(reg.detach())
    return OracleL2


def _touched(batches, key_ids=("seq", "pos", "neg")):
    ids = set()
    for b in batches:
        for k in key_ids:
            ids.update(np.unique(np.asarray(b[k])).tolist())
    return ids


def _untouched_rows(n_rows, touched):
    rows = [r for r in range(n_rows) if r not in touched or r == 0]
    return torch.tensor(rows, dtype=torch.int64)


def _check_tensors(got_sd, ref_sd, sd0, drift_max):
    for k, ref in ref_sd.items():
        got, p0 = got_sd[k].cpu().flatten(), sd0[k].flatten()
        ref = ref.flatten()
        if k.endswith("in_proj_bias"):                     # the key third's data gradient is rounding noise
            H = ref.numel() // 3
            sel = torch.cat([torch.arange(0, H), torch.arange(2 * H, 3 * H)])
            got, ref, p0 = got[sel], ref[sel], p0[sel]
        assert float((got - ref).abs().max()) <= drift_max, (k, float((got - ref).abs().max()))
        u, v = got - p0, ref - p0
        if u.numel() >= 64:
            cos = float(torch.dot(u, v) / (u.norm() * v.norm() + 1e-30))
            assert cos > 0.9, f"{k}: update direction cosine {cos:.3f}"


@pytest.mark.gpu
@pytest.mark.parametrize("l2", [1e-4, 1e-2])
@pytest.mark.parametrize("policy", ["soft", "none"])
def test_fused_l2_matches_oracle(l2, policy):
    """5 steps from the reference init: loss (with the regulariser) within 5e-3; item rows without a data gradient --
    row 0 included -- equal to the oracle's to 1e-6 after every step (pure fp32 Adam on coef * p); every other tensor
    within the bars of test_fused_trainer_* (direction cosine > 0.9; drift 6.5e-3 after 3 steps, 2 * 5 * lr + 5e-4
    after 5: an element whose data gradient sits below the bf16 noise floor may take the opposite sign each step)."""
    from oracle import srfrd_oracle as O
    from srfrd_b200.trainer import FusedTrainer, discriminator_weights
    data, smp = _c2_like()
    m = _srfr_reference_init(data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    orc = _oracle_l2(O)(sd0, "SRFR", 1, l2)
    tr = FusedTrainer(m, use_graph=True, l2_emb=l2)
    key = tr.spec.item_key
    batches = []
    for step in range(5):
        nb = smp.next_batch(256)
        batches.append(nb)
        tb = {k: torch.from_numpy(v) for k, v in nb.items()}
        w_cpu = O.discriminator_weights(tb["pos"], tb["p_fake"], policy) if policy != "none" else None
        ref_loss = orc.step(tb, w_cpu)
        cb = {k: v.cuda() for k, v in tb.items()}
        w = discriminator_weights(cb["pos"], cb["p_fake"], policy) if policy != "none" else None
        loss = float(tr.step(cb, w_pos=w))
        assert math.isfinite(loss) and abs(loss - ref_loss) < 5e-3, f"step {step}: {loss} vs oracle {ref_loss}"
        assert torch.isfinite(tr.P.data).all()
        rows = _untouched_rows(data.itemnum + 1, _touched(batches))
        got = m.state_dict()[key].cpu()[rows]
        ref = orc.sd[key].detach()[rows]
        assert len(rows) > 20
        assert float((got - ref).abs().max()) <= 1e-6, f"step {step}: untouched rows {float((got - ref).abs().max()):.3e}"
        assert float((got[0] - sd0[key][0]).abs().median()) > 0.5e-3   # ... and they did move, the pad row too
        if step == 2:
            _check_tensors(m.state_dict(), orc.state_dict(), sd0, 6.5e-3)
    _check_tensors(m.state_dict(), orc.state_dict(), sd0, 2 * 5 * 1e-3 + 5e-4)


@pytest.mark.gpu
def test_loss_gains_exactly_the_regulariser():
    """Same parameters and batch: loss(l2 = x) - loss(l2 = 0) == x * sum_p ||p||.  x = 1 keeps the term large next to
    the fp32 resolution of the ~1.4 BCE part it is added to; the kernel's own reg is checked at l2 = 1e-4."""
    from srfrd_b200.trainer import FusedTrainer
    data, smp = _c2_like()
    nb = smp.next_batch(256)
    cb = {k: torch.from_numpy(v).cuda() for k, v in nb.items()}
    m0, m1, m2 = (_srfr_reference_init(data.itemnum) for _ in range(3))
    norms = _seg_norms64(m0.flat_parameters().data, m0.flat_parameters().segments())
    t0 = FusedTrainer(m0, use_graph=False)
    t1 = FusedTrainer(m1, use_graph=False, l2_emb=1.0)
    t2 = FusedTrainer(m2, use_graph=False, l2_emb=1e-4)
    d = float(t1.step(cb)) - float(t0.step(cb))
    want = math.fsum(norms)
    assert abs(d - want) <= 1e-6 * want, (d, want)
    t2.step(cb)
    assert abs(float(t2._l2.reg) - 1e-4 * want) <= 1e-6 * 1e-4 * want
    coef = t2._l2.coef.cpu()
    assert all(float(coef[t]) == 0.0 for t, n in enumerate(norms) if n == 0.0)   # zero-initialised biases: no NaN
    assert sum(1 for n in norms if n == 0.0) >= 6


@pytest.mark.gpu
def test_l2_adds_one_launch_per_step():
    """With l2_emb = 0 the step launches exactly what it did before; l2 > 0 adds the norm kernel only."""
    from srfrd_b200 import _lib
    from srfrd_b200.trainer import FusedTrainer
    data, smp = _c2_like()
    cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
    counts = []
    for l2 in (0.0, 1e-3):
        tr = FusedTrainer(_srfr_reference_init(data.itemnum), use_graph=False, l2_emb=l2)
        tr.step(cb)
        c0 = _lib.launch_count
        tr.step(cb)
        counts.append(_lib.launch_count - c0)
    assert counts[1] == counts[0] + 1, counts


def _model(kind, N, seed=3):
    from srfrd_b200 import SRFR_model as M
    torch.manual_seed(seed)
    m = {"SRFR": lambda: M.SRFR(N, 50, 64, 16, 0.0, 2, 1, "cuda"), "SRFRN": lambda: M.SRFRN(N, 50, 64, 16, 0.0, 2, 1, "cuda"),
         "SASRec": lambda: M.SASRec(N, 50, 64, 0.0, 2, 2, "cuda"),
         "SRFU_F": lambda: M.SRFU_F(N, 50, 64, 51, 0.0, 2, 1, "cuda")}[kind]()
    for _, p in m.named_parameters():
        if p.dim() >= 2:
            torch.nn.init.xavier_normal_(p.data)
    return m.to("cuda")


def _drop_in_step(m, opt, cb, l2):
    """The reference loop body (trainer.py:26-44) on our module, as simulate() runs it."""
    h, zp, zn = m(None, cb["seq"], cb["rsq"], cb["pos"], cb["prs"], cb["neg"], cb["nrs"])
    idx = torch.where(cb["pos"] != 0)
    crit = torch.nn.BCEWithLogitsLoss()
    opt.zero_grad()
    loss = crit(zp[idx], torch.ones_like(zp[idx])) + crit(zn[idx], torch.zeros_like(zn[idx]))
    for param in m.parameters():
        loss += l2 * torch.norm(param)
    loss.backward()
    opt.step()
    return float(loss.detach())


def _compare_with_drop_in(kind, tr, m_ref, step_fn, n_steps, l2, sd0):
    opt = torch.optim.Adam(m_ref.parameters(), lr=1e-3, betas=(0.9, 0.98))
    key = tr.spec.item_key
    seen = []
    for step in range(n_steps):
        loss, cb = step_fn()
        seen.append({k: cb[k].cpu().numpy() for k in ("seq", "pos", "neg")})
        ref = _drop_in_step(m_ref, opt, cb, l2)
        assert abs(loss - ref) < 5e-3, f"{kind} step {step}: {loss} vs drop-in {ref}"
        rows = _untouched_rows(m_ref.spec.item_number + 1, _touched(seen))
        got, want = tr.model.state_dict()[key].cpu()[rows], m_ref.state_dict()[key].cpu()[rows]
        assert float((got - want).abs().max()) <= 1e-6, f"{kind} step {step}: untouched rows differ"
    ref_sd = {k: v.detach().cpu() for k, v in m_ref.state_dict().items()}
    _check_tensors(tr.model.state_dict(), ref_sd, sd0, 6.5e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["SRFR", "SRFRN", "SASRec", "SRFU_F"])
@pytest.mark.parametrize("packed,graph", [(True, True), (True, False), (False, True), (False, False)])
def test_fused_l2_matches_drop_in_autograd_loop(kind, packed, graph):
    from srfrd_b200.trainer import FusedTrainer
    l2 = 1e-3
    data, smp = _c2_like()
    m, m_ref = _model(kind, data.itemnum), _model(kind, data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    tr = FusedTrainer(m, use_graph=graph, packed=packed, l2_emb=l2)

    def step_fn():
        cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
        return float(tr.step(cb)), cb
    _compare_with_drop_in(kind, tr, m_ref, step_fn, 3, l2, sd0)


@pytest.mark.gpu
def test_fused_l2_step_sampled_matches_drop_in_autograd_loop():
    from srfrd_b200.trainer import DeviceSampler, FusedTrainer
    l2 = 1e-3
    data, _ = _c2_like()
    smp = DeviceSampler(data, 50, "cuda", seed=5)
    m, m_ref = _model("SRFR", data.itemnum), _model("SRFR", data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    tr = FusedTrainer(m, use_graph=True, l2_emb=l2)

    def step_fn():
        loss = float(tr.step_sampled(smp, 256))
        return loss, {k: tr._static[k].clone() for k in FusedTrainer._KEYS}
    _compare_with_drop_in("SRFR", tr, m_ref, step_fn, 3, l2, sd0)
