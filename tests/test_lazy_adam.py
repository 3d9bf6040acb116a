"""Lazy Adam for the item table (FusedTrainer(lazy_item_adam=True)): srfrd_touch_rows, srfrd_adam_step_fused_rows and
srfrd_dp_adam_step_rows, and the trainer built on them.

A step looks up R_s: the non-zero ids of seq, pos and neg (loss="bce"), or of seq and pos plus the drawn negatives
(loss="gbce").  Rows in R_s get exactly the dense Adam update (global-step bias corrections), every other item row keeps
p, m and v bit for bit.

GPU: the touch kernel against numpy; the gated Adam against the dense kernel bit for bit (stamped rows, unstamped rows,
the rest of the buffer, the zeroed bucket, loss read-out and step state); the gated data-parallel kernel at world 1 (the
suite's only GPU coverage of srfrd_dp_adam_step_rows: its grid barrier needs every block resident, so two ranks cannot
share one GPU); the trainer against the oracle with Adam applied to R_s only; epochs under graph replay; no leaked
gradient; lazy equals dense on the same gradients when every row is looked up; the refusals.
CPU: the stamp union collective of parallel.py over gloo.
"""
import math
import os

import numpy as np
import pytest
import torch


# ------------------------------------------------------------------------------------------------------------ helpers
def _state8(step: int):
    """Adam state8 after `step` steps: {step, bc1, bc2, uint32 step bits, counter 0, ...}."""
    s = torch.zeros(8, dtype=torch.float32)
    s[0], s[1], s[2] = float(step), 1 - 0.9 ** step, 1 - 0.98 ** step
    s.view(torch.int32)[3] = step
    return s.cuda()


def _epoch(state8) -> int:
    return int(state8.cpu().view(torch.int32)[3]) + 1


# ------------------------------------------------------------------------------------------------------------ 1. touch
@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["dense", "packed"])
@pytest.mark.parametrize("B,L", [(0, 50), (1, 1), (7, 50), (256, 50)])
def test_touch_rows_matches_numpy(layout, B, L):
    """Stamped rows are exactly the in-range non-zero ids (duplicates, ids 1 and N, out-of-range ids skipped, an empty
    batch); every other stamp keeps its old value.  'packed': the three arrays are views of one pack_batch buffer."""
    from srfrd_b200 import ops
    from srfrd_b200.trainer import FusedTrainer
    N = 1000
    rng = np.random.default_rng(B * 31 + L)
    arrs = [rng.integers(-3, N + 4, (B, L)) for _ in range(3)]
    for a in arrs:
        if a.size:
            a.flat[0], a.flat[-1] = 1, N                                 # ids 1 and N
            a[a < 0] = np.int64(-(2 ** 40))                              # out of range below and far above
            a[a > N] = N + 1 + 2 ** 33 * (a[a > N] - N)
            a[rng.random(a.shape) < 0.3] = 0                             # padding
            a.flat[a.size // 2] = a.flat[0]                              # a duplicate
    ids = rng.integers(-2, N + 3, 40)
    st = _state8(17)
    epoch = _epoch(st)
    old = rng.integers(0, epoch - 1, N + 1).astype(np.int32)             # never the current epoch
    stamp = torch.from_numpy(old.copy()).cuda()
    if layout == "packed":
        flat = torch.zeros(7 * B * L, dtype=torch.int64, device="cuda")
        views = FusedTrainer._carve(flat, B, L)
        for k, a in zip(("seq", "pos", "neg"), arrs):
            views[k].copy_(torch.from_numpy(a))
        dev = [views[k].view(-1) for k in ("seq", "pos", "neg")]
    else:
        dev = [torch.from_numpy(a).cuda().view(-1) for a in arrs]
    ops.touch_rows(stamp, st, N, *dev, ids=torch.from_numpy(ids).cuda())
    want = old.copy()
    for a in arrs + [ids]:
        v = a.reshape(-1)
        want[v[(v >= 1) & (v <= N)]] = epoch
    assert np.array_equal(stamp.cpu().numpy(), want)
    # the list alone, and the three arrays alone
    stamp2 = torch.from_numpy(old.copy()).cuda()
    ops.touch_rows(stamp2, st, N, dev[0], None, None)
    want2 = old.copy()
    v = arrs[0].reshape(-1)
    want2[v[(v >= 1) & (v <= N)]] = epoch
    assert np.array_equal(stamp2.cpu().numpy(), want2)


# ------------------------------------------------------------------------------------------------------------ 2. gated Adam
def _operands(N, D, share, seed):
    """A flat buffer: 36 encoder floats, the (N + 1, D) table, then 10 more encoder floats starting right after the table
    (they share its last float4 when (N + 1) D is not a multiple of 4) and zero padding to a multiple of 4.  m and v are
    stale and non-zero everywhere; the gradient is non-zero outside the table and on the stamped rows, except on a few
    stamped rows whose gradient is all zero."""
    g_ = torch.Generator(device="cuda").manual_seed(seed)
    rows, off = N + 1, 36
    n = (off + rows * D + 10 + 3) // 4 * 4
    p = torch.randn(n + 4, generator=g_, device="cuda")
    m = torch.randn(n, generator=g_, device="cuda") * 1e-2
    v = torch.rand(n, generator=g_, device="cuda") * 1e-4
    g = torch.randn(n + 4, generator=g_, device="cuda") * 1e-2
    st = _state8(6)
    epoch = _epoch(st)
    rng = np.random.default_rng(seed)
    hit = np.zeros(rows, bool)
    if share == "all":
        hit[:] = True
    elif share == "part":
        hit[rng.choice(np.arange(1, rows), max(1, (rows - 1) // 5), replace=False)] = True
    stamp = np.where(hit, epoch, rng.integers(0, epoch, rows)).astype(np.int32)
    zero_rows = np.nonzero(hit)[0][::7]                                   # stamped, but an all-zero gradient
    tab = g[off:off + rows * D].view(rows, D)
    keep = torch.from_numpy(hit).cuda()
    keep[torch.from_numpy(zero_rows).cuda().long()] = False
    tab.mul_(keep[:, None].float())
    g[n:n + 2] = torch.tensor([3.0, 5.0], device="cuda")                 # loss accumulators in the bucket's tail
    return dict(p=p, m=m, v=v, g=g, st=st, n=n, off=off, rows=rows, D=D, hit=hit, stamp=torch.from_numpy(stamp).cuda(),
                norm=torch.tensor([2.0, 4.0], device="cuda"))


def _clone(o):
    return {k: (v.clone() if torch.is_tensor(v) else v) for k, v in o.items()}


def _dense(o):
    from srfrd_b200 import ops
    n = o["n"]
    ops.adam_step_fused(o["p"][:n], o["g"][:n], o["m"], o["v"], 1e-3, 0.9, 0.98, 1e-8, o["st"], acc2=o["g"][n:n + 2],
                        norm2=o["norm"], loss=o["p"][n:n + 1])


def _gated(o):
    from srfrd_b200 import ops
    n = o["n"]
    ops.adam_step_fused_rows(o["p"][:n], o["g"][:n], o["m"], o["v"], 1e-3, 0.9, 0.98, 1e-8, o["st"], o["off"], o["rows"],
                             o["D"], o["stamp"], acc2=o["g"][n:n + 2], norm2=o["norm"], loss=o["p"][n:n + 1])


def _check_gated(got, dense, inp):
    off, rows, D, n = inp["off"], inp["rows"], inp["D"], inp["n"]
    hit = torch.from_numpy(inp["hit"]).cuda()
    tab = lambda t: t[off:off + rows * D].view(rows, D)
    rest = lambda t: torch.cat([t[:off], t[off + rows * D:n]])
    for k in ("p", "m", "v"):
        assert torch.equal(tab(got[k])[hit], tab(dense[k])[hit]), f"stamped rows of {k}"
        assert torch.equal(tab(got[k])[~hit], tab(inp[k])[~hit]), f"unstamped rows of {k} moved"
        assert torch.equal(rest(got[k]), rest(dense[k])), f"non-table part of {k}"
    assert not torch.any(got["g"][:n + 2]), "gradient bucket not zeroed"
    assert torch.equal(got["p"][n], dense["p"][n]), "loss read-out"
    assert torch.equal(got["st"][:4], dense["st"][:4]) and int(got["st"].view(torch.int32)[4]) == 0, "step state"
    if inp["hit"].all():
        for k in ("p", "m", "v", "g", "st"):
            assert torch.equal(got[k], dense[k]), f"every row stamped: {k} differs from the dense call"


@pytest.mark.gpu
@pytest.mark.parametrize("share", ["none", "part", "all"])
@pytest.mark.parametrize("N", [1, 129, 1_000_000])
@pytest.mark.parametrize("D", [50, 64, 256])
def test_gated_adam_equals_dense_on_stamped_rows(D, N, share):
    inp = _operands(N, D, share, seed=D + N)
    dense, got = _clone(inp), _clone(inp)
    _dense(dense)
    _gated(got)
    torch.cuda.synchronize()
    assert not torch.equal(dense["p"][inp["off"]:inp["off"] + D * (N + 1)], inp["p"][inp["off"]:inp["off"] + D * (N + 1)])
    _check_gated(got, dense, inp)


# ------------------------------------------------------------------------------------------------------------ 3. DP kernel
@pytest.mark.gpu
@pytest.mark.parametrize("share", ["none", "part", "all"])
@pytest.mark.parametrize("N,D", [(129, 64), (12101, 64), (1000, 256)])
def test_dp_rows_kernel_world1_equals_gated_kernel(N, D, share):
    """srfrd_dp_adam_step_rows with one-element pointer arrays to this rank's own buffers equals
    srfrd_adam_step_fused_rows bit for bit.  This is the only GPU coverage of the gated data-parallel kernel in the suite:
    its grid barrier needs every block resident, so two 'ranks' cannot be co-scheduled on one GPU; the multi-GPU
    check is tools/dp_check.py --lazy.  The kernel takes D % 4 == 0 only (FusedTrainer sends other widths down the
    NCCL path); the refusal is checked too."""
    from srfrd_b200 import ops
    inp = _operands(N, D, share, seed=3 * N + D)
    ref, got = _clone(inp), _clone(inp)
    _gated(ref)
    n = inp["n"]
    ptr = lambda t: torch.tensor([t.data_ptr()], dtype=torch.int64, device="cuda")
    sig = torch.zeros(64, dtype=torch.int32, device="cuda")
    local = torch.zeros(4, dtype=torch.int32, device="cuda")
    arrs = [ptr(got["g"]), ptr(got["p"]), ptr(sig), ptr(got["stamp"])]
    ops.dp_adam_step_rows(arrs[0].data_ptr(), arrs[1].data_ptr(), arrs[2].data_ptr(), 0, 1, n, got["m"], got["v"], 1e-3, 0.9,
                          0.98, 1e-8, got["st"], inp["norm"], local, inp["off"], inp["rows"], D, arrs[3].data_ptr())
    torch.cuda.synchronize()
    for k in ("p", "m", "v"):
        assert torch.equal(got[k][:n], ref[k][:n]), k
    assert torch.equal(got["p"][n], ref["p"][n]), "loss read-out"
    assert not torch.any(got["g"][:n + 2])
    assert torch.equal(got["st"][:4], ref["st"][:4])
    with pytest.raises(RuntimeError, match="multiple of 4"):
        ops.dp_adam_step_rows(arrs[0].data_ptr(), arrs[1].data_ptr(), arrs[2].data_ptr(), 0, 1, n, got["m"], got["v"], 1e-3,
                              0.9, 0.98, 1e-8, got["st"], inp["norm"], local, inp["off"], inp["rows"] * D // 50, 50,
                              arrs[3].data_ptr())


# ------------------------------------------------------------------------------------------------------------ 4. trainer
def _lazy_oracle(O, base):
    class OracleLazy(base):
        """The oracle step with Adam's update of the item table kept only on the rows in R_s: torch.optim.Adam steps
        every tensor, then the table rows outside R_s get back their parameters and moments."""

        def lazy_step(self, rows, *args):
            key = O._emb_keys(self.kind)[0]
            E = self.sd[key]
            st = self.opt.state.get(E, {})
            old = (E.detach().clone(), st["exp_avg"].clone() if st else torch.zeros_like(E),
                   st["exp_avg_sq"].clone() if st else torch.zeros_like(E))
            loss = self.step(*args)
            st = self.opt.state[E]
            out = torch.ones(E.shape[0], dtype=torch.bool)
            out[rows] = False
            with torch.no_grad():
                for t, o in zip((E, st["exp_avg"], st["exp_avg_sq"]), old):
                    t[out] = o[out]
            return loss
    return OracleLazy


def _rows(tb, lists):
    ids = torch.cat([tb[k].flatten() for k in lists])
    return torch.unique(ids[ids != 0])


LAZY_CASES = [("SRFR", True, True, "bce"), ("SRFR", False, False, "gbce"), ("SASRec", True, False, "gbce"),
              ("SASRec", False, True, "bce"), ("SRFU_F", True, True, "gbce"), ("SRFU_F", False, False, "bce"),
              ("SRFRN", True, True, "bce"), ("SRFRN", False, False, "bce")]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,packed,graph,loss", LAZY_CASES)
def test_fused_trainer_lazy_matches_oracle(kind, packed, graph, loss):
    """5 steps against the oracle with the item table's Adam applied to R_s only, within the bounds of
    test_fused_trainer_gbce_matches_oracle; item rows no step looked up equal their initial values bit for bit, and the
    gradient bucket is all zero after every step."""
    from oracle import srfrd_oracle as O
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_gbce import _oracle_gbce
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, smp = _c2_like()
    m = _model(kind, data.itemnum)
    heads = 2 if kind == "SASRec" else 1
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    kw = dict(loss="gbce", num_negatives=128) if loss == "gbce" else {}
    tr = FusedTrainer(m, use_graph=graph, packed=packed, lazy_item_adam=True, **kw)
    base = _oracle_gbce(O, tr, 128, 0.75) if loss == "gbce" else O.OracleTrainer
    orc = _lazy_oracle(O, base)(sd0, kind, heads)
    seen = torch.zeros(data.itemnum + 1, dtype=torch.bool)
    for step in range(5):
        tb = {k: torch.from_numpy(v) for k, v in smp.next_batch(256).items()}
        got = float(tr.step({k: v.cuda() for k, v in tb.items()}))
        assert not torch.any(tr.P.grad_bucket), f"step {step}: gradient left in the bucket"
        rows = _rows(tb, ("seq", "pos", "neg") if loss == "bce" else ("seq", "pos"))
        if loss == "gbce":
            rows = torch.unique(torch.cat([rows, tr._gbce_ws["ids"].cpu()]))
        seen[rows] = True
        ref = orc.lazy_step(rows, tb)
        assert math.isfinite(got) and abs(got - ref) < 5e-3 * max(1.0, abs(ref)), f"{kind} step {step}: {got} vs {ref}"
    assert 0 < int(seen.sum()) < data.itemnum
    _check_tensors(m.state_dict(), orc.state_dict(), sd0, 2 * 5 * 1e-3 + 5e-4)
    key = O._emb_keys(kind)[0]
    assert torch.equal(m.state_dict()[key].cpu()[~seen], sd0[key][~seen]), "a row no step looked up moved"


@pytest.mark.gpu
@pytest.mark.parametrize("loss", ["bce", "gbce"])
def test_fused_trainer_lazy_step_sampled_soft_weights(loss):
    from oracle import srfrd_oracle as O
    from srfrd_b200.trainer import DeviceSampler, FusedTrainer
    from tests.test_gbce import _oracle_gbce
    from tests.test_l2_emb import _c2_like, _check_tensors, _model
    data, _ = _c2_like()
    smp = DeviceSampler(data, 50, "cuda", seed=5)
    m = _model("SRFR", data.itemnum)
    sd0 = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    kw = dict(loss="gbce") if loss == "gbce" else {}
    tr = FusedTrainer(m, use_graph=True, lazy_item_adam=True, **kw)
    orc = _lazy_oracle(O, _oracle_gbce(O, tr, 256, 0.75) if loss == "gbce" else O.OracleTrainer)(sd0, "SRFR", 1)
    for step in range(5):
        got = float(tr.step_sampled(smp, 256, policy="soft"))
        assert not torch.any(tr.P.grad_bucket)
        tb = {k: tr._static[k].cpu().clone() for k in FusedTrainer._KEYS}
        w = tr._static["w_pos"].cpu().clone()
        rows = _rows(tb, ("seq", "pos", "neg") if loss == "bce" else ("seq", "pos"))
        if loss == "gbce":
            rows = torch.unique(torch.cat([rows, tr._gbce_ws["ids"].cpu()]))
        ref = orc.lazy_step(rows, tb, w)
        assert math.isfinite(got) and abs(got - ref) < 5e-3 * max(1.0, abs(ref)), f"step {step}: {got} vs {ref}"
    _check_tensors(m.state_dict(), orc.state_dict(), sd0, 2 * 5 * 1e-3 + 5e-4)


# ------------------------------------------------------------------------------------------------------------ 5. replays
def _table(tr, buf, r):
    off, rows, D = tr._table
    return buf[off:off + rows * D].view(rows, D)[r].clone()


@pytest.mark.gpu
@pytest.mark.parametrize("packed", [True, False])
def test_epochs_advance_under_graph_replay(packed):
    """Row r is looked up in step 1 only and row q in steps 1 and 3; steps 2 and 3 run from the captured graph.  After
    step 3, r's p, m and v are bit-identical to after step 1 and q's have moved."""
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, smp = _c2_like()
    tr = FusedTrainer(_model("SRFR", data.itemnum), use_graph=True, packed=packed, lazy_item_adam=True)
    batches = [{k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()} for _ in range(3)]
    used = torch.zeros(data.itemnum + 1, dtype=torch.bool)
    for b in batches:
        for k in ("seq", "pos", "neg"):
            used[b[k].flatten().cpu()] = True
    free = torch.nonzero(~used[1:]).flatten() + 1
    assert free.numel() >= 2
    r, q = int(free[0]), int(free[1])
    batches[0]["seq"][0, -1] = r
    batches[0]["neg"][1, -1] = q
    batches[2]["pos"][2, -1] = q
    tr.step(batches[0])
    after1 = [_table(tr, t, [r, q]) for t in (tr.P.data, tr.m, tr.v)]
    assert all(bool(torch.any(a != 0)) for a in after1[1:])
    tr.step(batches[1])
    assert tr._graph is not None
    tr.step(batches[2])
    torch.cuda.synchronize()
    after3 = [_table(tr, t, [r, q]) for t in (tr.P.data, tr.m, tr.v)]
    for a1, a3 in zip(after1, after3):
        assert torch.equal(a1[0], a3[0]), "a row not looked up since step 1 moved"
        assert not torch.equal(a1[1], a3[1]), "a row looked up again in step 3 did not move"
    assert int(tr.stamp[r]) == 1 and int(tr.stamp[q]) == 3


# ------------------------------------------------------------------------------------------------------------ 6. no leak
@pytest.mark.gpu
@pytest.mark.parametrize("kind,loss,packed", [("SRFR", "bce", True), ("SRFR", "gbce", False), ("SRFRN", "bce", True),
                                              ("SRFU_F", "gbce", True), ("SASRec", "bce", False)])
def test_no_leaked_gradient(kind, loss, packed):
    """After every lazy step the whole gradient bucket is zero: a row the backward wrote but the touch kernel did not
    stamp would keep its gradient."""
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, smp = _c2_like()
    kw = dict(loss="gbce") if loss == "gbce" else {}
    tr = FusedTrainer(_model(kind, data.itemnum), use_graph=True, packed=packed, lazy_item_adam=True, **kw)
    flat = tr.pack_batch({k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()})
    for step in range(4):
        if step % 2:
            tr.step_packed(flat)
        else:
            tr.prefetch({k: torch.from_numpy(v).pin_memory() for k, v in smp.next_batch(256).items()})
            tr.step_prefetched()
        torch.cuda.synchronize()
        assert not torch.any(tr.P.grad_bucket), f"step {step}: {int(torch.count_nonzero(tr.P.grad_bucket))} floats left"


# ------------------------------------------------------------------------------------------------------------ 7. all rows
@pytest.mark.gpu
@pytest.mark.parametrize("loss", ["bce", "gbce"])
def test_lazy_equals_dense_when_every_row_is_looked_up(loss, monkeypatch):
    """A tiny catalogue every batch covers.  Inside the captured step the operands of the gated Adam (p, the gradient
    bucket, m, v, state) are copied aside; after each replay the dense kernel on those copies must give the lazy step's
    result bit for bit.  (Two separately trained models cannot be compared bit for bit: the LayerNorm weight gradients
    are fp32 atomics.)"""
    from srfrd_b200 import ops, synth
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _model
    N = 40
    data = synth.make_interactions(3, 500, N, 5, 4.0, 50)
    smp = synth.BatchSampler(data, 50, 3)
    kw = dict(loss="gbce", num_negatives=16) if loss == "gbce" else {}
    tr = FusedTrainer(_model("SRFR", N), use_graph=True, lazy_item_adam=True, **kw)
    P = tr.P
    saved = dict(p=torch.empty_like(P.data_ext), g=torch.empty_like(P.grad_bucket), m=torch.empty_like(tr.m),
                 v=torch.empty_like(tr.v), st=torch.empty_like(tr.eng.step_state))
    real = ops.adam_step_fused_rows

    def spy(*a, **k):
        for key, src in (("p", P.data_ext), ("g", P.grad_bucket), ("m", tr.m), ("v", tr.v), ("st", tr.eng.step_state)):
            saved[key].copy_(src)
        real(*a, **k)
    monkeypatch.setattr(ops, "adam_step_fused_rows", spy)
    n = P.numel
    for step in range(4):
        b = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
        b["neg"][0, :N] = torch.arange(1, N + 1)                          # every row looked up
        tr.step(b)
        torch.cuda.synchronize()
        assert bool((tr.stamp[1:] == _epoch(saved["st"])).all()) and int(tr.stamp[0]) == 0
        d = {k: v.clone() for k, v in saved.items()}
        ops.adam_step_fused(d["p"][:n], d["g"][:n], d["m"], d["v"], tr.lr, tr.betas[0], tr.betas[1], tr.eps, d["st"],
                            acc2=d["g"][n:n + 2], norm2=tr.scal[0:2], loss=tr.scal[4:5].clone())
        torch.cuda.synchronize()
        assert torch.equal(d["p"][:n], P.data) and torch.equal(d["m"], tr.m) and torch.equal(d["v"], tr.v), step
        assert torch.equal(d["st"][:4], tr.eng.step_state[:4])
    assert tr._graph is not None


# ------------------------------------------------------------------------------------------------------------ 8. refusals
@pytest.mark.gpu
def test_refusals_before_any_launch():
    from srfrd_b200 import _lib
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, _ = _c2_like()
    models = [_model("SRFR", data.itemnum) for _ in range(2)]
    torch.cuda.synchronize()
    c0 = _lib.launch_count
    with pytest.raises(ValueError, match="l2_emb"):
        FusedTrainer(models[0], lazy_item_adam=True, l2_emb=1e-4)
    with pytest.raises(ValueError, match="ce"):
        FusedTrainer(models[1], lazy_item_adam=True, loss="ce")
    assert _lib.launch_count == c0


@pytest.mark.gpu
def test_dense_step_launches_unchanged_and_lazy_adds_the_touch():
    from srfrd_b200 import _lib
    from srfrd_b200.trainer import FusedTrainer
    from tests.test_l2_emb import _c2_like, _model
    data, smp = _c2_like()
    cb = {k: torch.from_numpy(v).cuda() for k, v in smp.next_batch(256).items()}
    counts = {}
    for loss in ("bce", "gbce"):
        for lazy in (False, True):
            tr = FusedTrainer(_model("SRFR", data.itemnum), use_graph=False, loss=loss, lazy_item_adam=lazy)
            tr.step(cb)
            c0 = _lib.launch_count
            tr.step(cb)
            counts[loss, lazy] = _lib.launch_count - c0
    assert counts["bce", True] == counts["bce", False] + 1, counts        # touch; the gated Adam replaces the dense one
    assert counts["gbce", True] == counts["gbce", False] + 2, counts      # touch of the batch + touch of the drawn ids


# ------------------------------------------------------------------------------------------------------------ 9. gloo
def _worker(rank, world, port, ret):
    import torch.distributed as dist
    from srfrd_b200 import parallel
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        stamp = torch.tensor([0, 3, 2, 1, 0, 4, 4, 3], dtype=torch.int32)  # epoch 4; rows 1 and 7 carry an old epoch
        if rank == 1:
            stamp[[1, 2, 4]] = 4
        parallel.union_row_stamps_(stamp, dist.group.WORLD)
        ret[rank] = stamp.tolist()
    finally:
        dist.destroy_process_group()


def test_union_row_stamps_gloo():
    import torch.multiprocessing as mp
    torch.set_num_threads(1)
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, 29623, ret), nprocs=2, join=True)
    want = [0, 4, 4, 1, 4, 4, 4, 3]
    assert ret[0] == want and ret[1] == want
    assert [i for i, e in enumerate(want) if e == 4] == [1, 2, 4, 5, 6]   # the union of both ranks' rows of epoch 4
