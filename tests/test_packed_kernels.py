"""Each kernel of the packed token layout (csrc/pack.cu) against an fp64 reference of its own, on the device.

The packed layout keeps, per sequence, one pad-representative row followed by the kept tokens; filler rows round the
row count rows[0] up to a multiple of 128 (DESIGN.md section 3).  References are computed in torch.float64 from exactly
the bf16 / fp32 operands the kernel reads.  Every output starts as NaN and every input row in [rows[0], cap) holds
finite garbage (the last attention tile reads those rows): rows below rows[0] must be finite and match, and the
kernels that write packed rows must leave the rows from rows[0] on untouched."""
import math

import numpy as np
import pytest
import torch

from tests.test_dropout_mask import drop_scale, keep_mask, masked
from tests.test_gpu_round2 import _ragged_batch

pytestmark = pytest.mark.gpu

bf16, f64 = torch.bfloat16, torch.float64
U = 2.0 ** -8                 # bf16 keeps 8 significant bits: one rounding is within 2^-9 relative, two within 2^-8

# (B, L, keep=pos): B = 1; the C2 shape; L = 127, where a full sequence plus its representative fills one tile exactly;
# B = 16384, several tiles per CTA; and a plan without keep ids
SHAPES = [(1, 50, True), (4096, 50, True), (37, 127, True), (16384, 50, True), (300, 20, False)]


def _plan(B, L, keep, seed, N=500):
    from srfrd_b200 import ops
    if B == 1:        # _ragged_batch's first row is empty: take one of its rows that holds a few tokens
        b = _ragged_batch(16, L, N, seed)
        r = next(i for i in range(1, 16) if int((b["seq"][i] != 0).sum()) > 4)
        b = {k: v[r:r + 1].contiguous() for k, v in b.items()}
    else:
        b = _ragged_batch(B, L, N, seed)
    plan = ops.PackedPlan(B, L, "cuda")
    plan.build(b["seq"], b["pos"] if keep else None)
    torch.cuda.synchronize()
    M, Tp = (int(x) for x in plan.rows[:2].cpu())
    assert 0 < M <= plan.cap and M % 128 == 0 and Tp <= M
    return b, plan, M, Tp


def _maps(plan):
    """Host view of the plan: row_tok (cap), tok_row (B * L), seq_first (B + 1), pad weight of every row (cap)."""
    info = plan.row_info.view(-1, 4)
    return dict(row_tok=plan.row_tok.long(), tok_row=plan.tok_row.long(), seq_first=plan.seq_first.long(),
                mult=info[:, 2].contiguous().view(torch.float32).double())


def _rand(rows, cols, seed, scale=1.0, dtype=bf16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(rows, cols, generator=g, device="cuda") * scale).to(dtype)


def _nan(rows, cols, dtype=bf16):
    return torch.full((rows, cols), float("nan"), dtype=dtype, device="cuda")


def _zero(t):
    return t.numel() == 0 or float(t.float().abs().max()) == 0.0


def _check(name, got, ref, rtol, atol):
    """|got - ref| <= rtol |ref| + atol elementwise, got finite; reports the worst ratio error / bound."""
    got = got.double()
    assert bool(torch.isfinite(got).all()), f"{name}: non-finite values"
    bound = rtol * ref.abs() + atol
    ratio = float(((got - ref).abs() / bound.clamp_min(1e-300)).max()) if got.numel() else 0.0
    assert ratio <= 1.0, f"{name}: error {ratio:.3g} x the bound"


def _untouched(name, out, M):
    assert bool(torch.isnan(out[M:].float()).all()), f"{name}: rows >= rows[0] were written"


# --------------------------------------------------------------------------------------------------------- attention
def _groups(B, M, Tp, maps):
    """Row groups of the attention definition: each sequence (representative + kept tokens), then each filler row alone."""
    sf = maps["seq_first"]
    start = torch.cat([sf[:B], torch.arange(Tp, M, device="cuda")])
    n = torch.cat([sf[1:B + 1], torch.arange(Tp + 1, M + 1, device="cuda")]) - start
    W = int(n.max())
    j = torch.arange(W, device="cuda")
    valid = j[None, :] < n[:, None]
    idx = torch.where(valid, start[:, None] + j[None, :], start[:, None])
    return idx, valid


def _packed_attention_ref(q, k, v, dO, idx, valid, mult, heads, drop=None):
    """fp64 packed attention: the query at row a of a group sees the group's rows 0..a; column 0 (the representative)
    weighs mult(query row) -- the number of dropped pads before the query's position -- and is left out when that is 0;
    one dropout factor covers the aggregated column (DESIGN.md section 9).  Returns o, dq, dk, dv on the packed rows."""
    G, W = idx.shape
    H = q.shape[1]
    hd = H // heads
    gather = lambda x: x[idx].double().view(G, W, heads, hd).transpose(1, 2).requires_grad_(True)
    Q, K, V = gather(q), gather(k), gather(v)
    a = torch.arange(W, device="cuda")
    w = torch.where(a[None, None, :] == 0, mult[idx][:, :, None], torch.ones((), dtype=f64, device="cuda"))   # (G, Wq, Wk)
    allowed = (a[None, :, None] >= a[None, None, :]) & valid[:, :, None] & valid[:, None, :] & (w > 0)
    w = (w * allowed)[:, None]
    S = (Q @ K.transpose(-1, -2)) / math.sqrt(hd)
    S = S.masked_fill(~allowed[:, None], -1e300)
    E = torch.exp(S - S.amax(-1, keepdim=True)) * w
    P = E / E.sum(-1, keepdim=True).clamp_min(1e-300)
    if drop is not None:
        P = P * drop
    O = P @ V
    dOg = dO[idx].double().view(G, W, heads, hd).transpose(1, 2) * valid[:, None, :, None]
    (O * dOg).sum().backward()
    out = {}
    for name, t in (("o", O.detach()), ("dq", Q.grad), ("dk", K.grad), ("dv", V.grad)):
        r = torch.zeros(q.shape[0], H, dtype=f64, device="cuda")
        r[idx[valid]] = t.transpose(1, 2).reshape(G, W, H)[valid]
        out[name] = r
    return out


def _packed_drop(idx, valid, heads, p, seed, stream, step):
    """Dropout factors of the packed kernels: element ((row * heads + h) * 256 + key column - group's first row)."""
    G, W = idx.shape
    rows = idx.cpu().numpy().astype(np.int64)
    h = np.arange(heads, dtype=np.int64)
    col = np.arange(W, dtype=np.int64)
    e = ((rows[:, None, :, None] * heads + h[None, :, None, None]) * 256 + col[None, None, None, :])
    return masked(torch.ones(e.shape, dtype=torch.float32), keep_mask(seed, stream, e, p, step), p).cuda().double()


def _dense_attention_ref(q, k, v, dO, maps, B, L, heads):
    """fp64 causal attention on the dense (B, L) layout in which every dropped pad slot holds its sequence's
    representative row (SRFR_model.py: a pad slot is a key with k = b_k, v = b_v, and its query output is dead)."""
    tr = maps["tok_row"]
    kept = tr >= 0
    rep = maps["seq_first"][:B].repeat_interleave(L)
    src = torch.where(kept, tr, rep)
    H = q.shape[1]
    hd = H // heads
    split = lambda x: x.view(B, L, heads, hd).transpose(1, 2)
    Q, K, V = (split(x[src].double()).requires_grad_(True) for x in (q, k, v))
    S = (Q @ K.transpose(-1, -2)) / math.sqrt(hd)
    S = S.masked_fill(~torch.ones(L, L, dtype=torch.bool, device="cuda").tril(), float("-inf"))
    O = torch.softmax(S, -1) @ V
    dOd = split(dO[src].double() * kept[:, None])
    (O * dOd).sum().backward()
    merge = lambda x: x.transpose(1, 2).reshape(B * L, H)
    return kept, tr, rep, merge(O.detach()), merge(Q.grad), merge(K.grad), merge(V.grad)


ATTN = [(B, L, keep, H, heads, p) for (B, L, keep) in SHAPES[:2] for (H, heads) in ((64, 1), (80, 1), (128, 1), (128, 2))
        for p in (0.0, 0.3)]
ATTN += [(37, 127, True, 80, 1, 0.0), (37, 127, True, 80, 1, 0.3), (37, 127, True, 128, 2, 0.3),
         (16384, 50, True, 80, 1, 0.3), (16384, 50, True, 128, 2, 0.0), (300, 20, False, 64, 1, 0.3)]


@pytest.mark.parametrize("B,L,keep,H,heads,p", ATTN)
def test_attention_packed(B, L, keep, H, heads, p):
    from srfrd_b200 import ops
    b, plan, M, Tp = _plan(B, L, keep, B + L + H)
    maps = _maps(plan)
    cap = plan.cap
    q, kv = _rand(cap, H, 1, 0.7), _rand(cap, 2 * H, 2, 0.7)
    k, v = kv[:, :H], kv[:, H:]
    dO = _rand(cap, H, 3)
    dO[:M][maps["row_tok"][:M] < 0] = 0                     # representative and filler rows: dead queries, as in the engine
    seed, stream, step = 4321, 9, 5.0
    stp = torch.tensor([step], device="cuda")
    o, dq, dkv = _nan(cap, H), _nan(cap, H), _nan(cap, 2 * H)
    args = (plan, L, H, heads, p, seed, stream, stp)
    ops.attention_fwd_packed(q, k, v, o, *args)
    ops.attention_bwd_packed(dO, q, k, v, dq, dkv[:, :H], dkv[:, H:], *args)
    torch.cuda.synchronize()
    idx, valid = _groups(B, M, Tp, maps)
    drop = _packed_drop(idx, valid, heads, p, seed, stream, step) if p else None
    ref = _packed_attention_ref(q, k, v, dO, idx, valid, maps["mult"], heads, drop)
    got = dict(o=o, dq=dq, dk=dkv[:, :H], dv=dkv[:, H:])
    # o: P is rounded to bf16 before P V (2^-9 of sum P |v| <= 2^-9 max|v|, times the dropout scale) and o itself once
    # more (2^-9 |o|); ex2.approx and fp32 accumulation are far below that
    vmax = float(v[:M].abs().max()) * drop_scale(p)
    _check("o", got["o"][:M], ref["o"][:M], U, U * vmax)
    # gradients: P and dS = P (dP - delta) reach the MMAs as bf16 and the outputs are bf16: a few 2^-9 roundings of
    # terms bounded by the tensor's scale -- 2^-7 of its largest magnitude, 2^-8 of each element
    for name in ("dq", "dk", "dv"):
        _check(name, got[name][:M], ref[name][:M], U, 2 * U * float(ref[name][:M].abs().max()))
    for name, t in got.items():
        _untouched(name, t, M)
    if p == 0.0:
        # the packed definition is the dense model's attention: o and dq of every kept token, dk / dv of every kept token,
        # and the representative's dk / dv equal the sum over the dropped pad slots it stands for
        kept, tr, rep, Od, dQd, dKd, dVd = _dense_attention_ref(q, k, v, dO, maps, B, L, heads)
        # (same bounds as above: the gradients' scale is the largest packed row, which is usually a representative's sum)
        scale = {n: vmax if n == "o" else 2 * float(ref[n][:M].abs().max()) for n in got}
        for name, dense in (("o", Od), ("dq", dQd), ("dk", dKd), ("dv", dVd)):
            _check("dense " + name, got[name][tr[kept]], dense[kept], U, U * scale[name])
        for name, dense in (("dk", dKd), ("dv", dVd)):
            pad_sum = torch.zeros(cap, H, dtype=f64, device="cuda").index_add_(0, rep[~kept], dense[~kept])
            reps = maps["seq_first"][:B]
            _check("dense pad sum " + name, got[name][reps], pad_sum[reps], U, U * scale[name])


def _ln64(x, w, b, eps):
    x = x.double()
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    rstd = 1.0 / torch.sqrt(var + eps)
    return (x - mean) * rstd * w.double() + b.double(), mean[:, 0], rstd[:, 0]


@pytest.mark.parametrize("B,L,p", [(4096, 50, 0.0), (4096, 50, 0.3), (37, 127, 0.0), (16384, 50, 0.3)])
def test_attention_packed_out_projection(B, L, p):
    """The folded out-projection: forward r = o Wo^T + bo + res and y = LayerNorm(r) with its (mean, rstd); backward
    dO = dr Wo formed in the kernel, then the packed attention gradients."""
    from srfrd_b200 import ops
    H = 80
    b, plan, M, Tp = _plan(B, L, True, B + L)
    maps = _maps(plan)
    cap = plan.cap
    q, kv, res, dr = _rand(cap, H, 4, 0.7), _rand(cap, 2 * H, 5, 0.7), _rand(cap, H, 6), _rand(cap, H, 7)
    dr[:M][maps["row_tok"][:M] < 0] = 0
    k, v = kv[:, :H], kv[:, H:]
    wo = _rand(H, H, 8, 0.15)
    woT = wo.t().contiguous()
    g = torch.Generator(device="cuda").manual_seed(9)
    bo, ln_w, ln_b = (torch.randn(H, generator=g, device="cuda") * s + c for s, c in ((0.1, 0.0), (0.1, 1.0), (0.1, 0.0)))
    eps, seed, stream, stp = 1e-8, 77, 10, torch.tensor([2.0], device="cuda")
    o, r, y, st, dq, dkv = _nan(cap, H), _nan(cap, H), _nan(cap, H), _nan(cap, 2, torch.float32), _nan(cap, H), _nan(cap, 2 * H)
    args = (plan, L, H, 1, p, seed, stream, stp)
    with ops.row_limit(plan.rows):
        ops.attention_fwd_packed(q, k, v, o, *args, wo=wo, bias=bo, residual=res, r=r, y=y, ln_w=ln_w, ln_b=ln_b, ln_eps=eps,
                                 ln_stats=st)
        ops.attention_bwd_packed(None, q, k, v, dq, dkv[:, :H], dkv[:, H:], *args, dr=dr, woT=woT)
    torch.cuda.synchronize()
    # r from the kernel's own bf16 o: one bf16 rounding of r plus fp32 accumulation of H products
    r_ref = o[:M].double() @ wo.double().T + bo.double() + res[:M].double()
    _check("r", r[:M], r_ref, U, 1e-5 * float((o[:M].double().abs() @ wo.double().abs().T).max()))
    # y and the statistics from the kernel's rounded r (the LayerNorm reads the rounded row, as gemm_tn's does)
    y_ref, mean, rstd = _ln64(r[:M], ln_w, ln_b, eps)
    _check("y", y[:M], y_ref, U, U * float(ln_b.abs().max()) + 1e-5)
    _check("mean", st[:M, 0], mean, 1e-5, 1e-6 * float(r[:M].float().abs().max()))
    _check("rstd", st[:M, 1], rstd, 1e-5, 0.0)
    idx, valid = _groups(B, M, Tp, maps)
    drop = _packed_drop(idx, valid, 1, p, seed, stream, 2.0) if p else None
    dO = (dr.float() @ wo.float()).to(bf16)                # what gemm_tn(dr, woT) writes: the kernel's bf16 dO
    ref = _packed_attention_ref(q, k, v, dO, idx, valid, maps["mult"], 1, drop)
    _check("o", o[:M], ref["o"][:M], U, U * float(v[:M].abs().max()) * drop_scale(p))
    for name, t in (("dq", dq), ("dk", dkv[:, :H]), ("dv", dkv[:, H:])):
        _check(name, t[:M], ref[name][:M], U, 2 * U * float(ref[name][:M].abs().max()))
    for name, t in (("o", o), ("r", r), ("y", y), ("stats", st), ("dq", dq), ("dkv", dkv)):
        _untouched(name, t, M)


# --------------------------------------------------------------------------------------------------------- embedding
def _tables(mode, D, F, N, L, B, seed):
    g = torch.Generator().manual_seed(seed)
    E, P = torch.randn(N + 1, D, generator=g).cuda(), torch.randn(L, D, generator=g).cuda()
    aux, aux_ids = None, None
    if mode == 1:
        aux, aux_ids = torch.randn(3, F, generator=g).cuda(), None
    if mode == 2:
        aux, aux_ids = torch.randn(7, D, generator=g).cuda(), torch.randint(0, 7, (B,), generator=g).cuda()
    return E, P, aux, aux_ids


EMB = [(mode, p, B, L) for mode in (0, 1, 2) for p in (0.0, 0.3) for (B, L) in ((4096, 50), (37, 127))] + [(1, 0.3, 1, 50),
                                                                                                       (0, 0.0, 16384, 50)]


@pytest.mark.parametrize("mode,p,B,L", EMB)
def test_embed_ln_fwd_packed(mode, p, B, L):
    """x0, q and the LayerNorm statistics of every packed row.  Mode 0 is SASRec (item_scale sqrt(D)), mode 1 SRFR (fake
    table), mode 2 SRFU (user-label table).  At p = 0 x0 is bit-equal to the dense kernel's row of the same token; with
    dropout the packed kernel hashes the packed row index, so x0 is checked against the host mask instead."""
    from srfrd_b200 import ops
    D, F = 64, (16 if mode == 1 else 0)
    H = D + F
    b, plan, M, Tp = _plan(B, L, True, B + L + mode)
    maps = _maps(plan)
    E, P, aux, aux_ids = _tables(mode, D, 16, 500, L, B, mode)
    if mode == 1:
        aux_ids = b["rsq"]
    scale = D ** 0.5 if mode == 0 else 1.0
    g = torch.Generator().manual_seed(1)
    ln_w, ln_b = (torch.randn(H, generator=g) * 0.2 + 1.0).cuda(), (torch.randn(H, generator=g) * 0.2).cuda()
    seed, stream, step = 555, 3, 4.0
    stp = torch.tensor([step], device="cuda")
    x_dense = torch.empty(B * L, H, device="cuda")            # the exact pre-dropout tensor of every dense token
    xb_dense = torch.empty(B * L, H, dtype=bf16, device="cuda")
    ops.embed_ln_fwd(E, P, aux, mode, b["seq"], aux_ids, scale, None, None, 1e-8, x0_bf16=xb_dense, x0_f32=x_dense)
    cap = plan.cap
    x0, qo, st = _nan(cap, H), _nan(cap, H), _nan(cap, 2, torch.float32)
    ops.embed_ln_fwd_packed(E, P, aux, mode, b["seq"], aux_ids, scale, ln_w, ln_b, 1e-8, x0, qo, st, plan, drop_p=p,
                            drop_seed=seed, drop_stream=stream, drop_step=stp)
    torch.cuda.synchronize()
    rt = maps["row_tok"][:M]
    tok = rt >= 0
    x32 = torch.zeros(M, H, device="cuda")
    x32[tok] = x_dense[rt[tok]]
    if p:
        x32 = masked(x32, keep_mask(seed, stream, np.arange(M * H).reshape(M, H), p, step), p)
    else:
        assert torch.equal(x0[:M][tok], xb_dense[rt[tok]])
    assert torch.equal(x0[:M], x32.to(bf16))
    live = x32.abs().amax(1) > 0
    assert _zero(x0[:M][~tok])          # representative and filler rows (and kept rows whose input id is 0): x0 = 0 ...
    assert torch.equal(qo[:M][~live], ln_b.to(bf16).expand(int((~live).sum()), H))   # ... so q is ln_b
    # q: LayerNorm of the fp32 row, rounded to bf16 once (2^-9 relative), plus fp32 statistics (~1e-6 of the row's scale)
    y_ref, mean, rstd = _ln64(x32, ln_w, ln_b, 1e-8)
    _check("q", qo[:M][live], y_ref[live], U, 1e-5 * float(y_ref.abs().max()))
    _check("mean", st[:M, 0][live], mean[live], 1e-5, 1e-6 * float(x32.abs().max()))
    _check("rstd", st[:M, 1][live], rstd[live], 1e-5, 0.0)
    for name, t in (("x0", x0), ("q", qo), ("stats", st)):
        _untouched(name, t, M)


@pytest.mark.parametrize("mode,B,L", [(0, 4096, 50), (1, 4096, 50), (2, 4096, 50), (1, 37, 127), (2, 1, 50), (1, 16384, 50)])
def test_embed_bwd_packed(mode, B, L):
    """dE, the fake (mode 1) or user-label (mode 2) table and d_pos: the fp64 scatter of the packed rows' dx0 over
    the dense tokens they hold.  A kept row whose input id is 0 (keep=pos) and the representative / filler rows add
    nothing, and rows 0 of dE and of the fake table get nothing."""
    from srfrd_b200 import ops
    D, F, N = 64, (16 if mode == 1 else 0), 500
    H = D + F
    b, plan, M, Tp = _plan(B, L, True, B + L + 10 * mode)
    maps = _maps(plan)
    cap = plan.cap
    scale = D ** 0.5 if mode == 0 else 1.0
    aux_ids = {0: None, 1: b["rsq"], 2: torch.randint(0, 7, (B,), device="cuda")}[mode]
    dx0 = _rand(cap, H, 11)
    d_item = torch.zeros(N + 1, D, device="cuda")
    d_aux = torch.zeros(3, F, device="cuda") if mode == 1 else (torch.zeros(7, D, device="cuda") if mode == 2 else None)
    d_pos = torch.zeros(L, D, device="cuda")
    ops.embed_bwd_packed(dx0, b["seq"], aux_ids, plan, D, F, mode, scale, d_item, d_aux, d_pos)
    torch.cuda.synchronize()
    rt = maps["row_tok"][:M]
    tok = rt.clamp_min(0)
    ids = torch.where(rt >= 0, b["seq"].view(-1)[tok], torch.zeros_like(rt))
    live = ids != 0
    assert bool((live <= (rt >= 0)).all())
    g = dx0[:M].double()[live]
    t = tok[live]

    def scatter(n, index, vals):
        ref = torch.zeros(n, vals.shape[1], dtype=f64, device="cuda").index_add_(0, index, vals)
        mag = torch.zeros_like(ref).index_add_(0, index, vals.abs())
        return ref, mag

    # fp32 atomic sums: each added term is exact, the running sum rounds once per add -- within n 2^-24 of the sum of
    # |terms| in the worst order, and in practice within 2^-14 of it for the n <= 16384 terms of one d_pos row
    checks = [("dE", d_item, *scatter(N + 1, ids[live], g[:, :D] * scale)),
              ("d_pos", d_pos, *scatter(L, t % L, g[:, :D]))]
    if mode == 1:
        f = b["rsq"].view(-1)[t]
        sel = f > 0
        checks.append(("d_fake", d_aux, *scatter(3, f[sel], g[sel][:, D:])))
    if mode == 2:
        checks.append(("d_label", d_aux, *scatter(7, aux_ids[t // L], g[:, :D])))
    for name, got, ref, mag in checks:
        _check(name, got, ref, 0.0, 2.0 ** -14 * mag + 1e-30)
    assert float(d_item[0].abs().max()) == 0.0
    if mode == 1:
        assert float(d_aux[0].abs().max()) == 0.0
    if mode == 0:                                              # kept rows with input id 0 exist in this batch and add nothing
        assert bool(((rt >= 0) & ~live).any())


# --------------------------------------------------------------------------------------------------------- repacking
@pytest.mark.parametrize("B,L,keep", SHAPES)
def test_unpack_pack_rows(B, L, keep):
    """unpack_rows: dense[t] = packed[tok_row[t]]; a dropped pad slot takes the representative row (mode 0) or zeros
    (mode 1).  pack_rows: packed[r] = dense[row_tok[r]]; representative and filler rows zero (mode 0), or the
    representative holds the sum over its sequence's dropped pad slots (mode 1) and filler rows zero."""
    from srfrd_b200 import ops
    b, plan, M, Tp = _plan(B, L, keep, B + L + 20)
    maps = _maps(plan)
    cap, T = plan.cap, B * L
    tr = maps["tok_row"]
    kept = tr >= 0
    rep = maps["seq_first"][:B].repeat_interleave(L)
    src0, src1 = _rand(cap, 80, 21), _rand(cap, 128, 22)
    d0, d1 = _nan(T, 80), _nan(T, 128)
    ops.unpack_rows([(src0, d0, 80, 0), (src1, d1, 128, 1)], plan)
    torch.cuda.synchronize()
    assert torch.equal(d0, src0[torch.where(kept, tr, rep)])
    assert torch.equal(d1[kept], src1[tr[kept]])
    assert _zero(d1[~kept])
    dense0, dense1, dense2 = _rand(T, 80, 23), _rand(T, 160, 24), _rand(T, 64, 25, 4.0)
    p0, p1, p2 = _nan(cap, 80), _nan(cap, 160), _nan(cap, 64)
    ops.pack_rows([(dense0, p0, 80, 0), (dense1, p1, 160, 1), (dense2, p2, 64, 1)], plan)
    torch.cuda.synchronize()
    rt = maps["row_tok"][:M]
    tok = rt >= 0
    for out, dense, mode in ((p0, dense0, 0), (p1, dense1, 1), (p2, dense2, 1)):
        assert torch.equal(out[:M][tok], dense[rt[tok]])
        assert _zero(out[Tp:M])                              # filler rows
        reps = maps["seq_first"][:B]
        if mode == 0:
            assert _zero(out[reps])
        else:
            ref = torch.zeros(cap, dense.shape[1], dtype=f64, device="cuda").index_add_(0, rep[~kept], dense[~kept].double())[reps]
            # fp32 accumulation of at most L bf16 rows, rounded once to bf16: within one bf16 ulp of the fp64 sum
            ulp = torch.exp2(torch.floor(torch.log2(ref.abs().clamp_min(1e-30))) - 7)
            err = (out[reps].double() - ref).abs()
            assert bool((err <= ulp).all()), float((err / ulp).max())
        _untouched("pack_rows", out, M)


# --------------------------------------------------------------------------------------------------------- loss
@pytest.mark.parametrize("B,L,srfrn,w_neg", [(4096, 50, False, False), (4096, 50, True, True), (37, 127, True, False),
                                             (1, 50, False, True), (16384, 50, False, False)])
def test_score_loss_fused_packed(B, L, srfrn, w_neg):
    """BCE of every dense token with a positive or negative weight, read through the packed h rows: the loss sums, dh of
    every packed row (0 where the row has no loss term), dE and (SRFRN) the fake-table gradient dF."""
    from srfrd_b200 import ops
    D, F, N = 64, (16 if srfrn else 0), 500
    W = D + F
    b, plan, M, Tp = _plan(B, L, True, B + L + 30)
    maps = _maps(plan)
    cap = plan.cap
    g = torch.Generator(device="cuda").manual_seed(31)
    E = torch.randn(N + 1, D, generator=g, device="cuda") * 0.3
    fake = torch.randn(3, F, generator=g, device="cuda") * 0.3 if srfrn else None
    h = torch.randn(cap, W, generator=g, device="cuda")
    pos, neg = b["pos"], b["neg"]
    wp = (torch.rand(B, L, generator=g, device="cuda") * (pos != 0)).contiguous()             # soft weights
    wn = (torch.rand(B, L, generator=g, device="cuda") * (pos != 0)).contiguous() if w_neg else None
    norm = torch.stack([wp.sum(), (wn if w_neg else wp).sum()]).float()
    acc = torch.zeros(2, device="cuda")
    dh = _nan(cap, W, torch.float32)
    dE = torch.zeros(N + 1, D, device="cuda")
    dF = torch.zeros(3, F, device="cuda") if srfrn else None
    ops.score_loss_fused_packed(h, E, fake, pos, neg, b["prs"], b["nrs"], wp, wn, norm, acc, dh, dE, dF, plan)
    torch.cuda.synchronize()
    # the fp64 reference on the dense tokens: every token with a loss term must be a packed row (keep=pos)
    tr = maps["tok_row"]
    a64, b64 = wp.view(-1).double(), (wn if w_neg else wp).view(-1).double()
    active = (a64 != 0) | (b64 != 0)
    assert bool((tr[active] >= 0).all())
    t = torch.nonzero(active)[:, 0]
    r = tr[t]
    hv = h[r].double()
    pid, nid = pos.view(-1)[t], neg.view(-1)[t]
    ep, en = E.double()[pid], E.double()[nid]
    if srfrn:
        ep = torch.cat([ep, fake.double()[b["prs"].view(-1)[t]]], 1)
        en = torch.cat([en, fake.double()[b["nrs"].view(-1)[t]]], 1)
    zp, zn = (hv * ep).sum(1), (hv * en).sum(1)
    wa, wb = a64[t], b64[t]
    sp = torch.nn.functional.softplus
    lp, ln = wa * sp(-zp), wb * sp(zn)
    # loss sums: fp32 terms (__expf / log1pf, ~2^-21 relative) summed in fp32 over <= 1e5 terms
    _check("loss+", acc[0:1], lp.sum()[None], 1e-5, 0.0)
    _check("loss-", acc[1:2], ln.sum()[None], 1e-5, 0.0)
    n0, n1 = float(norm[0]), float(norm[1])
    dzp, dzn = wa * (torch.sigmoid(zp) - 1) / n0, wb * torch.sigmoid(zn) / n1
    dh_ref = torch.zeros(M, W, dtype=f64, device="cuda")
    dh_ref[r] = dzp[:, None] * ep + dzn[:, None] * en
    # dh: one fp32 product-sum of two terms; the logit carries fp32 dot-product error (~1e-6 of |h||e|) into sigmoid
    _check("dh", dh[:M], dh_ref, 1e-4, 1e-5 * float(dh_ref.abs().max()))
    _untouched("dh", dh, M)
    dE_ref = torch.zeros(N + 1, D, dtype=f64, device="cuda")
    mag = torch.zeros_like(dE_ref)
    for ids, dz in ((pid, dzp), (nid, dzn)):
        sel = ids != 0
        dE_ref.index_add_(0, ids[sel], dz[sel, None] * hv[sel, :D])
        mag.index_add_(0, ids[sel], (dz[sel, None] * hv[sel, :D]).abs())
    # atomic fp32 sums of terms that carry ~1e-4 relative error each (the sigmoid of an fp32 logit)
    _check("dE", dE, dE_ref, 0.0, 1e-4 * mag + 1e-30)
    assert float(dE[0].abs().max()) == 0.0
    if srfrn:
        dF_ref = torch.zeros(3, F, dtype=f64, device="cuda")
        magF = torch.zeros_like(dF_ref)
        for ids, dz in ((b["prs"].view(-1)[t], dzp), (b["nrs"].view(-1)[t], dzn)):
            sel = ids != 0
            dF_ref.index_add_(0, ids[sel], dz[sel, None] * hv[sel, D:])
            magF.index_add_(0, ids[sel], (dz[sel, None] * hv[sel, D:]).abs())
        _check("dF", dF, dF_ref, 0.0, 1e-4 * magF + 1e-30)
        assert float(dF[0].abs().max()) == 0.0


# --------------------------------------------------------------------------------------------------------- last position
@pytest.mark.parametrize("B,L,keep", SHAPES)
def test_layernorm_fwd_rows_last_position(B, L, keep):
    """layernorm_fwd_rows at plan.last_row: the fp32 LayerNorm of the packed row that holds each sequence's last
    position (the representative for a sequence whose last slot is a dropped pad)."""
    from srfrd_b200 import ops
    H = 80
    b, plan, M, Tp = _plan(B, L, keep, B + L + 40)
    maps = _maps(plan)
    x = _rand(plan.cap, H, 41)
    g = torch.Generator().manual_seed(42)
    w, bb = (torch.randn(H, generator=g) * 0.2 + 1.0).cuda(), (torch.randn(H, generator=g) * 0.2).cuda()
    y = _nan(B, H, torch.float32)
    ops.layernorm_fwd_rows(x, w, bb, 1e-8, y, plan.last_row, B, H)
    torch.cuda.synchronize()
    last = plan.last_row.long()
    tr = maps["tok_row"].view(B, L)[:, -1]
    assert torch.equal(last, torch.where(tr >= 0, tr, maps["seq_first"][:B]))
    ref, _, _ = _ln64(x[last], w, bb, 1e-8)
    # fp32 statistics and an fp32 output: ~1e-6 of the normalised row's scale
    _check("y", y, ref, 1e-5, 1e-5 * float(ref.abs().max()))
