"""Per-kernel parity on the B200: every CUDA entry point (called through the C ABI via srfrd_b200.ops)
against the CPU oracle / plain fp32 torch on the same seeded inputs.  Integer and index results are
compared bit-exactly; floating point within the tolerance written next to each assertion."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

bf16 = torch.bfloat16


@pytest.fixture(scope="module")
def ops():
    from srfrd_b200 import ops as _ops
    return _ops


def rnd(shape, seed, scale=1.0, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dtype).cuda()


# ------------------------------------------------------------------------------------------- GEMMs
@pytest.mark.parametrize("M,N,K", [(128, 16, 16), (300, 80, 80), (1000, 160, 80), (257, 240, 96), (200, 272, 272),
                                   (64, 64, 80), (4096, 80, 80), (130, 544, 272), (50000, 80, 80),
                                   # several tiles per CTA with more K blocks than pipeline stages / with 3 merged K blocks
                                   (40000, 272, 272), (30000, 80, 160), (30000, 160, 80)])
def test_gemm_tn_plain(ops, M, N, K):
    A, B = rnd((M, K), 1, dtype=bf16), rnd((N, K), 2, 0.2, bf16)
    out = torch.full((M, N), float("nan"), device="cuda")
    ops.gemm_tn(A, B, out_f32=out)
    ref = A.float() @ B.float().T
    # bf16 products are exact in fp32; only the accumulation order differs -> 1e-4 relative to the row scale
    torch.testing.assert_close(out, ref, rtol=1e-4, atol=1e-4 * math.sqrt(K))
    simt = torch.empty_like(out)
    ops.gemm_ref(A, B, simt)
    torch.testing.assert_close(simt, ref, rtol=1e-4, atol=1e-4 * math.sqrt(K))


def test_gemm_tn_epilogue_variants(ops):
    M, N, K = 777, 80, 80
    A, B = rnd((M, K), 3, dtype=bf16), rnd((N, K), 4, 0.2, bf16)
    bias, res, gate = rnd((N,), 5), rnd((M, N), 6, dtype=bf16), rnd((M, N), 7, dtype=bf16)
    ids = (torch.arange(M, device="cuda") % 3 != 0).long()
    base = A.float() @ B.float().T
    # bias + relu -> bf16
    o = torch.empty(M, N, dtype=bf16, device="cuda")
    ops.gemm_tn(A, B, out_bf16=o, bias=bias, relu=True)
    torch.testing.assert_close(o.float(), torch.relu(base + bias), rtol=1e-2, atol=1e-2)
    # bias + residual + row mask
    ops.gemm_tn(A, B, out_bf16=o, bias=bias, residual=res, row_ids=ids)
    torch.testing.assert_close(o.float(), (base + bias + res.float()) * (ids != 0).float()[:, None], rtol=1e-2, atol=1e-2)
    # gate (relu backward) -> fp32
    of = torch.empty(M, N, device="cuda")
    ops.gemm_tn(A, B, out_f32=of, gate=gate)
    torch.testing.assert_close(of, base * (gate.float() > 0), rtol=1e-4, atol=1e-3)
    # strided operand / output views (kv halves)
    big = torch.zeros(M, 2 * N, dtype=bf16, device="cuda")
    ops.gemm_tn(A, B, out_bf16=big[:, N:], bias=bias)
    torch.testing.assert_close(big[:, N:].float(), base + bias, rtol=1e-2, atol=1e-2)
    assert float(big[:, :N].abs().max()) == 0.0


@pytest.mark.parametrize("T,Mo,No", [(72, 80, 80), (1000, 160, 80), (5000, 64, 80), (3000, 272, 272), (64, 16, 16),
                                     (100000, 80, 80), (700, 544, 272)])
def test_gemm_wgrad(ops, T, Mo, No):
    dY, X = rnd((T, Mo), 8, dtype=bf16), rnd((T, No), 9, dtype=bf16)
    dW = torch.zeros(Mo, No, device="cuda")
    ops.gemm_wgrad(dY, X, dW)
    ref = dY.float().T @ X.float()
    torch.testing.assert_close(dW, ref, rtol=1e-3, atol=2e-3 * math.sqrt(T))
    simt = torch.empty_like(dW)
    ops.gemm_ref(dY, X, simt, a_mn_major=True, b_mn_major=True)
    torch.testing.assert_close(simt, ref, rtol=1e-3, atol=2e-3 * math.sqrt(T))
    db = torch.zeros(Mo, device="cuda")
    ops.gemm_wgrad(dY, X, dW, db)         # accumulates; bias gradient from the fused all-ones MMA
    torch.testing.assert_close(dW, 2 * ref, rtol=1e-3, atol=4e-3 * math.sqrt(T))
    torch.testing.assert_close(db, dY.float().sum(0), rtol=1e-3, atol=2e-3 * math.sqrt(T))


@pytest.mark.parametrize("M,N,K,drop", [(300, 80, 80, 0.0), (20000, 80, 80, 0.0), (5000, 64, 64, 0.0), (3000, 96, 160, 0.0),
                                        (4100, 80, 80, 0.3), (777, 128, 128, 0.0)])
def test_gemm_tn_fused_layernorm(ops, M, N, K, drop):
    """The LayerNorm folded into the residual GEMM's epilogue equals GEMM followed by the LayerNorm kernel."""
    A, B = rnd((M, K), 50, dtype=bf16), rnd((N, K), 51, 0.2, bf16)
    bias, res = rnd((N,), 52), rnd((M, N), 53, dtype=bf16)
    w, b = rnd((N,), 54) * 0.3 + 1.0, rnd((N,), 55) * 0.1
    ids = (torch.arange(M, device="cuda") % 7 != 0).long()
    kw = dict(bias=bias, residual=res, row_ids=ids, drop_p=drop, drop_seed=99, drop_stream=3)
    x_ref = torch.empty(M, N, dtype=bf16, device="cuda")
    y_ref = torch.empty_like(x_ref)
    st_ref = torch.empty(M, 2, device="cuda")
    ops.gemm_tn(A, B, out_bf16=x_ref, **kw)
    ops.layernorm_fwd(x_ref, w, b, 1e-8, y_bf16=y_ref, stats=st_ref)
    x, y, st = torch.empty_like(x_ref), torch.empty_like(x_ref), torch.empty_like(st_ref)
    ops.gemm_tn(A, B, out_bf16=x, ln_out=y, ln_w=w, ln_b=b, ln_eps=1e-8, ln_stats=st, **kw)
    assert torch.equal(x, x_ref)
    torch.testing.assert_close(st[:, 0], st_ref[:, 0], rtol=1e-4, atol=1e-5)
    live = ids.bool()                                     # masked rows are all-zero: rstd = eps^-1/2 amplifies rounding noise
    torch.testing.assert_close(st[live, 1], st_ref[live, 1], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(y.float(), y_ref.float(), rtol=1.6e-2, atol=1e-2)
    assert float((y.float() - y_ref.float()).abs().mean()) < 1e-3


# ------------------------------------------------------------------------------------------- K1
@pytest.mark.parametrize("kind", ["SRFR", "SRFRN", "SRFU_B", "SRFU_F", "SRFU_R", "SASRec"])
def test_embed_gather_bit_exact(ops, kind):
    """Pre-LayerNorm tensor must equal the reference's embedding arithmetic bit for bit (north_star)."""
    from oracle import srfrd_oracle as O
    from tests.conftest import load_golden
    fx = load_golden(kind)
    N, L, D, Fw = (int(v) for v in fx["meta"][:4])
    sd, i = fx["param"], fx["in"]
    ref = O.embed(sd, kind, i["seq"], i["rsq"])
    ik, pk = O._emb_keys(kind)
    mode = 1 if kind in ("SRFR", "SRFRN") else (2 if kind.startswith("SRFU") else 0)
    aux = None
    aux_ids = None
    if mode == 1:
        aux, aux_ids = sd["embedding_layer.fake_embed.weight"].cuda(), i["rsq"].cuda()
    if mode == 2:
        aux = sd["embedding_layer.user_label_embed.weight"].cuda()
        aux_ids = torch.empty(i["seq"].shape[0], dtype=torch.int64, device="cuda")
        ops.srfu_labels(i["rsq"].cuda(), {"SRFU_B": 0, "SRFU_F": 1, "SRFU_R": 2}[kind], aux_ids)
        assert torch.equal(aux_ids.cpu(), O.srfu_labels(kind, i["rsq"]).long())
    H = ref.shape[-1]
    x32 = torch.empty(ref.shape[0] * L, H, device="cuda")
    xb = torch.empty(ref.shape[0] * L, H, dtype=bf16, device="cuda")
    q = torch.empty_like(xb)
    st = torch.empty(ref.shape[0] * L, 2, device="cuda")
    w, b = sd["attention_layernorms.0.weight"].cuda(), sd["attention_layernorms.0.bias"].cuda()
    ops.embed_ln_fwd(sd[ik].cuda(), sd[pk].cuda(), aux, mode, i["seq"].cuda(), aux_ids, D ** 0.5 if kind == "SASRec" else 1.0,
                     w, b, 1e-8, x0_bf16=xb, x0_f32=x32, q_bf16=q, stats=st)
    assert torch.equal(x32.cpu().view_as(ref), ref)                      # bit-exact gather + positional add
    assert torch.equal(xb.cpu(), ref.view(-1, H).to(bf16))                # and its bf16 rounding
    qref = torch.nn.functional.layer_norm(ref, (H,), sd["attention_layernorms.0.weight"], sd["attention_layernorms.0.bias"], 1e-8)
    torch.testing.assert_close(q.float().cpu().view_as(qref), qref, rtol=1e-2, atol=1e-2)   # bf16 output


def test_embed_large_bit_exact(ops):
    g = torch.Generator().manual_seed(11)
    N, L, D, Fw, B = 5000, 50, 64, 16, 257
    E, P, Fe = torch.randn(N + 1, D, generator=g), torch.randn(L, D, generator=g), torch.randn(3, Fw, generator=g)
    seq = torch.randint(0, N + 1, (B, L), generator=g)
    seq[:, :20] = 0
    rsq = torch.randint(0, 3, (B, L), generator=g)
    ref = torch.cat([E[seq] + P[None], Fe[rsq]], -1) * (seq != 0)[..., None]
    out = torch.empty(B * L, D + Fw, device="cuda")
    ops.embed_ln_fwd(E.cuda(), P.cuda(), Fe.cuda(), 1, seq.cuda(), rsq.cuda(), 1.0, None, None, 1e-8, x0_f32=out)
    assert torch.equal(out.cpu().view_as(ref), ref)


# ------------------------------------------------------------------------------------------- LayerNorm
@pytest.mark.parametrize("T,H", [(100, 80), (1000, 64), (333, 272), (64, 16)])
def test_layernorm_fwd_bwd(ops, T, H):
    x = rnd((T, H), 20, dtype=bf16)
    w, b = rnd((H,), 21) * 0.3 + 1.0, rnd((H,), 22) * 0.1
    y32 = torch.empty(T, H, device="cuda")
    yb = torch.empty(T, H, dtype=bf16, device="cuda")
    st = torch.empty(T, 2, device="cuda")
    ops.layernorm_fwd(x, w, b, 1e-8, y_f32=y32, stats=st)
    ops.layernorm_fwd(x, w, b, 1e-8, y_bf16=yb)
    xr = x.float().clone().requires_grad_(True)
    wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    ref = torch.nn.functional.layer_norm(xr, (H,), wr, br, 1e-8)
    torch.testing.assert_close(y32, ref.detach(), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(yb.float(), ref.detach(), rtol=1e-2, atol=1e-2)
    # last-position-only variant
    L = 4 if T % 4 == 0 else 1
    ylast = torch.empty(T // L, H, device="cuda")
    ops.layernorm_fwd(x, w, b, 1e-8, y_f32=ylast, T=T // L, H=H, row_stride=L, row_offset=L - 1)
    torch.testing.assert_close(ylast, ref.detach().view(T // L, L, H)[:, -1], rtol=1e-5, atol=1e-5)
    # backward, fp32 and bf16 upstream gradients, with add + row mask
    dy = rnd((T, H), 23)
    add = rnd((T, H), 24, dtype=bf16)
    ids = (torch.arange(T, device="cuda") % 4 != 1).long()
    ref.backward(dy)
    dx = torch.empty(T, H, dtype=bf16, device="cuda")
    dw, db = torch.zeros(H, device="cuda"), torch.zeros(H, device="cuda")
    ops.layernorm_bwd(dy, x, st, w, dx, dw, db, add=add, row_ids=ids)
    dx_ref = (xr.grad + add.float()) * (ids != 0).float()[:, None]
    torch.testing.assert_close(dx.float(), dx_ref, rtol=2e-2, atol=2e-2)
    torch.testing.assert_close(dw, wr.grad, rtol=1e-3, atol=1e-3 * math.sqrt(T))
    torch.testing.assert_close(db, br.grad, rtol=1e-3, atol=1e-3 * math.sqrt(T))
    dw.zero_(); db.zero_()
    ops.layernorm_bwd(dy.to(bf16), x, st, w, dx, dw, db)
    torch.testing.assert_close(dx.float(), xr.grad, rtol=3e-2, atol=3e-2)


def test_ragged_widths_gather_layernorm_wgrad(ops):
    """Widths that are not multiples of 8 / 16 (the reference's own 45 + 5): operands carry zero padding columns up to
    the padded leading dimension; gather stays bit-exact, LayerNorm statistics use the true width."""
    from oracle import srfrd_oracle as O
    from tests.conftest import load_golden
    fx = load_golden("SRFR_w50")
    N, L, D, Fw = (int(v) for v in fx["meta"][:4])
    H, Hp = D + Fw, 64
    sd, i = fx["param"], fx["in"]
    ref = O.embed(sd, "SRFR", i["seq"], i["rsq"])
    T = ref.shape[0] * L
    x32 = torch.empty(T, H, device="cuda")
    xb = torch.full((T, Hp), 7.0, dtype=bf16, device="cuda")
    q = torch.full((T, Hp), 7.0, dtype=bf16, device="cuda")
    st = torch.empty(T, 2, device="cuda")
    w, b = sd["attention_layernorms.0.weight"].cuda(), sd["attention_layernorms.0.bias"].cuda()
    ops.embed_ln_fwd(sd["embedding_layer.item_embed.weight"].cuda(), sd["embedding_layer.pos_embed.weight"].cuda(),
                     sd["embedding_layer.fake_embed.weight"].cuda(), 1, i["seq"].cuda(), i["rsq"].cuda(), 1.0, w, b, 1e-8,
                     x0_bf16=xb, x0_f32=x32, q_bf16=q, stats=st)
    assert torch.equal(x32.cpu().view_as(ref), ref)                       # bit-exact gather + positional add
    assert torch.equal(xb[:, :H].cpu(), ref.view(-1, H).to(bf16))
    assert float(xb[:, H:56].abs().max()) == 0.0 and float(q[:, H:56].abs().max()) == 0.0   # chunk padding written as 0
    qref = torch.nn.functional.layer_norm(ref, (H,), w.cpu(), b.cpu(), 1e-8)
    torch.testing.assert_close(q[:, :H].float().cpu().view_as(qref), qref, rtol=1e-2, atol=1e-2)
    # LayerNorm forward / backward on a zero-padded (T, 64) operand with true width 50
    x = torch.zeros(300, Hp, dtype=bf16, device="cuda")
    x[:, :H] = rnd((300, H), 25, dtype=bf16)
    y = torch.full((300, Hp), 3.0, dtype=bf16, device="cuda")
    st2 = torch.empty(300, 2, device="cuda")
    ops.layernorm_fwd(x, w, b, 1e-8, y_bf16=y, stats=st2, H=H)
    xr = x[:, :H].float().clone().requires_grad_(True)
    wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    yr = torch.nn.functional.layer_norm(xr, (H,), wr, br, 1e-8)
    torch.testing.assert_close(y[:, :H].float(), yr.detach(), rtol=1e-2, atol=1e-2)
    assert float(y[:, H:56].abs().max()) == 0.0
    dy = torch.zeros(300, Hp, dtype=bf16, device="cuda")
    dy[:, :H] = rnd((300, H), 26, dtype=bf16)
    yr.backward(dy[:, :H].float())
    dx = torch.full((300, Hp), 5.0, dtype=bf16, device="cuda")
    dw, db = torch.zeros(H, device="cuda"), torch.zeros(H, device="cuda")
    ops.layernorm_bwd(dy, x, st2, w, dx, dw, db, H=H)
    torch.testing.assert_close(dx[:, :H].float(), xr.grad, rtol=3e-2, atol=3e-2)
    assert float(dx[:, H:56].abs().max()) == 0.0
    torch.testing.assert_close(dw, wr.grad, rtol=1e-3, atol=2e-2)
    torch.testing.assert_close(db, br.grad, rtol=1e-3, atol=2e-2)
    # weight gradient with true widths 50 x 45 inside padded operands
    dY = torch.zeros(700, Hp, dtype=bf16, device="cuda"); dY[:, :H] = rnd((700, H), 27, dtype=bf16)
    X = torch.zeros(700, 48, dtype=bf16, device="cuda"); X[:, :D] = rnd((700, D), 28, dtype=bf16)
    dW, dbias = torch.zeros(H, D, device="cuda"), torch.zeros(H, device="cuda")
    ops.gemm_wgrad(dY, X, dW, dbias, Mo=H, No=D)
    torch.testing.assert_close(dW, dY[:, :H].float().T @ X[:, :D].float(), rtol=1e-3, atol=2e-3 * math.sqrt(700))
    torch.testing.assert_close(dbias, dY[:, :H].float().sum(0), rtol=1e-3, atol=2e-3 * math.sqrt(700))


# ------------------------------------------------------------------------------------------- attention
def _attn_ref(q, k, v, heads):
    from oracle import srfrd_oracle as O
    return O.attention(q, k, v, heads)


def _attn_ref_dropout(q, k, v, heads, factor):
    """fp64 causal attention whose probabilities are multiplied by the dropout factors (B, heads, L, L) after the
    softmax, as every attention kernel does (F.dropout on the attention weights, SRFR_model.py:112)."""
    B, L, H = q.shape
    hd = H // heads
    split = lambda x: x.view(B, L, heads, hd).transpose(1, 2)
    s = split(q) @ split(k).transpose(-1, -2) / math.sqrt(hd)
    s = s.masked_fill(~torch.ones(L, L, dtype=torch.bool).tril(), float("-inf"))
    return ((torch.softmax(s, -1) * factor) @ split(v)).transpose(1, 2).reshape(B, L, H)


_ATTN_CASES = [(3, 12, 32, 1), (5, 50, 80, 1), (2, 50, 80, 2), (2, 200, 272, 1), (4, 7, 16, 4), (64, 50, 64, 1), (7, 50, 64, 2),
               (3, 128, 64, 1), (5, 100, 128, 1), (300, 50, 80, 1), (9, 33, 96, 3), (2, 240, 32, 1),
               # 128 < maxlen <= 256: two query tiles per sequence, FlashAttention-2 style backward
               (3, 129, 64, 1), (2, 256, 128, 2), (5, 200, 80, 1), (160, 200, 272, 1), (3, 150, 96, 2)]
# dropout p = 0.3 with two heads on each kernel: SIMT (head width 20), the tile kernel (L <= 128), the long kernel (L > 128)
_ATTN_DROP = [(6, 20, 40, 2), (7, 50, 128, 2), (3, 150, 128, 2)]


@pytest.mark.parametrize("B,L,H,heads,drop", [c + (0.0,) for c in _ATTN_CASES] + [c + (0.3,) for c in _ATTN_DROP],
                         ids=["-".join(map(str, c)) for c in _ATTN_CASES] + ["-".join(map(str, c)) + "-drop0.3" for c in _ATTN_DROP])
def test_attention_fwd_bwd(ops, B, L, H, heads, drop):
    from tests.test_dropout_mask import keep_mask, masked
    T = B * L
    q, kv = rnd((T, H), 30, 0.7, bf16), rnd((T, 2 * H), 31, 0.7, bf16)
    o = torch.empty(T, H, dtype=bf16, device="cuda")
    stats = torch.zeros(T * heads, 4, device="cuda") if L > 128 else None
    seed, stream, step = 2024, 6, 3.0
    dkw = dict(drop_p=drop, seed=seed, stream_id=stream, drop_step=torch.tensor([step], device="cuda")) if drop else {}
    ops.attention_fwd(q, kv[:, :H], kv[:, H:], o, B, L, H, heads, stats=stats, **dkw)
    dt = torch.float64 if drop else torch.float32
    qr = q.to(dt).cpu().view(B, L, H).requires_grad_(True)
    kr = kv[:, :H].to(dt).cpu().view(B, L, H).requires_grad_(True)
    vr = kv[:, H:].to(dt).cpu().view(B, L, H).requires_grad_(True)
    if drop:
        # dense kernels hash element ((b * heads + h) * L + query) * L + key
        keep = keep_mask(seed, stream, np.arange(B * heads * L * L).reshape(B, heads, L, L), drop, step)
        ref = _attn_ref_dropout(qr, kr, vr, heads, masked(torch.ones(keep.shape), keep, drop).double())
    else:
        ref = _attn_ref(qr, kr, vr, heads)
    torch.testing.assert_close(o.to(dt).cpu().view(B, L, H), ref.detach(), rtol=2e-2, atol=1e-2)   # bf16 output
    ntri = (L * (L + 1) // 2 + 3) // 4 * 4      # SIMT path (no stats given): packed causal triangles of P and dS in smem
    if L > 128 and 2 * ntri * 4 + 4 * L * 34 > 227 * 1024:
        with pytest.raises(RuntimeError, match="shared memory"):
            ops.attention_bwd(o, q, kv[:, :H], kv[:, H:], o, kv[:, :H], kv[:, H:], B, L, H, heads)
    do = rnd((T, H), 32, dtype=bf16)
    ref.backward(do.to(dt).cpu().view(B, L, H))
    dq = torch.empty(T, H, dtype=bf16, device="cuda")
    dkv = torch.empty(T, 2 * H, dtype=bf16, device="cuda")
    ops.attention_bwd(do, q, kv[:, :H], kv[:, H:], dq, dkv[:, :H], dkv[:, H:], B, L, H, heads, o=o, stats=stats, **dkw)
    for got, want in ((dq, qr.grad), (dkv[:, :H], kr.grad), (dkv[:, H:], vr.grad)):
        w = want.view(T, H)
        torch.testing.assert_close(got.to(dt).cpu(), w, rtol=3e-2, atol=2e-2 * float(w.abs().max()))


def test_attention_dropout_is_consistent(ops):
    B, L, H = 8, 20, 32
    T = B * L
    q, kv = rnd((T, H), 33, 0.5, bf16), rnd((T, 2 * H), 34, 0.5, bf16)
    o1, o2, o3 = (torch.empty(T, H, dtype=bf16, device="cuda") for _ in range(3))
    step = torch.tensor([3.0], device="cuda")
    ops.attention_fwd(q, kv[:, :H], kv[:, H:], o1, B, L, H, 1, 0.5, 77, 5, step)
    ops.attention_fwd(q, kv[:, :H], kv[:, H:], o2, B, L, H, 1, 0.5, 77, 5, step)
    step += 1
    ops.attention_fwd(q, kv[:, :H], kv[:, H:], o3, B, L, H, 1, 0.5, 77, 5, step)
    assert torch.equal(o1, o2) and not torch.equal(o1, o3)
    # maxlen > 128 (tile-pair kernels): the backward regenerates the forward's mask from (seed, step, element), so the
    # gradient of sum(o * do) w.r.t. v equals P_dropped^T do -- checked through a finite linear probe in v
    B, L, H = 3, 200, 64
    T = B * L
    q, kv = rnd((T, H), 35, 0.5, bf16), rnd((T, 2 * H), 36, 0.5, bf16)
    st = torch.zeros(T, 4, device="cuda")
    oa, ob = torch.empty(T, H, dtype=bf16, device="cuda"), torch.empty(T, H, dtype=bf16, device="cuda")
    ops.attention_fwd(q, kv[:, :H], kv[:, H:], oa, B, L, H, 1, 0.3, 99, 6, step, stats=st)
    ops.attention_fwd(q, kv[:, :H], kv[:, H:], ob, B, L, H, 1, 0.3, 99, 6, step, stats=st)
    assert torch.equal(oa, ob)
    do = rnd((T, H), 37, dtype=bf16)
    dq, dkv = torch.empty(T, H, dtype=bf16, device="cuda"), torch.empty(T, 2 * H, dtype=bf16, device="cuda")
    ops.attention_bwd(do, q, kv[:, :H], kv[:, H:], dq, dkv[:, :H], dkv[:, H:], B, L, H, 1, 0.3, 99, 6, step, o=oa, stats=st)
    dv_dir = rnd((T, H), 38, 0.25, bf16)                      # o is linear in v: <do, o(v + e) - o(v)> == <dv, e>
    kv2 = kv.clone()
    kv2[:, H:] = (kv[:, H:].float() + dv_dir.float()).to(bf16)
    e = kv2[:, H:].float() - kv[:, H:].float()
    ops.attention_fwd(q, kv2[:, :H], kv2[:, H:], ob, B, L, H, 1, 0.3, 99, 6, step, stats=torch.zeros_like(st))
    lhs = float((do.float() * (ob.float() - oa.float())).sum())
    rhs = float((dkv[:, H:].float() * e).sum())
    assert abs(lhs - rhs) <= 0.03 * max(abs(lhs), abs(rhs)) + 0.5, (lhs, rhs)


# ------------------------------------------------------------------------------------------- K4 scoring / loss
@pytest.mark.parametrize("srfrn", [False, True])
def test_score_loss_fused_and_split(ops, srfrn):
    from oracle import srfrd_oracle as O
    g = torch.Generator().manual_seed(40)
    T, N, D, Fw = 999, 300, 64, 16
    W = D + (Fw if srfrn else 0)
    h = torch.randn(T, W, generator=g)
    E, Fe = torch.randn(N + 1, D, generator=g) * 0.3, torch.randn(3, Fw, generator=g) * 0.3
    pos = torch.randint(0, N + 1, (T,), generator=g)
    pos[torch.rand(T, generator=g) < 0.5] = 0
    neg = torch.where(pos != 0, torch.randint(1, N + 1, (T,), generator=g), torch.zeros_like(pos))
    prs, nrs = torch.randint(1, 3, (T,), generator=g) * (pos != 0), (pos != 0).long()
    wpos = torch.rand(T, generator=g) * (pos != 0)
    wneg = torch.rand(T, generator=g) * (pos != 0)

    def rows(ids, fids):
        r = E[ids]
        return torch.cat([r, Fe[fids]], -1) if srfrn else r

    for use_w in (False, True):
        hr, Er, Fr = h.clone().requires_grad_(True), E.clone().requires_grad_(True), Fe.clone().requires_grad_(True)
        r_p = torch.cat([Er[pos], Fr[prs]], -1) if srfrn else Er[pos]
        r_n = torch.cat([Er[neg], Fr[nrs]], -1) if srfrn else Er[neg]
        zp, zn = (hr * r_p).sum(-1), (hr * r_n).sum(-1)
        if use_w:
            loss = O.weighted_loss(zp, zn, wpos, wneg)
        else:
            loss = O.reference_loss(zp, zn, pos)           # trainer.py:36-38
        loss.backward()
        Er.grad[0] = 0                                      # padding_idx
        if srfrn:
            Fr.grad[0] = 0
        c = lambda t: None if t is None else t.cuda()
        ft = c(Fe) if srfrn else None
        norm = torch.zeros(2, device="cuda")
        ops.weight_sums(c(pos), c(wpos) if use_w else None, c(wneg) if use_w else None, norm)
        acc = torch.zeros(2, device="cuda")
        dh = torch.full((T, W), float("nan"), device="cuda")
        dE, dF = torch.zeros(N + 1, D, device="cuda"), torch.zeros(3, Fw, device="cuda")
        zpo, zno = torch.empty(T, device="cuda"), torch.empty(T, device="cuda")
        ops.score_loss_fused(c(h), c(E), ft, c(pos), c(neg), c(prs) if srfrn else None, c(nrs) if srfrn else None,
                             c(wpos) if use_w else None, c(wneg) if use_w else None, norm, acc, dh, dE,
                             dF if srfrn else None, zpo, zno)
        out = torch.zeros(1, device="cuda")
        ops.loss_finalize(acc, norm, out)
        assert abs(float(out) - float(loss)) < 1e-5 * max(1.0, abs(float(loss)))       # fp32 loss
        torch.testing.assert_close(zpo.cpu(), zp.detach(), rtol=1e-5, atol=1e-5)
        torch.testing.assert_close(dh.cpu(), hr.grad, rtol=1e-4, atol=1e-7)
        torch.testing.assert_close(dE.cpu(), Er.grad, rtol=1e-4, atol=1e-7)
        if srfrn:
            torch.testing.assert_close(dF.cpu(), Fr.grad, rtol=1e-4, atol=1e-6)
        # split path: logits forward, then backward from given dz
        z1, z2 = torch.empty(T, device="cuda"), torch.empty(T, device="cuda")
        ops.score_fwd(c(h), c(E), ft, c(pos), c(neg), c(prs) if srfrn else None, c(nrs) if srfrn else None, z1, z2)
        torch.testing.assert_close(z2.cpu(), zn.detach(), rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------------------------------- K5 / colsum / Adam
def test_embed_bwd_and_positional_colsum(ops):
    g = torch.Generator().manual_seed(50)
    B, L, N, D, Fw = 37, 12, 90, 32, 16
    H = D + Fw
    E, P, Fe = (torch.randn(s, generator=g).requires_grad_(True) for s in ((N + 1, D), (L, D), (3, Fw)))
    seq = torch.randint(0, N + 1, (B, L), generator=g)
    seq[:, :3] = 0
    rsq = torch.randint(0, 3, (B, L), generator=g)
    x0 = torch.cat([E[seq] + P[None], Fe[rsq]], -1) * (seq != 0)[..., None]
    dx = (torch.randn(B, L, H, generator=g) * (seq != 0)[..., None]).to(bf16)
    x0.backward(dx.float())
    E.grad[0] = 0
    Fe.grad[0] = 0
    dE, dF, dP = torch.zeros(N + 1, D, device="cuda"), torch.zeros(3, Fw, device="cuda"), torch.zeros(L, D, device="cuda")
    dxc = dx.cuda().view(B * L, H)
    ops.embed_bwd(dxc, seq.cuda(), rsq.cuda(), D, Fw, 1, 1.0, dE, dF)
    tmp = torch.zeros(L * H, device="cuda")
    ops.colsum(dxc, tmp, M=B, N=L * H, ld=L * H)
    ops.add_segments(tmp, L * H, H, D, dP)
    torch.testing.assert_close(dE.cpu(), E.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(dF.cpu(), Fe.grad, rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(dP.cpu(), P.grad, rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("M,N", [(1000, 80), (77, 160), (5000, 64), (33, 4000)])
def test_colsum(ops, M, N):
    X = rnd((M, N), 60, dtype=bf16)
    out = torch.zeros(N, device="cuda")
    ops.colsum(X, out)
    torch.testing.assert_close(out, X.float().sum(0), rtol=1e-4, atol=1e-3 * math.sqrt(M))


def test_adam_matches_torch(ops):
    n = 10007
    p0, grads = rnd((n,), 70), [rnd((n,), 71 + i) for i in range(3)]
    ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-3, betas=(0.9, 0.98))
    npad = (n + 3) // 4 * 4
    p, g, m, v = (torch.zeros(npad, device="cuda") for _ in range(4))
    p[:n] = p0
    state = torch.zeros(4, device="cuda")
    for gi in grads:
        ref.grad = gi.clone()
        opt.step()
        g[:n] = gi
        ops.adam_tick(state, 0.9, 0.98)
        ops.adam_step(p, g, m, v, 1e-3, 0.9, 0.98, 1e-8, state, zero_grad=True)
        assert float(g.abs().max()) == 0.0
    torch.testing.assert_close(p[:n], ref.detach(), rtol=1e-6, atol=1e-7)


def test_cast_weights_and_dropout_apply(ops):
    W = rnd((48, 32), 80)
    d, dt = torch.zeros(48, 32, dtype=bf16, device="cuda"), torch.zeros(32, 48, dtype=bf16, device="cuda")
    tab, n = ops.make_cast_table([(W, d, dt)], "cuda")
    ops.cast_weights(tab, n)
    assert torch.equal(d, W.to(bf16)) and torch.equal(dt, W.to(bf16).T.contiguous())
    x = torch.ones(4096, 64, dtype=bf16, device="cuda")
    y = torch.empty_like(x)
    ops.dropout_apply(x, y, 64, 0.5, 123, 7)
    keep = float((y != 0).float().mean())
    assert abs(keep - 0.5) < 0.01 and float(y.max()) == 2.0
    # the GEMM epilogue draws the same mask for the same (seed, stream, element)
    A, B = torch.eye(64, dtype=bf16, device="cuda").repeat(64, 1), torch.eye(64, dtype=bf16, device="cuda")
    o = torch.empty(4096, 64, dtype=bf16, device="cuda")
    ops.gemm_tn(A, B, out_bf16=o, drop_p=0.5, drop_seed=123, drop_stream=7)
    y2 = torch.empty_like(x)
    ops.dropout_apply(A.contiguous(), y2, 64, 0.5, 123, 7)
    assert torch.equal(o, y2)


# ------------------------------------------------------------------------------------------- K8 / K9
def _dyadic(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(-16, 17, shape, generator=g).float() / 8.0


@pytest.mark.parametrize("U,N,D", [(5, 300, 16), (200, 5000, 64), (130, 70000, 64), (64, 1000, 256)])
def test_catalogue_topk_bit_exact_on_dyadic_inputs(ops, U, N, D):
    """Entries k/8 with |k| <= 16: every partial sum is exact in fp32, so scores are identical under any
    accumulation order and the top-10 ids must match the oracle exactly, ties broken by lower id."""
    from oracle import srfrd_oracle as O
    from srfrd_b200 import evaluation as EV
    feats, table = _dyadic((U, D), 90), _dyadic((N + 1, D), 91)
    table[5] = table[9]                                   # force exact ties
    v_ref, i_ref = O.catalogue_topk(feats, table, 10)
    idx = EV.CatalogueIndex(table.cuda(), 0)
    s, i = EV.local_topk(feats.cuda(), idx, n_split=1)
    assert np.array_equal(i.cpu().numpy(), i_ref)
    assert np.array_equal(s.cpu().numpy(), v_ref.astype(np.float32))


def test_catalogue_topk_gaussian_and_split_precision(ops):
    from oracle import srfrd_oracle as O
    from srfrd_b200 import evaluation as EV
    g = torch.Generator().manual_seed(92)
    U, N, D = 300, 40000, 64
    feats = torch.randn(U, D, generator=g)
    table = (torch.randn(N + 1, D, generator=g) * 0.05).to(bf16).float()       # table exactly bf16 (C3)
    idx = EV.CatalogueIndex(table.cuda(), 0)
    # n_split=1: operands rounded to bf16; oracle fed the same rounded operands, fp64 accumulate
    v_ref, i_ref = O.catalogue_topk(feats, table, 10, operand_dtype=bf16)
    s, i = EV.local_topk(feats.cuda(), idx, 1)
    got_i, got_s = i.cpu().numpy(), s.cpu().numpy()
    mism = got_i != i_ref
    # any index mismatch must be a near-tie: score gap below fp32 accumulation noise
    assert np.all(np.abs(got_s - v_ref)[mism] < 1e-5) and mism.mean() < 0.01
    np.testing.assert_allclose(got_s, v_ref, rtol=1e-5, atol=1e-5)
    # n_split=3: user features kept to ~fp32 accuracy -> matches the fp32 oracle
    v32, i32 = O.catalogue_topk(feats, table, 10)
    s3, i3 = EV.local_topk(feats.cuda(), idx, 3)
    m3 = i3.cpu().numpy() != i32
    assert m3.mean() < 0.01 and np.all(np.abs(s3.cpu().numpy() - v32)[m3] < 1e-5)
    np.testing.assert_allclose(s3.cpu().numpy(), v32, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("U,N,G", [(150, 9000, 8), (64, 40, 8)])
def test_sharded_topk_equals_unsharded(ops, U, N, G):
    """Row shards emulated on one GPU: per-shard top-10 + merge == unsharded top-10, bit-exact.  N = 40 over 8 ranks leaves
    ranks with a handful of rows and one with none (more ranks than table rows is legal)."""
    from oracle import srfrd_oracle as O
    from srfrd_b200 import evaluation as EV
    D = 64
    feats, table = _dyadic((U, D), 93), _dyadic((N + 1, D), 94)
    _, i_ref = O.catalogue_topk(feats, table, 10)
    ss, ii = [], []
    for r in range(G):
        lo, hi = EV.CatalogueIndex.shard_bounds(N + 1, r, G)
        s, i = EV.local_topk(feats.cuda(), EV.CatalogueIndex(table[lo:hi].cuda(), lo), 1)
        ss.append(s); ii.append(i)
    ms, mi = EV.merge_shards(torch.stack(ss, 1), torch.stack(ii, 1))
    assert np.array_equal(mi.cpu().numpy(), i_ref)
    ndcg, hr = EV.hr_ndcg_from_topk(mi, torch.from_numpy(i_ref[:, 3]))
    assert hr == 1.0 and abs(ndcg - 1 / np.log2(5)) < 1e-12


def test_invalid_arguments_fail_loudly(ops):
    A, B = rnd((10, 20), 95, dtype=bf16), rnd((16, 20), 96, dtype=bf16)    # K = 20 is not a multiple of 8
    with pytest.raises(RuntimeError, match="gemm_tn"):
        ops.gemm_tn(A, B, out_f32=torch.empty(10, 16, device="cuda"))
    with pytest.raises(RuntimeError):
        ops.embed_ln_fwd(torch.zeros(4, 8), torch.zeros(2, 8), None, 0, torch.zeros(1, 2, dtype=torch.int64), None, 1.0,
                         None, None, 1e-8, x0_f32=torch.zeros(2, 8))      # CPU tensors: no fallback
