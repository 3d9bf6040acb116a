"""The packed attention kernels with the out-projection folded in (srfrd_attention_fwd_packed / _bwd_packed with their
trailing out-projection arguments) against the two launches they replace: attention + gemm_tn(o, wo, residual, fused
LayerNorm) forward, gemm_tn(dr, woT) + attention backward.  Same K order, add order and rounding, so every output row
the kernels own is bit-identical; outputs start as NaN so that a row the fused kernel misses fails."""
import numpy as np
import pytest
import torch


def _lib():
    from srfrd_b200 import _lib
    return _lib.load()


def test_oproj_plan():
    """Which shapes fold the out-projection in (host arithmetic only: no device needed)."""
    lib = _lib()
    sup = lambda L, H, heads: lib.srfrd_attention_packed_oproj_supported(L, H, heads)
    assert sup(50, 80, 1) == 3                  # C2: forward and backward
    assert sup(127, 112, 1) == 3
    assert sup(50, 128, 1) == 1                 # backward: 2 x 16 KB of Wo^T no longer fit next to its 196 KB
    assert sup(50, 128, 2) == 0 and sup(50, 80, 2) == 0     # multi-head: separate launches
    assert sup(128, 80, 1) == 0                 # L + 1 > 128: no tile layout
    assert sup(50, 72, 1) == 0                  # head width not a multiple of 16


def _batch(B, L, rng):
    seq = np.zeros((B, L), np.int64)
    for b in range(B):
        n = 0 if b % 13 == 5 else int(rng.integers(1, L + 1))
        if b % 17 == 3:
            n = L                                    # full-length sequences: at L = 127 one sequence fills a tile
        if n:
            seq[b, L - n:] = rng.integers(1, 1000, n)
    return torch.from_numpy(seq).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,drop", [(4096, 50, 0.0), (4096, 50, 0.5), (37, 127, 0.0), (300, 9, 0.0),
                                      (16384, 50, 0.0)])              # the last: several tiles per CTA, forward too
def test_fused_out_projection_matches_separate_launches(B, L, drop):
    from srfrd_b200 import ops
    H = 80
    rng = np.random.default_rng(B + L)
    plan = ops.PackedPlan(B, L, "cuda")
    plan.build(_batch(B, L, rng))
    torch.cuda.synchronize()
    M, T = int(plan.rows[0]), plan.cap
    assert 0 < M <= T
    g = torch.Generator(device="cuda").manual_seed(7)
    rnd = lambda *s, sc=0.5: torch.randn(*s, generator=g, device="cuda") * sc
    q, kv, Q, dr = (rnd(T, w).to(torch.bfloat16) for w in (H, 2 * H, H, H))
    wo = rnd(H, H, sc=0.15).to(torch.bfloat16)
    woT = wo.t().contiguous()
    bo, ln_w, ln_b = rnd(H, sc=0.1), 1.0 + rnd(H, sc=0.1), rnd(H, sc=0.1)
    eps, seed, step = 1e-8, 1234, torch.full((1,), 3.0, device="cuda")
    nan = lambda w, dt=torch.bfloat16: torch.full((T, w), float("nan"), dtype=dt, device="cuda")
    out = {}
    for mode in ("separate", "fused"):
        o, r, y, st2, dq, dkv = nan(H), nan(H), nan(H), nan(2, torch.float32), nan(H), nan(2 * H)
        # dO is an intermediate, not an output: the last tile also multiplies rows past M (P = 0 there), which gemm_tn
        # leaves untouched, so they must hold finite values as the engine's workspace does
        dO = torch.zeros(T, H, dtype=torch.bfloat16, device="cuda")
        args = (plan, L, H, 1, drop, seed, 10, step)
        with ops.row_limit(plan.rows):
            if mode == "separate":
                ops.attention_fwd_packed(q, kv[:, :H], kv[:, H:], o, *args)
                ops.gemm_tn(o, wo, out_bf16=r, bias=bo, residual=Q, ln_out=y, ln_w=ln_w, ln_b=ln_b, ln_eps=eps, ln_stats=st2)
                ops.gemm_tn(dr, woT, out_bf16=dO)
                ops.attention_bwd_packed(dO, q, kv[:, :H], kv[:, H:], dq, dkv[:, :H], dkv[:, H:], *args)
            else:
                ops.attention_fwd_packed(q, kv[:, :H], kv[:, H:], o, *args, wo=wo, bias=bo, residual=Q, r=r, y=y,
                                         ln_w=ln_w, ln_b=ln_b, ln_eps=eps, ln_stats=st2)
                ops.attention_bwd_packed(None, q, kv[:, :H], kv[:, H:], dq, dkv[:, :H], dkv[:, H:], *args, dr=dr, woT=woT)
        torch.cuda.synchronize()
        out[mode] = dict(o=o, r=r, y=y, st2=st2, dq=dq, dk=dkv[:, :H], dv=dkv[:, H:])
    for name in ("o", "r", "y", "st2", "dq", "dk", "dv"):
        a, b = out["separate"][name][:M], out["fused"][name][:M]
        assert not torch.isnan(a.float()).any(), name
        assert torch.equal(a, b), (name, int((a != b).any(1).sum()), M)
    assert float(out["fused"]["dq"][:M].float().abs().max()) > 0


@pytest.mark.gpu
def test_multi_head_keeps_separate_launches():
    from srfrd_b200 import ops
    assert ops.attention_packed_oproj_supported(50, 128, 2) == 0
    B, L, H = 64, 50, 128
    plan = ops.PackedPlan(B, L, "cuda")
    plan.build(_batch(B, L, np.random.default_rng(0)))
    T = plan.cap
    z = lambda w: torch.zeros(T, w, dtype=torch.bfloat16, device="cuda")
    q, kv, o, w = z(H), z(2 * H), z(H), torch.zeros(H, H, dtype=torch.bfloat16, device="cuda")
    f = torch.ones(H, device="cuda")
    with pytest.raises(RuntimeError, match="out-projection"):
        ops.attention_fwd_packed(q, kv[:, :H], kv[:, H:], o, plan, L, H, 2, wo=w, residual=z(H), r=z(H), y=z(H),
                                 ln_w=f, ln_b=f)
