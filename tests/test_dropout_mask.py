"""Every in-kernel dropout mask against a host restatement of the hash, bit for bit.

The mask is a pure function (csrc/common.cuh): element `idx` of a launch with (seed, stream, step) is kept when
    hash_u32(mix_seed(seed, step), stream, idx) >= (uint32)((double)(float)p * 2^32)
and a kept value is multiplied by the fp32 scale 1 / (1 - p).  `keep_mask` restates it in numpy (uint32 wrap-around
arithmetic), so each kernel's element index -- written next to its dropout_keep call -- is checked exactly, not only
its keep rate (test_gpu_round2.test_dropout_keep_rate_and_mean_preservation) or its self-consistency.
Operands are chosen so that the pre-dropout values are exact in fp32, which makes the whole output an exact comparison."""
import numpy as np
import pytest
import torch

bf16 = torch.bfloat16
_M32 = 0xFFFFFFFF
_M64 = 0xFFFFFFFFFFFFFFFF


def keep_mask(seed, stream, idx, p, step=None):
    """numpy bool array: True where the kernels keep element `idx` (any integer array) of a launch with (seed, stream),
    dropout probability p and optional device step value `step` (mix_seed reads the raw bits of the fp32 step)."""
    seed = int(seed) & _M64
    if step is not None:
        bits = int(np.float32(step).view(np.uint32))
        seed ^= (bits * 0xD6E8FEB86659FD93) & _M64
    idx = np.asarray(idx).astype(np.uint64)
    lo = (idx & np.uint64(_M32)).astype(np.uint32)
    hi = (idx >> np.uint64(32)).astype(np.uint32)
    u = np.uint32
    const = (seed & _M32) ^ (((seed >> 32) * 0xC2B2AE3D) & _M32) ^ (((int(stream) & _M32) * 0x27D4EB2F) & _M32)
    x = (lo * u(0x9E3779B1)) ^ (hi * u(0x85EBCA77)) ^ u(const)
    x ^= x >> u(16); x *= u(0x7FEB352D)
    x ^= x >> u(15); x *= u(0x846CA68B)
    x ^= x >> u(16)
    return x >= u(int(float(np.float32(p)) * 4294967296.0))


def drop_scale(p):
    """The kernels' fp32 scale of a kept value, 1.f / (1.f - p)."""
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


def masked(x32, keep, p):
    """x (fp32 tensor) through the mask: kept values times the fp32 scale (fp32 product, as in the kernels), else 0."""
    k = torch.from_numpy(np.ascontiguousarray(keep)).to(x32.device)
    return torch.where(k, x32 * torch.tensor(drop_scale(p), dtype=torch.float32, device=x32.device), torch.zeros_like(x32))


# (seed, stream, step): two seeds, two streams, a zero and a non-zero step; p = 0.3 and 0.5
CASES = [(1234, 11, None, 0.3), (1234, 12, 3.0, 0.3), (987654321987, 11, 7.0, 0.5), (987654321987, 12, None, 0.5)]


def _step(step):
    return None if step is None else torch.tensor([step], dtype=torch.float32, device="cuda")


def _ints(shape, lo, hi, gen, scale=1.0):
    """Small integers (times a power of two): bf16-exact, and their products and short sums are exact in fp32."""
    return (torch.randint(lo, hi + 1, shape, generator=gen).float() * scale).cuda()


def test_keep_mask_rate_and_threshold():
    """The host restatement itself (no device): keep rate 1 - p within 4 sigma, and the threshold's edge cases."""
    idx = np.arange(1 << 20, dtype=np.int64) + (5 << 32)
    for seed, stream, step, p in CASES:
        k = keep_mask(seed, stream, idx, p, step)
        assert abs(k.mean() - (1 - p)) < 4 * np.sqrt(p * (1 - p) / k.size)
    assert keep_mask(1, 2, idx[:100], 0.0).all()                 # threshold 0 keeps everything
    assert not np.array_equal(keep_mask(1, 2, idx, 0.5), keep_mask(1, 2, idx, 0.5, 0.0 + 1.0))
    assert np.array_equal(keep_mask(1, 2, idx, 0.5), keep_mask(1, 2, idx, 0.5, 0.0))   # step 0.0: bits 0, seed unchanged


@pytest.mark.gpu
@pytest.mark.parametrize("seed,stream,step,p", CASES)
def test_dropout_apply_mask_is_exact(seed, stream, step, p):
    """srfrd_dropout_apply, element index r * N + c, on strided input and output views."""
    from srfrd_b200 import ops
    M, N = 1000, 80
    g = torch.Generator().manual_seed(seed % 1000 + stream)
    big = (torch.randn(M, 2 * N, generator=g) + 3.0).to(bf16).cuda()           # no zeros among the inputs
    x = big[:, N:]
    out_big = torch.full((M, N + 16), float("nan"), dtype=bf16, device="cuda")
    out = out_big[:, 8:8 + N]
    ops.dropout_apply(x, out, N, p, seed, stream, _step(step))
    keep = keep_mask(seed, stream, np.arange(M * N).reshape(M, N), p, step)
    assert torch.equal(out, masked(x.float(), keep, p).to(bf16))             # zeros where dropped, bf16(x * scale) else
    assert torch.isnan(out_big[:, :8].float()).all() and torch.isnan(out_big[:, 8 + N:].float()).all()


@pytest.mark.gpu
@pytest.mark.parametrize("seed,stream,step,p", CASES)
def test_gemm_tn_dropout_mask_is_exact(seed, stream, step, p):
    """The gemm_tn epilogue, element index row * N + n (N = the output's width, not its leading dimension): a strided
    output view, M not a multiple of the 128-row tile, several column tiles.  bias + A B^T is exact in fp32."""
    from srfrd_b200 import ops
    M, N, K = 777, 160, 80
    g = torch.Generator().manual_seed(seed % 1000 + stream)
    A, B = _ints((M, K), -3, 3, g).to(bf16), _ints((N, K), -3, 3, g, 0.25).to(bf16)
    bias = _ints((N,), -40, 40, g, 0.125) + 0.0625                            # never zero: x != 0 everywhere
    x = A.double() @ B.double().T + bias.double()
    assert float((x - x.float().double()).abs().max()) == 0.0                 # exactly representable in fp32
    big = torch.full((M, 2 * N + 8), float("nan"), dtype=bf16, device="cuda")
    out = big[:, N:2 * N]
    ops.gemm_tn(A, B, out_bf16=out, bias=bias, drop_p=p, drop_seed=seed, drop_stream=stream, drop_step=_step(step))
    keep = keep_mask(seed, stream, np.arange(M * N).reshape(M, N), p, step)
    assert torch.equal(out, masked(x.float(), keep, p).to(bf16))
    assert torch.isnan(big[:, :N].float()).all() and torch.isnan(big[:, 2 * N:].float()).all()


@pytest.mark.gpu
@pytest.mark.parametrize("seed,stream,step,p", CASES[:2])
def test_mlp2_tn_dropout_masks_are_exact(seed, stream, step, p):
    """srfrd_mlp2_tn, both stages, element index row * N + c with each stage's own stream.  Stage 1 (relu(drop1(A W1^T +
    b1))) is exact in fp32 and compared bit for bit.  Stage 2 (drop2(mid W2^T + b2)) is compared with the fp64 product of
    the kernel's own bf16 intermediate: the zeros must sit exactly where the host mask drops, and the kept values are
    within bf16 rounding of ref * scale."""
    from srfrd_b200 import ops
    M, N = 1000, 80
    s1, s2 = stream, stream + 7
    g = torch.Generator().manual_seed(seed % 1000 + stream)
    A, W1 = _ints((M, N), -3, 3, g).to(bf16), _ints((N, N), -3, 3, g, 0.25).to(bf16)
    W2 = (torch.randn(N, N, generator=g) * 0.2).to(bf16).cuda()
    b1 = _ints((N,), -40, 40, g, 0.125) + 0.0625
    b2 = (torch.randn(N, generator=g) * 0.1).cuda()
    mid = torch.full((M, N), float("nan"), dtype=bf16, device="cuda")
    out = torch.full((M, N), float("nan"), dtype=bf16, device="cuda")
    ops.mlp2_tn(A, W1, W2, mid, out, bias1=b1, bias2=b2, relu1=True, drop1_p=p, drop2_p=p, drop1_stream=s1, drop2_stream=s2,
                drop_seed=seed, drop_step=_step(step))
    idx = np.arange(M * N).reshape(M, N)
    x1 = (A.double() @ W1.double().T + b1.double()).float()
    assert torch.equal(mid, torch.relu(masked(x1, keep_mask(seed, s1, idx, p, step), p)).to(bf16))
    k2 = keep_mask(seed, s2, idx, p, step)
    x2 = mid.double() @ W2.double().T + b2.double()
    ref = torch.where(torch.from_numpy(k2).cuda(), x2 * drop_scale(p), torch.zeros_like(x2))
    got = out.double()
    assert torch.equal(got[torch.from_numpy(~k2).cuda()], torch.zeros(int((~k2).sum()), dtype=torch.float64, device="cuda"))
    # kept: bf16 output rounding (2^-9 relative) plus the fp32 accumulation of N products of bf16 operands (~1e-6 of the
    # row's sum of |mid| |W2|); a kept value is never 0 unless its pre-dropout value is
    tol = 2.0 ** -8 * ref.abs() + 1e-5 * (mid.double().abs() @ W2.double().abs().T)
    assert bool(((got - ref).abs() <= tol).all()), float(((got - ref).abs() - tol).max())


@pytest.mark.gpu
@pytest.mark.parametrize("mode,D,F", [(0, 64, 0), (1, 64, 16), (2, 64, 0), (1, 45, 5)])
@pytest.mark.parametrize("seed,stream,step,p", CASES[1:3])
def test_embed_dropout_mask_is_exact(mode, D, F, seed, stream, step, p):
    """embed_ln_fwd (SASRec emb_dropout on the dense layout): element index t * H + col, after the positional add, with
    the vector kernel (D multiple of 8) and the generic one (the reference's 45 + 5).  The fp32 x0 equals the p = 0 x0 of
    the same launch through the host mask, bit for bit; its bf16 copy is that value rounded."""
    from srfrd_b200 import ops
    B, L, N = 67, 50, 500
    H = D + (F if mode == 1 else 0)
    g = torch.Generator().manual_seed(mode * 10 + D)
    E, P = torch.randn(N + 1, D, generator=g).cuda(), torch.randn(L, D, generator=g).cuda()
    seq = torch.randint(0, N + 1, (B, L), generator=g)
    seq[:, :20] = 0
    seq = seq.cuda()
    aux, aux_ids = None, None
    if mode == 1:
        aux, aux_ids = torch.randn(3, F, generator=g).cuda(), torch.randint(0, 3, (B, L), generator=g).cuda()
    if mode == 2:
        aux, aux_ids = torch.randn(5, D, generator=g).cuda(), torch.randint(0, 5, (B,), generator=g).cuda()
    scale = D ** 0.5 if mode == 0 else 1.0
    x_ref = torch.empty(B * L, H, device="cuda")
    ops.embed_ln_fwd(E, P, aux, mode, seq, aux_ids, scale, None, None, 1e-8, x0_f32=x_ref)
    x32 = torch.full((B * L, H), float("nan"), device="cuda")
    Hp = (H + 7) // 8 * 8                          # bf16 rows are padded to whole 16-byte chunks (45 + 5 -> 56 columns)
    xb = torch.full((B * L, Hp), float("nan"), dtype=bf16, device="cuda")
    ops.embed_ln_fwd(E, P, aux, mode, seq, aux_ids, scale, None, None, 1e-8, x0_bf16=xb, x0_f32=x32, drop_p=p, drop_seed=seed,
                     drop_stream=stream, drop_step=_step(step))
    want = masked(x_ref, keep_mask(seed, stream, np.arange(B * L * H).reshape(B * L, H), p, step), p)
    assert torch.equal(x32, want)
    assert torch.equal(xb[:, :H], want.to(bf16))
    assert Hp == H or float(xb[:, H:].float().abs().max()) == 0.0            # padding columns written as 0
