// Causal self-attention on tcgen05 for maxlen <= 128 (SURVEY.md 2.3 row k2; SRFR_model.py:112).
//
// A tile is a window of 128 consecutive tokens that holds spt = floor(128 / L) whole sequences, so the
// queries AND the keys/values of those sequences live in the same window:
//     S[128 x 128] = Q K^T   (tcgen05, fp32 in TMEM)   -> per-row causal/same-sequence softmax in registers
//     O[128 x hd ] = P V     (P written to smem as a bf16 K-major operand, V read MN-major from its TMA tile)
// One thread owns one query row (TMEM lane), so max / sum / delta need no cross-thread reduction, and the
// (L x L) probabilities never touch HBM.  Backward recomputes S and P and runs five MMAs per tile:
//     S = Q K^T, dP = dO V^T, dQ = dS K, dK = dS^T Q, dV = P^T dO
// where the SAME 128-byte-swizzled [128 tokens x 64 features] TMA tile serves as a K-major operand (rows = M/N)
// and as an MN-major operand (rows = K) -- only the descriptor changes.
// Warp roles (192 threads): warp 0 TMA producer, warp 1 MMA issuer, warps 2..5 softmax + epilogue.
#include <stdlib.h>

#include "common.cuh"
#include "srfrd_b200.h"

namespace srfrd {

int attn_fwd_simt(const void* q, int ldq, const void* k, const void* v, int ldkv, void* o, int ldo, int64_t B, int L,
                  int H, int heads, float drop_p, uint64_t seed, uint32_t stream_id, const float* drop_step, void* stream);
int attn_bwd_simt(const void* dout, int lddo, const void* q, int ldq, const void* k, const void* v, int ldkv, void* dq,
                  int lddq, void* dk, void* dv, int lddkv, int64_t B, int L, int H, int heads, float drop_p,
                  uint64_t seed, uint32_t stream_id, const float* drop_step, void* stream);

bool attn_long_supported(int64_t B, int L, int H, int heads, int ldq, int ldkv);
int attn_long_fwd(const void* q, int ldq, const void* k, const void* v, int ldkv, void* o, int ldo, float* stats, int64_t B,
                  int L, int H, int heads, float drop_p, uint64_t seed, uint32_t stream_id, const float* drop_step,
                  void* stream);
int attn_long_bwd(const void* dout, int lddo, const void* q, int ldq, const void* k, const void* v, int ldkv, const void* o,
                  int ldo, float* stats, void* dq, int lddq, void* dk, void* dv, int lddkv, int64_t B, int L, int H, int heads,
                  float drop_p, uint64_t seed, uint32_t stream_id, const float* drop_step, void* stream);

static constexpr int TILE = 128;
static constexpr int OPB = TILE * 64 * 2;     // operand block: 128 rows x 64 bf16 = 16 KB
static constexpr int ATC_THREADS = 192;

struct AttnTc {
  int64_t T;
  int L, hd, heads, spt, n_tiles, kblocks;
  int tma_o;                              // forward output leaves through TMA stores (heads == 1 or hd % 64 == 0)
  int debug;
  float scale, scale_log2e;
  bf16* o; int ldo;                       // forward output
  bf16 *dq, *dk, *dv; int lddq, lddkv;    // backward outputs
  uint64_t drop_seed; uint32_t drop_thresh, drop_stream; float drop_scale; const float* drop_step;
  // packed token layout (pack.cu): tiles start at pk_tile_row0[tile] and hold whole variable-length sequences; per row
  // pk_info = {first row of its sequence, one past its last row, float bits of the pad column's weight, position}
  const int* pk_rows;                     // device {M, T', n_tiles}
  const int4* pk_info;
  const int* pk_tile_row0;
  // fused out-projection (packed layout, heads == 1; SRFR_model.py:112-113, the out_proj of F.multi_head_attention_forward
  // and the residual + forward LayerNorm that follow it):
  //   forward : r = o Wo^T + bo + res,  y = LayerNorm(r) * ln_w + ln_b,  ln_stats = (mean, rstd)   (o is still written)
  //   backward: dO = dr Wo, computed in the kernel instead of read from memory
  const float *op_bias, *ln_w, *ln_b; float* ln_stats; float ln_eps;
  bf16 *op_r, *op_y; int ldr, ldy;
};

// byte offset of element (row r, column c) inside a [128 x 64] bf16 block with the 128-byte swizzle
__device__ __forceinline__ uint32_t sw128(int r, int c) {
  return (uint32_t)(r * 128 + ((((c >> 3) ^ (r & 7)) << 4) | ((c & 7) << 1)));
}

struct RowInfo {
  int r; int64_t t; bool owned; int jlo, jhi, l; int64_t bh;
  float pm;        // packed layout: weight of the key column at the window start (the pad representative stands for
                   // `pm` dropped pad slots); 1 otherwise
  int jbase;       // packed layout: un-shifted window start (dropout hash index)
};
// Packed layout.  Row r of the tile that starts at packed row `row0`: the row is owned when its whole sequence lies inside
// the tile (tiles start at sequence boundaries; a trailing partial sequence belongs to the next tile).  Keys: the rows of
// the same sequence up to the row itself; the first of them is the pad representative, weighted by the number of
// dropped pad slots before this row's position -- with weight 0 the window simply starts one column later.
__device__ __forceinline__ RowInfo row_info_pk(const AttnTc& p, int row0, int M, int h, int quarter, int lane) {
  RowInfo ri;
  ri.r = quarter * 32 + lane;
  ri.t = (int64_t)row0 + ri.r;
  int4 inf = make_int4(0, 0, 0, 0);
  const bool in = ri.t < M;
  if (in) inf = __ldg(p.pk_info + ri.t);
  ri.owned = in && inf.x >= row0 && inf.y <= row0 + TILE;
  const float mult = __int_as_float(inf.z);
  ri.jbase = inf.x - row0;
  ri.jlo = ri.jbase + (mult == 0.f ? 1 : 0);
  ri.jhi = ri.r;
  ri.pm = mult == 0.f ? 1.f : mult;
  ri.l = 0;
  ri.bh = ri.t * p.heads + h;
  return ri;
}
__device__ __forceinline__ RowInfo row_info(const AttnTc& p, int tile, int h, int quarter, int lane) {
  RowInfo ri;
  ri.r = quarter * 32 + lane;
  ri.t = (int64_t)tile * p.spt * p.L + ri.r;
  ri.owned = ri.r < p.spt * p.L && ri.t < p.T;
  const int sidx = ri.r / p.L;
  ri.l = ri.r - sidx * p.L;
  ri.jlo = sidx * p.L;
  ri.jhi = ri.jlo + ri.l;
  ri.bh = (ri.t / p.L) * p.heads + h;
  ri.pm = 1.f;
  ri.jbase = ri.jlo;
  return ri;
}
__device__ __forceinline__ float drop_f(const AttnTc& p, const RowInfo& ri, int col) {
  if (!p.drop_thresh) return 1.f;
  const uint64_t idx = p.pk_info ? (uint64_t)ri.bh * 256u + (uint64_t)(col - ri.jbase)
                                 : ((uint64_t)ri.bh * p.L + ri.l) * p.L + (col - ri.jlo);
  return dropout_keep(p.drop_seed, p.drop_stream, idx, p.drop_thresh) ? p.drop_scale : 0.f;
}

// row max and sum of exp over the causal window of this thread's row (two passes over the S accumulator)
__device__ __forceinline__ void row_softmax_stats(uint32_t tS, const AttnTc& p, const RowInfo& ri, float& m, float& sum) {
  m = -INFINITY;
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t raw[32];
    tmem_ld32(tS + c * 32, raw);
    tmem_ld_wait();
    const int lo = ri.jlo - c * 32;
    const unsigned span = (unsigned)(ri.jhi - ri.jlo);
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if ((unsigned)(j - lo) <= span) m = fmaxf(m, __uint_as_float(raw[j]));
  }
  sum = 0.f;
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t raw[32];
    tmem_ld32(tS + c * 32, raw);
    tmem_ld_wait();
    const int lo = ri.jlo - c * 32;
    const unsigned span = (unsigned)(ri.jhi - ri.jlo);
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if ((unsigned)(j - lo) <= span) sum += exp2f((__uint_as_float(raw[j]) - m) * p.scale_log2e);
  }
}

__device__ __forceinline__ void store_row32(uint8_t* blk_base, int r, int c, const float* v) {
  // 32 consecutive keys [c*32, c*32+32) of row r -> 4 x 16 B into the swizzled K-major block pair
  uint8_t* blk = blk_base + (c >> 1) * OPB;
  const int col0 = (c & 1) * 32;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const uint4 w = make_uint4(pack_bf16x2(v[8 * u], v[8 * u + 1]), pack_bf16x2(v[8 * u + 2], v[8 * u + 3]),
                               pack_bf16x2(v[8 * u + 4], v[8 * u + 5]), pack_bf16x2(v[8 * u + 6], v[8 * u + 7]));
    *reinterpret_cast<uint4*>(blk + sw128(r, col0 + 8 * u)) = w;
  }
}

__device__ __forceinline__ void store_out_row(bf16* dst, uint32_t tacc, int hd, float mul) {
  for (int c = 0; c < hd; c += 16) {
    uint32_t raw[16];
    tmem_ld16(tacc + c, raw);
    tmem_ld_wait();
    if (dst) {
      uint4* o = reinterpret_cast<uint4*>(dst + c);
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(raw[j]) * mul;
      o[0] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      o[1] = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]),
                        pack_bf16x2(v[14], v[15]));
    }
  }
}

// =============================================================================================== forward
// profiling experiments only (SRFRD_ATTN_DEBUG=5): clock64 timeline of CTA 0, [event][item]
__device__ long long g_attn_dbg[16 * 16];
#define AT_STAMP(ev, n) do { if (p.debug == 5 && blockIdx.x == 0 && (n) < 16) { if (elect_one()) g_attn_dbg[(ev) * 16 + (n)] = clock64(); } } while (0)

__device__ __forceinline__ void named_bar_sync_a(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void tma_store_2d_a(const CUtensorMap* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tmap),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_wait_read_all() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Packed layout: a tile owns a data-dependent number of rows, so its results leave through coalesced 16-byte stores of the
// owned rows (all 256 epilogue threads) instead of a TMA store with a fixed box.
__device__ __forceinline__ void store_staged_rows(bf16* dst, int ld, int64_t row0, int col0, const uint8_t* blocks, int hd,
                                                  int n_own, int tid256) {
  const int cpr = hd >> 3;                                   // 16-byte chunks per row
  for (int i = tid256; i < n_own * cpr; i += 256) {
    const int r = i / cpr, ch = i - r * cpr;
    const uint4 v = *reinterpret_cast<const uint4*>(blocks + (ch >> 3) * OPB + sw128(r, (ch & 7) * 8));
    *reinterpret_cast<uint4*>(dst + (row0 + r) * ld + col0 + ch * 8) = v;
  }
}

static constexpr int AF_THREADS = 320;   // forward: 8 softmax / epilogue warps + TMA warp + MMA warp

// Forward out-projection epilogue of one tile (OP), run by the 256 epilogue threads: thread (row r, part) takes the
// 32-column chunks c = 32 part, 32 part + 64, ... of its row, as gemm_tn's LNF epilogue does (half = part), so the
// partial row sums and their combination are the same.  On entry every thread has stored its share of o from Qs.
__device__ __forceinline__ void out_proj_epilogue(const AttnTc& p, uint8_t* Qs, uint8_t* Vs, float* xsum, float* xsq,
                                               const float* sop, uint32_t tacc, uint64_t* proj_full, uint64_t* w_full,
                                               uint32_t ph, int r, int part, int quarter, int row0, int n_own) {
  mbar_wait2(proj_full, ph, w_full, ph);   // r accumulator complete, residual tile landed
  tc_fence_after();
  float ln_sum = 0.f, ln_sq = 0.f;
#pragma unroll 1
  for (int c = part * 32; c < p.hd; c += 64) {
    uint32_t raw[32];
    tmem_ld32(tacc + c, raw);
    uint8_t* blk = Vs + (c >> 6) * OPB;
    uint4 ax[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (c + 8 * j < p.hd) ax[j] = *reinterpret_cast<const uint4*>(blk + sw128(r, (c & 63) + 8 * j));
    tmem_ld_wait();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (c + 8 * j >= p.hd) break;
      float v[8], a[8];
      unpack_bf16x8(ax[j], a);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = (__uint_as_float(raw[8 * j + i]) + sop[c + 8 * j + i]) + a[i];
      const uint4 pk = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
      *reinterpret_cast<uint4*>(blk + sw128(r, (c & 63) + 8 * j)) = pk;   // r in place over the residual
      lnf_accum8(pk, ln_sum, ln_sq);
    }
  }
  tc_fence_before();
  xsum[part * TILE + r] = ln_sum;          // (the softmax's exchange arrays: every thread has read them)
  xsq[part * TILE + r] = ln_sq;
  named_bar_sync_a(9, 256);                // partner's partial sums visible; every thread has read o out of Qs
  float mean, rstd, nb;
  lnf_stats(ln_sum, ln_sq, xsum[(part ^ 1) * TILE + r], xsq[(part ^ 1) * TILE + r], p.hd, p.ln_eps, mean, rstd, nb);
#pragma unroll 1
  for (int c = part * 32; c < p.hd; c += 64) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (c + 8 * j >= p.hd) break;
      const uint32_t off = (c >> 6) * OPB + sw128(r, (c & 63) + 8 * j);
      *reinterpret_cast<uint4*>(Qs + off) =
          lnf_apply8(*reinterpret_cast<const uint4*>(Vs + off), rstd, nb, sop + TILE + c + 8 * j, sop + 2 * TILE + c + 8 * j);
    }
  }
  if (part == 0 && r < n_own && p.ln_stats) *reinterpret_cast<float2*>(p.ln_stats + 2 * (size_t)(row0 + r)) = make_float2(mean, rstd);
  named_bar_sync_a(9, 256);                // r and y complete in Vs / Qs
  store_staged_rows(p.op_r, p.ldr, row0, 0, Vs, p.hd, n_own, threadIdx.x);
  store_staged_rows(p.op_y, p.ldy, row0, 0, Qs, p.hd, n_own, threadIdx.x);
}

// Forward, two CTAs per SM (smem <= 98 KB, 256 TMEM columns each): a tile is a chain of TMA -> S MMA -> softmax ->
// PV MMA -> output latencies, so a second resident CTA fills the gaps.  Shared memory is reused in place: P overwrites
// K (dead once S is complete), O overwrites Q and leaves through a TMA store whose box has exactly spt*L rows.
// Softmax: the rows of TMEM lane quarter q need the key chunks (32 columns) c_lo(q)..q only (causal, same sequence);
// the two warps of a quarter split them (chunk parity), keep them in registers (one TMEM round trip), exchange
// partial row maxima / sums through shared memory, and split the O epilogue by column chunk the same way.
// Measured (clock64 timeline): with one thread per row and three TMEM passes the softmax alone was 10 k cycles of a
// 17 k-cycle tile -- single-warp instruction latency, not bandwidth.
// Warp roles (320 threads): warps 0..7 softmax + epilogue (quarter = warp & 3, part = warp >> 2), warp 8 TMA,
// warp 9 MMA (control warps have the highest ids: the scheduler favours them).
// Fused out-projection (OP, packed layout, heads == 1): once the PV MMA has released K's and V's blocks (kv_free), the TMA
// warp loads Wo (B operand, hd rows x K = hd) into K's blocks and the residual tile into V's; the MMA warp multiplies the
// staged O (Q's blocks, already the K-major A operand) by Wo^T into S's TMEM columns (dead since the softmax); the epilogue
// adds bias and residual, writes r in place over the residual, normalises it into Q's blocks (y) and stores o, r, y and
// the statistics of the tile's owned rows.  Same K order (64 + 16 at hd = 80), add order and LayerNorm arithmetic as
// gemm_tn's LNF epilogue, so the results are bit-identical to the separate launch.  A tile is then done only when its
// y has left: q_free alone gates the next item's loads.
template <bool DROP, bool PK, bool OP>
__global__ void __launch_bounds__(AF_THREADS, 2)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmO,
                   const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmR, AttnTc p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int opbytes = p.kblocks * OPB;
  uint8_t* Qs = smem;                              // Q, later O (bf16, swizzled, stored by TMA)
  uint8_t* Ks = Qs + opbytes;                      // K, later P (2 key blocks)
  uint8_t* Vs = Ks + max(p.kblocks, 2) * OPB;
  float* smax = reinterpret_cast<float*>(Vs + opbytes);   // [2 parts][128 rows] partial row maxima
  float* ssum = smax + 2 * TILE;                          // [2 parts][128 rows] partial row sums
  uint64_t* bars = reinterpret_cast<uint64_t*>(ssum + 2 * TILE);
  uint64_t *qk_full = bars, *v_full = bars + 1, *s_full = bars + 2, *p_full = bars + 3, *o_full = bars + 4,
           *kv_free = bars + 5, *q_free = bars + 6;
  uint64_t *w_full = bars + 7, *o_staged = bars + 8, *proj_full = bars + 9;   // OP: Wo + residual landed, O staged, r ready
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10);
  float* sop = reinterpret_cast<float*>(bars + 16);        // OP: bias, LayerNorm weight, LayerNorm bias [3][TILE]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmO);
    if (OP) { tma_prefetch_desc(&tmW); tma_prefetch_desc(&tmR); }
    mbar_init(qk_full, 1); mbar_init(v_full, 1); mbar_init(s_full, 1); mbar_init(p_full, 8); mbar_init(o_full, 1);
    mbar_init(kv_free, 1); mbar_init(q_free, 1);
    mbar_init(w_full, 1); mbar_init(o_staged, 1); mbar_init(proj_full, 1);
    fence_barrier_init();
  }
  if (warp == 9) { tmem_alloc(tmem_slot, 256); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tS = tmem_base, tO = tmem_base + 128;
  pdl_prologue_done();
  if (DROP) p.drop_seed = mix_seed(p.drop_seed, p.drop_step);
  const int pk_M = PK ? __ldg(p.pk_rows) : 0;
  const int n_items = (PK ? __ldg(p.pk_rows + 2) : p.n_tiles) * p.heads;

  if (warp == 8) {
    uint32_t ph = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ph ^= 1) {
      const int tile = it / p.heads, h = it % p.heads;
      const int row0 = PK ? __ldg(p.pk_tile_row0 + tile) : tile * p.spt * p.L, col0 = h * p.hd;
      mbar_wait(q_free, ph ^ 1);                   // O of the previous item has left Q's smem
      if (!OP) mbar_wait(kv_free, ph ^ 1);         // previous PV MMA is done with P (K's smem) and V (OP: implied)
      AT_STAMP(0, it / gridDim.x);
      if (elect_one()) {
        mbar_expect_tx(qk_full, 2 * opbytes);
        for (int kb = 0; kb < p.kblocks; ++kb) {
          tma_load_2d(Qs + kb * OPB, &tmQ, qk_full, col0 + kb * 64, row0, SRFRD_EVICT_FIRST);
          tma_load_2d(Ks + kb * OPB, &tmK, qk_full, col0 + kb * 64, row0, SRFRD_EVICT_FIRST);
        }
        mbar_expect_tx(v_full, opbytes);
        for (int kb = 0; kb < p.kblocks; ++kb)
          tma_load_2d(Vs + kb * OPB, &tmV, v_full, col0 + kb * 64, row0, SRFRD_EVICT_FIRST);
        // (no L2 prefetch of the next item here: two CTAs per SM already overlap one item's loads with the other's
        //  compute, and the extra live values spill at the 96-register cap that two CTAs per SM impose)
      }
      __syncwarp();
      if (OP) {
        mbar_wait(kv_free, ph);                    // this item's PV MMA is done with K's and V's blocks
        if (elect_one()) {
          mbar_expect_tx(w_full, p.kblocks * (p.hd * 128 + OPB));
          for (int kb = 0; kb < p.kblocks; ++kb) {
            tma_load_2d(Ks + kb * OPB, &tmW, w_full, kb * 64, 0, SRFRD_EVICT_LAST);
            tma_load_2d(Vs + kb * OPB, &tmR, w_full, kb * 64, row0, SRFRD_EVICT_FIRST);
          }
        }
        __syncwarp();
      }
    }
  } else if (warp == 9) {
    const uint32_t idS = umma_idesc_bf16(TILE, TILE, 0, 0);
    const uint32_t idO = umma_idesc_bf16(TILE, p.hd, 0, 1);
    const uint32_t idW = umma_idesc_bf16(TILE, p.hd, 0, 0);       // OP: O Wo^T, both operands K-major
    const uint64_t dQ = umma_smem_desc(smem_u32(Qs), 0, 1024), dK = umma_smem_desc(smem_u32(Ks), 0, 1024);
    const uint64_t dP = umma_smem_desc(smem_u32(Ks), 0, 1024), dV = umma_smem_desc(smem_u32(Vs), OPB, 1024);
    uint32_t ph = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ph ^= 1) {
      mbar_wait(qk_full, ph);
      tc_fence_after();
      AT_STAMP(1, it / gridDim.x);
      if (elect_one()) {
        for (int kb = 0; kb < p.kblocks; ++kb) {
          const int ksteps = min(4, (p.hd - kb * 64) / 16);
          for (int k = 0; k < ksteps; ++k)
            umma_bf16(tS, dQ + (uint64_t)(kb * (OPB >> 4) + 2 * k), dK + (uint64_t)(kb * (OPB >> 4) + 2 * k), idS, (kb | k) != 0);
        }
        umma_commit(s_full);
      }
      __syncwarp();
      AT_STAMP(2, it / gridDim.x);
      mbar_wait(p_full, ph);
      mbar_wait(v_full, ph);
      tc_fence_after();
      AT_STAMP(3, it / gridDim.x);
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)     // K = 128 keys; V tile read MN-major (rows = K): 16 rows = 2048 B
          umma_bf16(tO, dP + (uint64_t)((ks >> 2) * (OPB >> 4) + (ks & 3) * 2), dV + (uint64_t)(ks * 128), idO, ks != 0);
        umma_commit(kv_free);
        umma_commit(o_full);
      }
      __syncwarp();
      AT_STAMP(4, it / gridDim.x);
      if (OP) {                              // r = O Wo^T into S's columns: A = staged O (Q's blocks), B = Wo (K's blocks)
        mbar_wait2(o_staged, ph, w_full, ph);
        tc_fence_after();
        if (elect_one()) {
          for (int kb = 0; kb < p.kblocks; ++kb) {
            const int ksteps = min(4, (p.hd - kb * 64) / 16);
            for (int k = 0; k < ksteps; ++k)
              umma_bf16(tS, dQ + (uint64_t)(kb * (OPB >> 4) + 2 * k), dK + (uint64_t)(kb * (OPB >> 4) + 2 * k), idW, (kb | k) != 0);
          }
          umma_commit(proj_full);
        }
        __syncwarp();
      }
    }
  } else {
    const int quarter = warp & 3, part = warp >> 2;
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    // key chunks (32 columns) that any row of this quarter needs: from the first row's window start to the quarter's
    // own diagonal chunk (causal: row r needs columns jlo..r); this warp takes c_lo + part, c_lo + part + 2
    const int r_first = quarter * 32;
    // packed layout: a sequence has at most L + 1 rows, so a row's window starts at most L columns before it
    const int c_lo = PK ? (max(0, r_first - p.L) >> 5) : min(((r_first / p.L) * p.L) >> 5, quarter), c_hi = quarter;
    if (OP)                                // read by the epilogue only after several barriers of these 256 threads
      for (int i = threadIdx.x; i < TILE; i += 256) {
        sop[i] = (p.op_bias && i < p.hd) ? __ldg(p.op_bias + i) : 0.f;
        sop[TILE + i] = i < p.hd ? __ldg(p.ln_w + i) : 0.f;
        sop[2 * TILE + i] = i < p.hd ? __ldg(p.ln_b + i) : 0.f;
      }
    uint32_t ph = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ph ^= 1) {
      const int tile = it / p.heads, h = it % p.heads;
      const int pk_row0 = PK ? __ldg(p.pk_tile_row0 + tile) : 0;
      RowInfo ri = PK ? row_info_pk(p, pk_row0, pk_M, h, quarter, lane) : row_info(p, tile, h, quarter, lane);
      if (!ri.owned) { ri.jlo = 1 << 20; ri.jhi = ri.jlo; }         // empty window; TMEM loads stay warp-collective
      const unsigned span = (unsigned)(ri.jhi - ri.jlo);
      mbar_wait(s_full, ph);
      tc_fence_after();
      if (warp == 0) AT_STAMP(5, it / gridDim.x);
      // chunk indices of this warp; an index past the window re-reads the last chunk with an empty mask so the
      // TMEM loads stay unconditional
      const int c0 = c_lo + part, c1 = c_lo + part + 2;
      const int lo0 = (c0 <= c_hi) ? ri.jlo - c0 * 32 : (1 << 20);
      const int lo1 = (c1 <= c_hi) ? ri.jlo - c1 * 32 : (1 << 20);
      uint32_t raw0[32], raw1[32];
      tmem_ld32(tS + lane_off + min(c0, c_hi) * 32, raw0);
      tmem_ld32(tS + lane_off + min(c1, c_hi) * 32, raw1);
      tmem_ld_wait();
      float m = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        m = ((unsigned)(j - lo0) <= span) ? fmaxf(m, __uint_as_float(raw0[j])) : m;
        m = ((unsigned)(j - lo1) <= span) ? fmaxf(m, __uint_as_float(raw1[j])) : m;
      }
      smax[part * TILE + ri.r] = m;
      named_bar_sync_a(1 + quarter, 64);           // the two warps of this quarter
      m = fmaxf(m, smax[(part ^ 1) * TILE + ri.r]);
      const float mb = m * p.scale_log2e;
      float sum = 0.f;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int c = u ? c1 : c0;
        const uint32_t (&raw)[32] = u ? raw1 : raw0;
        if (c <= c_hi) {
          const int lo = u ? lo1 : lo0;
          uint8_t* blk = Ks + (c >> 1) * OPB;
          const int col0 = (c & 1) * 32;
#pragma unroll
          for (int g = 0; g < 4; ++g) {            // 8 keys -> one 16-byte chunk of the swizzled K-major P block
            float e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int j = 8 * g + i;
              float x = ex2_approx(fmaf(__uint_as_float(raw[j]), p.scale_log2e, -mb));   // un-normalised; O is scaled by 1/sum
              x = ((unsigned)(j - lo) <= span) ? x : 0.f;
              if (PK) x = (j == lo) ? x * ri.pm : x;       // the pad representative's column counts pm times
              sum += x;
              if (DROP) x *= drop_f(p, ri, c * 32 + j);
              e[i] = x;
            }
            *reinterpret_cast<uint4*>(blk + sw128(ri.r, col0 + 8 * g)) =
                make_uint4(pack_bf16x2(e[0], e[1]), pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
          }
        }
      }
      ssum[part * TILE + ri.r] = sum;
      for (int c = part; c < 4; c += 2)            // key chunks outside the quarter's window: P = 0 (chunk parity = part)
        if (c < c_lo || c > c_hi) {
          uint8_t* blk = Ks + (c >> 1) * OPB;
#pragma unroll
          for (int g = 0; g < 4; ++g)
            *reinterpret_cast<uint4*>(blk + sw128(ri.r, (c & 1) * 32 + 8 * g)) = make_uint4(0u, 0u, 0u, 0u);
        }
      tc_fence_before();
      fence_proxy_async();                 // generic-proxy smem writes -> visible to the MMA (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
      if (warp == 0) AT_STAMP(6, it / gridDim.x);
      mbar_wait(o_full, ph);
      tc_fence_after();
      if (warp == 0) AT_STAMP(7, it / gridDim.x);
      named_bar_sync_a(1 + quarter, 64);           // partner's partial sum is visible
      const float tot = ssum[ri.r] + ssum[TILE + ri.r];
      const float inv = ri.owned ? 1.f / tot : 0.f;
      if (!p.tma_o) {                      // head slices narrower than a 64-column store box: direct row stores
        if (part == 0) store_out_row(ri.owned ? p.o + ri.t * p.ldo + h * p.hd : nullptr, tO + lane_off, p.hd, inv);
        tc_fence_before();
        named_bar_sync_a(9, 256);
        if (warp == 0 && lane == 0) mbar_arrive(q_free);
        __syncwarp();
        continue;
      }
      // O = (P V) / sum -> bf16 into Q's smem blocks (same 128-byte swizzle the TMA store expects); 32-column chunks
      // alternate between the two warps of the quarter
#pragma unroll 1
      for (int c = part * 32; c < p.hd; c += 64) {
        uint32_t ro[32];
        tmem_ld32(tO + lane_off + c, ro);
        tmem_ld_wait();
        uint8_t* blk = Qs + (c >> 6) * OPB;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (c + 8 * u >= p.hd) break;
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(ro[8 * u + j]) * inv;
          *reinterpret_cast<uint4*>(blk + sw128(ri.r, (c & 63) + 8 * u)) =
              make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
        }
      }
      tc_fence_before();
      fence_proxy_async();
      named_bar_sync_a(9, 256);
      if (warp == 0) AT_STAMP(8, it / gridDim.x);
      if (PK) {
        if (OP && warp == 0 && lane == 0) mbar_arrive(o_staged);   // the out-projection MMA may read O
        const int n_own = __ldg(p.pk_tile_row0 + tile + 1) - pk_row0;
        store_staged_rows(p.o, p.ldo, pk_row0, h * p.hd, Qs, p.hd, n_own, threadIdx.x);
        if (OP) out_proj_epilogue(p, Qs, Vs, smax, ssum, sop, tS + lane_off, proj_full, w_full, ph, ri.r, part, quarter,
                                  pk_row0, n_own);
        named_bar_sync_a(9, 256);                  // every thread has read its chunks: Q's smem may be refilled
        if (warp == 0 && lane == 0) mbar_arrive(q_free);
      } else if (warp == 0 && lane == 0) {
        const int row0 = tile * p.spt * p.L, col0 = h * p.hd;
        for (int kb = 0; kb < p.kblocks; ++kb) tma_store_2d_a(&tmO, Qs + kb * OPB, col0 + kb * 64, row0);
        bulk_commit_wait_read_all();
        mbar_arrive(q_free);
      }
      __syncwarp();
      if (warp == 0) AT_STAMP(9, it / gridDim.x);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) { tc_fence_after(); tmem_dealloc(tmem_base, 256); }
}

// =============================================================================================== backward
// One CTA per SM (S, dP, dQ need 256 + hd TMEM columns; Q, K, V, dO, P, dS fill shared memory).  Same structure as
// the forward: 8 softmax warps split the key chunks of a lane quarter, keep their S and dP chunks in registers (one
// TMEM round trip), and exchange row max, row sum and delta = sum_j P_ij dP_ij through shared memory.  dQ / dK / dV
// leave through TMA stores from the (dead) dO / K / Q operand blocks.
// Warp roles (320 threads): warps 0..7 softmax + epilogue (quarter = warp & 3, part = warp >> 2), warp 8 TMA, warp 9 MMA.
// Fused out-projection (OP, packed layout, heads == 1): tmDO maps dr instead of dO.  The dr tile lands in P's blocks (dead
// until the softmax backward), Wo^T (B operand, hd rows x K = hd) is loaded once into its own blocks, and the MMA warp
// computes dO = dr Wo into TMEM columns [384, 384 + hd) before S; the epilogue warps write it as bf16 into dO's blocks
// (the layout a TMA load would have left) and the dP MMA follows.  Same K order and rounding as gemm_tn without bias.
template <bool DROP, bool PK, bool OP>
__global__ void __launch_bounds__(AF_THREADS, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                   const __grid_constant__ CUtensorMap tmV, const __grid_constant__ CUtensorMap tmDO,
                   const __grid_constant__ CUtensorMap tmDQ, const __grid_constant__ CUtensorMap tmDK,
                   const __grid_constant__ CUtensorMap tmDV, const __grid_constant__ CUtensorMap tmWT, AttnTc p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int opbytes = p.kblocks * OPB;
  uint8_t* Qs = smem;                            // Q, later dV staging
  uint8_t* Ks = Qs + opbytes;                    // K, later dK staging
  uint8_t* Vs = Ks + opbytes;
  uint8_t* Ds = Vs + opbytes;                    // dO, later dQ staging
  uint8_t* Ps = Ds + opbytes;                    // P * dropout mask, 2 key blocks
  uint8_t* Gs = Ps + 2 * OPB;                    // dS, 2 key blocks
  float* xch = reinterpret_cast<float*>(Gs + 2 * OPB);   // [3 values][2 parts][128 rows]: max, sum, delta numerator
  uint64_t* bars = reinterpret_cast<uint64_t*>(xch + 6 * TILE);
  uint64_t *in_full = bars, *in_free = bars + 1, *sdp_full = bars + 2, *ds_full = bars + 3, *out_full = bars + 4;
  uint64_t *w_full = bars + 5, *do_full = bars + 6, *do_staged = bars + 7;    // OP: Wo^T landed, dr Wo done, dO staged
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8);
  uint8_t* Ws = smem + (4 * p.kblocks + 4) * OPB + 4096;  // OP: Wo^T, kblocks x [hd x 64] (after xch and the barriers)
  const int wblk = p.hd * 128;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV); tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmDQ); tma_prefetch_desc(&tmDK); tma_prefetch_desc(&tmDV);
    if (OP) tma_prefetch_desc(&tmWT);
    mbar_init(in_full, 1); mbar_init(in_free, 1); mbar_init(sdp_full, 1); mbar_init(ds_full, 8); mbar_init(out_full, 1);
    mbar_init(w_full, 1); mbar_init(do_full, 1); mbar_init(do_staged, 8);
    fence_barrier_init();
  }
  if (warp == 9) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();
  if (DROP) p.drop_seed = mix_seed(p.drop_seed, p.drop_step);
  const int pk_M = PK ? __ldg(p.pk_rows) : 0;
  const int n_items = (PK ? __ldg(p.pk_rows + 2) : p.n_tiles) * p.heads;
  // S and dP live in columns [0,128) and [128,256); once the softmax backward has consumed them the same
  // columns receive dK and dV, and dQ goes to [256, 256+hd).
  const uint32_t tS = tmem_base, tDP = tmem_base + 128, tDK = tmem_base, tDV = tmem_base + 128, tDQ = tmem_base + 256;
  const uint32_t tDO = tmem_base + 384;    // OP: dO = dr Wo (hd <= 128 columns)

  if (warp == 8) {
    if (OP) {
      if (elect_one()) {
        mbar_expect_tx(w_full, p.kblocks * wblk);
        for (int kb = 0; kb < p.kblocks; ++kb) tma_load_2d(Ws + kb * wblk, &tmWT, w_full, kb * 64, 0, SRFRD_EVICT_LAST);
      }
      __syncwarp();
    }
    uint32_t ph = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ph ^= 1) {
      const int tile = it / p.heads, h = it % p.heads;
      const int row0 = PK ? __ldg(p.pk_tile_row0 + tile) : tile * p.spt * p.L, col0 = h * p.hd;
      mbar_wait(in_free, ph ^ 1);            // previous item's outputs have left the operand blocks
      if (elect_one()) {
        mbar_expect_tx(in_full, 4 * opbytes);
        for (int kb = 0; kb < p.kblocks; ++kb) {
          tma_load_2d(Qs + kb * OPB, &tmQ, in_full, col0 + kb * 64, row0, SRFRD_EVICT_FIRST);
          tma_load_2d(Ks + kb * OPB, &tmK, in_full, col0 + kb * 64, row0, SRFRD_EVICT_FIRST);
          tma_load_2d(Vs + kb * OPB, &tmV, in_full, col0 + kb * 64, row0, SRFRD_EVICT_FIRST);
          tma_load_2d((OP ? Ps : Ds) + kb * OPB, &tmDO, in_full, col0 + kb * 64, row0, SRFRD_EVICT_FIRST);   // OP: dr
        }
        if (!(p.debug & 256) && it + (int)gridDim.x < n_items) {        // next item's operands: HBM -> L2 while this one computes
          const int itn = it + gridDim.x;
          const int rown = PK ? __ldg(p.pk_tile_row0 + itn / p.heads) : (itn / p.heads) * p.spt * p.L, coln = (itn % p.heads) * p.hd;
          for (int kb = 0; kb < p.kblocks; ++kb) {
            tma_prefetch_l2_2d(&tmQ, coln + kb * 64, rown);
            tma_prefetch_l2_2d(&tmK, coln + kb * 64, rown);
            tma_prefetch_l2_2d(&tmV, coln + kb * 64, rown);
            tma_prefetch_l2_2d(&tmDO, coln + kb * 64, rown);
          }
        }
      }
      __syncwarp();
    }
  } else if (warp == 9) {
    const uint32_t idKK = umma_idesc_bf16(TILE, TILE, 0, 0);      // S, dP : both operands K-major
    const uint32_t idKM = umma_idesc_bf16(TILE, p.hd, 0, 1);      // dQ    : A = dS K-major, B = K MN-major
    const uint32_t idMM = umma_idesc_bf16(TILE, p.hd, 1, 1);      // dK, dV: A = dS^T / P^T MN-major, B MN-major
    // K-major views (+2 per 16-column K step, +OPB>>4 per 64-column block) and MN-major views (+128 per 16-row K step)
    const uint64_t kQ = umma_smem_desc(smem_u32(Qs), 0, 1024), kK = umma_smem_desc(smem_u32(Ks), 0, 1024);
    const uint64_t kV = umma_smem_desc(smem_u32(Vs), 0, 1024), kD = umma_smem_desc(smem_u32(Ds), 0, 1024);
    const uint64_t kG = umma_smem_desc(smem_u32(Gs), 0, 1024);
    const uint64_t mK = umma_smem_desc(smem_u32(Ks), OPB, 1024), mQ = umma_smem_desc(smem_u32(Qs), OPB, 1024);
    const uint64_t mD = umma_smem_desc(smem_u32(Ds), OPB, 1024), mG = umma_smem_desc(smem_u32(Gs), OPB, 1024);
    const uint64_t mP = umma_smem_desc(smem_u32(Ps), OPB, 1024);
    const uint64_t kP = umma_smem_desc(smem_u32(Ps), 0, 1024), kW = umma_smem_desc(smem_u32(Ws), 0, 1024);   // OP: dr, Wo^T
    const uint32_t idW = umma_idesc_bf16(TILE, p.hd, 0, 0);
    if (OP) { mbar_wait(w_full, 0); }
    uint32_t ph = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ph ^= 1) {
      mbar_wait(in_full, ph);                // (implies the previous item's dK / dV were read out of the S / dP columns)
      tc_fence_after();
      if (OP) {                              // dO = dr Wo first (it gates dP), then S while the epilogue stages dO
        if (elect_one()) {
          for (int kb = 0; kb < p.kblocks; ++kb) {
            const int ksteps = min(4, (p.hd - kb * 64) / 16);
            for (int k = 0; k < ksteps; ++k)
              umma_bf16(tDO, kP + (uint64_t)(kb * (OPB >> 4) + 2 * k), kW + (uint64_t)(kb * (wblk >> 4) + 2 * k), idW, (kb | k) != 0);
          }
          umma_commit(do_full);
          for (int kb = 0; kb < p.kblocks; ++kb) {
            const int ksteps = min(4, (p.hd - kb * 64) / 16);
            for (int k = 0; k < ksteps; ++k) {
              const uint64_t o = (uint64_t)(kb * (OPB >> 4) + 2 * k);
              umma_bf16(tS, kQ + o, kK + o, idKK, (kb | k) != 0);
            }
          }
        }
        __syncwarp();
        mbar_wait(do_staged, ph);
        tc_fence_after();
      }
      if (elect_one()) {
        for (int kb = 0; kb < p.kblocks; ++kb) {
          const int ksteps = min(4, (p.hd - kb * 64) / 16);
          for (int k = 0; k < ksteps; ++k) {
            const uint64_t o = (uint64_t)(kb * (OPB >> 4) + 2 * k);
            if (!OP) umma_bf16(tS, kQ + o, kK + o, idKK, (kb | k) != 0);
            umma_bf16(tDP, kD + o, kV + o, idKK, (kb | k) != 0);
          }
        }
        umma_commit(sdp_full);
      }
      __syncwarp();
      mbar_wait(ds_full, ph);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < 8; ++ks) {
          const uint64_t ko = (uint64_t)((ks >> 2) * (OPB >> 4) + (ks & 3) * 2);   // K-major A: key block, 32 B per step
          const uint64_t mo = (uint64_t)(ks * 128);                                // MN-major: 16 rows = 2048 B
          umma_bf16(tDQ, kG + ko, mK + mo, idKM, ks != 0);      // dQ[i, :] += dS[i, keys] K[keys, :]
          umma_bf16(tDK, mG + mo, mQ + mo, idMM, ks != 0);      // dK[j, :] += dS[rows, j]^T Q[rows, :]
          umma_bf16(tDV, mP + mo, mD + mo, idMM, ks != 0);      // dV[j, :] += P[rows, j]^T dO[rows, :]
        }
        umma_commit(out_full);
      }
      __syncwarp();
    }
  } else {
    const int quarter = warp & 3, part = warp >> 2;
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    const int r_first = quarter * 32;
    const int c_lo = PK ? (max(0, r_first - p.L) >> 5) : min(((r_first / p.L) * p.L) >> 5, quarter), c_hi = quarter;
    float* xmax = xch; float* xsum = xch + 2 * TILE; float* xdel = xch + 4 * TILE;
    uint32_t ph = 0;
    for (int it = blockIdx.x; it < n_items; it += gridDim.x, ph ^= 1) {
      const int tile = it / p.heads, h = it % p.heads;
      const int pk_row0 = PK ? __ldg(p.pk_tile_row0 + tile) : 0;
      RowInfo ri = PK ? row_info_pk(p, pk_row0, pk_M, h, quarter, lane) : row_info(p, tile, h, quarter, lane);
      const bool own = ri.owned;
      if (!own) { ri.jlo = 1 << 20; ri.jhi = ri.jlo; }              // empty window, loads stay warp-collective
      const unsigned span = (unsigned)(ri.jhi - ri.jlo);
      const int c0 = c_lo + part, c1 = c_lo + part + 2;
      const int lo0 = (c0 <= c_hi) ? ri.jlo - c0 * 32 : (1 << 20);
      const int lo1 = (c1 <= c_hi) ? ri.jlo - c1 * 32 : (1 << 20);
      if (OP) {                              // dO -> bf16 into dO's blocks (gemm_tn's rounding: + 0 bias, then bf16)
        mbar_wait(do_full, ph);
        tc_fence_after();
#pragma unroll 1
        for (int c = part * 32; c < p.hd; c += 64) {
          uint32_t ro[32];
          tmem_ld32(tDO + lane_off + c, ro);
          tmem_ld_wait();
          uint8_t* blk = Ds + (c >> 6) * OPB;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (c + 8 * u >= p.hd) break;
            float v[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(ro[8 * u + j]) + 0.f;
            *reinterpret_cast<uint4*>(blk + sw128(ri.r, (c & 63) + 8 * u)) =
                make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
          }
        }
        tc_fence_before();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(do_staged);
      }
      mbar_wait(sdp_full, ph);
      tc_fence_after();
      uint32_t s0[32], s1[32], g0[32], g1[32];
      tmem_ld32(tS + lane_off + min(c0, c_hi) * 32, s0);
      tmem_ld32(tS + lane_off + min(c1, c_hi) * 32, s1);
      tmem_ld32(tDP + lane_off + min(c0, c_hi) * 32, g0);
      tmem_ld32(tDP + lane_off + min(c1, c_hi) * 32, g1);
      tmem_ld_wait();
      float m = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        m = ((unsigned)(j - lo0) <= span) ? fmaxf(m, __uint_as_float(s0[j])) : m;
        m = ((unsigned)(j - lo1) <= span) ? fmaxf(m, __uint_as_float(s1[j])) : m;
      }
      xmax[part * TILE + ri.r] = m;
      named_bar_sync_a(1 + quarter, 64);
      m = fmaxf(m, xmax[(part ^ 1) * TILE + ri.r]);
      const float mb = m * p.scale_log2e;
      // e_j = exp(s_j - m) (kept in s*), partial sum and partial sum_j e_j * dP_j * mask_j (dropout mask folded into g*)
      float sum = 0.f, dsum = 0.f;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        float e0 = ex2_approx(fmaf(__uint_as_float(s0[j]), p.scale_log2e, -mb));
        float e1 = ex2_approx(fmaf(__uint_as_float(s1[j]), p.scale_log2e, -mb));
        e0 = ((unsigned)(j - lo0) <= span) ? e0 : 0.f;
        e1 = ((unsigned)(j - lo1) <= span) ? e1 : 0.f;
        if (PK) {                                   // the pad representative's column counts pm times (P is the total mass)
          e0 = (j == lo0) ? e0 * ri.pm : e0;
          e1 = (j == lo1) ? e1 * ri.pm : e1;
        }
        float d0 = __uint_as_float(g0[j]), d1 = __uint_as_float(g1[j]);
        if (DROP) {
          const float k0 = drop_f(p, ri, c0 * 32 + j), k1 = drop_f(p, ri, c1 * 32 + j);
          d0 *= k0; d1 *= k1;                       // dA = dAd * M
          g0[j] = __float_as_uint(k0); g1[j] = __float_as_uint(k1);
          sum += e0 + e1;
          dsum = fmaf(e0, d0, fmaf(e1, d1, dsum));
          s0[j] = __float_as_uint(e0); s1[j] = __float_as_uint(e1);
          // without dropout g* keeps dP; with dropout we need both the mask (for P) and dP*mask: recompute below
        } else {
          sum += e0 + e1;
          dsum = fmaf(e0, d0, fmaf(e1, d1, dsum));
          s0[j] = __float_as_uint(e0); s1[j] = __float_as_uint(e1);
        }
      }
      xsum[part * TILE + ri.r] = sum;
      xdel[part * TILE + ri.r] = dsum;
      named_bar_sync_a(1 + quarter, 64);
      sum += xsum[(part ^ 1) * TILE + ri.r];
      dsum += xdel[(part ^ 1) * TILE + ri.r];
      const float inv = own ? 1.f / sum : 0.f;
      const float delta = dsum * inv;
      if (DROP) {                                   // g* currently holds the dropout factor; rebuild dP * mask
        uint32_t t0[32], t1[32];
        tmem_ld32(tDP + lane_off + min(c0, c_hi) * 32, t0);
        tmem_ld32(tDP + lane_off + min(c1, c_hi) * 32, t1);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float k0 = __uint_as_float(g0[j]), k1 = __uint_as_float(g1[j]);
          // P_drop = p * k ; dS = p * (dP * k - delta) * scale
          const float p0 = __uint_as_float(s0[j]) * inv, p1 = __uint_as_float(s1[j]) * inv;
          g0[j] = __float_as_uint(p0 * (__uint_as_float(t0[j]) * k0 - delta) * p.scale);
          g1[j] = __float_as_uint(p1 * (__uint_as_float(t1[j]) * k1 - delta) * p.scale);
          s0[j] = __float_as_uint(p0 * k0); s1[j] = __float_as_uint(p1 * k1);
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float p0 = __uint_as_float(s0[j]) * inv, p1 = __uint_as_float(s1[j]) * inv;
          g0[j] = __float_as_uint(p0 * (__uint_as_float(g0[j]) - delta) * p.scale);      // S = scale * q k^T
          g1[j] = __float_as_uint(p1 * (__uint_as_float(g1[j]) - delta) * p.scale);
          s0[j] = __float_as_uint(p0); s1[j] = __float_as_uint(p1);
        }
      }
      if (c0 <= c_hi) {
        store_row32(Ps, ri.r, c0, reinterpret_cast<const float*>(s0));
        store_row32(Gs, ri.r, c0, reinterpret_cast<const float*>(g0));
      }
      if (c1 <= c_hi) {
        store_row32(Ps, ri.r, c1, reinterpret_cast<const float*>(s1));
        store_row32(Gs, ri.r, c1, reinterpret_cast<const float*>(g1));
      }
      for (int c = part; c < 4; c += 2)            // key chunks outside the quarter's window: P = dS = 0
        if (c < c_lo || c > c_hi) {
          const uint32_t off = (c >> 1) * OPB;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const uint32_t a = off + sw128(ri.r, (c & 1) * 32 + 8 * g);
            *reinterpret_cast<uint4*>(Ps + a) = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(Gs + a) = make_uint4(0u, 0u, 0u, 0u);
          }
        }
      tc_fence_before();
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(ds_full);
      mbar_wait(out_full, ph);
      tc_fence_after();
      if (!p.tma_o) {                      // head slices narrower than a 64-column store box: direct row stores
        if (part == 0) {
          store_out_row(own ? p.dq + ri.t * p.lddq + h * p.hd : nullptr, tDQ + lane_off, p.hd, 1.f);
          store_out_row(own ? p.dk + ri.t * p.lddkv + h * p.hd : nullptr, tDK + lane_off, p.hd, 1.f);
          store_out_row(own ? p.dv + ri.t * p.lddkv + h * p.hd : nullptr, tDV + lane_off, p.hd, 1.f);
        }
        tc_fence_before();
        named_bar_sync_a(9, 256);
        if (warp == 0 && lane == 0) mbar_arrive(in_free);
        __syncwarp();
        continue;
      }
      // dQ -> dO's blocks, dK -> K's blocks, dV -> Q's blocks (all operands are dead once out_full fires);
      // 32-column chunks alternate between the two warps of the quarter
#pragma unroll 1
      for (int o = 0; o < 3; ++o) {
        const uint32_t tsrc = (o == 0 ? tDQ : (o == 1 ? tDK : tDV)) + lane_off;
        uint8_t* dst = o == 0 ? Ds : (o == 1 ? Ks : Qs);
#pragma unroll 1
        for (int c = part * 32; c < p.hd; c += 64) {
          uint32_t ro[32];
          tmem_ld32(tsrc + c, ro);
          tmem_ld_wait();
          uint8_t* blk = dst + (c >> 6) * OPB;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            if (c + 8 * u >= p.hd) break;
            *reinterpret_cast<uint4*>(blk + sw128(ri.r, (c & 63) + 8 * u)) =
                make_uint4(pack_bf16x2(__uint_as_float(ro[8 * u]), __uint_as_float(ro[8 * u + 1])),
                           pack_bf16x2(__uint_as_float(ro[8 * u + 2]), __uint_as_float(ro[8 * u + 3])),
                           pack_bf16x2(__uint_as_float(ro[8 * u + 4]), __uint_as_float(ro[8 * u + 5])),
                           pack_bf16x2(__uint_as_float(ro[8 * u + 6]), __uint_as_float(ro[8 * u + 7])));
          }
        }
      }
      tc_fence_before();
      fence_proxy_async();
      named_bar_sync_a(9, 256);
      if (PK) {
        const int n_own = __ldg(p.pk_tile_row0 + tile + 1) - pk_row0;
        store_staged_rows(p.dq, p.lddq, pk_row0, h * p.hd, Ds, p.hd, n_own, threadIdx.x);
        store_staged_rows(p.dk, p.lddkv, pk_row0, h * p.hd, Ks, p.hd, n_own, threadIdx.x);
        store_staged_rows(p.dv, p.lddkv, pk_row0, h * p.hd, Qs, p.hd, n_own, threadIdx.x);
        named_bar_sync_a(9, 256);                  // every thread has read its chunks: the operand blocks may be refilled
        if (warp == 0 && lane == 0) mbar_arrive(in_free);
      } else if (warp == 0 && lane == 0) {
        const int row0 = tile * p.spt * p.L, col0 = h * p.hd;
        for (int kb = 0; kb < p.kblocks; ++kb) {
          tma_store_2d_a(&tmDQ, Ds + kb * OPB, col0 + kb * 64, row0);
          tma_store_2d_a(&tmDK, Ks + kb * OPB, col0 + kb * 64, row0);
          tma_store_2d_a(&tmDV, Qs + kb * OPB, col0 + kb * 64, row0);
        }
        bulk_commit_wait_read_all();
        mbar_arrive(in_free);
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

static bool tc_supported(int L, int H, int heads, int ldq, int ldkv) {
  if (heads <= 0 || H % heads) return false;
  const int hd = H / heads;
  return L >= 1 && L <= TILE && hd % 16 == 0 && hd <= 128 && ldq % 8 == 0 && ldkv % 8 == 0;
}

static int fill(AttnTc& p, int64_t B, int L, int H, int heads, float drop_p, uint64_t seed, uint32_t stream_id,
                const float* drop_step) {
  p.T = B * L; p.L = L; p.heads = heads; p.hd = H / heads;
  p.spt = TILE / L;
  p.n_tiles = (int)((B + p.spt - 1) / p.spt);
  p.kblocks = (p.hd + 63) / 64;
  p.scale = 1.0f / sqrtf((float)p.hd);
  p.scale_log2e = p.scale * 1.4426950408889634f;
  p.drop_seed = seed; p.drop_stream = stream_id; p.drop_step = drop_step; p.drop_thresh = 0; p.drop_scale = 1.f;
  if (drop_p > 0.f) {
    SRFRD_REQUIRE(drop_p < 1.f, "attention: dropout p must be < 1");
    p.drop_thresh = (uint32_t)((double)drop_p * 4294967296.0);
    p.drop_scale = 1.f / (1.f - drop_p);
  }
  return 0;
}

}  // namespace srfrd

using namespace srfrd;

extern "C" int srfrd_attn_debug_read(long long* host_dst) {
  SRFRD_CUDA(cudaDeviceSynchronize());
  SRFRD_CUDA(cudaMemcpyFromSymbol(host_dst, g_attn_dbg, sizeof(long long) * 16 * 16));
  return 0;
}

extern "C" int srfrd_attention_fwd(const void* q, int ldq, const void* k, const void* v, int ldkv, void* o, int ldo,
                                   float* stats, int64_t B, int L, int H, int heads, float drop_p, uint64_t seed,
                                   uint32_t stream_id, const float* drop_step, void* stream) {
  SRFRD_REQUIRE(q && k && v && o, "attention_fwd: null pointer");
  if (B == 0 || L == 0) return 0;
  if (attn_long_supported(B, L, H, heads, ldq, ldkv) && ldo % 8 == 0 && ((uintptr_t)o & 15) == 0 && !getenv("SRFRD_ATTN_SIMT"))
    return attn_long_fwd(q, ldq, k, v, ldkv, o, ldo, stats, B, L, H, heads, drop_p, seed, stream_id, drop_step, stream);
  if (!tc_supported(L, H, heads, ldq, ldkv) || ldo % 8 || ((uintptr_t)o & 15))
    return attn_fwd_simt(q, ldq, k, v, ldkv, o, ldo, B, L, H, heads, drop_p, seed, stream_id, drop_step, stream);
  AttnTc p = {};
  if (int rc = fill(p, B, L, H, heads, drop_p, seed, stream_id, drop_step)) return rc;
  p.o = (bf16*)o; p.ldo = ldo;
  p.tma_o = (heads == 1 || p.hd % 64 == 0) ? 1 : 0;
  { const char* dbg = getenv("SRFRD_ATTN_DEBUG"); p.debug = dbg ? atoi(dbg) : 0; }
  { const char* l2 = getenv("SRFRD_L2_PREFETCH"); if (l2 && atoi(l2) == 0) p.debug |= 256; }   // bit 8: no L2 prefetch (backward)
  CUtensorMap tmQ, tmK, tmV, tmO;
  if (int rc = make_tmap_bf16_2d(&tmQ, q, p.T, H, ldq, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmK, k, p.T, H, ldkv, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmV, v, p.T, H, ldkv, TILE, 64)) return rc;
  // the store box covers exactly the spt*L rows a tile owns (rows beyond belong to the next tile's sequences)
  if (int rc = make_tmap_bf16_2d(&tmO, o, p.T, H, ldo, p.spt * L, 64)) return rc;
  const size_t smem = (size_t)(2 * p.kblocks + (p.kblocks > 2 ? p.kblocks : 2)) * OPB + 4 * TILE * sizeof(float) + 1024 + 256;
  static bool attr = false;
  if (!attr) {
    SRFRD_CUDA(cudaFuncSetAttribute(attn_fwd_tc_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_fwd_tc_kernel<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 113 * 1024));
    attr = true;
  }
  int grid = p.n_tiles * heads;
  if (grid > 2 * num_sms()) grid = 2 * num_sms();
  if (p.drop_thresh)
    SRFRD_CUDA(launch_pdl(attn_fwd_tc_kernel<true, false, false>, dim3(grid), dim3(AF_THREADS), smem, (cudaStream_t)stream, tmQ, tmK, tmV, tmO,
                          tmO, tmO, p));
  else
    SRFRD_CUDA(launch_pdl(attn_fwd_tc_kernel<false, false, false>, dim3(grid), dim3(AF_THREADS), smem, (cudaStream_t)stream, tmQ, tmK, tmV, tmO,
                          tmO, tmO, p));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_attention_bwd(const void* dout, int lddo, const void* q, int ldq, const void* k, const void* v,
                                   int ldkv, const void* o, int ldo, float* stats, void* dq, int lddq, void* dk, void* dv,
                                   int lddkv, int64_t B, int L, int H, int heads, float drop_p, uint64_t seed,
                                   uint32_t stream_id, const float* drop_step, void* stream) {
  SRFRD_REQUIRE(dout && q && k && v && dq && dk && dv, "attention_bwd: null pointer");
  if (B == 0 || L == 0) return 0;
  if (attn_long_supported(B, L, H, heads, ldq, ldkv) && o && stats && !getenv("SRFRD_ATTN_SIMT"))
    return attn_long_bwd(dout, lddo, q, ldq, k, v, ldkv, o, ldo, stats, dq, lddq, dk, dv, lddkv, B, L, H, heads, drop_p, seed,
                         stream_id, drop_step, stream);
  if (!tc_supported(L, H, heads, ldq, ldkv) || lddo % 8 || lddq % 8 || lddkv % 8)
    return attn_bwd_simt(dout, lddo, q, ldq, k, v, ldkv, dq, lddq, dk, dv, lddkv, B, L, H, heads, drop_p, seed,
                         stream_id, drop_step, stream);
  AttnTc p = {};
  if (int rc = fill(p, B, L, H, heads, drop_p, seed, stream_id, drop_step)) return rc;
  p.dq = (bf16*)dq; p.dk = (bf16*)dk; p.dv = (bf16*)dv; p.lddq = lddq; p.lddkv = lddkv;
  p.tma_o = ((heads == 1 || p.hd % 64 == 0) && (((uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) & 15) == 0) ? 1 : 0;
  CUtensorMap tmQ, tmK, tmV, tmDO, tmDQ, tmDK, tmDV;
  if (int rc = make_tmap_bf16_2d(&tmQ, q, p.T, H, ldq, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmK, k, p.T, H, ldkv, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmV, v, p.T, H, ldkv, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmDO, dout, p.T, H, lddo, TILE, 64)) return rc;
  tmDQ = tmQ; tmDK = tmQ; tmDV = tmQ;
  if (p.tma_o) {      // store boxes cover exactly the spt*L rows a tile owns
    if (int rc = make_tmap_bf16_2d(&tmDQ, dq, p.T, H, lddq, p.spt * L, 64)) return rc;
    if (int rc = make_tmap_bf16_2d(&tmDK, dk, p.T, H, lddkv, p.spt * L, 64)) return rc;
    if (int rc = make_tmap_bf16_2d(&tmDV, dv, p.T, H, lddkv, p.spt * L, 64)) return rc;
  }
  const size_t smem = (size_t)(4 * p.kblocks + 4) * OPB + 6 * TILE * sizeof(float) + 1024 + 256;
  static bool attr = false;
  if (!attr) {
    SRFRD_CUDA(cudaFuncSetAttribute(attn_bwd_tc_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_bwd_tc_kernel<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr = true;
  }
  int grid = p.n_tiles * heads;
  if (grid > num_sms()) grid = num_sms();
  if (p.drop_thresh)
    SRFRD_CUDA(launch_pdl(attn_bwd_tc_kernel<true, false, false>, dim3(grid), dim3(AF_THREADS), smem, (cudaStream_t)stream, tmQ, tmK, tmV,
                          tmDO, tmDQ, tmDK, tmDV, tmDV, p));
  else
    SRFRD_CUDA(launch_pdl(attn_bwd_tc_kernel<false, false, false>, dim3(grid), dim3(AF_THREADS), smem, (cudaStream_t)stream, tmQ, tmK, tmV,
                          tmDO, tmDQ, tmDK, tmDV, tmDV, p));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Packed token layout (pack.cu): the same kernels with tiles, row windows and the pad column's weight read from the
// device-resident plan; q / k / v / o (and the gradients) are (capacity, ld) buffers of packed rows.
static int packed_supported(int L, int H, int heads, int ldq, int ldkv) {
  if (!tc_supported(L, H, heads, ldq, ldkv)) return 0;
  const int hd = H / heads;
  return (L + 1 <= TILE) && (heads == 1 || hd % 64 == 0);
}

extern "C" int srfrd_attention_packed_supported(int L, int H, int heads) {
  return packed_supported(L, H, heads, 8, 8) && !getenv("SRFRD_ATTN_SIMT");
}

// Shared memory of the packed kernels (1024 B of slack for the 1024-byte alignment of the operand blocks)
static size_t fwd_smem(int kblocks, bool op) {
  return (size_t)(2 * kblocks + (kblocks > 2 ? kblocks : 2)) * OPB + 4 * TILE * sizeof(float) + 1024 + 256 +
         (op ? 3 * TILE * sizeof(float) : 0);
}
static size_t bwd_smem(int kblocks, int hd, bool op) {
  return op ? (size_t)(4 * kblocks + 4) * OPB + 4096 + (size_t)kblocks * hd * 128 + 1024
            : (size_t)(4 * kblocks + 4) * OPB + 6 * TILE * sizeof(float) + 1024 + 256;
}
static constexpr size_t FWD_SMEM_MAX = 113 * 1024;       // two CTAs per SM
static constexpr size_t BWD_SMEM_MAX = 227 * 1024;

// Which packed kernels can fold the attention out-projection in: bit 0 forward, bit 1 backward.  One head (a CTA owns
// whole rows, so the LayerNorm of the forward epilogue sees all columns), at most 128 columns (the kernels' operand
// blocks and TMEM plan), and the shared-memory plan has to fit.
static int oproj_supported(int L, int H, int heads) {
  if (!packed_supported(L, H, heads, 8, 8) || heads != 1 || H > 128) return 0;
  const int kblocks = (H + 63) / 64;
  return (fwd_smem(kblocks, true) <= FWD_SMEM_MAX ? 1 : 0) | (bwd_smem(kblocks, H, true) <= BWD_SMEM_MAX ? 2 : 0);
}

extern "C" int srfrd_attention_packed_oproj_supported(int L, int H, int heads) {
  return getenv("SRFRD_ATTN_SIMT") ? 0 : oproj_supported(L, H, heads);
}

extern "C" int srfrd_attention_fwd_packed(const void* q, int ldq, const void* k, const void* v, int ldkv, void* o, int ldo,
                                          const srfrd_pack_t* pk, int L, int H, int heads, float drop_p, uint64_t seed,
                                          uint32_t stream_id, const float* drop_step, void* stream, const void* wo, int ldw,
                                          const float* bo, const void* res, int ldres, const float* ln_w, const float* ln_b,
                                          float ln_eps, float* ln_stats, void* r, int ldr, void* y, int ldy) {
  SRFRD_REQUIRE(q && k && v && o && pk && pk->rows && pk->row_info && pk->tile_row0, "attention_fwd_packed: null pointer");
  SRFRD_REQUIRE(packed_supported(L, H, heads, ldq, ldkv) && ldo % 8 == 0 && ((uintptr_t)o & 15) == 0,
                "attention_fwd_packed: unsupported shape (L=%d H=%d heads=%d)", L, H, heads);
  const bool op = wo != nullptr;
  if (op) {
    SRFRD_REQUIRE(oproj_supported(L, H, heads) & 1, "attention_fwd_packed: no fused out-projection for H=%d heads=%d", H, heads);
    SRFRD_REQUIRE(res && ln_w && ln_b && r && y, "attention_fwd_packed: fused out-projection needs residual, LayerNorm, r and y");
    SRFRD_REQUIRE(ldw % 8 == 0 && ldw >= H && ldres % 8 == 0 && ldr % 8 == 0 && ldy % 8 == 0 &&
                      (((uintptr_t)res | (uintptr_t)r | (uintptr_t)y | (uintptr_t)wo) & 15) == 0,
                  "attention_fwd_packed: bad out-projection operands");
  }
  AttnTc p = {};
  if (int rc = fill(p, 1, L, H, heads, drop_p, seed, stream_id, drop_step)) return rc;
  p.T = pk->cap;
  p.o = (bf16*)o; p.ldo = ldo; p.tma_o = 1;
  p.pk_rows = pk->rows; p.pk_info = (const int4*)pk->row_info; p.pk_tile_row0 = pk->tile_row0;
  CUtensorMap tmQ, tmK, tmV, tmW, tmR;
  if (int rc = make_tmap_bf16_2d(&tmQ, q, p.T, H, ldq, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmK, k, p.T, H, ldkv, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmV, v, p.T, H, ldkv, TILE, 64)) return rc;
  tmW = tmQ; tmR = tmQ;
  if (op) {
    if (int rc = make_tmap_bf16_2d(&tmW, wo, H, H, ldw, H, 64)) return rc;        // the whole [H x H] weight in one box row
    if (int rc = make_tmap_bf16_2d(&tmR, res, p.T, H, ldres, TILE, 64)) return rc;
    p.op_bias = bo; p.ln_w = ln_w; p.ln_b = ln_b; p.ln_stats = ln_stats; p.ln_eps = ln_eps;
    p.op_r = (bf16*)r; p.op_y = (bf16*)y; p.ldr = ldr; p.ldy = ldy;
  }
  const size_t smem = fwd_smem(p.kblocks, op);
  static bool attr = false;
  if (!attr) {
    SRFRD_CUDA(cudaFuncSetAttribute(attn_fwd_tc_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM_MAX));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_fwd_tc_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM_MAX));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_fwd_tc_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM_MAX));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_fwd_tc_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FWD_SMEM_MAX));
    attr = true;
  }
  int64_t grid = (pk->cap / 64 + 1) * heads;               // more tiles than this cannot exist
  if (grid > 2 * num_sms()) grid = 2 * num_sms();
  auto kern = p.drop_thresh ? (op ? attn_fwd_tc_kernel<true, true, true> : attn_fwd_tc_kernel<true, true, false>)
                            : (op ? attn_fwd_tc_kernel<false, true, true> : attn_fwd_tc_kernel<false, true, false>);
  SRFRD_CUDA(launch_pdl(kern, dim3((unsigned)grid), dim3(AF_THREADS), smem, (cudaStream_t)stream, tmQ, tmK, tmV, tmQ, tmW, tmR, p));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_attention_bwd_packed(const void* dout, int lddo, const void* q, int ldq, const void* k, const void* v,
                                          int ldkv, void* dq, int lddq, void* dk, void* dv, int lddkv, const srfrd_pack_t* pk,
                                          int L, int H, int heads, float drop_p, uint64_t seed, uint32_t stream_id,
                                          const float* drop_step, void* stream, const void* dr, int lddr, const void* woT,
                                          int ldw) {
  const bool op = dr != nullptr;
  SRFRD_REQUIRE((op ? (woT != nullptr) : (dout != nullptr)) && q && k && v && dq && dk && dv && pk && pk->rows &&
                    pk->row_info && pk->tile_row0,
                "attention_bwd_packed: null pointer");
  SRFRD_REQUIRE(packed_supported(L, H, heads, ldq, ldkv) && (op || lddo % 8 == 0) && lddq % 8 == 0 && lddkv % 8 == 0 &&
                    (((uintptr_t)dq | (uintptr_t)dk | (uintptr_t)dv) & 15) == 0,
                "attention_bwd_packed: unsupported shape (L=%d H=%d heads=%d)", L, H, heads);
  if (op) {
    SRFRD_REQUIRE(oproj_supported(L, H, heads) & 2, "attention_bwd_packed: no fused out-projection for H=%d heads=%d", H, heads);
    SRFRD_REQUIRE(lddr % 8 == 0 && ldw % 8 == 0 && ldw >= H && (((uintptr_t)dr | (uintptr_t)woT) & 15) == 0,
                  "attention_bwd_packed: bad out-projection operands");
  }
  AttnTc p = {};
  if (int rc = fill(p, 1, L, H, heads, drop_p, seed, stream_id, drop_step)) return rc;
  p.T = pk->cap;
  p.dq = (bf16*)dq; p.dk = (bf16*)dk; p.dv = (bf16*)dv; p.lddq = lddq; p.lddkv = lddkv; p.tma_o = 1;
  p.pk_rows = pk->rows; p.pk_info = (const int4*)pk->row_info; p.pk_tile_row0 = pk->tile_row0;
  { const char* l2 = getenv("SRFRD_L2_PREFETCH"); if (l2 && atoi(l2) == 0) p.debug |= 256; }
  CUtensorMap tmQ, tmK, tmV, tmDO, tmWT;
  if (int rc = make_tmap_bf16_2d(&tmQ, q, p.T, H, ldq, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmK, k, p.T, H, ldkv, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmV, v, p.T, H, ldkv, TILE, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmDO, op ? dr : dout, p.T, H, op ? lddr : lddo, TILE, 64)) return rc;   // OP: dr
  tmWT = tmQ;
  if (op) if (int rc = make_tmap_bf16_2d(&tmWT, woT, H, H, ldw, H, 64)) return rc;
  const size_t smem = bwd_smem(p.kblocks, p.hd, op);
  static bool attr = false;
  if (!attr) {
    SRFRD_CUDA(cudaFuncSetAttribute(attn_bwd_tc_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM_MAX));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_bwd_tc_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM_MAX));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_bwd_tc_kernel<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM_MAX));
    SRFRD_CUDA(cudaFuncSetAttribute(attn_bwd_tc_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, BWD_SMEM_MAX));
    attr = true;
  }
  int64_t grid = (pk->cap / 64 + 1) * heads;
  if (grid > num_sms()) grid = num_sms();
  auto kern = p.drop_thresh ? (op ? attn_bwd_tc_kernel<true, true, true> : attn_bwd_tc_kernel<true, true, false>)
                            : (op ? attn_bwd_tc_kernel<false, true, true> : attn_bwd_tc_kernel<false, true, false>);
  SRFRD_CUDA(launch_pdl(kern, dim3((unsigned)grid), dim3(AF_THREADS), smem, (cudaStream_t)stream, tmQ, tmK, tmV, tmDO, tmQ, tmQ,
                        tmQ, tmWT, p));
  SRFRD_LAUNCH_CHECK();
  return 0;
}
