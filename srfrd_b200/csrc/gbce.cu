// gSASRec's gBCE loss over k negatives shared by every row of a step, on tcgen05.  For h rows r with positive pos_r,
// weight w_r and negatives n_1..n_k (uniform with replacement over 1..N):
//   alpha = k / (N - 1),  beta = 1 - t (1 - alpha),  z_r = <h_r, E[pos_r]>,  s_rj = <h_r, E[n_j]>,
//   m_rj  = 0 if n_j occurs in row r's sequence (its seq or pos ids), else 1,     W = sum_r w_r = norm[0]
//   loss  = ( sum_r w_r beta softplus(-z_r) + sum_r w_r sum_j m_rj softplus(s_rj) ) / W
//   dz_r  = w_r beta (sigmoid(z_r) - 1) / W,      ds_rj = w_r m_rj sigmoid(s_rj) / W
// Because the negatives are shared, S = h N^T is a real GEMM (k <= 256 columns) and so are dh = dS N and dN = dS^T h.
//   gbce_draw_kernel   draws the ids from a hash of (seed, device step counter), gathers their rows from the fp32 item
//                      table into a zero-padded (Kp, Dp) bf16 K-major table (Kp = k rounded up to 128), and builds the
//                      per-sequence exclusion bitmask (n_seq, ceil(k / 32)) uint32 (bit j set: n_j occurs in the sequence)
//   GB_DH              one CTA per 128-row tile of h, the skeleton of catalogue_ce.cu's CE_DH with the negatives as the
//                      streamed blocks: S into a double-buffered TMEM S, the negative loss term into loss_acc[1],
//                      X = m sigmoid(S) (bf16, smem), dh_acc += X N (TMEM).  The epilogue adds the positive term: z_r
//                      as a per-row dot of the resident h tile with bf16(E[pos]), its loss into loss_acc[0], dz E[pos] into
//                      dh and dz h into d_item[pos] (red.add, as score_loss_fused does)
//   GB_DN              one CTA per (128-negative block, split of the row tiles), the skeleton of CE_DE: for each row tile
//                      of its split, S, X = (w / W) m sigmoid(S), dN_acc += X^T h; the (Kp, Dp) partial of the split is
//                      written to a workspace.  TMEM: S 2 x 128 + Dp <= 512 columns; S, dh and dN at once would not fit
//   gbce_scatter_kernel sums the partials of each negative over the splits and over its duplicate draws in a fixed order
//                      and adds the sum to d_item[n_j] once per distinct id: the negatives' part of dE is deterministic
// The read-out acc[0] / norm[0] + acc[1] / norm[1] of the Adam kernels then gives the loss, since norm[1] == norm[0] when
// there is no w_neg.
#include "common.cuh"
#include "srfrd_b200.h"

namespace srfrd {
namespace {

constexpr int GT = 128;                   // rows of a tile: h rows or negatives
constexpr int GTB = GT * 64 * 2;          // one [128 x 64] bf16 tile
constexpr int GB_THREADS = 320;
constexpr int GB_MAX_STAGES = 8;
constexpr int GB_MAX_K = 256;
constexpr size_t GB_SMEM_LIMIT = 227 * 1024;
constexpr uint32_t GB_SALT = 0x67BCE5u;   // hash stream of the draw (the batch sampler and dropout use others)
enum { GB_DH = 0, GB_DN = 1 };

struct GbParams {
  int64_t cap;                  // rows of the h buffer
  const int* rows_dev;          // device row count (packed layout) or null: rows = min(cap, *rows_dev)
  const int* row_tok;           // packed layout: dense token of h row r (-1: no token) or null (identity)
  const int64_t* pos;           // positive item per dense token
  const float* w_pos;           // weight per dense token, or null -> 1[pos != 0]
  const float* norm;            // norm[0] = W
  const uint32_t* excl;         // (n_seq, kw) exclusion bits, or null (no exclusion)
  int kw, L;                    // words per sequence; dense tokens per sequence (sequence of token t = t / L)
  int k, Kp, n_split;
  int Dp, kb, stages, D;
  float beta;
  const float* item; int ldi;   // fp32 item table (positive rows)
  int64_t n_items;
  float* loss_acc;              // [0] += positive terms, [1] += negative terms (unnormalised)
  float* dh; int lddh;          // (cap, lddh) fp32, first D columns written
  float* d_item; int ldd;       // (N + 1, ldd) fp32, positive rows added to (null: no dE)
  float* part;                  // (n_split, Kp, Dp) fp32 partials of dN
};

__device__ __forceinline__ uint32_t gb_sw128(int r, int c) {      // byte offset of (row r, column c) in a swizzled tile
  return (uint32_t)(r * 128 + ((((c >> 3) ^ (r & 7)) << 4) | ((c & 7) << 1)));
}
__device__ __forceinline__ void gb_bar(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ float gb_sigmoid(float x) { return 1.f / (1.f + __expf(-x)); }
__device__ __forceinline__ float gb_softplus(float x) { return fmaxf(x, 0.f) + log1pf(__expf(-fabsf(x))); }
__device__ __forceinline__ float gb_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
// 32 values of row r, 32-column chunk c of the [128 x 128] X -> the swizzled K-major tile pair at `base`
__device__ __forceinline__ void gb_store32(uint8_t* base, int r, int c, const float* v) {
  uint8_t* blk = base + (c >> 1) * GTB;
  const int col0 = (c & 1) * 32;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    *reinterpret_cast<uint4*>(blk + gb_sw128(r, col0 + 8 * u)) =
        make_uint4(pack_bf16x2(v[8 * u], v[8 * u + 1]), pack_bf16x2(v[8 * u + 2], v[8 * u + 3]),
                   pack_bf16x2(v[8 * u + 4], v[8 * u + 5]), pack_bf16x2(v[8 * u + 6], v[8 * u + 7]));
}

__device__ __forceinline__ int64_t gb_draw(uint64_t seed, int j, int64_t n_items) {
  return 1 + (int64_t)(hash_u32(seed, GB_SALT, (uint64_t)j) % (uint32_t)n_items);
}

__device__ __forceinline__ int gb_rows(const GbParams& p) {
  return (int)(p.rows_dev ? min(p.cap, (int64_t)__ldg(p.rows_dev)) : p.cap);
}
// unnormalised weight of h row r (< rows), its positive and its sequence; 0 = the row carries no loss term (no token,
// pos outside 1..N, zero weight)
__device__ __forceinline__ float gb_row(const GbParams& p, int64_t r, int64_t& tgt, int64_t& sq) {
  tgt = 0; sq = 0;
  const int64_t tok = p.row_tok ? (int64_t)__ldg(p.row_tok + r) : r;
  if (tok < 0) return 0.f;
  const int64_t t = __ldg(p.pos + tok);
  if (t < 1 || t > p.n_items) return 0.f;
  const float w = p.w_pos ? __ldg(p.w_pos + tok) : 1.f;
  if (w != 0.f) { tgt = t; sq = tok / p.L; }
  return w;
}
// bits of negatives j0 .. j0 + 31 (j0 % 32 == 0) that enter row's loss: drawn (j < k) and not excluded for sequence sq
__device__ __forceinline__ uint32_t gb_keep(const GbParams& p, int64_t sq, int j0) {
  if (j0 >= p.k) return 0u;
  const uint32_t valid = p.k - j0 >= 32 ? 0xffffffffu : ((1u << (p.k - j0)) - 1u);
  const uint32_t ex = p.excl ? __ldg(p.excl + sq * p.kw + (j0 >> 5)) : 0u;
  return valid & ~ex;
}

template <int MODE>
__global__ void __launch_bounds__(GB_THREADS, 1)
gbce_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmN, GbParams p) {
  pdl_prologue_done();
  const int rows = gb_rows(p);
  const int n_rt = (rows + GT - 1) / GT;
  int unit, rt0 = 0, nstream;
  if (MODE == GB_DH) {
    unit = blockIdx.x;
    if (unit >= n_rt) return;                                   // CTA-uniform, before any barrier
    nstream = p.Kp / GT;
  } else {
    unit = blockIdx.y;
    rt0 = (int)((int64_t)blockIdx.x * n_rt / p.n_split);
    nstream = (int)((int64_t)(blockIdx.x + 1) * n_rt / p.n_split) - rt0;
    if (nstream <= 0) {                                         // an empty split still owns its partial
      float* dst = p.part + ((int64_t)blockIdx.x * p.Kp + (int64_t)unit * GT) * p.Dp;
      for (int i = threadIdx.x; i < GT * p.Dp; i += blockDim.x) dst[i] = 0.f;
      return;
    }
  }

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* res = smem;                                          // resident block: h rows (DH) or negative rows (DN)
  uint8_t* ring = res + p.kb * GTB;                             // stages x kb tiles of the streamed operand
  uint8_t* Xs = ring + p.stages * p.kb * GTB;                   // X [128 x 128] bf16; DH epilogue: row exchange
  float* xch = reinterpret_cast<float*>(Xs);
  uint64_t* bars = reinterpret_cast<uint64_t*>(Xs + 2 * GTB);
  uint64_t* full = bars;
  uint64_t* empty = bars + p.stages;
  uint64_t* res_full = bars + 2 * p.stages;
  uint64_t* s_full = res_full + 1;                              // [2]
  uint64_t* s_free = res_full + 3;                              // [2]
  uint64_t* x_full = res_full + 5;
  uint64_t* x_free = res_full + 6;
  uint64_t* acc_full = res_full + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 8);
  constexpr uint32_t TMEM_COLS = 512;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmH); tma_prefetch_desc(&tmN);
    for (int i = 0; i < p.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(res_full, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_free[i], 8); }
    mbar_init(x_full, 8); mbar_init(x_free, 1); mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 9) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tS = tmem_base, tACC = tmem_base + 2 * GT;     // S: 2 x 128 columns; output accumulator: Dp columns

  if (warp == 8) {
    // ---------------------------------------------------------------- TMA producer
    const CUtensorMap* tmRes = MODE == GB_DN ? &tmN : &tmH;
    const CUtensorMap* tmStr = MODE == GB_DN ? &tmH : &tmN;
    const int str0 = MODE == GB_DN ? rt0 : 0;
    if (elect_one()) {
      mbar_expect_tx(res_full, p.kb * GTB);
      for (int kb = 0; kb < p.kb; ++kb) tma_load_2d(res + kb * GTB, tmRes, res_full, kb * 64, unit * GT, SRFRD_EVICT_FIRST);
    }
    __syncwarp();
    int slot = 0; uint32_t ph = 0;
    for (int n = 0; n < nstream; ++n) {
      mbar_wait(&empty[slot], ph ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&full[slot], p.kb * GTB);
        for (int kb = 0; kb < p.kb; ++kb)
          tma_load_2d(ring + (slot * p.kb + kb) * GTB, tmStr, &full[slot], kb * 64, (str0 + n) * GT, SRFRD_EVICT_LAST);
      }
      __syncwarp();
      if (++slot == p.stages) { slot = 0; ph ^= 1; }
    }
  } else if (warp == 9) {
    // ---------------------------------------------------------------- MMA issuer
    const uint32_t idS = umma_idesc_bf16(GT, GT, 0, 0);
    const uint64_t dRes = umma_smem_desc(smem_u32(res), 0, 1024);       // K-major views
    const uint64_t dRing = umma_smem_desc(smem_u32(ring), 0, 1024);
    const uint64_t mRing = umma_smem_desc(smem_u32(ring), GTB, 1024);   // MN-major view of a ring tile (rows = K)
    const uint64_t kX = umma_smem_desc(smem_u32(Xs), 0, 1024);          // X as K-major A (DH: X N)
    const uint64_t mX = umma_smem_desc(smem_u32(Xs), GTB, 1024);        // X^T as MN-major A (DN: X^T h)
    mbar_wait(res_full, 0);
    // second product of streamed block m, whose tiles sit in ring slot st
    auto out_mma = [&](int m, int st) {
      mbar_wait(x_full, m & 1);
      tc_fence_after();
      if (elect_one()) {
        for (int cb = 0; cb < p.kb; ++cb) {
          const int ncols = min(64, p.Dp - cb * 64);
          const uint64_t bq = mRing + (uint64_t)((st * p.kb + cb) * (GTB >> 4));
          if (MODE == GB_DH) {
            const uint32_t id = umma_idesc_bf16(GT, ncols, 0, 1);
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma_bf16(tACC + cb * 64, kX + (uint64_t)((ks >> 2) * (GTB >> 4) + (ks & 3) * 2), bq + (uint64_t)(ks * 128), id,
                        (m | ks) != 0);
          } else {
            const uint32_t id = umma_idesc_bf16(GT, ncols, 1, 1);
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma_bf16(tACC + cb * 64, mX + (uint64_t)(ks * 128), bq + (uint64_t)(ks * 128), id, (m | ks) != 0);
          }
        }
        umma_commit(&empty[st]);
        umma_commit(x_free);
      }
      __syncwarp();
    };
    int slot = 0, prev = 0; uint32_t ph = 0;
    for (int n = 0; n < nstream; ++n) {
      const int buf = n & 1;
      mbar_wait(&s_free[buf], ((n >> 1) & 1) ^ 1);               // the epilogue warps have read this S buffer's last use
      mbar_wait(&full[slot], ph);
      tc_fence_after();
      if (elect_one()) {
        for (int kb = 0; kb < p.kb; ++kb) {
          const int ksteps = min(4, (p.Dp - kb * 64) / 16);
          const uint64_t rt = dRes + (uint64_t)(kb * (GTB >> 4));
          const uint64_t st = dRing + (uint64_t)((slot * p.kb + kb) * (GTB >> 4));
          const uint64_t a = MODE == GB_DN ? st : rt, b = MODE == GB_DN ? rt : st;   // A: h rows, B: negative rows
          for (int k = 0; k < ksteps; ++k) umma_bf16(tS + buf * GT, a + 2 * k, b + 2 * k, idS, (kb | k) != 0);
        }
        umma_commit(&s_full[buf]);
      }
      __syncwarp();
      if (n > 0) out_mma(n - 1, prev);                           // S of block n runs while X of block n - 1 is formed
      prev = slot;
      if (++slot == p.stages) { slot = 0; ph ^= 1; }
    }
    out_mma(nstream - 1, prev);
    if (elect_one()) umma_commit(acc_full);
    __syncwarp();
  } else {
    // ---------------------------------------------------------------- epilogue: warp w reads TMEM lanes 32 (w & 3) ..
    // + 31 and the 64 S columns of half `part`
    const int quarter = warp & 3, part = warp >> 2;
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    const int r = quarter * 32 + lane;
    const float nv = __ldg(p.norm);
    const float inv_norm = nv > 0.f ? 1.f / nv : 0.f;
    auto read_s = [&](int n, float (&v)[64]) {
      const int buf = n & 1;
      mbar_wait(&s_full[buf], (n >> 1) & 1);
      tc_fence_after();
      uint32_t a[32], b[32];
      tmem_ld32(tS + lane_off + buf * GT + part * 64, a);
      tmem_ld32(tS + lane_off + buf * GT + part * 64 + 32, b);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_free[buf]);
#pragma unroll
      for (int j = 0; j < 32; ++j) { v[j] = __uint_as_float(a[j]); v[32 + j] = __uint_as_float(b[j]); }
    };
    // X chunk pair of this half <- x (after the previous block's second product has read X)
    auto store_x = [&](int n, const float (&x)[64]) {
      mbar_wait(x_free, (n & 1) ^ 1);
      gb_store32(Xs, r, 2 * part, x);
      gb_store32(Xs, r, 2 * part + 1, x + 32);
      tc_fence_before();
      fence_proxy_async();                                        // generic-proxy smem writes -> visible to the MMA
      __syncwarp();
      if (lane == 0) mbar_arrive(x_full);
    };

    if (MODE == GB_DH) {
      const int64_t row = (int64_t)unit * GT + r;
      const bool in = row < rows;
      int64_t tgt = 0, sq = 0;
      const float w = in ? gb_row(p, row, tgt, sq) : 0.f;
      float lneg = 0.f;
      for (int n = 0; n < nstream; ++n) {
        float v[64];
        read_s(n, v);
        const int j0 = n * GT + part * 64;
        const uint32_t k0 = w != 0.f ? gb_keep(p, sq, j0) : 0u, k1 = w != 0.f ? gb_keep(p, sq, j0 + 32) : 0u;
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const bool keep = ((j < 32 ? k0 >> j : k1 >> (j - 32)) & 1u) != 0;
          lneg += keep ? gb_softplus(v[j]) : 0.f;
          v[j] = keep ? gb_sigmoid(v[j]) : 0.f;
        }
        store_x(n, v);
      }
      const float tneg = warp_sum(w * lneg);
      if (lane == 0 && tneg != 0.f) red_add_f32(p.loss_acc + 1, tneg);
      mbar_wait(acc_full, 0);
      mbar_wait(res_full, 0);                                     // the resident h tile is read directly below
      tc_fence_after();
      // positive logit: this thread's column blocks of the resident bf16 h row against bf16(E[pos]); the two warps of a
      // lane quarter exchange their halves through X, which no MMA reads any more
      const float* Ep = p.item + tgt * p.ldi;
      float zp = 0.f;
      if (w != 0.f) {
        for (int cb = part; cb < p.kb; cb += 2) {
          const int nc = min(64, p.D - cb * 64);
          for (int j = 0; j < nc; ++j)
            zp = fmaf(bf2f(*reinterpret_cast<const bf16*>(res + cb * GTB + gb_sw128(r, j))), gb_round(__ldg(Ep + cb * 64 + j)),
                      zp);
        }
      }
      xch[part * GT + r] = zp;
      gb_bar(1 + quarter, 64);
      const float z = xch[r] + xch[GT + r];
      const float dz = w != 0.f ? w * p.beta * (gb_sigmoid(z) - 1.f) * inv_norm : 0.f;
      if (part == 0) {
        const float tpos = warp_sum(w != 0.f ? w * p.beta * gb_softplus(-z) : 0.f);
        if (lane == 0 && tpos != 0.f) red_add_f32(p.loss_acc, tpos);
      }
      const float coef = w * inv_norm;
      for (int cb = part; cb < p.kb; cb += 2) {
        uint32_t a[32], b[32];
        tmem_ld32(tACC + lane_off + cb * 64, a);
        tmem_ld32(tACC + lane_off + cb * 64 + 32, b);
        tmem_ld_wait();
        if (in) {
          float* dst = p.dh + row * p.lddh + cb * 64;
          float* de = p.d_item && dz != 0.f ? p.d_item + tgt * p.ldd + cb * 64 : nullptr;
          const int nc = min(64, p.D - cb * 64);
#pragma unroll
          for (int j = 0; j < 64; ++j) {
            const uint32_t u = j < 32 ? a[j] : b[j - 32];
            if (j < nc) {
              dst[j] = w != 0.f ? fmaf(dz, gb_round(__ldg(Ep + cb * 64 + j)), coef * __uint_as_float(u)) : 0.f;
              if (de) red_add_f32(de + j, dz * bf2f(*reinterpret_cast<const bf16*>(res + cb * GTB + gb_sw128(r, j))));
            }
          }
        }
      }
    } else {
      // GB_DN: S lanes are the rows of streamed tile rt0 + n, columns this CTA's negatives
      for (int n = 0; n < nstream; ++n) {
        const int64_t row = (int64_t)(rt0 + n) * GT + r;
        int64_t tgt = 0, sq = 0;
        const float w = row < rows ? gb_row(p, row, tgt, sq) : 0.f;
        const float coef = w * inv_norm;
        const int j0 = unit * GT + part * 64;
        const uint32_t k0 = coef != 0.f ? gb_keep(p, sq, j0) : 0u, k1 = coef != 0.f ? gb_keep(p, sq, j0 + 32) : 0u;
        float v[64];
        read_s(n, v);
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const bool keep = ((j < 32 ? k0 >> j : k1 >> (j - 32)) & 1u) != 0;
          v[j] = keep ? coef * gb_sigmoid(v[j]) : 0.f;
        }
        store_x(n, v);
      }
      mbar_wait(acc_full, 0);
      tc_fence_after();
      // accumulator lanes are this CTA's negatives
      float* dst0 = p.part + ((int64_t)blockIdx.x * p.Kp + (int64_t)unit * GT + r) * p.Dp;
      for (int cb = part; cb < p.kb; cb += 2) {
        uint32_t a[32], b[32];
        tmem_ld32(tACC + lane_off + cb * 64, a);
        tmem_ld32(tACC + lane_off + cb * 64 + 32, b);
        tmem_ld_wait();
        const int nc = min(64, p.Dp - cb * 64);
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const uint32_t u = j < 32 ? a[j] : b[j - 32];
          if (j < nc) dst0[cb * 64 + j] = __uint_as_float(u);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

// Blocks 0 .. Kp - 1: negative row j (drawn id, or the given one) -> bf16 row j of the table, zeros past k and D.
// Blocks Kp ..: one warp per sequence; lane j % 32 holds negatives j, each of the sequence's ids is broadcast and
// compared, and a ballot per 32 negatives gives one word of the exclusion mask.
struct GbDraw {
  const float* item; int ldi; int64_t n_items; int D, Dp, k, Kp, kw;
  uint64_t seed; const float* step; int draw;
  int64_t* ids; bf16* nb;
  const int64_t* ex_a; int len_a; const int64_t* ex_b; int len_b; int64_t n_seq;
  uint32_t* excl;
};

__global__ void __launch_bounds__(128) gbce_draw_kernel(GbDraw q) {
  const uint64_t seed = mix_seed(q.seed, q.step);
  if ((int)blockIdx.x < q.Kp) {
    const int j = blockIdx.x;
    int64_t id = 0;
    if (j < q.k) {
      id = q.draw ? gb_draw(seed, j, q.n_items) : __ldg(q.ids + j);
      if (q.draw && threadIdx.x == 0) q.ids[j] = id;
    }
    const float* src = q.item + id * q.ldi;
    for (int c = threadIdx.x; c < q.Dp; c += blockDim.x)
      q.nb[(int64_t)j * q.Dp + c] = f2bf(j < q.k && c < q.D ? __ldg(src + c) : 0.f);
    return;
  }
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)(blockIdx.x - q.Kp) * 4 + (threadIdx.x >> 5);
  if (b >= q.n_seq) return;                                     // warp-uniform
  int64_t ng[GB_MAX_K / 32];
  bool hit[GB_MAX_K / 32];
#pragma unroll
  for (int i = 0; i < GB_MAX_K / 32; ++i) {
    const int j = 32 * i + lane;
    ng[i] = j < q.k ? (q.draw ? gb_draw(seed, j, q.n_items) : __ldg(q.ids + j)) : -1;
    hit[i] = false;
  }
  const int tot = q.len_a + q.len_b;
  for (int t0 = 0; t0 < tot; t0 += 32) {
    const int t = t0 + lane;
    int64_t x = -2;
    if (t < q.len_a) x = __ldg(q.ex_a + b * q.len_a + t);
    else if (t < tot) x = __ldg(q.ex_b + b * q.len_b + (t - q.len_a));
    const int cnt = min(32, tot - t0);
    for (int s = 0; s < cnt; ++s) {
      const int64_t y = __shfl_sync(0xffffffffu, x, s);
#pragma unroll
      for (int i = 0; i < GB_MAX_K / 32; ++i) hit[i] |= ng[i] == y;
    }
  }
#pragma unroll
  for (int i = 0; i < GB_MAX_K / 32; ++i) {
    const uint32_t word = __ballot_sync(0xffffffffu, hit[i]);
    if (lane == 0 && i < q.kw) q.excl[b * q.kw + i] = word;
  }
}

// Block j: negative j adds the sum of the partials of every draw of its id (j and its later duplicates, each over the
// splits in order) to d_item[id], unless an earlier draw has the same id and does it.
__global__ void __launch_bounds__(128) gbce_scatter_kernel(const int64_t* ids, int k, const float* part, int n_split, int Kp,
                                                           int Dp, int D, float* d_item, int ldd) {
  __shared__ int64_t sid[GB_MAX_K];
  for (int i = threadIdx.x; i < k; i += blockDim.x) sid[i] = __ldg(ids + i);
  __syncthreads();
  const int j = blockIdx.x;
  const int64_t id = sid[j];
  for (int i = 0; i < j; ++i)
    if (sid[i] == id) return;                                   // block-uniform
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float acc = 0.f;
    for (int jj = j; jj < k; ++jj) {
      if (sid[jj] != id) continue;
#pragma unroll 8
      for (int s = 0; s < n_split; ++s) acc += __ldg(part + ((int64_t)s * Kp + jj) * Dp + c);
    }
    d_item[id * ldd + c] += acc;
  }
}

struct GbPlan { int Kp, n_split, kb, stages; size_t smem; };

int gb_plan(int k, int Dp, int64_t cap_rows, GbPlan& pl) {
  SRFRD_REQUIRE(k >= 1 && k <= GB_MAX_K, "gbce: k = %d negatives outside 1..%d", k, GB_MAX_K);
  SRFRD_REQUIRE(Dp >= 16 && Dp <= 256 && Dp % 16 == 0, "gbce: padded width Dp = %d must be a multiple of 16 in [16, 256]",
                Dp);
  SRFRD_REQUIRE(cap_rows >= 0 && cap_rows < (1ll << 31) - GT, "gbce: cap_rows = %lld out of range", (long long)cap_rows);
  pl.Kp = (k + GT - 1) / GT * GT;
  pl.kb = (Dp + 63) / 64;
  // resident block + X (2 tiles) + barriers + alignment slack; the ring takes the rest, at least two stages
  const size_t fixed = (size_t)(pl.kb + 2) * GTB + 256 + 1024;
  pl.stages = (int)((GB_SMEM_LIMIT - fixed) / ((size_t)pl.kb * GTB));
  if (pl.stages > GB_MAX_STAGES) pl.stages = GB_MAX_STAGES;
  pl.smem = fixed + (size_t)pl.stages * pl.kb * GTB;
  // the dN pass: (Kp / 128) negative blocks x n_split row ranges, about one CTA per SM
  const int nblk = pl.Kp / GT;
  const int n_rt = ceil_div(cap_rows, GT);
  pl.n_split = max(1, min(max(n_rt, 1), num_sms() / nblk));
  return 0;
}

template <int MODE>
int gb_launch(const CUtensorMap& tmH, const CUtensorMap& tmN, const GbParams& p, const GbPlan& pl, cudaStream_t stream) {
  static bool attr = false;
  if (!attr) {
    SRFRD_CUDA(cudaFuncSetAttribute(gbce_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GB_SMEM_LIMIT));
    attr = true;
  }
  const dim3 grid = MODE == GB_DN ? dim3(pl.n_split, pl.Kp / GT) : dim3(ceil_div(p.cap, GT));
  SRFRD_CUDA(launch_pdl(gbce_kernel<MODE>, grid, dim3(GB_THREADS), pl.smem, stream, tmH, tmN, p));
  return 0;
}

}  // namespace
}  // namespace srfrd

extern "C" int srfrd_gbce_plan(int k, int Dp, int64_t cap_rows, int* neg_rows, int* n_split, int64_t* smem_bytes,
                               int* ring_stages) {
  srfrd::GbPlan pl;
  if (int rc = srfrd::gb_plan(k, Dp, cap_rows, pl)) return rc;
  if (neg_rows) *neg_rows = pl.Kp;
  if (n_split) *n_split = pl.n_split;
  if (smem_bytes) *smem_bytes = (int64_t)pl.smem;
  if (ring_stages) *ring_stages = pl.stages;
  return 0;
}

extern "C" int srfrd_gbce_draw(const float* item, int ldi, int64_t n_items, int D, int Dp, int k, uint64_t seed,
                               const float* step, int draw, int64_t* neg_ids, void* neg_bf16, const int64_t* ex_a,
                               int len_a, const int64_t* ex_b, int len_b, int64_t n_seq, uint32_t* excl, void* stream) {
  using namespace srfrd;
  GbPlan pl;
  if (int rc = gb_plan(k, Dp, 0, pl)) return rc;
  SRFRD_REQUIRE(item && neg_ids && neg_bf16, "gbce_draw: null pointer");
  SRFRD_REQUIRE(n_items >= 1 && n_items + 1 < (1ll << 31), "gbce_draw: n_items = %lld out of range", (long long)n_items);
  SRFRD_REQUIRE(D >= 1 && D <= Dp && ldi >= D, "gbce_draw: D = %d, ldi = %d, Dp = %d", D, ldi, Dp);
  SRFRD_REQUIRE(n_seq >= 0 && len_a >= 0 && len_b >= 0, "gbce_draw: negative sizes");
  SRFRD_REQUIRE(n_seq == 0 || (excl && (len_a == 0 || ex_a) && (len_b == 0 || ex_b)), "gbce_draw: null exclusion operand");
  GbDraw q;
  q.item = item; q.ldi = ldi; q.n_items = n_items; q.D = D; q.Dp = Dp; q.k = k; q.Kp = pl.Kp; q.kw = (k + 31) / 32;
  q.seed = seed; q.step = step; q.draw = draw; q.ids = neg_ids; q.nb = reinterpret_cast<bf16*>(neg_bf16);
  q.ex_a = ex_a; q.len_a = len_a; q.ex_b = ex_b; q.len_b = len_b; q.n_seq = n_seq; q.excl = excl;
  const int64_t blocks = pl.Kp + (n_seq + 3) / 4;
  gbce_draw_kernel<<<(unsigned)blocks, 128, 0, (cudaStream_t)stream>>>(q);
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_gbce_loss(const void* h_bf16, int ldh, const void* neg_bf16, const int64_t* neg_ids, int k, int Dp,
                               int D, const float* item, int ldi, int64_t n_items, const int64_t* pos, const float* w_pos,
                               const float* norm, const uint32_t* excl, int L, const int* row_tok, const int* rows_dev,
                               int64_t cap_rows, float beta, float* loss_acc, float* dh, int lddh, float* d_item, int ldd,
                               float* part, void* stream) {
  using namespace srfrd;
  GbPlan pl;
  if (int rc = gb_plan(k, Dp, cap_rows, pl)) return rc;
  SRFRD_REQUIRE(h_bf16 && neg_bf16 && neg_ids && item && pos && norm && loss_acc && dh, "gbce_loss: null pointer");
  SRFRD_REQUIRE(n_items >= 1 && n_items + 1 < (1ll << 31), "gbce_loss: n_items = %lld out of range", (long long)n_items);
  SRFRD_REQUIRE(D >= 1 && D <= Dp && ldi >= D && lddh >= D && ldh >= Dp, "gbce_loss: D = %d, Dp = %d, ldi = %d, lddh = %d, "
                "ldh = %d", D, Dp, ldi, lddh, ldh);
  SRFRD_REQUIRE(!d_item || (ldd >= D && part), "gbce_loss: d_item needs ldd >= D and the partial workspace");
  SRFRD_REQUIRE(L >= 1, "gbce_loss: L = %d", L);
  SRFRD_REQUIRE(!row_tok || rows_dev, "gbce_loss: a row map needs the device row count");
  if (cap_rows == 0) return 0;
  GbParams p = GbParams{};
  p.cap = cap_rows; p.rows_dev = rows_dev; p.row_tok = row_tok; p.pos = pos; p.w_pos = w_pos; p.norm = norm;
  p.excl = excl; p.kw = (k + 31) / 32; p.L = L; p.k = k; p.Kp = pl.Kp; p.n_split = pl.n_split;
  p.Dp = Dp; p.kb = pl.kb; p.stages = pl.stages; p.D = D; p.beta = beta; p.item = item; p.ldi = ldi; p.n_items = n_items;
  p.loss_acc = loss_acc; p.dh = dh; p.lddh = lddh; p.d_item = d_item; p.ldd = ldd; p.part = part;
  CUtensorMap tmH, tmN;
  if (int rc = make_tmap_bf16_2d(&tmH, h_bf16, cap_rows, Dp, ldh, GT, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmN, neg_bf16, pl.Kp, Dp, Dp, GT, 64)) return rc;
  if (int rc = gb_launch<GB_DH>(tmH, tmN, p, pl, (cudaStream_t)stream)) return rc;
  if (!d_item) return 0;
  if (int rc = gb_launch<GB_DN>(tmH, tmN, p, pl, (cudaStream_t)stream)) return rc;
  gbce_scatter_kernel<<<k, 128, 0, (cudaStream_t)stream>>>(neg_ids, k, part, pl.n_split, pl.Kp, Dp, D, d_item, ldd);
  SRFRD_LAUNCH_CHECK();
  return 0;
}
