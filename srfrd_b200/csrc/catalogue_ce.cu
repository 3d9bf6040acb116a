// Full-catalogue softmax cross-entropy on tcgen05: loss = sum_t w_t (LSE_j z_tj - z_t,pos) / sum_t w_t with
// z_tj = <h_t, E_j> over every item j = 1..N (row 0, the pad item, is never a candidate), and its two gradients
//   dh_t = (w_t / sum w) (sum_j p_tj E_j - E_pos),      dE_j = sum_t (w_t / sum w) (p_tj - 1[j = pos_t]) h_t.
// The (rows, N) logits are never written to memory: this is the FlashAttention-2 decomposition of attention_long.cu with
// the item table as keys and values, no mask but the catalogue's ends, scale 1 and many key tiles.  Three passes, each
// a template instance of ONE kernel (warps 0-7: softmax / epilogue, 8: TMA, 9: MMA):
//   CE_LSE  one CTA per 128-row tile of h: S = h E_j^T per 128-item tile into a double-buffered TMEM S, one online
//           (max, exp2-sum) per row and column half; writes LSE and adds sum_t w_t (LSE_t - z_t,pos) to loss_acc[0]
//   CE_DH   one CTA per row tile: S again, X = P - onehot(pos) (bf16, smem), dh_acc += X E_j (TMEM, Dp columns);
//           dh = (w / sum w) dh_acc
//   CE_DE   one CTA per 128-item tile: for every row tile, S, X = (w / sum w)(P - onehot), dE_acc += X^T h_i; the CTA
//           owns its items, so dE is added without atomics and is deterministic
// Every operand moves as [128 rows x 64 columns] bf16 TMA tiles (16 KB, 128-byte swizzle); a streamed tile serves as the
// K-major operand of S and, unchanged, as the MN-major operand of the second product.  One ring stage holds the kb =
// Dp / 64 tiles of one streamed 128-row block.
#include "common.cuh"
#include "srfrd_b200.h"

namespace srfrd {
namespace {

constexpr int CT = 128;                   // rows of a tile: h rows or items
constexpr int CTB = CT * 64 * 2;          // one [128 x 64] bf16 tile
constexpr int CE_THREADS = 320;
constexpr int CE_MAX_STAGES = 8;
constexpr size_t CE_SMEM_LIMIT = 227 * 1024;
constexpr float CE_LOG2E = 1.4426950408889634f;
constexpr float CE_LN2 = 0.6931471805599453f;
enum { CE_LSE = 0, CE_DH = 1, CE_DE = 2 };

struct CeParams {
  int64_t cap;                  // rows of the h buffer
  const int* rows_dev;          // device row count (packed layout) or null: rows = min(cap, *rows_dev)
  const int* row_tok;           // packed layout: dense token of h row r (-1: no token) or null (identity)
  const int64_t* pos;           // target item per dense token
  const float* w_pos;           // weight per dense token, or null -> 1[pos != 0]
  const float* norm;            // norm[0] = sum of the weights (bwd)
  int64_t n_items;              // N: table rows 0..N
  int Dp, kb, stages, D;
  float* lse;                   // (cap) natural log-sum-exp of each row (written by CE_LSE, read by CE_DH / CE_DE)
  float* loss_acc;              // [0] += sum_t w_t (LSE_t - z_t,pos)
  float* dh; int lddh;          // (cap, lddh) fp32, first D columns
  float* d_item; int ldd;       // (N + 1, ldd) fp32, first D columns, added to
};

__device__ __forceinline__ uint32_t ce_sw128(int r, int c) {      // byte offset of (row r, column c) in a swizzled tile
  return (uint32_t)(r * 128 + ((((c >> 3) ^ (r & 7)) << 4) | ((c & 7) << 1)));
}
__device__ __forceinline__ float ce_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void ce_bar(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
// 32 values of row r, 32-column chunk c of the [128 x 128] X -> the swizzled K-major tile pair at `base`
__device__ __forceinline__ void ce_store32(uint8_t* base, int r, int c, const float* v) {
  uint8_t* blk = base + (c >> 1) * CTB;
  const int col0 = (c & 1) * 32;
#pragma unroll
  for (int u = 0; u < 4; ++u)
    *reinterpret_cast<uint4*>(blk + ce_sw128(r, col0 + 8 * u)) =
        make_uint4(pack_bf16x2(v[8 * u], v[8 * u + 1]), pack_bf16x2(v[8 * u + 2], v[8 * u + 3]),
                   pack_bf16x2(v[8 * u + 4], v[8 * u + 5]), pack_bf16x2(v[8 * u + 6], v[8 * u + 7]));
}

__device__ __forceinline__ int ce_rows(const CeParams& p) {
  return (int)(p.rows_dev ? min(p.cap, (int64_t)__ldg(p.rows_dev)) : p.cap);
}
// unnormalised weight of h row r (< rows) and its target; 0 = the row carries no loss term (no token, pos outside 1..N,
// zero weight)
__device__ __forceinline__ float ce_row(const CeParams& p, int64_t r, int64_t& tgt) {
  tgt = 0;
  const int64_t tok = p.row_tok ? (int64_t)__ldg(p.row_tok + r) : r;
  if (tok < 0) return 0.f;
  const int64_t t = __ldg(p.pos + tok);
  if (t < 1 || t > p.n_items) return 0.f;
  const float w = p.w_pos ? __ldg(p.w_pos + tok) : 1.f;
  if (w != 0.f) tgt = t;
  return w;
}

template <int MODE>
__global__ void __launch_bounds__(CE_THREADS, 1)
catalogue_ce_kernel(const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmE, CeParams p) {
  pdl_prologue_done();
  const int rows = ce_rows(p);
  const int n_rt = (rows + CT - 1) / CT;
  const int n_it = (int)((p.n_items + CT) / CT);                // item tiles over table rows 0..N
  const int unit = blockIdx.x;
  if (MODE == CE_DE ? (unit >= n_it || n_rt == 0) : unit >= n_rt) return;     // CTA-uniform, before any barrier
  const int nstream = MODE == CE_DE ? n_rt : n_it;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* res = smem;                                          // resident block: h rows (LSE, DH) or item rows (DE)
  uint8_t* ring = res + p.kb * CTB;                             // stages x kb tiles of the streamed operand
  uint8_t* Xs = ring + p.stages * p.kb * CTB;                   // X [128 x 128] bf16 (DH, DE); LSE: row statistics
  float* xch = reinterpret_cast<float*>(Xs);
  uint64_t* bars = reinterpret_cast<uint64_t*>(Xs + 2 * CTB);
  uint64_t* full = bars;
  uint64_t* empty = bars + p.stages;
  uint64_t* res_full = bars + 2 * p.stages;
  uint64_t* s_full = res_full + 1;                              // [2]
  uint64_t* s_free = res_full + 3;                              // [2]
  uint64_t* x_full = res_full + 5;
  uint64_t* x_free = res_full + 6;
  uint64_t* acc_full = res_full + 7;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_full + 8);
  constexpr uint32_t TMEM_COLS = MODE == CE_LSE ? 256 : 512;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmH); tma_prefetch_desc(&tmE);
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
  const uint32_t tS = tmem_base, tACC = tmem_base + 2 * CT;     // S: 2 x 128 columns; output accumulator: Dp columns

  if (warp == 8) {
    // ---------------------------------------------------------------- TMA producer
    const CUtensorMap* tmRes = MODE == CE_DE ? &tmE : &tmH;
    const CUtensorMap* tmStr = MODE == CE_DE ? &tmH : &tmE;
    if (elect_one()) {
      mbar_expect_tx(res_full, p.kb * CTB);
      for (int kb = 0; kb < p.kb; ++kb) tma_load_2d(res + kb * CTB, tmRes, res_full, kb * 64, unit * CT, SRFRD_EVICT_FIRST);
    }
    __syncwarp();
    int slot = 0; uint32_t ph = 0;
    for (int n = 0; n < nstream; ++n) {
      mbar_wait(&empty[slot], ph ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&full[slot], p.kb * CTB);
        for (int kb = 0; kb < p.kb; ++kb)
          tma_load_2d(ring + (slot * p.kb + kb) * CTB, tmStr, &full[slot], kb * 64, n * CT, SRFRD_EVICT_LAST);
      }
      __syncwarp();
      if (++slot == p.stages) { slot = 0; ph ^= 1; }
    }
  } else if (warp == 9) {
    // ---------------------------------------------------------------- MMA issuer
    const uint32_t idS = umma_idesc_bf16(CT, CT, 0, 0);
    const uint64_t dRes = umma_smem_desc(smem_u32(res), 0, 1024);       // K-major views
    const uint64_t dRing = umma_smem_desc(smem_u32(ring), 0, 1024);
    const uint64_t mRing = umma_smem_desc(smem_u32(ring), CTB, 1024);   // MN-major view of a ring tile (rows = K)
    const uint64_t kX = umma_smem_desc(smem_u32(Xs), 0, 1024);          // X as K-major A (DH: X E)
    const uint64_t mX = umma_smem_desc(smem_u32(Xs), CTB, 1024);        // X^T as MN-major A (DE: X^T h)
    mbar_wait(res_full, 0);
    // second product of streamed block m, whose tiles sit in ring slot st
    auto out_mma = [&](int m, int st) {
      mbar_wait(x_full, m & 1);
      tc_fence_after();
      if (elect_one()) {
        for (int cb = 0; cb < p.kb; ++cb) {
          const int ncols = min(64, p.Dp - cb * 64);
          const uint64_t bq = mRing + (uint64_t)((st * p.kb + cb) * (CTB >> 4));
          if (MODE == CE_DH) {
            const uint32_t id = umma_idesc_bf16(CT, ncols, 0, 1);
#pragma unroll
            for (int ks = 0; ks < 8; ++ks)
              umma_bf16(tACC + cb * 64, kX + (uint64_t)((ks >> 2) * (CTB >> 4) + (ks & 3) * 2), bq + (uint64_t)(ks * 128), id,
                        (m | ks) != 0);
          } else {
            const uint32_t id = umma_idesc_bf16(CT, ncols, 1, 1);
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
      mbar_wait(&s_free[buf], ((n >> 1) & 1) ^ 1);               // the softmax warps have read this S buffer's last use
      mbar_wait(&full[slot], ph);
      tc_fence_after();
      if (elect_one()) {
        for (int kb = 0; kb < p.kb; ++kb) {
          const int ksteps = min(4, (p.Dp - kb * 64) / 16);
          const uint64_t rt = dRes + (uint64_t)(kb * (CTB >> 4));
          const uint64_t st = dRing + (uint64_t)((slot * p.kb + kb) * (CTB >> 4));
          const uint64_t a = MODE == CE_DE ? st : rt, b = MODE == CE_DE ? rt : st;   // A: h rows, B: item rows
          for (int k = 0; k < ksteps; ++k) umma_bf16(tS + buf * CT, a + 2 * k, b + 2 * k, idS, (kb | k) != 0);
        }
        umma_commit(&s_full[buf]);
        if (MODE == CE_LSE) umma_commit(&empty[slot]);
      }
      __syncwarp();
      if (MODE != CE_LSE && n > 0) out_mma(n - 1, prev);          // S of block n runs while X of block n - 1 is formed
      prev = slot;
      if (++slot == p.stages) { slot = 0; ph ^= 1; }
    }
    if (MODE != CE_LSE) {
      out_mma(nstream - 1, prev);
      if (elect_one()) umma_commit(acc_full);
      __syncwarp();
    }
  } else {
    // ---------------------------------------------------------------- softmax (+ epilogue): warp w reads TMEM lanes
    // 32 (w & 3) .. + 31 and the 64 S columns of half `part`
    const int quarter = warp & 3, part = warp >> 2;
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    const int r = quarter * 32 + lane;
    float inv_norm = 0.f;
    if (MODE != CE_LSE) { const float nv = __ldg(p.norm); inv_norm = nv > 0.f ? 1.f / nv : 0.f; }
    // columns [lo, hi) of this half of item block `blk` are items 1..N
    auto item_range = [&](int blk, int& lo, int& hi, int64_t& id0) {
      id0 = (int64_t)blk * CT + part * 64;
      lo = id0 == 0 ? 1 : 0;
      hi = (int)max((int64_t)0, min((int64_t)64, p.n_items + 1 - id0));
    };
    auto read_s = [&](int n, float (&v)[64]) {
      const int buf = n & 1;
      mbar_wait(&s_full[buf], (n >> 1) & 1);
      tc_fence_after();
      uint32_t a[32], b[32];
      tmem_ld32(tS + lane_off + buf * CT + part * 64, a);
      tmem_ld32(tS + lane_off + buf * CT + part * 64 + 32, b);
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
      ce_store32(Xs, r, 2 * part, x);
      ce_store32(Xs, r, 2 * part + 1, x + 32);
      tc_fence_before();
      fence_proxy_async();                                        // generic-proxy smem writes -> visible to the MMA
      __syncwarp();
      if (lane == 0) mbar_arrive(x_full);
    };

    if (MODE == CE_LSE || MODE == CE_DH) {
      const int64_t row = (int64_t)unit * CT + r;
      const bool in = row < rows;
      int64_t tgt = 0;
      const float w = in ? ce_row(p, row, tgt) : 0.f;
      if (MODE == CE_LSE) {
        float m = -INFINITY, s = 0.f, zp = 0.f;                   // running max (log2 units) and sum of this half
        for (int n = 0; n < nstream; ++n) {
          float v[64];
          read_s(n, v);
          int lo, hi; int64_t id0;
          item_range(n, lo, hi, id0);
          float mx = -INFINITY;
#pragma unroll
          for (int j = 0; j < 64; ++j) mx = (j >= lo && j < hi) ? fmaxf(mx, v[j]) : mx;
          if (mx > -INFINITY) {
            const float mn = fmaxf(m, mx * CE_LOG2E);
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < 64; ++j) {
              const float e = ce_ex2(fmaf(v[j], CE_LOG2E, -mn));
              acc += (j >= lo && j < hi) ? e : 0.f;
            }
            s = s * ce_ex2(m - mn) + acc;
            m = mn;
          }
          const int64_t pc = tgt - id0;
          if (pc >= 0 && pc < 64) {
#pragma unroll
            for (int j = 0; j < 64; ++j) zp = (j == (int)pc) ? v[j] : zp;
          }
        }
        xch[(part * 3 + 0) * CT + r] = m;
        xch[(part * 3 + 1) * CT + r] = s;
        xch[(part * 3 + 2) * CT + r] = zp;
        ce_bar(1 + quarter, 64);                                  // the two warps of this lane quarter
        if (part == 0) {
          const float m1 = xch[3 * CT + r], s1 = xch[4 * CT + r], z1 = xch[5 * CT + r];
          const float M = fmaxf(m, m1);
          const float S = (m > -INFINITY ? s * ce_ex2(m - M) : 0.f) + (m1 > -INFINITY ? s1 * ce_ex2(m1 - M) : 0.f);
          const float lse = (M + log2f(S)) * CE_LN2;
          if (in) p.lse[row] = lse;
          const float term = w != 0.f ? w * (lse - (zp + z1)) : 0.f;
          const float tot = warp_sum(term);
          if (lane == 0 && tot != 0.f) red_add_f32(p.loss_acc, tot);
        }
      } else {
        const float lse2 = w != 0.f ? __ldg(p.lse + row) * CE_LOG2E : 0.f;
        for (int n = 0; n < nstream; ++n) {
          float v[64];
          read_s(n, v);
          int lo, hi; int64_t id0;
          item_range(n, lo, hi, id0);
          const int pc = (int)max((int64_t)-1, min((int64_t)64, tgt - id0));
#pragma unroll
          for (int j = 0; j < 64; ++j) {
            const float e = (j >= lo && j < hi) ? ce_ex2(fmaf(v[j], CE_LOG2E, -lse2)) : 0.f;
            v[j] = w != 0.f ? e - (j == pc ? 1.f : 0.f) : 0.f;
          }
          store_x(n, v);
        }
        mbar_wait(acc_full, 0);
        tc_fence_after();
        const float coef = w * inv_norm;
        for (int cb = part; cb < p.kb; cb += 2) {
          uint32_t a[32], b[32];
          tmem_ld32(tACC + lane_off + cb * 64, a);
          tmem_ld32(tACC + lane_off + cb * 64 + 32, b);
          tmem_ld_wait();
          if (in) {
            float* dst = p.dh + row * p.lddh + cb * 64;
            const int nc = min(64, p.D - cb * 64);
#pragma unroll
            for (int j = 0; j < 64; ++j) {
              const uint32_t u = j < 32 ? a[j] : b[j - 32];
              if (j < nc) dst[j] = w != 0.f ? coef * __uint_as_float(u) : 0.f;
            }
          }
        }
      }
    } else {
      // CE_DE: S lanes are the rows of streamed block n, columns this CTA's items
      int lo, hi; int64_t id0;
      item_range(unit, lo, hi, id0);
      for (int n = 0; n < nstream; ++n) {
        const int64_t row = (int64_t)n * CT + r;
        int64_t tgt = 0;
        const float w = row < rows ? ce_row(p, row, tgt) : 0.f;
        const float coef = w * inv_norm;
        const float lse2 = w != 0.f ? __ldg(p.lse + row) * CE_LOG2E : 0.f;
        const int pc = (int)max((int64_t)-1, min((int64_t)64, tgt - id0));
        float v[64];
        read_s(n, v);
#pragma unroll
        for (int j = 0; j < 64; ++j) {
          const float e = (j >= lo && j < hi) ? ce_ex2(fmaf(v[j], CE_LOG2E, -lse2)) : 0.f;
          v[j] = coef != 0.f ? coef * (e - (j == pc ? 1.f : 0.f)) : 0.f;
        }
        store_x(n, v);
      }
      mbar_wait(acc_full, 0);
      tc_fence_after();
      const int64_t item = (int64_t)unit * CT + r;                // accumulator lanes are this CTA's items
      for (int cb = part; cb < p.kb; cb += 2) {
        uint32_t a[32], b[32];
        tmem_ld32(tACC + lane_off + cb * 64, a);
        tmem_ld32(tACC + lane_off + cb * 64 + 32, b);
        tmem_ld_wait();
        if (item >= 1 && item <= p.n_items) {
          float* dst = p.d_item + item * p.ldd + cb * 64;
          const int nc = min(64, p.D - cb * 64);
#pragma unroll
          for (int j = 0; j < 64; ++j) {
            const uint32_t u = j < 32 ? a[j] : b[j - 32];
            if (j < nc) dst[j] += __uint_as_float(u);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
}

struct CePlan { int kb, stages; size_t smem; };

int ce_plan(int Dp, CePlan& pl) {
  SRFRD_REQUIRE(Dp >= 16 && Dp <= 256 && Dp % 16 == 0,
                "catalogue_ce: padded width Dp = %d must be a multiple of 16 in [16, 256]", Dp);
  pl.kb = (Dp + 63) / 64;
  // resident block + X (2 tiles) + barriers + alignment slack; the ring takes the rest, at least two stages
  const size_t fixed = (size_t)(pl.kb + 2) * CTB + 256 + 1024;
  pl.stages = (int)((CE_SMEM_LIMIT - fixed) / ((size_t)pl.kb * CTB));
  if (pl.stages > CE_MAX_STAGES) pl.stages = CE_MAX_STAGES;
  SRFRD_REQUIRE(pl.stages >= 2, "catalogue_ce: Dp = %d leaves %d ring stages (need 2)", Dp, pl.stages);
  pl.smem = fixed + (size_t)pl.stages * pl.kb * CTB;
  return 0;
}

int ce_setup(CeParams& p, CUtensorMap& tmH, CUtensorMap& tmE, CePlan& pl, const void* h, int ldh, const void* table, int ldt,
             int64_t n_items, int Dp, const int64_t* pos, const float* w_pos, const int* row_tok, const int* rows_dev,
             int64_t cap_rows) {
  if (int rc = ce_plan(Dp, pl)) return rc;
  SRFRD_REQUIRE(h && table && pos, "catalogue_ce: null pointer");
  SRFRD_REQUIRE(n_items >= 1 && n_items + 1 < (1ll << 31), "catalogue_ce: n_items = %lld out of range", (long long)n_items);
  SRFRD_REQUIRE(cap_rows >= 0 && cap_rows < (1ll << 31) - CT, "catalogue_ce: cap_rows = %lld out of range",
                (long long)cap_rows);
  SRFRD_REQUIRE(ldh >= Dp && ldt >= Dp, "catalogue_ce: leading dimensions (%d, %d) below Dp = %d", ldh, ldt, Dp);
  SRFRD_REQUIRE(!row_tok || rows_dev, "catalogue_ce: a row map needs the device row count");
  p = CeParams{};
  p.cap = cap_rows; p.rows_dev = rows_dev; p.row_tok = row_tok; p.pos = pos; p.w_pos = w_pos; p.n_items = n_items;
  p.Dp = Dp; p.kb = pl.kb; p.stages = pl.stages;
  if (cap_rows > 0)
    if (int rc = make_tmap_bf16_2d(&tmH, h, cap_rows, Dp, ldh, CT, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmE, table, n_items + 1, Dp, ldt, CT, 64)) return rc;
  return 0;
}

template <int MODE>
int ce_launch(const CUtensorMap& tmH, const CUtensorMap& tmE, const CeParams& p, const CePlan& pl, cudaStream_t stream) {
  static bool attr = false;
  if (!attr) {
    SRFRD_CUDA(cudaFuncSetAttribute(catalogue_ce_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CE_SMEM_LIMIT));
    attr = true;
  }
  const int grid = MODE == CE_DE ? ceil_div(p.n_items + 1, CT) : ceil_div(p.cap, CT);
  SRFRD_CUDA(launch_pdl(catalogue_ce_kernel<MODE>, dim3(grid), dim3(CE_THREADS), pl.smem, stream, tmH, tmE, p));
  return 0;
}

}  // namespace
}  // namespace srfrd

extern "C" int srfrd_catalogue_ce_plan(int Dp, int64_t* smem_bytes, int* ring_stages, int* tmem_cols) {
  srfrd::CePlan pl;
  if (int rc = srfrd::ce_plan(Dp, pl)) return rc;
  if (smem_bytes) *smem_bytes = (int64_t)pl.smem;
  if (ring_stages) *ring_stages = pl.stages;
  if (tmem_cols) *tmem_cols = 512;
  return 0;
}

extern "C" int srfrd_catalogue_ce_fwd(const void* h_bf16, int ldh, const void* table_bf16, int ldt, int64_t n_items, int Dp,
                                      const int64_t* pos, const float* w_pos, const int* row_tok, const int* rows_dev,
                                      int64_t cap_rows, float* lse, float* loss_acc, void* stream) {
  using namespace srfrd;
  CeParams p; CePlan pl; CUtensorMap tmH, tmE;
  if (int rc = ce_setup(p, tmH, tmE, pl, h_bf16, ldh, table_bf16, ldt, n_items, Dp, pos, w_pos, row_tok, rows_dev, cap_rows))
    return rc;
  SRFRD_REQUIRE(lse && loss_acc, "catalogue_ce_fwd: null output");
  if (cap_rows == 0) return 0;
  p.lse = lse; p.loss_acc = loss_acc;
  return ce_launch<CE_LSE>(tmH, tmE, p, pl, (cudaStream_t)stream);
}

extern "C" int srfrd_catalogue_ce_bwd(const void* h_bf16, int ldh, const void* table_bf16, int ldt, int64_t n_items, int Dp,
                                      int D, const int64_t* pos, const float* w_pos, const float* norm, const int* row_tok,
                                      const int* rows_dev, int64_t cap_rows, const float* lse, float* dh, int lddh,
                                      float* d_item, int ldd, void* stream) {
  using namespace srfrd;
  CeParams p; CePlan pl; CUtensorMap tmH, tmE;
  if (int rc = ce_setup(p, tmH, tmE, pl, h_bf16, ldh, table_bf16, ldt, n_items, Dp, pos, w_pos, row_tok, rows_dev, cap_rows))
    return rc;
  SRFRD_REQUIRE(lse && norm, "catalogue_ce_bwd: null lse / norm");
  SRFRD_REQUIRE(D >= 1 && D <= Dp, "catalogue_ce_bwd: D = %d outside 1..Dp = %d", D, Dp);
  SRFRD_REQUIRE(!dh || lddh >= D, "catalogue_ce_bwd: lddh = %d below D = %d", lddh, D);
  SRFRD_REQUIRE(!d_item || ldd >= D, "catalogue_ce_bwd: ldd = %d below D = %d", ldd, D);
  if (cap_rows == 0) return 0;
  p.lse = const_cast<float*>(lse); p.norm = norm; p.D = D;
  p.dh = dh; p.lddh = lddh; p.d_item = d_item; p.ldd = ldd;
  if (dh)
    if (int rc = ce_launch<CE_DH>(tmH, tmE, p, pl, (cudaStream_t)stream)) return rc;
  if (d_item)
    if (int rc = ce_launch<CE_DE>(tmH, tmE, p, pl, (cudaStream_t)stream)) return rc;
  return 0;
}
