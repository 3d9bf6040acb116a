// tcgen05 / TMEM / TMA GEMMs for the encoder's dense contractions (SURVEY.md 2.3 rows k2-k4, k7).
//
//  gemm_tn   : C[M,N] = epilogue(A[M,K] * B[N,K]^T)   both operands K-major (row-major, K contiguous)
//              forward linears (A = activations, B = weight (out,in)) and data-gradients
//              (A = dY, B = W^T shadow).  Persistent CTAs, 128-row tiles, 640 threads (roles at the kernel), optional
//              LayerNorm of the result row folded into the epilogue.
//  gemm_wgrad: dW[Mo,No] += sum_t A[t,Mo] * B[t,No]   both operands MN-major (token index = K)
//              weight gradients, split-K over tokens, 16-byte vector red.add into the flat fp32 gradient buffer.
//              192 threads: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue
//              (TMEM lane quarter = warp_idx & 3).
#include <stdlib.h>

#include "common.cuh"
#include "srfrd_b200.h"

namespace srfrd {

// ffn.cu: the lean one-tile-per-CTA path for small inputs (see srfrd_gemm_tn)
bool gemm_small_eligible(int M, int N, int K, const srfrd_gemm_epilogue_t* ep, int lda, int ldb);
int gemm_small_launch(const void* A, int lda, const void* B, int ldb, int M, int N, int K, const srfrd_gemm_epilogue_t* ep,
                      cudaStream_t stream);

static constexpr int BLOCK_M = 128;
static constexpr int BLOCK_K = 64;                       // 64 bf16 = one 128-byte swizzle row
static constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB
static constexpr int GEMM_THREADS = 192;                 // gemm_wgrad
static constexpr int TN_THREADS = 640;                   // gemm_tn: 2 epilogue sets of 8 warps + 4 control warps
static constexpr int TMEM_COLS = 512;
static constexpr int EPI_BLK_BYTES = BLOCK_M * 64 * 2;   // one [128 rows x 64 cols] bf16 epilogue block, 16 KB
static constexpr int TN_MAX_BLOCK_N = 192;               // <= 3 epilogue blocks per tile and per set
static constexpr int MAX_BIAS = 1024;
static constexpr int MAX_LN = 128;                       // widest row of the fused LayerNorm epilogue (two staging blocks x 2)

struct GemmEpilogue {
  const float* bias;        // [N] or null
  const bf16* residual;     // [M, ldr] or null
  const bf16* gate;         // [M, ldg] or null : v *= (gate > 0)      (ReLU backward)
  const int64_t* row_ids;   // [M] or null      : v *= (row_ids[m] != 0) (pad re-mask, SRFR_model.py:121)
  bf16* out_bf16;           // [M, ldc] or null
  float* out_f32;           // [M, ldc] or null
  int ldr, ldg, ldc;
  int relu;
  uint64_t drop_seed;       // dropout (drop_thresh == 0 -> off): v = keep ? v * drop_scale : 0
  uint32_t drop_thresh, drop_stream;
  float drop_scale;
  const float* drop_step;
  const float* ln_w;        // fused LayerNorm of the result row (LNF kernels): weight / bias [N], stats [M, 2] or null
  const float* ln_b;
  float* ln_stats;
  float ln_eps;
};

// profiling experiments only (SRFRD_GEMM_DEBUG=5): clock64 timeline of CTA 0, [event][tile], read by srfrd_gemm_debug_read
__device__ long long g_gemm_dbg[32 * 16];
__device__ long long g_gemm_cta[2 * 160];     // per-CTA start / end globaltimer (SRFRD_GEMM_DEBUG=5); end stamp | smid << 48
#define TN_STAMP(ev, tile) do { if (s.debug == 5 && blockIdx.x == 0 && (tile) < 16) { if (elect_one()) g_gemm_dbg[(ev) * 16 + (tile)] = clock64(); } } while (0)

struct GemmShape {
  const int* rows_dev;      // dynamic row count: M = min(M, *rows_dev) (packed token layout), or null
  int M, N, K;
  int block_n, m_tiles, n_tiles, stages;
  int has_aux;              // residual or gate present: the tile's aux block(s) arrive by TMA in the set's tile buffer
  int tma_out;              // bf16 output written IN PLACE over the aux block(s) and stored with TMA
  int buf_blocks;           // 64-column blocks per set's tile buffer (0 if neither aux nor TMA output)
  int debug;                // SRFRD_GEMM_DEBUG (profiling experiments only): 1 = no TMA store, 2 = no epilogue math, 5 = timeline
  int b_resident;           // the whole B operand (one column tile, all K blocks) is loaded once and stays in shared memory
  int sched_slot;           // which {next tile, CTAs done} pair of g_tn_sched this launch uses
  int kgroup;               // K blocks per pipeline stage / barrier (resident B, K <= 192: the whole K in one stage)
  int nacc;                 // TMEM accumulator stages: 4 x 128 columns when the tile is <= 128 wide, else 2 x 256
  int dynamic;              // draw tile ids from the atomic counter (experiment switch, see the producer warp)
  int l2_prefetch;          // TMA-prefetch the residual / gate tile (and the next A tile) into L2 ahead of the real load
  int nbuf;                 // tile buffers: 2 (one per epilogue set) or 4 (two per set: residual prefetch and the TMA store's
                            // read latency leave the epilogue's chain); tile n uses buffer n % nbuf
};

// Dynamic tile scheduler state (SRFRD_GEMM_DYNAMIC=1, off by default: no measured gain).  Per-CTA durations on identical
// work spread by up to 40 % (per-SM globaltimer stamps; whole GPCs are slower than others).  The last CTA to exit resets
// its pair; launches rotate through the pairs so that kernels running concurrently on two streams never share one.
static constexpr int TN_SCHED_SLOTS = 64;
__device__ int g_tn_sched[TN_SCHED_SLOTS * 2];
static constexpr int TN_RING = 16;                       // tile-id ring between the producer and the other warps

// byte offset of the 16-byte chunk j (8 bf16 columns) of row r inside a 128-byte-swizzled [128 x 64] bf16 block
__device__ __forceinline__ uint32_t sw128_chunk(int r, int j) { return (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4)); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tmap, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tmap),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

// C = epilogue(A B^T).  Persistent CTAs over 128-row tiles.  All global traffic is asynchronous bulk copies:
// A / B tiles and the residual-or-gate ("aux") tile arrive by TMA, the bf16 result is written IN PLACE over the
// aux tile (same thread, same 16-byte chunk) and leaves by TMA stores, so the epilogue threads only touch TMEM
// and shared memory and nothing in the per-tile critical path waits on an HBM round trip.
//   warps 0..7 / 8..15: epilogue set 0 / 1 (tiles alternate between the sets).  Tile n uses accumulator stage n % nacc
//     (4 x 128 TMEM columns for tiles <= 128 wide, else 2 x 256) and tile buffer n % nbuf (2, or 4 for residual / gate
//     tiles: the store of a tile is then only waited for when the set issues its NEXT store).  Warp (quarter q, half h)
//     owns TMEM lanes [32q, 32q+32) and the 32-column chunks with chunk % 2 == h.  Four epilogue warps per scheduler:
//     measured, the epilogue is a chain of TMEM / barrier latencies, not bandwidth.
//   warp 16: TMA producer for A (and B: loaded once and kept when there is one column tile and K <= 192, else per stage);
//            publishes the tile ids in a small ring (static round-robin order; an atomic counter behind a switch)
//   warp 17: TMEM allocator + MMA issuer   warp 19: second MMA issuer (alternate tiles) when a stage holds a tile's whole K
//   warp 18: TMA producer for the aux tile, L2-prefetched as soon as the tile id is known
//     The control warps have the HIGHEST warp ids: the scheduler favours high ids, and with low ids the MMA issuer
//     took ~700 cycles to issue five MMAs while the epilogue warps of its scheduler were busy (clock64 timeline).
// AUX: 0 none, 1 residual (v += aux), 2 gate (v = aux > 0 ? v : 0).  bias / ReLU / row mask are branch-free.
// LNF: the LayerNorm that follows the residual add is computed in the epilogue.  While packing its columns to bf16 a
// thread accumulates sum and sum of squares of the ROUNDED values (what a separate LayerNorm kernel would read back);
// the two warps of a row exchange them through shared memory at the set's named barrier; each thread then re-reads its
// own chunks from the staging buffer, normalises them into a second staging buffer and a second TMA store writes it.
template <int AUX, bool DROP, bool LNF>
__global__ void __launch_bounds__(TN_THREADS, 1)
gemm_tn_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmAux, const __grid_constant__ CUtensorMap tmOut,
               const __grid_constant__ CUtensorMap tmLn, GemmShape s, GemmEpilogue e) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int b_stage_bytes = ((s.block_n * BLOCK_K * 2) + 1023) & ~1023;
  uint8_t* smA = smem;
  const int kblocks = (s.K + BLOCK_K - 1) / BLOCK_K;
  const int a_stage_bytes = s.kgroup * A_STAGE_BYTES;
  uint8_t* smB = smA + s.stages * a_stage_bytes;         // [stages] or, resident, [kblocks]
  uint8_t* smBuf = smB + (s.b_resident ? kblocks : s.stages) * b_stage_bytes;   // [set][buf_blocks][16 KB]
  uint8_t* smY = smBuf + s.nbuf * s.buf_blocks * EPI_BLK_BYTES;   // LNF: [set][buf_blocks][16 KB] LayerNorm output staging
  float* sbias = reinterpret_cast<float*>(smY + (LNF ? 2 * s.buf_blocks * EPI_BLK_BYTES : 0));
  float* sln = sbias + MAX_BIAS;                             // LNF: weight [MAX_LN], bias [MAX_LN]
  float* sxch = sln + (LNF ? 2 * MAX_LN : 0);                // LNF: [set][half][128 rows] (sum, sum of squares)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sxch + (LNF ? 2 * 2 * BLOCK_M * 2 : 0));
  uint64_t* full = bars;
  uint64_t* empty = bars + s.stages;
  uint64_t* tfull = bars + 2 * s.stages;
  uint64_t* tempty = tfull + 4;                          // [nacc <= 4] accumulator stages (tile tl uses stage tl % nacc)
  uint64_t* xfull = tempty + 4;                          // [nbuf <= 4] aux tile landed
  uint64_t* bfree = xfull + 4;                           // [nbuf] tile buffer free again (TMA store has read it)
  uint64_t* sfull = bfree + 4;                           // [TN_RING] tile id published
  uint64_t* bres = sfull + TN_RING;                      // resident B landed
  int* ring = reinterpret_cast<int*>(bres + 1);          // [TN_RING] tile ids, -1 = no more tiles
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ring + TN_RING);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* sched = g_tn_sched + 2 * s.sched_slot;

  if (warp == 16) {                                      // barrier initialisation spread over the lanes
    if (lane == 0) {
      tma_prefetch_desc(&tmA);
      tma_prefetch_desc(&tmB);
      if (s.has_aux) tma_prefetch_desc(&tmAux);
      if (s.tma_out) tma_prefetch_desc(&tmOut);
      if (LNF) tma_prefetch_desc(&tmLn);
    }
    if (lane < s.stages) { mbar_init(&full[lane], 1); mbar_init(&empty[lane], 1); }
    if (lane >= 8 && lane < 12) {
      const int i = lane - 8;
      mbar_init(&xfull[i], 1); mbar_init(&bfree[i], 1);
    }
    if (lane >= 12 && lane < 16) { mbar_init(&tfull[lane - 12], 1); mbar_init(&tempty[lane - 12], 8); }
    if (lane >= 16) mbar_init(&sfull[lane - 16], 1);
    if (lane == 10) mbar_init(bres, 1);
    fence_barrier_init();
  }
  if (s.debug == 5 && threadIdx.x == 0) {
    unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    if (blockIdx.x == 0) { g_gemm_dbg[10 * 16] = (long long)gt; g_gemm_dbg[10 * 16 + 1] = clock64(); }
    if (blockIdx.x < 160) g_gemm_cta[2 * blockIdx.x] = (long long)gt;
  }
  if (warp == 17) { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  pdl_prologue_done();                                   // everything below may read what earlier kernels wrote
  if (s.rows_dev) {                                      // data-dependent row count (packed layout): capacity stays static
    s.M = min(s.M, __ldg(s.rows_dev));
    s.m_tiles = (s.M + BLOCK_M - 1) / BLOCK_M;
  }
  const int total_tiles = s.m_tiles * s.n_tiles;
  for (int i = threadIdx.x; i < MAX_BIAS; i += blockDim.x) sbias[i] = (e.bias && i < s.N) ? __ldg(e.bias + i) : 0.f;
  if (LNF) {
    for (int i = threadIdx.x; i < MAX_LN; i += blockDim.x) {
      sln[i] = i < s.N ? __ldg(e.ln_w + i) : 0.f;
      sln[MAX_LN + i] = i < s.N ? __ldg(e.ln_b + i) : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Warps 16..18 stay converged; only the issuing instructions are predicated on elect.sync so that barrier
  // addresses and descriptors live in uniform registers (see topk.cu for the measurement behind this).
  if (warp == 16) {
    int stage = 0; uint32_t phase = 0;
    if (s.b_resident) {
      if (elect_one()) {
        mbar_expect_tx(bres, kblocks * s.block_n * BLOCK_K * 2);
        for (int kb = 0; kb < kblocks; ++kb)
          tma_load_2d(smB + kb * b_stage_bytes, &tmB, bres, kb * BLOCK_K, 0, SRFRD_EVICT_LAST);
      }
      __syncwarp();
    }
    // Tile ids travel to the other warps through a small ring (one mbarrier per entry, -1 = end).  The producer fills it
    // with the static round-robin order; SRFRD_GEMM_DYNAMIC=1 draws the ids from an atomic counter instead (first two
    // tiles static).  Measured at C2 the dynamic order gains nothing: a tile has to be claimed when its loads are issued,
    // 4-6 tiles before it completes, which is as long as the imbalance it could correct.
    int t = blockIdx.x, t1 = blockIdx.x + (int)gridDim.x;
    if (t >= total_tiles) t = -1;                        // (dynamic row count: this CTA may have nothing to do)
    if (t1 >= total_tiles) t1 = -1;
    for (int tl = 0;; ++tl) {
      int fetched = -1;
      if (lane == 0) {
        if (t >= 0 && t1 >= 0) fetched = s.dynamic ? atomicAdd(sched, 1) + 2 * (int)gridDim.x : t1 + (int)gridDim.x;
        ring[tl & (TN_RING - 1)] = t;
        mbar_arrive(&sfull[tl & (TN_RING - 1)]);
        if (t < 0) {                                     // end marker twice: each epilogue set reads every other entry
          ring[(tl + 1) & (TN_RING - 1)] = -1;
          mbar_arrive(&sfull[(tl + 1) & (TN_RING - 1)]);
        }
      }
      __syncwarp();
      if (t < 0) break;
      const int m0 = (t / s.n_tiles) * BLOCK_M, n0 = (t % s.n_tiles) * s.block_n;
      for (int kb = 0; kb < kblocks; kb += s.kgroup) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (kb == 0) TN_STAMP(0, tl);
        if (elect_one()) {
          if (s.b_resident) {
            const int ng = min(s.kgroup, kblocks - kb);
            mbar_expect_tx(&full[stage], ng * A_STAGE_BYTES);
            for (int j = 0; j < ng; ++j)
              tma_load_2d(smA + stage * a_stage_bytes + j * A_STAGE_BYTES, &tmA, &full[stage], (kb + j) * BLOCK_K, m0,
                          SRFRD_EVICT_FIRST);
          } else {
            mbar_expect_tx(&full[stage], A_STAGE_BYTES + s.block_n * BLOCK_K * 2);
            tma_load_2d(smA + stage * A_STAGE_BYTES, &tmA, &full[stage], kb * BLOCK_K, m0, SRFRD_EVICT_FIRST);
            tma_load_2d(smB + stage * b_stage_bytes, &tmB, &full[stage], kb * BLOCK_K, n0, SRFRD_EVICT_LAST);
          }
        }
        __syncwarp();
        if (++stage == s.stages) { stage = 0; phase ^= 1; }
      }
      if (s.l2_prefetch && s.stages * s.kgroup < 2 * kblocks + 2 && t1 >= 0 && elect_one()) {   // shallow A pipeline (fused LN)
        const int m1 = (t1 / s.n_tiles) * BLOCK_M;
        for (int kb = 0; kb < kblocks; ++kb) tma_prefetch_l2_2d(&tmA, kb * BLOCK_K, m1);
      }
      __syncwarp();
      t = t1;
      t1 = __shfl_sync(0xffffffffu, fetched, 0);
      if (t1 >= total_tiles) t1 = -1;
    }
  } else if (warp == 17 || warp == 19) {
    // MMA issuers.  The per-tile issue chain (barrier tests, five MMAs, two commits: ~1 650 cycles, clock64 timeline) was
    // the CTA's critical path, so with one stage per tile and an even number of stages two warps take alternate tiles:
    // issuer p owns accumulator stage p and the stages of equal parity, so every barrier still has a single waiter.
    const bool two = (s.kgroup * 1 >= kblocks) && (s.stages % 2 == 0);
    const int p = warp == 19 ? 1 : 0, step = two ? 2 : 1;
    if (two || p == 0) {
      const uint64_t adesc0 = umma_smem_desc(smem_u32(smA), 0, 1024), bdesc0 = umma_smem_desc(smem_u32(smB), 0, 1024);
      if (s.b_resident) { mbar_wait(bres, 0); tc_fence_after(); }
      mbar_wait(&sfull[p], 0);
      int t = ring[p];
      int stage = two ? p : 0; uint32_t phase = 0;
      const int acc_cols = 512 / s.nacc;
      for (int tl = p; t >= 0; tl += step) {
        const int as = tl % s.nacc;                      // accumulator stage: up to nacc - 1 tiles ahead of the epilogues
        const uint32_t aphase = (tl / s.nacc) & 1;
        const int n0 = (t % s.n_tiles) * s.block_n;
        int bn = min(s.block_n, s.N - n0);
        bn = (bn + 15) & ~15;
        const uint32_t idesc = umma_idesc_bf16(BLOCK_M, bn, 0, 0);
        // this issuer's next ring entry is published once the loads of the tile before it are issued, which never waits
        // on this tile: one overlapped test for the ring entry, the accumulator stage and the operands
        // (only with one stage per tile: otherwise the producer may need this tile's stages back before it can finish
        // issuing the tile, and the next entry is read after the last K block instead)
        const int nx = tl + step;
        const bool merged = s.kgroup >= kblocks;
        if (merged) {
          mbar_wait3(&sfull[nx & (TN_RING - 1)], (nx / TN_RING) & 1, &tempty[as], aphase ^ 1, &full[stage], phase);
          t = ring[nx & (TN_RING - 1)];
        } else {
          mbar_wait2(&tempty[as], aphase ^ 1, &full[stage], phase);
        }
        tc_fence_after();
        TN_STAMP(1, tl);
        const uint32_t tacc = tmem_base + as * acc_cols;
        for (int kb = 0; kb < kblocks; kb += s.kgroup) {
          if (kb) mbar_wait(&full[stage], phase);
          tc_fence_after();
          if (kb == 0) TN_STAMP(2, tl);
          const bool last = kb + s.kgroup >= kblocks;
          if (last) TN_STAMP(3, tl);
          if (elect_one()) {
            for (int j = 0; j < s.kgroup && kb + j < kblocks; ++j) {
              // K-major SW128: 8-row groups are 1024 B apart (SBO); +32 B (= 2 in descriptor units) per UMMA_K = 16
              const uint64_t ad = adesc0 + (uint64_t)((stage * a_stage_bytes + j * A_STAGE_BYTES) >> 4);
              const uint64_t bd = bdesc0 + (uint64_t)((s.b_resident ? kb + j : stage) * (b_stage_bytes >> 4));
              const int ksteps = min(BLOCK_K / 16, (s.K - (kb + j) * BLOCK_K + 15) / 16);
#pragma unroll
              for (int k = 0; k < BLOCK_K / 16; ++k)
                if (k < ksteps) umma_bf16(tacc, ad + 2 * k, bd + 2 * k, idesc, ((kb + j) | k) != 0);
            }
            umma_commit(&empty[stage]);
            if (last) umma_commit(&tfull[as]);
          }
          __syncwarp();
          if (two) { stage += 2; if (stage >= s.stages) { stage -= s.stages; phase ^= 1; } }
          else if (++stage == s.stages) { stage = 0; phase ^= 1; }
        }
        if (!merged) {
          mbar_wait(&sfull[nx & (TN_RING - 1)], (nx / TN_RING) & 1);
          t = ring[nx & (TN_RING - 1)];
        }
      }
    }
  } else if (warp == 18) {
    if (AUX) {
      for (int n_local = 0;; ++n_local) {
        mbar_wait(&sfull[n_local & (TN_RING - 1)], (n_local / TN_RING) & 1);
        const int t = ring[n_local & (TN_RING - 1)];
        if (t < 0) break;
        const int m0 = (t / s.n_tiles) * BLOCK_M, n0 = (t % s.n_tiles) * s.block_n;
        const int nblk = (min(s.block_n, s.N - n0) + 63) >> 6;
        const int b = n_local % s.nbuf;
        const uint32_t bph = (n_local / s.nbuf) & 1;       // use count of buffer b -> parity
        // The tile id is known several tiles before the buffer is free again: pull the tile into L2 now, so that the
        // load issued once the buffer is free costs an L2 hit instead of an HBM round trip in the epilogue's chain.
        if (s.l2_prefetch && elect_one())
          for (int blk = 0; blk < nblk; ++blk) tma_prefetch_l2_2d(&tmAux, n0 + blk * 64, m0);
        __syncwarp();
        mbar_wait(&bfree[b], bph ^ 1);                   // first use of a buffer: passes at once (fresh barrier)
        if (elect_one()) {
          mbar_expect_tx(&xfull[b], nblk * EPI_BLK_BYTES);
          for (int blk = 0; blk < nblk; ++blk)
            tma_load_2d(smBuf + (b * s.buf_blocks + blk) * EPI_BLK_BYTES, &tmAux, &xfull[b], n0 + blk * 64, m0,
                        SRFRD_EVICT_FIRST);
        }
        __syncwarp();
      }
    }
  } else if (warp < 16) {
    const int set = warp >> 3, quarter = warp & 3, half = (warp >> 2) & 1;
    const int r = quarter * 32 + lane;                   // row inside the tile == TMEM lane
    const bool issuer = (quarter == 0) && (half == 0) && (lane == 0);
    const bool stamp = (quarter == 0) && (half == 0);
    const bool use_buf = AUX || s.tma_out;
    int pending_b = -1;                                  // issuer, nbuf == 4: buffer whose TMA store may still be reading
    if (DROP) e.drop_seed = mix_seed(e.drop_seed, e.drop_step);
    const float relu_floor = e.relu ? 0.f : -INFINITY;
    for (int n_local = set;; n_local += 2) {             // tiles alternate between the sets
      mbar_wait(&sfull[n_local & (TN_RING - 1)], (n_local / TN_RING) & 1);
      const int t = ring[n_local & (TN_RING - 1)];
      if (t < 0) break;
      const int m0 = (t / s.n_tiles) * BLOCK_M, n0 = (t % s.n_tiles) * s.block_n;
      const int bn = min(s.block_n, s.N - n0);           // multiple of 16
      const int nblk = (bn + 63) >> 6;
      const int row = m0 + r;
      const bool row_ok = row < s.M;
      float rowm = 1.f;
      if (e.row_ids && row_ok) rowm = (__ldg(e.row_ids + row) != 0) ? 1.f : 0.f;
      if (stamp) TN_STAMP(4, n_local);
      // accumulator ready AND (aux tile landed, which implies the buffer was free | previous store has read the buffer)
      const int as = n_local % s.nacc;
      const uint32_t aph = (n_local / s.nacc) & 1;
      const int b = n_local % s.nbuf;                    // tile buffer (nbuf even: a buffer always belongs to one set)
      const uint32_t tph = (n_local / s.nbuf) & 1;       // its use count -> parity
      uint8_t* buf = smBuf + b * s.buf_blocks * EPI_BLK_BYTES;
      if (AUX) mbar_wait2(&tfull[as], aph, &xfull[b], tph);
      else if (s.tma_out) mbar_wait2(&tfull[as], aph, &bfree[b], tph ^ 1);
      else mbar_wait(&tfull[as], aph);
      tc_fence_after();
      if (stamp) TN_STAMP(5, n_local);
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + as * (512 / s.nacc);
      float ln_sum = 0.f, ln_sq = 0.f;
      if (s.debug != 2) {
#pragma unroll 1
        for (int c = half * 32; c < bn; c += 64) {       // this warp's 32-column chunks of the tile
          uint8_t* blkp = buf + (c >> 6) * EPI_BLK_BYTES;
          const int cj = (c & 63) >> 3;                  // first 16-byte chunk inside the 64-column block
          uint32_t raw[32];
          tmem_ld32(taddr + c, raw);
          uint4 ax[4];
          if (AUX) {
#pragma unroll
            for (int j = 0; j < 4; ++j) ax[j] = *reinterpret_cast<const uint4*>(blkp + sw128_chunk(r, cj + j));
          }
          const int nc = n0 + c;
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (c + 8 * j >= bn) break;                  // bn is a multiple of 16: chunks come in pairs
            float v[8], a[8];
            if (AUX) unpack_bf16x8(ax[j], a);
            const float4 b0 = *reinterpret_cast<const float4*>(sbias + nc + 8 * j);
            const float4 b1 = *reinterpret_cast<const float4*>(sbias + nc + 8 * j + 4);
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float x = __uint_as_float(raw[8 * j + i]) + bb[i];
              if (DROP) {
                const int n = nc + 8 * j + i;
                x = dropout_keep(e.drop_seed, e.drop_stream, (uint64_t)row * (uint64_t)s.N + (uint64_t)n, e.drop_thresh)
                        ? x * e.drop_scale : 0.f;
              }
              x = fmaxf(x, relu_floor);
              if (AUX == 2) x = a[i] > 0.f ? x : 0.f;
              if (AUX == 1) x += a[i];
              v[i] = x * rowm;
            }
            if (s.tma_out) {
              const uint4 pk = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
              *reinterpret_cast<uint4*>(blkp + sw128_chunk(r, cj + j)) = pk;
              if (LNF) lnf_accum8(pk, ln_sum, ln_sq);    // row statistics of the ROUNDED values (common.cuh)
            } else if (row_ok) {
              const int n = nc + 8 * j;
              if (e.out_bf16)
                *reinterpret_cast<uint4*>(e.out_bf16 + (size_t)row * e.ldc + n) =
                    make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
              if (e.out_f32) {
                float4* o = reinterpret_cast<float4*>(e.out_f32 + (size_t)row * e.ldc + n);
                o[0] = make_float4(v[0], v[1], v[2], v[3]);
                o[1] = make_float4(v[4], v[5], v[6], v[7]);
              }
            }
          }
        }
      }
      if (stamp) TN_STAMP(6, n_local);
      tc_fence_before();                                 // accumulator fully read: hand the TMEM stage back
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
      if (use_buf) {
        if (s.tma_out) fence_proxy_async();              // generic-proxy smem writes -> visible to the TMA store
        if (LNF) *reinterpret_cast<float2*>(sxch + ((set * 2 + half) * BLOCK_M + r) * 2) = make_float2(ln_sum, ln_sq);
        if (stamp) TN_STAMP(7, n_local);
        named_bar_sync(1 + set, 256);                    // every warp of the set is done with the tile buffer
        if (stamp) TN_STAMP(8, n_local);
        if (LNF) {
          if (issuer && s.debug != 1) {                  // x leaves while the row statistics are computed
            for (int blk = 0; blk < nblk; ++blk) tma_store_2d(&tmOut, buf + blk * EPI_BLK_BYTES, n0 + blk * 64, m0);
            bulk_commit();
          }
          uint8_t* ybuf = smY + set * s.buf_blocks * EPI_BLK_BYTES;
          // one-pass statistics: the two warps of a row exchange (sum, sum of squares) of their columns
          const float2 other = *reinterpret_cast<const float2*>(sxch + ((set * 2 + (half ^ 1)) * BLOCK_M + r) * 2);
          float mean, rstd, nb;
          lnf_stats(ln_sum, ln_sq, other.x, other.y, bn, e.ln_eps, mean, rstd, nb);
#pragma unroll 1
          for (int c = half * 32; c < bn; c += 64) {
            const int cj = (c & 63) >> 3;
            const uint32_t boff = (uint32_t)((c >> 6) * EPI_BLK_BYTES);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (c + 8 * j >= bn) break;
              const uint32_t off = boff + sw128_chunk(r, cj + j);
              const float* w = sln + c + 8 * j;
              *reinterpret_cast<uint4*>(ybuf + off) =
                  lnf_apply8(*reinterpret_cast<const uint4*>(buf + off), rstd, nb, w, w + MAX_LN);
            }
          }
          if (half == 0 && row_ok && e.ln_stats) *reinterpret_cast<float2*>(e.ln_stats + 2 * (size_t)row) = make_float2(mean, rstd);
          fence_proxy_async();
          named_bar_sync(1 + set, 256);                  // LayerNorm rows complete in the second staging buffer
          if (issuer) {
            if (s.debug != 1) {
              for (int blk = 0; blk < nblk; ++blk) tma_store_2d(&tmLn, ybuf + blk * EPI_BLK_BYTES, n0 + blk * 64, m0);
              bulk_commit();
              bulk_wait_read<0>();                       // both stores have read their buffers
            }
            mbar_arrive(&bfree[b]);
          }
          __syncwarp();
        } else {
        if (issuer) {
          if (s.nbuf == 4 && s.tma_out) {
            // two buffers per set: do not wait for THIS store to read its buffer (1 300 - 1 800 cycles, during which the
            // whole set would stand at its next named barrier); the set's previous store has long finished -- release
            // that buffer now.  It is next needed four tiles after its use, i.e. by the set's tile after next.
            if (s.debug != 1) {
              for (int blk = 0; blk < nblk; ++blk) tma_store_2d(&tmOut, buf + blk * EPI_BLK_BYTES, n0 + blk * 64, m0);
              bulk_commit();
              if (pending_b >= 0) bulk_wait_read<1>();   // all but the newest group have read their source
            }
            if (pending_b >= 0) mbar_arrive(&bfree[pending_b]);
            pending_b = b;
          } else {
            if (s.tma_out && s.debug != 1) {
              for (int blk = 0; blk < nblk; ++blk) tma_store_2d(&tmOut, buf + blk * EPI_BLK_BYTES, n0 + blk * 64, m0);
              bulk_commit();
              bulk_wait_read<0>();                       // smem has been read: the buffer may be refilled
            }
            mbar_arrive(&bfree[b]);
          }
        }
        __syncwarp();
        }
      }
      if (stamp) TN_STAMP(9, n_local);
    }
    if (issuer && pending_b >= 0) {                      // smem must outlive the last store's read
      bulk_wait_read<0>();
      mbar_arrive(&bfree[pending_b]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (s.debug == 5 && threadIdx.x == 0) {
    unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    if (blockIdx.x == 0) { g_gemm_dbg[11 * 16] = (long long)gt; g_gemm_dbg[11 * 16 + 1] = clock64(); }
    unsigned smid; asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    if (blockIdx.x < 160) g_gemm_cta[2 * blockIdx.x + 1] = (long long)((gt & 0xffffffffffffull) | ((unsigned long long)smid << 48));
  }
  if (warp == 17) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_COLS); }
  if (s.dynamic && threadIdx.x == 0) {                   // last CTA out rearms the scheduler pair for its next user
    __threadfence();
    if (atomicAdd(sched + 1, 1) == (int)gridDim.x - 1) { sched[0] = 0; sched[1] = 0; __threadfence(); }
  }
}

// ---------------------------------------------------------------------------------------------
// weight gradient: split-K over tokens, MN-major operands
// ---------------------------------------------------------------------------------------------
struct WgradShape {
  const int* rows_dev; // dynamic token count: T = min(T, *rows_dev), a multiple of 128 (packed token layout), or null.
                       // Written by the pack-plan kernels at the very start of a step, never by the preceding kernel.
  int T, Mo, No;       // tokens, output rows (dY width), output cols (X width)
  int block_n;         // columns per CTA tile (multiple of 16, <= 256)
  int a_atoms, b_atoms;  // 64-wide MN atoms per stage
  int stages, k_splits;
  float* out;          // [Mo, ldw] fp32, accumulated with red.add
  int ldw;
  float* dbias;        // [Mo] or null: column sums of dY, computed by one extra N=16 MMA per K step against a
                       // constant all-ones operand (the bias gradient for free, no second pass over dY)
};

__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_wgrad_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, WgradShape s) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int ATOM_BYTES = BLOCK_K * 128;             // 64 k-rows x 128 B (64 bf16 along MN)
  const int a_bytes = s.a_atoms * ATOM_BYTES, b_bytes = s.b_atoms * ATOM_BYTES;
  uint8_t* smA = smem;
  uint8_t* smB = smem + s.stages * a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smB + s.stages * b_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + s.stages;
  uint64_t* tfull = bars + 2 * s.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull + 1);
  uint8_t* ones = smem + s.stages * (a_bytes + b_bytes) + 1024;      // 64 k-rows x 128 B of bf16 1.0 (after the barriers)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * BLOCK_M, n0 = blockIdx.z * s.block_n;
  const bool do_bias = s.dbias != nullptr && blockIdx.z == 0;
  if (do_bias) {
    for (int i = threadIdx.x; i < ATOM_BYTES / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(ones)[i] = 0x3F803F80u;
    fence_proxy_async();
  }
  // dynamic token count (packed layout): read before anything else so that a CTA without work skips cleanly
  const int T_eff = s.rows_dev ? min(s.T, *s.rows_dev) : s.T;
  const int kblocks_total = (T_eff + BLOCK_K - 1) / BLOCK_K;
  const int per = (kblocks_total + s.k_splits - 1) / s.k_splits;
  const int kb_begin = blockIdx.x * per, kb_end = min(kblocks_total, kb_begin + per);
  const int nkb = max(0, kb_end - kb_begin);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < s.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_prologue_done();
  constexpr int BIAS_COL = 496;                          // accumulator columns [496, 512): sum_t dY[t, row]

  if (nkb > 0) {
    if (warp == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&full[stage], a_bytes + b_bytes);
          for (int a = 0; a < s.a_atoms; ++a)
            tma_load_2d(smA + stage * a_bytes + a * ATOM_BYTES, &tmA, &full[stage], m0 + a * 64, kb * BLOCK_K,
                        SRFRD_EVICT_FIRST);
          for (int b = 0; b < s.b_atoms; ++b)
            tma_load_2d(smB + stage * b_bytes + b * ATOM_BYTES, &tmB, &full[stage], n0 + b * 64, kb * BLOCK_K,
                        SRFRD_EVICT_FIRST);
        }
        __syncwarp();
        if (++stage == s.stages) { stage = 0; phase ^= 1; }
      }
    } else if (warp == 1) {
      int bn = min(s.block_n, s.No - n0);
      bn = (bn + 15) & ~15;
      // a column tile wider than 256 (H = 272) takes two MMAs per K step: columns [0, 256) and [256, bn)
      const int bn1 = min(bn, 256), bn2 = bn - bn1;
      const uint32_t idesc = umma_idesc_bf16(BLOCK_M, bn1, 1, 1);
      const uint32_t idesc2 = umma_idesc_bf16(BLOCK_M, bn2 > 0 ? bn2 : 16, 1, 1);
      // MN-major SW128: 64-wide MN atoms are ATOM_BYTES apart (LBO); 8 k-rows = 1024 B (SBO);
      // one UMMA_K = 16 k-rows = 2048 B (= 128 in descriptor units)
      const uint64_t adesc0 = umma_smem_desc(smem_u32(smA), ATOM_BYTES, 1024);
      const uint64_t bdesc0 = umma_smem_desc(smem_u32(smB), ATOM_BYTES, 1024);
      const uint64_t onesdesc = umma_smem_desc(smem_u32(ones), ATOM_BYTES, 1024);
      const uint32_t idesc_ones = umma_idesc_bf16(BLOCK_M, 16, 1, 1);
      int stage = 0; uint32_t phase = 0;
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint64_t ad = adesc0 + (uint64_t)(stage * (a_bytes >> 4)), bd = bdesc0 + (uint64_t)(stage * (b_bytes >> 4));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BLOCK_K / 16; ++k)
            umma_bf16(tmem_base, ad + 128 * k, bd + 128 * k, idesc, (kb > kb_begin) || (k > 0));
          if (bn2 > 0) {
#pragma unroll
            for (int k = 0; k < BLOCK_K / 16; ++k)       // B atoms 4.. (columns 256..): 4 atoms further in the stage
              umma_bf16(tmem_base + 256, ad + 128 * k, bd + (uint64_t)(4 * (ATOM_BYTES >> 4)) + 128 * k, idesc2,
                        (kb > kb_begin) || (k > 0));
          }
          if (do_bias) {
#pragma unroll
            for (int k = 0; k < BLOCK_K / 16; ++k)
              umma_bf16(tmem_base + BIAS_COL, ad + 128 * k, onesdesc + 128 * k, idesc_ones, (kb > kb_begin) || (k > 0));
          }
          umma_commit(&empty[stage]);
          if (kb == kb_end - 1) umma_commit(tfull);
        }
        __syncwarp();
        if (++stage == s.stages) { stage = 0; phase ^= 1; }
      }
    } else {
      const int quarter = warp & 3;
      const int row = m0 + quarter * 32 + lane;
      const int bn = min(s.block_n, s.No - n0);
      mbar_wait(tfull, 0);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
      const bool vec_red = (s.ldw % 4 == 0) && ((reinterpret_cast<uintptr_t>(s.out) & 15) == 0);
      for (int c = 0; c < bn; c += 16) {
        uint32_t raw[16];
        tmem_ld16(taddr + c, raw);
        tmem_ld_wait();
        if (row < s.Mo) {
          float* o = s.out + (size_t)row * s.ldw + n0 + c;
          // 148 CTAs add into the same Mo x No block at the same moment: 16-byte vector reductions cut the number of
          // L2 atomic operations by four (ncu: the scalar version spent a third of the CTA's lifetime here)
          if (vec_red && n0 + c + 16 <= s.No) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + j), "f"(__uint_as_float(raw[j])),
                           "f"(__uint_as_float(raw[j + 1])), "f"(__uint_as_float(raw[j + 2])), "f"(__uint_as_float(raw[j + 3]))
                           : "memory");
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (n0 + c + j < s.No) red_add_f32(o + j, __uint_as_float(raw[j]));
          }
        }
      }
      if (do_bias) {                       // columns [240, 256) all hold sum_t dY[t, row]
        uint32_t raw[16];
        tmem_ld16(taddr + BIAS_COL, raw);
        tmem_ld_wait();
        if (row < s.Mo) red_add_f32(s.dbias + row, __uint_as_float(raw[0]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ---------------------------------------------------------------------------------------------
// plain SIMT reference GEMM: used ONLY by tests to cross-check the tensor-core kernels on device
// ---------------------------------------------------------------------------------------------
__global__ void gemm_ref_kernel(const bf16* A, int lda, const bf16* B, int ldb, float* C, int ldc, int M, int N, int K,
                                int a_mn_major, int b_mn_major) {
  int n = blockIdx.x * blockDim.x + threadIdx.x, m = blockIdx.y;
  if (n >= N || m >= M) return;
  float acc = 0.f;
  for (int k = 0; k < K; ++k) {
    float a = a_mn_major ? bf2f(A[(size_t)k * lda + m]) : bf2f(A[(size_t)m * lda + k]);
    float b = b_mn_major ? bf2f(B[(size_t)k * ldb + n]) : bf2f(B[(size_t)n * ldb + k]);
    acc = fmaf(a, b, acc);
  }
  C[(size_t)m * ldc + n] = acc;
}

static int pick_block_n(int N) {
  int tiles = (N + 255) / 256;
  int bn = ((N + tiles - 1) / tiles + 15) & ~15;
  return bn;
}
// gemm_tn: with more than one column tile the tile width is a multiple of 64, so the 64-column TMA store boxes of
// one tile never reach into its neighbour's columns
static int pick_block_n_tn(int N) {
  if (N <= TN_MAX_BLOCK_N) return (N + 15) & ~15;
  const int tiles = (N + TN_MAX_BLOCK_N - 1) / TN_MAX_BLOCK_N;
  const int bn = ((N + tiles - 1) / tiles + 63) & ~63;
  return bn > TN_MAX_BLOCK_N ? TN_MAX_BLOCK_N : bn;
}

}  // namespace srfrd

using namespace srfrd;

// Tile / pipeline plan of one gemm_tn launch: pure host arithmetic (no CUDA call), shared by the launcher and by
// srfrd_gemm_tn_plan(), through which the CPU tests check every shape's plan (shared memory, stage counts, issuer rule).
static int plan_gemm_tn(int M, int N, int K, bool has_aux, bool tma_out, bool lnf, GemmShape& s, size_t& smem_out) {
  s.M = M; s.N = N; s.K = K;
  s.block_n = pick_block_n_tn(N);
  s.n_tiles = (N + s.block_n - 1) / s.block_n;
  s.m_tiles = (M + BLOCK_M - 1) / BLOCK_M;
  s.has_aux = has_aux;
  s.tma_out = tma_out;
  const int b_stage_bytes = ((s.block_n * BLOCK_K * 2) + 1023) & ~1023;
  const int stage_bytes = A_STAGE_BYTES + b_stage_bytes;
  { const char* dbg = getenv("SRFRD_GEMM_DEBUG"); s.debug = dbg ? atoi(dbg) : 0; }
  s.buf_blocks = (s.has_aux || s.tma_out) ? (s.block_n + 63) / 64 : 0;
  SRFRD_REQUIRE(!lnf || s.n_tiles == 1, "gemm_tn: fused LayerNorm needs one column tile (N=%d)", N);
  // residual / gate tiles without the LayerNorm fusion: two tile buffers per set when a two-stage A pipeline still fits
  s.nbuf = 2;
  if (s.has_aux && s.tma_out && !lnf && s.n_tiles == 1) {
    const int kb_h = (K + BLOCK_K - 1) / BLOCK_K;
    const int need = 1024 + 4 * s.buf_blocks * EPI_BLK_BYTES + MAX_BIAS * 4 + 1024 + kb_h * b_stage_bytes + 2 * kb_h * A_STAGE_BYTES;
    if (need <= 227 * 1024 && kb_h * b_stage_bytes <= 48 * 1024) s.nbuf = 4;
    { const char* nb = getenv("SRFRD_GEMM_NBUF"); if (nb && atoi(nb) == 2) s.nbuf = 2; }
  }
  int fixed = 1024 + (lnf ? 4 : s.nbuf) * s.buf_blocks * EPI_BLK_BYTES + MAX_BIAS * 4 + (lnf ? 2 * MAX_LN * 4 + 2 * 2 * BLOCK_M * 2 * 4 : 0) + 1024;
  // B (the weight matrix) is identical for every row tile: with one column tile and few K blocks it is loaded once
  const int kblocks_h = (K + BLOCK_K - 1) / BLOCK_K;
  s.b_resident = (s.n_tiles == 1 && kblocks_h * b_stage_bytes <= 48 * 1024) ? 1 : 0;
  { const char* r = getenv("SRFRD_GEMM_BRES"); if (r) s.b_resident = s.b_resident && atoi(r); }
  s.kgroup = 1;
  if (s.b_resident) {
    fixed += kblocks_h * b_stage_bytes;
    // the whole K of a tile in one stage (one barrier round trip per tile instead of one per K block) while >= 3 fit
    if ((227 * 1024 - fixed) / (kblocks_h * A_STAGE_BYTES) >= ((lnf || s.nbuf == 4) ? 2 : 3)) s.kgroup = kblocks_h;
    { const char* g = getenv("SRFRD_GEMM_KGROUP"); if (g && atoi(g) == 0) s.kgroup = 1; }
    s.stages = (227 * 1024 - fixed) / (s.kgroup * A_STAGE_BYTES);
  } else {
    s.stages = (227 * 1024 - fixed) / stage_bytes;
  }
  if (s.stages > 6) s.stages = 6;
  SRFRD_REQUIRE(s.stages >= 2, "gemm_tn: tile does not fit shared memory");
  smem_out = (size_t)s.stages * (s.b_resident ? s.kgroup * A_STAGE_BYTES : stage_bytes) + fixed;
  { const char* d = getenv("SRFRD_GEMM_DYNAMIC"); s.dynamic = d ? atoi(d) : 0; }
  { const char* l = getenv("SRFRD_L2_PREFETCH"); s.l2_prefetch = l ? atoi(l) : 1; }
  s.nacc = s.block_n <= 128 ? 4 : 2;
  { const char* a = getenv("SRFRD_GEMM_NACC"); if (a && atoi(a) == 2) s.nacc = 2; }
  s.sched_slot = 0;
  return 0;
}

extern "C" int srfrd_gemm_tn_plan(int M, int N, int K, int has_aux, int bf16_out, int fused_ln, int* out) {
  SRFRD_REQUIRE(out && M > 0 && N > 0 && K > 0 && N % 16 == 0 && K % 8 == 0, "gemm_tn_plan: bad arguments");
  GemmShape s;
  s.rows_dev = nullptr;
  size_t smem = 0;
  if (int rc = plan_gemm_tn(M, N, K, has_aux != 0, bf16_out != 0, fused_ln != 0, s, smem)) return rc;
  const int kblocks = (K + BLOCK_K - 1) / BLOCK_K;
  out[0] = s.block_n; out[1] = s.n_tiles; out[2] = s.stages; out[3] = s.kgroup; out[4] = s.b_resident;
  out[5] = s.nacc; out[6] = s.nbuf; out[7] = s.buf_blocks; out[8] = (int)smem;
  out[9] = (s.kgroup >= kblocks && s.stages % 2 == 0) ? 1 : 0;      // second MMA issuer active (same rule as the kernel)
  out[10] = kblocks;
  return 0;
}

extern "C" int srfrd_gemm_tn(const void* A, int lda, const void* B, int ldb, int M, int N, int K,
                             const srfrd_gemm_epilogue_t* ep, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  SRFRD_REQUIRE(A && B && ep, "gemm_tn: null operand");
  SRFRD_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_tn: empty shape M=%d N=%d K=%d", M, N, K);
  SRFRD_REQUIRE(N % 16 == 0 && K % 8 == 0, "gemm_tn: need N %% 16 == 0 and K %% 8 == 0 (got N=%d K=%d)", N, K);
  SRFRD_REQUIRE(lda % 8 == 0 && ldb % 8 == 0 && lda >= K && ldb >= K, "gemm_tn: bad leading dims lda=%d ldb=%d", lda, ldb);
  SRFRD_REQUIRE(ep->out_bf16 || ep->out_f32, "gemm_tn: no output");
  SRFRD_REQUIRE(ep->ldc % 8 == 0 && ep->ldc >= N, "gemm_tn: bad ldc=%d", ep->ldc);
  SRFRD_REQUIRE(!ep->residual || ep->ldr % 8 == 0, "gemm_tn: bad ldr");
  SRFRD_REQUIRE(!ep->gate || ep->ldg % 8 == 0, "gemm_tn: bad ldg");
  SRFRD_REQUIRE(!(ep->residual && ep->gate), "gemm_tn: residual and gate cannot be combined (one aux operand)");
  SRFRD_REQUIRE(!ep->bias || N <= MAX_BIAS, "gemm_tn: bias with N=%d > %d unsupported", N, MAX_BIAS);
  if (gemm_small_eligible(M, N, K, ep, lda, ldb)) {
    SRFRD_REQUIRE(!(ep->drop_p > 0.f) || ep->drop_p < 1.f, "gemm_tn: dropout p must be < 1");
    return gemm_small_launch(A, lda, B, ldb, M, N, K, ep, stream);
  }
  GemmShape s;
  const void* aux = ep->residual ? ep->residual : ep->gate;
  const int ldaux = ep->residual ? ep->ldr : ep->ldg;
  // TMA store needs a 16-byte aligned bf16 output; the fp32 output (predict logits, tests) is stored directly
  const bool tma_out = ep->out_bf16 && !ep->out_f32 && (((uintptr_t)ep->out_bf16 & 15) == 0);
  SRFRD_REQUIRE(!aux || (((uintptr_t)aux & 15) == 0), "gemm_tn: residual / gate must be 16-byte aligned");
  const bool lnf = ep->ln_out_bf16 != nullptr;
  if (lnf) {
    SRFRD_REQUIRE(ep->residual && tma_out && N <= MAX_LN && ep->ln_w && ep->ln_b,
                  "gemm_tn: fused LayerNorm needs a residual, a bf16 output, N <= %d (N=%d) and ln_w / ln_b", MAX_LN, N);
    SRFRD_REQUIRE(ep->ld_ln % 8 == 0 && ep->ld_ln >= N && (((uintptr_t)ep->ln_out_bf16 & 15) == 0), "gemm_tn: bad ln_out");
  }
  size_t smem = 0;
  if (int rc = plan_gemm_tn(M, N, K, aux != nullptr, tma_out, lnf, s, smem)) return rc;
  s.rows_dev = row_limit();
  const int b_stage_bytes = ((s.block_n * BLOCK_K * 2) + 1023) & ~1023;
  (void)b_stage_bytes;
  static int next_slot = 0;
  s.sched_slot = next_slot;
  next_slot = (next_slot + 1) % TN_SCHED_SLOTS;
  CUtensorMap tmA, tmB, tmAux, tmOut, tmLn;
  if (int rc = make_tmap_bf16_2d(&tmA, A, M, K, lda, BLOCK_M, BLOCK_K)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmB, B, N, K, ldb, s.block_n, BLOCK_K)) return rc;
  tmAux = tmA; tmOut = tmA;
  if (s.has_aux) if (int rc = make_tmap_bf16_2d(&tmAux, aux, M, N, ldaux, BLOCK_M, 64)) return rc;
  if (s.tma_out) if (int rc = make_tmap_bf16_2d(&tmOut, ep->out_bf16, M, N, ep->ldc, BLOCK_M, 64)) return rc;
  tmLn = tmA;
  if (lnf) if (int rc = make_tmap_bf16_2d(&tmLn, ep->ln_out_bf16, M, N, ep->ld_ln, BLOCK_M, 64)) return rc;
  GemmEpilogue e;
  e.bias = ep->bias; e.residual = (const bf16*)ep->residual; e.gate = (const bf16*)ep->gate;
  e.row_ids = ep->row_ids; e.out_bf16 = (bf16*)ep->out_bf16; e.out_f32 = ep->out_f32;
  e.ldr = ep->ldr; e.ldg = ep->ldg; e.ldc = ep->ldc; e.relu = ep->relu;
  e.drop_seed = ep->drop_seed; e.drop_stream = ep->drop_stream; e.drop_step = ep->drop_step;
  e.drop_thresh = 0; e.drop_scale = 1.f;
  e.ln_w = ep->ln_w; e.ln_b = ep->ln_b; e.ln_stats = ep->ln_stats; e.ln_eps = ep->ln_eps;
  if (ep->drop_p > 0.f) {
    SRFRD_REQUIRE(ep->drop_p < 1.f, "gemm_tn: dropout p must be < 1");
    e.drop_thresh = (uint32_t)((double)ep->drop_p * 4294967296.0);
    e.drop_scale = 1.f / (1.f - ep->drop_p);
  }
  int grid = s.m_tiles * s.n_tiles;
  if (grid > num_sms()) grid = num_sms();
  const int aux_mode = ep->residual ? 1 : (ep->gate ? 2 : 0);
#define SRFRD_TN_LAUNCH(AUXM, DROPF, LNFF)                                                                            \
  do {                                                                                                                \
    static bool attr_set = false;                                                                                     \
    if (!attr_set) {                                                                                                  \
      SRFRD_CUDA(cudaFuncSetAttribute(gemm_tn_kernel<AUXM, DROPF, LNFF>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      227 * 1024));                                                                   \
      attr_set = true;                                                                                                \
    }                                                                                                                 \
    SRFRD_CUDA(launch_pdl(gemm_tn_kernel<AUXM, DROPF, LNFF>, dim3(grid), dim3(TN_THREADS), smem, stream, tmA, tmB,    \
                          tmAux, tmOut, tmLn, s, e));                                                                 \
  } while (0)
  const bool drop = e.drop_thresh != 0;
  if (lnf) { if (drop) SRFRD_TN_LAUNCH(1, true, true); else SRFRD_TN_LAUNCH(1, false, true); }
  else if (aux_mode == 0) { if (drop) SRFRD_TN_LAUNCH(0, true, false); else SRFRD_TN_LAUNCH(0, false, false); }
  else if (aux_mode == 1) { if (drop) SRFRD_TN_LAUNCH(1, true, false); else SRFRD_TN_LAUNCH(1, false, false); }
  else { if (drop) SRFRD_TN_LAUNCH(2, true, false); else SRFRD_TN_LAUNCH(2, false, false); }
#undef SRFRD_TN_LAUNCH
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_gemm_debug_read(long long* host_dst) {
  SRFRD_CUDA(cudaDeviceSynchronize());
  SRFRD_CUDA(cudaMemcpyFromSymbol(host_dst, g_gemm_dbg, sizeof(long long) * 32 * 16));
  SRFRD_CUDA(cudaMemcpyFromSymbol(host_dst + 32 * 16, g_gemm_cta, sizeof(long long) * 2 * 160));
  return 0;
}

extern "C" int srfrd_gemm_wgrad(const void* dY, int lda, const void* X, int ldb, int64_t T, int Mo, int No,
                                float* dW, int ldw, float* dbias, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  SRFRD_REQUIRE(dY && X && dW, "gemm_wgrad: null operand");
  SRFRD_REQUIRE(T > 0 && Mo > 0 && No > 0, "gemm_wgrad: empty shape");
  SRFRD_REQUIRE(lda % 8 == 0 && ldb % 8 == 0 && lda >= Mo && ldb >= No, "gemm_wgrad: leading dims must be multiples of 8 and cover the widths");
  SRFRD_REQUIRE(T < (1ll << 31), "gemm_wgrad: too many tokens");
  WgradShape s;
  s.rows_dev = row_limit();
  s.T = (int)T; s.Mo = Mo; s.No = No;
  // one column tile up to 480 columns (H = 272: X is then read once per 128-row tile of dY instead of once per
  // (row tile, column tile) pair); wider outputs are split evenly
  s.block_n = No <= 480 ? ((No + 15) & ~15) : pick_block_n((No + 15) & ~15);
  const int n_tiles = (No + s.block_n - 1) / s.block_n, m_tiles = (Mo + BLOCK_M - 1) / BLOCK_M;
  s.a_atoms = 2;
  s.b_atoms = (s.block_n + 63) / 64;
  const int stage_bytes = (s.a_atoms + s.b_atoms) * BLOCK_K * 128;
  s.stages = (190 * 1024) / stage_bytes;
  if (s.stages > 6) s.stages = 6;
  const int kblocks = (s.T + BLOCK_K - 1) / BLOCK_K;
  int splits = num_sms() / (n_tiles * m_tiles);
  if (splits < 1) splits = 1;
  if (splits > kblocks) splits = kblocks;
  s.k_splits = splits;
  s.out = dW; s.ldw = ldw; s.dbias = dbias;
  SRFRD_REQUIRE(s.block_n <= 480, "gemm_wgrad: column tile %d too wide", s.block_n);
  const size_t smem = (size_t)s.stages * stage_bytes + 1024 + 1024 + BLOCK_K * 128;
  CUtensorMap tmA, tmB;
  // MN-major: the TMA box is [64 tokens (rows), 64 features (cols)]
  if (int rc = make_tmap_bf16_2d(&tmA, dY, T, Mo, lda, BLOCK_K, 64)) return rc;
  if (int rc = make_tmap_bf16_2d(&tmB, X, T, No, ldb, BLOCK_K, 64)) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    SRFRD_CUDA(cudaFuncSetAttribute(gemm_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  dim3 grid(s.k_splits, m_tiles, n_tiles);
  SRFRD_CUDA(launch_pdl(gemm_wgrad_kernel, grid, dim3(GEMM_THREADS), smem, stream, tmA, tmB, s));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_gemm_ref(const void* A, int lda, const void* B, int ldb, float* C, int ldc, int M, int N, int K,
                              int a_mn_major, int b_mn_major, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  dim3 grid((N + 127) / 128, M);
  gemm_ref_kernel<<<grid, 128, 0, stream>>>((const bf16*)A, lda, (const bf16*)B, ldb, C, ldc, M, N, K, a_mn_major,
                                            b_mn_major);
  SRFRD_LAUNCH_CHECK();
  return 0;
}
