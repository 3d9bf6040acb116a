// K8: full-catalogue scoring  feats (U, D) x table (N, D)^T  on tcgen05 with a streaming per-row top-10; logits never
// reach HBM.  K9: merge of partial / per-shard candidate lists.
// (SURVEY.md rows A9/A10 + full-catalogue extension: == predict(..., label = arange(1, N+1)) + stable top-k
//  with the tie-break (score desc, item id asc).)
//
// Two phases.
//  1. Streaming (catalogue_unitmax_kernel; catalogue_tilemax_kernel is the round-1 form, kept for widths whose operands do
//     not fit the unit form and behind SRFRD_TOPK_UNIT=0): every CTA owns a run of (user group, item tile) pairs.
//     * The user tiles are STATIONARY IN TENSOR MEMORY: at the start of a run the epilogue warps copy their rows (bf16,
//       packed two per 32-bit column) into TMEM with tcgen05.st and every MMA takes its A operand from there
//       (tcgen05.mma TS form).  With A in shared memory the SS-form MMA of a 128 x N x 16 step reads 4 KB of A plus
//       N * 32 B of B, which saturates the 128 B/clk shared-memory port while TMA is also writing tiles.
//     * Every item tile (streamed through a TMA ring) is multiplied against both user tiles of the group, which halves
//       the L2 -> SM traffic per score; CTAs sweep the table in time-aligned windows so that it crosses the HBM bus
//       ~4 times per pass instead of ~28 (make_plan).
//     * The epilogue keeps, per user row, only the ten best RANKING UNITS (half an item tile: 56 consecutive rows at
//       D = 64) by their maximum score: the exact top-10 items provably live in them (see the proof at the kernel).
//  2. Exact re-scoring (catalogue_refine64_kernel / catalogue_refine_kernel): the 10 x 56 candidate rows of every user,
//     same bf16 operands, fp32 accumulation, order (score desc, id asc); writes the row's final list (and, for the
//     row-sharded protocol, the 80-byte wire format of the all-gather).
// n_split = 2/3 feeds hi/lo bf16 splits of the fp32 user features as extra K (near-fp32 scores).
// k <= 10 runs these top-10 kernels (a smaller k is the prefix of their lists).  10 < k <= KMAX runs compile-time k-list
// variants (catalogue_unitmax_kernel<.., KLIST = true>, catalogue_refine_k_kernel, merge_topk_k_kernel) with lists of k
// entries everywhere; only the unit form serves them, and the host plan refuses a k whose lists do not fit (topk_kmax).
// srfrd_catalogue_rank runs the unit form's rank variant (catalogue_unitmax_kernel<.., RANK = true>): no lists, each row
// counts the items ahead of its held-out item, one phase.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "srfrd_b200.h"

namespace srfrd {

static constexpr int TK = 10;               // list length kept per row
static constexpr int KMAX = SRFRD_TOPK_KMAX;  // longest list of the k-list kernels (k > TK)
static constexpr int KL_ROWS = 256;         // rows (epilogue threads) whose lists a unit-form CTA keeps in shared memory
static constexpr int TILE_U = 128;          // users per MMA (TMEM lanes)
static constexpr int KB = 64;               // k-block (bf16 elements)

struct TopkShape {
  int U, D;
  int n_split;            // 1..3 user-feature splits (each a (U, D) bf16 matrix stacked along rows: split s at row s*U_pad)
  int u_pad;              // row offset between splits in the feats tensor
  int row_lo, row_hi;     // candidate rows of the (local) table: [row_lo, row_hi)
  int64_t id_base;        // global item id of local row 0
  int kblocks;            // ceil(D / 64)
  int nt;                 // item rows per tile
  int tiles_total;        // item tiles over [row_lo, row_hi)
  int ugroups;            // user groups of UBS * 128 rows
  int64_t share;          // (user group, item tile) pairs per CTA: CTA i owns the linear range [i * share, (i + 1) * share)
  int slots;              // tile-maxima lists per row = 2 epilogue sets x max pieces a user group is cut into
  int stages;
  int debug;              // SRFRD_TOPK_DEBUG (profiling experiments only): 1 = never insert
  long long* trace;       // SRFRD_TOPK_TRACE (profiling only): clock64 stamps of CTA 0's work units [unit][12]
  const bf16* feats; int ld_feats;
  const bf16* table; int ld_table;
  float* out_scores;      // (U, slots, TK)  phase 1: tile maxima; phase 2 writes the row's exact top-10 into slot 0
  int* out_ids;           // (U, slots, TK)  phase 1: tile indices (-1 = empty); phase 2: global item ids in slot 0
  float* packed;          // optional (U, 2 * TK): the row's final list as TK fp32 scores followed by TK int32 global ids
                          // -- the send buffer of the row-sharded all-gather (80 B per user), written by phase 2
  int k;                  // list length of the k-list kernels (11 .. KMAX); the TK kernels never read it.  Every list
                          // buffer above is then k entries long instead of TK (last field: the TK kernels' parameter
                          // offsets are unchanged)
  // rank variant (catalogue_unitmax_kernel<.., RANK = true>) only; the list kernels never read these
  const bf16* target_rows; int ld_target;   // (U, D) bf16 row of each user's held-out item
  const int64_t* target_ids;                // (U,) global id of that item
  float* target_scores;                     // optional (U,): its SIMT score, written by the piece that holds tile 0
  int* rank_out;                            // (U,) items ahead of the target, summed over pieces with atomicAdd
};

// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync_t(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Sorted (value desc) list of TK entries per thread in shared memory, entry k of thread x at [k * stride + x].
// Keys reach a thread in increasing order, so the strict comparison keeps the lower key ahead on ties.
// All TK entries are loaded at once (one shared-memory latency instead of a dependent walk), the insertion
// position is a count of compares and the shift is a chain of selects.  Returns the new 10th best value.
__device__ __forceinline__ float list_insert_smem(float* ls, int* li, int stride, float sc, int id) {
  float v[TK]; int ix[TK];
#pragma unroll
  for (int k = 0; k < TK; ++k) { v[k] = ls[k * stride]; ix[k] = li[k * stride]; }
  int r = 0;                                   // entries that stay ahead of the new one
#pragma unroll
  for (int k = 0; k < TK; ++k) r += (v[k] >= sc) ? 1 : 0;
#pragma unroll
  for (int k = TK - 1; k >= 1; --k) {
    const bool shift = k > r, here = k == r;
    const float nv = shift ? v[k - 1] : (here ? sc : v[k]);
    const int ni = shift ? ix[k - 1] : (here ? id : ix[k]);
    if (k >= r) { ls[k * stride] = nv; li[k * stride] = ni; }
    v[k] = nv;
  }
  if (r == 0) { ls[0] = sc; li[0] = id; }
  return v[TK - 1];
}

// ---------------------------------------------------------------------------------------------------------------
// Phase 1 (tcgen05): per user row, the TK item tiles with the largest TILE MAXIMUM score.
//
// Why tile maxima are enough: order tiles by (max desc, tile index asc) and items by (score desc, id asc).  If an item
// x of tile T were in the row's top TK without T being among the TK best tiles, each of those TK tiles C would hold an
// item at least as good as x (its maximum: a larger score, or an equal score at a lower id because C < T and tiles are
// contiguous id ranges) -- TK items ahead of x, a contradiction.  So the exact top TK items all live in the TK best
// tiles, and phase 2 re-scores just those TK x NT items per row.  The streaming epilogue therefore needs ONE value per
// (row, tile) -- a chain of FMNMX3 over the row's NT scores -- and ONE compare against the row's current TK-th best
// tile maximum; an insertion handles a (value, tile index) pair, never a column search.
//
// One CTA per SM; every CTA owns an equal share of the linear (user group, item tile) space, cut into "pieces" at
// user-group boundaries (a piece = one user group x a run of item tiles; its user tiles are staged into TMEM once).
//   NACC accumulator stages (UBS x NT fp32 columns each) with ONE ISSUER WARP PER STAGE: a tile's MMAs cost a few
//     hundred cycles of barrier waits, fences and commits on the issuing thread, so the tensor pipe only stays busy
//     with three issuers working on consecutive tiles.
//   Two epilogue sets of 4 * UBS warps take alternate tiles.  A thread reads its row's NT scores out of TMEM in one
//     round trip and hands the accumulator back at once.  (Measured on this part: tcgen05.ld sustains > 800 B/clk/SM
//     with enough loads in flight, but a lone warp sees ~160 cycles per round trip -- the epilogue is a latency chain,
//     so it is split over many warps and kept off the accumulator's critical path.)  The per-thread lists live in
//     shared memory and are only touched on the rare insertion; the two threads that serve the same row (one per set)
//     publish their current threshold to each other: a tile below EITHER list's TK-th best cannot be a top-TK tile.
//   Control warps have the highest warp ids (the scheduler favours them).
// Barriers are never shared by waiters that would skip phases: smem stage s is always consumed by issuer
// (tile % NACC) because the ring length is a multiple of NACC * kblocks, and tfull is indexed [stage][set].
template <int UBS, int NT, int NACC>
__global__ void __launch_bounds__(32 * (8 * UBS + 4), 1)
catalogue_tilemax_kernel(const __grid_constant__ CUtensorMap tmE, TopkShape s) {
  constexpr int NEPI = 8 * UBS;                       // epilogue warps
  constexpr int ACC_STRIDE = UBS * NT;                // TMEM columns per accumulator stage
  constexpr int B_TILE_BYTES = NT * KB * 2;
  constexpr int LSTR = NEPI * 32;                     // list stride (threads)
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smB = smem;
  float* lsc = reinterpret_cast<float*>(smB + s.stages * B_TILE_BYTES);       // [TK][LSTR]
  int* lid = reinterpret_cast<int*>(lsc + TK * LSTR);
  float* lthr = reinterpret_cast<float*>(lid + TK * LSTR);                    // [LSTR] current TK-th best per thread
  uint64_t* bars = reinterpret_cast<uint64_t*>(lthr + LSTR);
  uint64_t* full = bars;
  uint64_t* empty = bars + s.stages;
  uint64_t* tfull = bars + 2 * s.stages;              // [NACC][2 sets]
  uint64_t* tempty = tfull + 2 * NACC;                // [NACC]
  uint64_t* afull = tempty + NACC;
  uint64_t* aempty = afull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int a_cols = s.n_split * (s.D / 2);           // 32-bit TMEM columns of one user tile
  const int64_t total = (int64_t)s.ugroups * s.tiles_total;
  const int64_t lin0 = (int64_t)blockIdx.x * s.share, lin1 = min(total, lin0 + s.share);

  if (warp == NEPI && lane == 0) {
    tma_prefetch_desc(&tmE);
    for (int i = 0; i < s.stages; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2 * NACC; ++i) mbar_init(&tfull[i], 1);
    for (int i = 0; i < NACC; ++i) mbar_init(&tempty[i], 4 * UBS);
    mbar_init(afull, 4 * UBS);
    mbar_init(aempty, NACC);
    fence_barrier_init();
  }
  if (warp == NEPI + 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tA = tmem_base + NACC * ACC_STRIDE;  // user tiles live after the accumulator stages

  if (warp == NEPI) {
    // ------------------------------------------------------------------ TMA producer (item tiles)
    int stage = 0; uint32_t phase = 0;
    for (int64_t lin = lin0; lin < lin1;) {
      const int t0 = (int)(lin % s.tiles_total);
      const int t1 = (int)min((int64_t)s.tiles_total, t0 + (lin1 - lin));
      for (int t = t0; t < t1; ++t) {
        for (int kb = 0; kb < s.kblocks; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (elect_one()) {
            mbar_expect_tx(&full[stage], B_TILE_BYTES);
            tma_load_2d(smB + stage * B_TILE_BYTES, &tmE, &full[stage], kb * KB, s.row_lo + t * NT, SRFRD_EVICT_NORMAL);
          }
          __syncwarp();
          if (++stage == s.stages) { stage = 0; phase ^= 1; }
        }
      }
      lin += t1 - t0;
    }
  } else if (warp > NEPI && warp <= NEPI + NACC) {
    // ------------------------------------------------------------------ MMA issuer w: tiles with n % NACC == w
    const int w = warp - NEPI - 1;
    const uint32_t idesc = umma_idesc_bf16(TILE_U, NT, 0, 0);
    const uint64_t bdesc0 = umma_smem_desc(smem_u32(smB), 0, 1024);
    const bool fast = s.D == 64 && s.n_split == 1;
    const uint32_t tacc = tmem_base + w * ACC_STRIDE;
    int stage = 0; uint32_t phase = 0, uphase = 0, aphase = 0;
    int n = 0;                                          // tiles seen by this CTA so far
    for (int64_t lin = lin0; lin < lin1;) {
      const int t0 = (int)(lin % s.tiles_total);
      const int t1 = (int)min((int64_t)s.tiles_total, t0 + (lin1 - lin));
      mbar_wait(afull, uphase);                         // user tiles of this piece are in TMEM
      uphase ^= 1;
      tc_fence_after();
      for (int t = t0; t < t1; ++t, ++n) {
        if (n % NACC != w) {                            // another issuer's tile: just advance the smem ring
          stage += s.kblocks;
          if (stage >= s.stages) { stage -= s.stages; phase ^= 1; }
          continue;
        }
        // the item tile usually landed long ago: take that (cheap) wait first so that nothing but the MMA issue sits
        // between the accumulator coming back (tempty) and the tensor pipe starting on it
        mbar_wait2(&tempty[w], aphase ^ 1, &full[stage], phase);   // both tests in flight together (~250 cycles each)
        aphase ^= 1;
        tc_fence_after();
        for (int kb = 0; kb < s.kblocks; ++kb) {
          if (kb > 0) mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint64_t bd = bdesc0 + (uint64_t)(stage * (B_TILE_BYTES >> 4));
          if (elect_one()) {
            if (fast) {                                   // D == 64, one split: 4 K-steps, everything unrolled
#pragma unroll
              for (int ub = 0; ub < UBS; ++ub)           // the item tile is reused for every user tile
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  umma_bf16_ts(tacc + ub * NT, tA + ub * 32 + k * 8, bd + 2 * k, idesc, k != 0);
            } else {
              const int ksteps = min(KB / 16, (s.D - kb * KB + 15) / 16);
              for (int ub = 0; ub < UBS; ++ub)
                for (int sp = 0; sp < s.n_split; ++sp)
                  for (int k = 0; k < ksteps; ++k)
                    umma_bf16_ts(tacc + ub * NT, tA + ub * a_cols + sp * (s.D / 2) + (kb * (KB / 16) + k) * 8,
                                 bd + 2 * k, idesc, (kb | sp | k) != 0);
            }
            if (kb == s.kblocks - 1) umma_commit(&tfull[w * 2 + (n & 1)]);      // the epilogue is the critical path
            umma_commit(&empty[stage]);
          }
          __syncwarp();
          if (++stage == s.stages) { stage = 0; phase ^= 1; }
        }
      }
      if (elect_one()) umma_commit(aempty);             // this warp's MMAs of the piece are done with the user tiles
      __syncwarp();
      lin += t1 - t0;
    }
  } else if (warp < NEPI) {
    // ------------------------------------------------------------------ epilogue: set = tile parity
    const int quarter = warp & 3, ub = (warp >> 2) % UBS, set = warp / (4 * UBS);
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    float* thr_mine = lthr + warp * 32 + lane;
    const float* thr_other = lthr + ((warp + 4 * UBS) % NEPI) * 32 + lane;   // same user row, other set
    uint32_t cnt[NACC];                                 // uses of tfull[a][set] so far -> wait parity
#pragma unroll
    for (int a = 0; a < NACC; ++a) cnt[a] = 0;
    uint32_t uphase = 0;
    int n = 0;
    for (int64_t lin = lin0; lin < lin1;) {
      const int ug = (int)(lin / s.tiles_total);
      const int t0 = (int)(lin % s.tiles_total);
      const int t1 = (int)min((int64_t)s.tiles_total, t0 + (lin1 - lin));
      const int piece = (int)(lin / s.share - ((int64_t)ug * s.tiles_total) / s.share);
      const int urow = (ug * UBS + ub) * TILE_U + quarter * 32 + lane;
      if (set == 0) {
        // ---- stage this thread's user row into tensor memory (A operand, K-major, 2 bf16 per column) ----
        mbar_wait(aempty, uphase ^ 1);                    // previous piece's MMAs no longer read the user tiles
        uphase ^= 1;
        tc_fence_after();
        for (int sp = 0; sp < s.n_split; ++sp) {
          const uint4* src = reinterpret_cast<const uint4*>(s.feats + ((size_t)sp * s.u_pad + urow) * s.ld_feats);
          for (int c = 0; c < s.D / 2; c += 8) {            // 8 columns = 16 features = one UMMA K step
            uint32_t v[8];
            uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
            if (urow < s.U) { lo = __ldg(src + c / 4); hi = __ldg(src + c / 4 + 1); }
            v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
            tmem_st8(tA + lane_off + ub * a_cols + sp * (s.D / 2) + c, v);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(afull);
      }
      float ts[TK]; int ti[TK];                       // this thread's TK best (tile maximum, tile index), sorted
#pragma unroll
      for (int r = 0; r < TK; ++r) { ts[r] = -INFINITY; ti[r] = -1; }
      float thr = -INFINITY;
      *thr_mine = -INFINITY;
      // both threads of a row start the piece together: the partner's published threshold always belongs to THIS piece
      named_bar_sync_t(1 + ub * 4 + quarter, 64);
      for (int t = t0; t < t1; ++t, ++n) {
        if ((n & 1) != set) continue;                     // the other set's tile
        const int a = n % NACC;
        uint32_t par = 0;
#pragma unroll
        for (int q = 0; q < NACC; ++q)
          if (q == a) { par = cnt[q] & 1; cnt[q]++; }
        const float thr_p = *thr_other;
        mbar_wait(&tfull[a * 2 + set], par);
        tc_fence_after();
        const uint32_t taddr = tmem_base + lane_off + a * ACC_STRIDE + ub * NT;
        uint32_t r0[32], r1[32];
        tmem_ld32(taddr, r0);
        if (NT > 32) tmem_ld32(taddr + 32, r1);
        tmem_ld_wait();
        tc_fence_before();                                // scores are in registers: hand the accumulator back now
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[a]);
        if (t == s.tiles_total - 1) {                     // last tile of the table: columns past row_hi are not items
          const int col_row0 = s.row_lo + t * NT;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (col_row0 + j >= s.row_hi) r0[j] = 0xff800000u;
            if (NT > 32 && col_row0 + 32 + j >= s.row_hi) r1[j] = 0xff800000u;
          }
        }
        // FMNMX3: two scores folded per ALU instruction
        float m0 = fmax3(__uint_as_float(r0[0]), __uint_as_float(r0[1]), __uint_as_float(r0[2]));
        float m1 = fmax3(__uint_as_float(r0[3]), __uint_as_float(r0[4]), __uint_as_float(r0[5]));
#pragma unroll
        for (int j = 6; j < 30; j += 4) {
          m0 = fmax3(m0, __uint_as_float(r0[j]), __uint_as_float(r0[j + 1]));
          m1 = fmax3(m1, __uint_as_float(r0[j + 2]), __uint_as_float(r0[j + 3]));
        }
        m0 = fmax3(m0, __uint_as_float(r0[30]), __uint_as_float(r0[31]));
        if (NT > 32) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            m0 = fmax3(m0, __uint_as_float(r1[j]), __uint_as_float(r1[j + 1]));
            m1 = fmax3(m1, __uint_as_float(r1[j + 2]), __uint_as_float(r1[j + 3]));
          }
        }
        const float tmax = fmaxf(m0, m1);
        thr = fmaxf(thr, thr_p);
        if (tmax > thr && s.debug != 1) {                 // rare after warm-up, thread-divergent
          ts[TK - 1] = tmax; ti[TK - 1] = t;
#pragma unroll
          for (int r = TK - 1; r > 0; --r) {              // strict: an equal maximum never overtakes an earlier tile
            if (ts[r] > ts[r - 1]) {
              const float fs = ts[r]; ts[r] = ts[r - 1]; ts[r - 1] = fs;
              const int is = ti[r]; ti[r] = ti[r - 1]; ti[r - 1] = is;
            }
          }
          thr = fmaxf(thr, ts[TK - 1]);
          *thr_mine = thr;
        }
      }
      if (urow < s.U) {
        const size_t o = ((size_t)urow * s.slots + piece * 2 + set) * TK;
#pragma unroll
        for (int r = 0; r < TK; ++r) {
          s.out_scores[o + r] = ts[r];
          s.out_ids[o + r] = ti[r];
        }
      }
      lin += t1 - t0;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NEPI + 1) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ---------------------------------------------------------------------------------------------------------------
// Phase 1, unit form (two user tiles; item tiles of MT = (512 - 2 * a_cols) / 4 rows rounded down to 16: 112 at D = 64).
//
// Tensor memory holds 448 accumulator columns = 896 cycles of tensor work, so the tensor pipe's share is bounded by
// 896 / (one accumulator round trip) -- release -> issuer sees it ~250 cycles, four tcgen05.mma issues ~320, commit ->
// epilogue sees it ~350, one round of tcgen05.ld ~200-340 -- and by the epilogue warps' own serial time per unit.  With
// K = 64 a score costs only four K steps, so this kernel is an epilogue / latency problem, not a tensor-throughput one
// (a quarter of the MMAs, SRFRD_TOPK_DEBUG=4, changes the time by 2 %).  Structure (clock64 stamps of one CTA:
// SRFRD_TOPK_TRACE, tools/topk_trace.py; A/B timings: tools/topk_ab.py):
//   * an MMA is 128 users x MT ITEMS x 16; a work unit is (one MT-item tile) x (ONE user tile); unit q = 2 * tile +
//     user_tile uses accumulator stage w = user_tile + 2 * (tile parity).  ONE ISSUER WARP PER STAGE: an issuer that
//     alternates between two stages in order holds the ready one back behind the late one.
//   * 8 epilogue + 4 issuer warps = 3 per scheduler -> 168 registers a thread: a thread owns one user row and reads
//     its whole MT scores in ONE round of tcgen05.ld (MT registers), hands the accumulator back, and only then reduces
//     them (FMNMX3, eight independent chains) to the maxima of the tile's two halves -- the ranking unit is a half
//     (list entries are 2 * tile + half, phase 2 re-scores 10 x MT / 2 items per row).  The four warps of user tile
//     ub serve all of its units, alternating between its two stages; the next unit's barrier is tested before the
//     reduction so that the test's latency hides under it.
//   * no producer warp: passing tempty[w] for tile n tells issuer w that ITS MMAs on tile n - 2 are complete; the
//     second of the two issuers of a tile parity to get there (shared-memory counter) re-fills that tile's ring slot,
//     after its own MMAs for tile n are issued.  (The same hand-over done by epilogue threads cost ~550 cycles on the
//     accumulator's critical path.)
//   * every barrier has one waiter group that consumes every phase (tfull[w]: the warps of user tile w & 1;
//     tempty[w]: issuer w; full[slot]: the two issuers of the slot's parity -- the ring length is even).
//   * per-row lists stay in REGISTERS and are offered to after the release.
// Measured at 16 384 users x 1 M items, streaming phase only (tools/topk_ab.py, same box, same data):
//     round-2 form (two issuers + producer, 16 epilogue warps x 96 registers, two ld rounds per unit)        2.18 ms
//     + one issuer per stage, lists in shared memory, offer under the next load's latency                   2.63 ms
//       (without insertions 1.92: the insertion of ~30 % of a warp's units delays the release)
//     MMAs of MT / 2 columns with a barrier pair per half (eight round trips in flight)                      2.77 ms
//     16 epilogue warps, a column half each, one ld round                                                    2.40 ms
//     this form                                                                                              1.93 ms
//     this form with quarter-tile ranking units (phase 2 halves, but four offers per unit: insertions 0.30)  2.10 ms
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}

//
// KLIST: the k-list variant (k = s.k in TK + 1 .. KMAX).  A k-long list per row does not fit in registers next to the MT
// scores, so the 256 rows' lists live in shared memory after the barriers, entry j of thread x at [j * 256 + x] (bank-
// conflict free), UNSORTED: an insertion overwrites the current worst entry (lowest maximum; among equal maxima the
// highest unit, which the order (max desc, unit asc) ranks last) and rescans the k entries for the new worst -- no shifts,
// no dependent chain.  The strict v > thr test stays: units reach a thread in increasing index order, so an equal maximum
// never displaces an earlier unit.  The proof above holds with TK replaced by k.  Everything else is the same code.
//
// RANK: the rank variant (srfrd_catalogue_rank).  No list: each row counts the items ahead of its held-out item t,
// score > score(t) or score == score(t) at a lower id, t itself excluded BY ID.  At the start of a piece a thread computes
// score(t) with SIMT arithmetic (target_score: catalogue_refine_kernel's loop) next to staging its user row; per unit,
// after the accumulator has been handed back, the unit's maximum decides: below score(t), nothing in the unit counts;
// otherwise the unit's columns are counted against one threshold (a unit entirely below t's id counts x >= score(t),
// i.e. x > the next float down; one entirely above counts x > score(t)) and the unit that holds t's id is corrected
// column by column.  At the end of the piece the row's count goes into rank_out with one integer atomicAdd (pieces of
// the same user group, and row shards launched one after another, add up exactly in any order).  The ring, barriers,
// refill and plan are those of the top-10 form.
//
// SIMT score of a (user row, item row) pair in catalogue_refine_kernel's order: per split, fmaf over the features in
// order, then the splits summed.
__device__ __forceinline__ float target_score(const bf16* feats, size_t split_stride, const bf16* item, int D,
                                              int n_split) {
  const uint4* e = reinterpret_cast<const uint4*>(item);
  float acc = 0.f;
  for (int sp = 0; sp < n_split; ++sp) {
    const uint4* f = reinterpret_cast<const uint4*>(feats + sp * split_stride);
    float a = 0.f;
    for (int c = 0; c < D / 8; ++c) {
      const uint4 fv = __ldg(f + c), ev = __ldg(e + c);
      const uint32_t fw[4] = {fv.x, fv.y, fv.z, fv.w}, ew[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 x = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&fw[q]));
        const float2 y = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ew[q]));
        a = fmaf(x.x, y.x, a);
        a = fmaf(x.y, y.y, a);
      }
    }
    acc += a;
  }
  return acc;
}

template <int MT, bool TRACE, bool KLIST = false, bool RANK = false>
__global__ void __launch_bounds__(384, 1)
catalogue_unitmax_kernel(const __grid_constant__ CUtensorMap tmE, TopkShape s) {
  constexpr int UBS = 2, NEPI = 8, NACC = 4;
  constexpr int HALF = MT / 2;                        // ranking unit (items) = columns one thread reads
  constexpr int B_TILE_BYTES = MT * KB * 2;
  constexpr int TR0 = 2000, TRN = 256;                // traced tiles of CTA 0
  static_assert(MT % 16 == 0 && HALF >= 32 && HALF < 64, "unit form: MT in {64 .. 112}");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smB = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smB + s.stages * B_TILE_BYTES);
  uint64_t* full = bars;
  int* rcnt = reinterpret_cast<int*>(bars + s.stages); // [stages] issuers done with the slot's tile (0..2)
  uint64_t* tfull = bars + 2 * s.stages;              // [NACC]
  uint64_t* tempty = tfull + NACC;                    // [NACC]
  uint64_t* afull = tempty + NACC;
  uint64_t* aempty = afull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aempty + 1);
  const int ring_tiles = s.stages / s.kblocks;        // item tiles the ring holds

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int a_cols = s.n_split * (s.D / 2);
  const int64_t total = (int64_t)s.ugroups * s.tiles_total;
  const int64_t lin0 = (int64_t)blockIdx.x * s.share, lin1 = min(total, lin0 + s.share);

  if (warp == NEPI && lane == 0) {
    tma_prefetch_desc(&tmE);
    for (int i = 0; i < s.stages; ++i) { mbar_init(&full[i], 1); rcnt[i] = 0; }
    for (int i = 0; i < NACC; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }
    mbar_init(afull, 4 * UBS);
    mbar_init(aempty, NACC);
    fence_barrier_init();
  }
  if (warp == NEPI + 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tA = tmem_base + NACC * MT;

  if (warp >= NEPI) {
    // ------------------------------------------------------------------ MMA issuer of stage w = user tile + 2 * tile parity
    const int w = warp - NEPI, ub = w & 1, par = w >> 1;
    if (w == 0 && elect_one()) {                        // fill the ring; afterwards the issuers refill a slot as it frees
      for (int64_t m = 0; m < ring_tiles && lin0 + m < lin1; ++m) {
        const int t = (int)((lin0 + m) % s.tiles_total);
        const int st0 = (int)(m * s.kblocks);
        for (int kb = 0; kb < s.kblocks; ++kb) {
          mbar_expect_tx(&full[st0 + kb], B_TILE_BYTES);
          tma_load_2d(smB + (st0 + kb) * B_TILE_BYTES, &tmE, &full[st0 + kb], kb * KB, s.row_lo + t * MT, SRFRD_EVICT_NORMAL);
        }
      }
    }
    __syncwarp();
    const uint32_t idesc = umma_idesc_bf16(TILE_U, MT, 0, 0);
    const uint64_t bdesc0 = umma_smem_desc(smem_u32(smB), 0, 1024);
    const bool fast = s.D == 64 && s.n_split == 1;
    const uint32_t tacc = tmem_base + w * MT;
    int stage = 0; uint32_t phase = 0, uphase = 0, aphase = 0;
    int n = 0;                                          // tiles seen by this CTA so far
    const int ntiles = (int)(lin1 - lin0);
    int rt = (int)((lin0 + ring_tiles - 2) % s.tiles_total);   // table tile that follows tile n - 2 in its ring slot
    for (int64_t lin = lin0; lin < lin1;) {
      const int t0 = (int)(lin % s.tiles_total);
      const int t1 = (int)min((int64_t)s.tiles_total, t0 + (lin1 - lin));
      mbar_wait(afull, uphase);                         // user tiles of this piece are in TMEM
      uphase ^= 1;
      tc_fence_after();
      for (int t = t0; t < t1; ++t, ++n) {
        const int rt_now = rt;
        if (++rt == s.tiles_total) rt = 0;
        if ((n & 1) == par) {
          const bool tr = TRACE && blockIdx.x == 0 && n >= TR0 && n < TR0 + TRN;
          long long* trq = s.trace + (size_t)(2 * (n - TR0) + ub) * 12;
          if (tr && lane == 0) trq[0] = clock64();
          mbar_wait2(&tempty[w], aphase ^ 1, &full[stage], phase);   // both tests in flight together
          aphase ^= 1;
          tc_fence_after();
          if (tr && lane == 0) trq[1] = clock64();
          for (int kb = 0; kb < s.kblocks; ++kb) {
            int st = stage + kb; uint32_t ph = phase;
            if (st >= s.stages) { st -= s.stages; ph ^= 1; }
            if (kb > 0) { mbar_wait(&full[st], ph); tc_fence_after(); }
            const uint64_t bd = bdesc0 + (uint64_t)(st * (B_TILE_BYTES >> 4));
            if (elect_one()) {
              if (fast) {                                   // D == 64, one split: 4 K-steps
#pragma unroll
                for (int k = 0; k < 4; ++k)
                  if (k == 0 || s.debug != 4) umma_bf16_ts(tacc, tA + ub * 32 + k * 8, bd + 2 * k, idesc, k != 0);
              } else {
                const int ksteps = min(KB / 16, (s.D - kb * KB + 15) / 16);
                for (int sp = 0; sp < s.n_split; ++sp)
                  for (int k = 0; k < ksteps; ++k)
                    umma_bf16_ts(tacc, tA + ub * a_cols + sp * (s.D / 2) + (kb * (KB / 16) + k) * 8, bd + 2 * k, idesc,
                                 (kb | sp | k) != 0);
              }
              if (tr) trq[2] = clock64();
              if (kb == s.kblocks - 1) umma_commit(&tfull[w]);
              if (tr) trq[3] = clock64();
            }
            __syncwarp();
          }
          if (n >= 2 && n - 2 + ring_tiles < ntiles && elect_one()) {
            int ps = stage - 2 * s.kblocks;
            if (ps < 0) ps += s.stages;
            if (atomicAdd(&rcnt[ps], 1) == 1) {
              rcnt[ps] = 0;
              __threadfence_block();
              for (int kb = 0; kb < s.kblocks; ++kb) {
                mbar_expect_tx(&full[ps + kb], B_TILE_BYTES);
                tma_load_2d(smB + (ps + kb) * B_TILE_BYTES, &tmE, &full[ps + kb], kb * KB, s.row_lo + rt_now * MT, SRFRD_EVICT_NORMAL);
              }
            }
          }
          __syncwarp();
        }
        stage += s.kblocks;
        if (stage >= s.stages) { stage -= s.stages; phase ^= 1; }
      }
      if (elect_one()) umma_commit(aempty);             // this warp's MMAs of the piece are done with the user tiles
      __syncwarp();
      lin += t1 - t0;
    }
  } else {
    // ------------------------------------------------------------------ epilogue: warp = (user tile, lane quarter)
    const int quarter = warp & 3, ub = warp >> 2;
    const uint32_t lane_off = (uint32_t)(quarter * 32) << 16;
    const uint32_t taddr0 = tmem_base + lane_off + ub * MT;                  // stage ub (even tiles); + 2 * MT: odd tiles
    uint32_t uphase = 0, tph0 = 0, tph1 = 0;
    int n = 0;
    for (int64_t lin = lin0; lin < lin1;) {
      const int ug = (int)(lin / s.tiles_total);
      const int t0 = (int)(lin % s.tiles_total);
      const int t1 = (int)min((int64_t)s.tiles_total, t0 + (lin1 - lin));
      const int piece = (int)(lin / s.share - ((int64_t)ug * s.tiles_total) / s.share);
      const int urow = (ug * UBS + ub) * TILE_U + quarter * 32 + lane;
      {
        // ---- stage this thread's user row into tensor memory (A operand, K-major, 2 bf16 per column) ----
        mbar_wait(aempty, uphase ^ 1);                    // previous piece's MMAs no longer read the user tiles
        uphase ^= 1;
        tc_fence_after();
        for (int sp = 0; sp < s.n_split; ++sp) {
          const uint4* src = reinterpret_cast<const uint4*>(s.feats + ((size_t)sp * s.u_pad + urow) * s.ld_feats);
          for (int c = 0; c < s.D / 2; c += 8) {            // 8 columns = 16 features = one UMMA K step
            uint32_t v[8];
            uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
            if (urow < s.U) { lo = __ldg(src + c / 4); hi = __ldg(src + c / 4 + 1); }
            v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
            tmem_st8(tA + lane_off + ub * a_cols + sp * (s.D / 2) + c, v);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(afull);
      }
      float tsc = INFINITY, tsc_dn = INFINITY;          // rank variant: the target's score and the next float below it
      int tid = -1, rcount = 0;                         //   (+inf for rows past U: nothing counts), its id, the count
      if constexpr (RANK) {
        if (urow < s.U) {                               // the MMAs of the piece are already running
          tid = (int)s.target_ids[urow];
          tsc = target_score(s.feats + (size_t)urow * s.ld_feats, (size_t)s.u_pad * s.ld_feats,
                             s.target_rows + (size_t)urow * s.ld_target, s.D, s.n_split);
          tsc_dn = nextafterf(tsc, -INFINITY);
          if (t0 == 0 && s.target_scores) s.target_scores[urow] = tsc;   // one piece per user group holds tile 0
        }
      }
      constexpr int TKR = (KLIST || RANK) ? 1 : TK;     // register list (unused by the k-list and rank variants)
      float ts[TKR]; int ti[TKR];                       // this row's TK best (unit maximum, unit index), sorted
#pragma unroll
      for (int r = 0; r < TKR; ++r) { ts[r] = -INFINITY; ti[r] = -1; }
      float thr = -INFINITY;
      float* kls = nullptr; int* kli = nullptr;         // k-list variant: this thread's list in shared memory
      int kworst = 0;                                   //   and the slot of its worst entry
      if constexpr (KLIST) {
        kls = reinterpret_cast<float*>(bars + 2 * s.stages + 32) + threadIdx.x;
        kli = reinterpret_cast<int*>(kls - threadIdx.x + s.k * KL_ROWS) + threadIdx.x;
        for (int j = 0; j < s.k; ++j) { kls[j * KL_ROWS] = -INFINITY; kli[j * KL_ROWS] = -1; }
      }
      auto offer = [&](float v, int id) {               // rare after warm-up, thread-divergent
        if (v > thr && s.debug != 1) {
          if constexpr (KLIST) {
            kls[kworst * KL_ROWS] = v; kli[kworst * KL_ROWS] = id;
            float wv = kls[0]; int wi = kli[0], wj = 0;
#pragma unroll 8
            for (int j = 1; j < s.k; ++j) {
              const float x = kls[j * KL_ROWS]; const int xi = kli[j * KL_ROWS];
              if (x < wv || (x == wv && xi > wi)) { wv = x; wi = xi; wj = j; }
            }
            thr = wv; kworst = wj;
          } else {
            ts[TK - 1] = v; ti[TK - 1] = id;
#pragma unroll
            for (int r = TK - 1; r > 0; --r) {          // strict: an equal maximum never overtakes an earlier unit
              if (ts[r] > ts[r - 1]) {
                const float fs = ts[r]; ts[r] = ts[r - 1]; ts[r - 1] = fs;
                const int is = ti[r]; ti[r] = ti[r - 1]; ti[r - 1] = is;
              }
            }
            thr = ts[TK - 1];
          }
        }
      };
      auto reduce_half = [&](uint32_t (&r0)[32], uint32_t (&r1)[16], uint32_t (&r2)[8], int limit) {
        if (limit < HALF) {                             // last tile of the table: columns past row_hi are not items
#pragma unroll
          for (int j = 0; j < 32; ++j) if (j >= limit) r0[j] = 0xff800000u;
          if constexpr ((HALF - 32) & 16) {
#pragma unroll
            for (int j = 0; j < 16; ++j) if (32 + j >= limit) r1[j] = 0xff800000u;
          }
          if constexpr ((HALF - 32) & 8) {
#pragma unroll
            for (int j = 0; j < 8; ++j) if (32 + ((HALF - 32) & 16) + j >= limit) r2[j] = 0xff800000u;
          }
        }
        float m[4];                                     // FMNMX3: two scores folded per ALU instruction, four chains
#pragma unroll
        for (int c = 0; c < 4; ++c) m[c] = fmaxf(__uint_as_float(r0[2 * c]), __uint_as_float(r0[2 * c + 1]));
#pragma unroll
        for (int j = 8; j < 32; j += 8) {
#pragma unroll
          for (int c = 0; c < 4; ++c) m[c] = fmax3(m[c], __uint_as_float(r0[j + 2 * c]), __uint_as_float(r0[j + 2 * c + 1]));
        }
        if constexpr ((HALF - 32) & 16) {
#pragma unroll
          for (int j = 0; j < 16; j += 8) {
#pragma unroll
            for (int c = 0; c < 4; ++c) m[c] = fmax3(m[c], __uint_as_float(r1[j + 2 * c]), __uint_as_float(r1[j + 2 * c + 1]));
          }
        }
        if constexpr ((HALF - 32) & 8) {
#pragma unroll
          for (int c = 0; c < 4; ++c) m[c] = fmax3(m[c], __uint_as_float(r2[2 * c]), __uint_as_float(r2[2 * c + 1]));
        }
        return fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3]));
      };
      // rank variant: items of one unit (columns already masked by reduce_half) ahead of the target; g0 = id of column 0
      auto count_half = [&](const uint32_t (&r0)[32], const uint32_t (&r1)[16], const uint32_t (&r2)[8], float m,
                            int g0) {
        auto col = [&](int j) {                         // j is a compile-time constant in the unrolled loops below
          return __uint_as_float(j < 32 ? r0[j] : (j < 32 + ((HALF - 32) & 16) ? r1[j - 32] : r2[j - 32 - ((HALF - 32) & 16)]));
        };
        int n = 0;
        if (m >= tsc) {                                 // else no item of the unit reaches the target's score
          const int p = tid - g0;                       // the target's column (outside 0 .. HALF - 1: another unit)
          const float thr = p >= HALF ? tsc_dn : tsc;   // all ids below the target's: ties count too
          int c[4] = {0, 0, 0, 0};
#pragma unroll
          for (int j = 0; j < HALF; ++j) c[j & 3] += col(j) > thr ? 1 : 0;
          n = (c[0] + c[1]) + (c[2] + c[3]);
          if (p >= 0 && p < HALF) {                     // the target's own unit: ties below its id count, it does not
#pragma unroll
            for (int j = 0; j < HALF; ++j) {
              const float x = col(j);
              n += (j < p && x == tsc) ? 1 : 0;
              n -= (j == p && x > tsc) ? 1 : 0;
            }
          }
        }
        return n;
      };
      bool ready = false;                               // this unit's tfull was already seen complete (tested a unit ahead)
      for (int t = t0; t < t1; ++t, ++n) {
        const int odd = n & 1, w = ub + 2 * odd;
        const bool tr = TRACE && blockIdx.x == 0 && n >= TR0 && n < TR0 + TRN && quarter == 0 && lane == 0;
        long long* trq = s.trace + (size_t)(2 * (n - TR0) + ub) * 12;
        if (tr) trq[4] = clock64();
        if (!ready) mbar_wait(&tfull[w], odd ? tph1 : tph0);
        if (odd) tph1 ^= 1; else tph0 ^= 1;
        tc_fence_after();
        if (tr) trq[5] = clock64();
        const int valid = s.row_hi - (s.row_lo + t * MT);   // real items in this tile (>= MT except in the last tile)
        float mA = 0.f, mB = 0.f;
        if (s.debug == 5) {                               // ablation: hand the accumulator back unread
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[w]);
          ready = false;
        } else {
          const uint32_t taddr = taddr0 + odd * (2 * MT);
          uint32_t a0[32], a1[16], a2[8], b0[32], b1[16], b2[8];
          tmem_ld32(taddr, a0);
          if constexpr ((HALF - 32) & 16) tmem_ld16(taddr + 32, a1);
          if constexpr ((HALF - 32) & 8) tmem_ld8(taddr + 32 + ((HALF - 32) & 16), a2);
          tmem_ld32(taddr + HALF, b0);
          if constexpr ((HALF - 32) & 16) tmem_ld16(taddr + HALF + 32, b1);
          if constexpr ((HALF - 32) & 8) tmem_ld8(taddr + HALF + 32 + ((HALF - 32) & 16), b2);
          tmem_ld_wait();
          tc_fence_before();                              // scores are in registers: hand the accumulator back now
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[w]);
          if (tr) trq[6] = clock64();
          // the next unit's barrier is tested now, its ~100-cycle answer is looked at after the maxima
          ready = t + 1 < t1 && mbar_try_wait(&tfull[ub + 2 * (odd ^ 1)], odd ? tph0 : tph1);
          mA = reduce_half(a0, a1, a2, valid);
          mB = reduce_half(b0, b1, b2, valid - HALF);
          if constexpr (RANK) {
            const int g0 = (int)(s.id_base + s.row_lo + t * MT);
            rcount += count_half(a0, a1, a2, mA, g0) + count_half(b0, b1, b2, mB, g0 + HALF);
          }
        }
        if (tr) trq[7] = clock64();
        if constexpr (!RANK) {
          offer(mA, 2 * t);
          offer(mB, 2 * t + 1);
        }
        if (tr) trq[8] = clock64();
      }
      if constexpr (RANK) {
        if (urow < s.U && rcount) atomicAdd(&s.rank_out[urow], rcount);
      } else if constexpr (KLIST) {
        if (urow < s.U) {
          const size_t o = ((size_t)urow * s.slots + piece * 2) * s.k;  // unsorted; phase 2 selects from it
          for (int r = 0; r < s.k; ++r) {
            s.out_scores[o + r] = kls[r * KL_ROWS];
            s.out_ids[o + r] = kli[r * KL_ROWS];
          }
        }
      } else if (urow < s.U) {
        const size_t o = ((size_t)urow * s.slots + piece * 2) * TK;     // the piece's second list slot stays empty
#pragma unroll
        for (int r = 0; r < TK; ++r) {
          s.out_scores[o + r] = ts[r];
          s.out_ids[o + r] = ti[r];
        }
      }
      lin += t1 - t0;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NEPI + 1) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ---------------------------------------------------------------------------------------------------------------
// Phase 2: one warp per user row.  Merge the row's tile-maxima lists into the TK best tiles (max desc, tile asc),
// re-score their TK x NT items with the same bf16 operands (fp32 accumulation), keep the exact top TK by
// (score desc, id asc) and write it into slot 0 of the row's list buffer (global ids); the other slots are emptied
// so that the merge kernel K9 sees one list per row and shard.
__device__ __forceinline__ bool better(float sa, int ia, float sb, int ib) {       // (score desc, id asc); id < 0 = empty
  if (ib < 0) return ia >= 0;
  if (ia < 0) return false;
  return sa > sb || (sa == sb && ia < ib);
}

__global__ void __launch_bounds__(256) catalogue_refine_kernel(TopkShape s) {
  const int lane = threadIdx.x & 31;
  const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= s.U) return;
  float* osc = s.out_scores + (size_t)u * s.slots * TK;
  int* oid = s.out_ids + (size_t)u * s.slots * TK;
  const int nent = s.slots * TK;
  // ---- 1. the TK best tiles: TK rounds of warp arg-best over the (value, tile) pairs, each lane holding a strided share
  int tiles[TK];
  float last_v = INFINITY; int last_t = -1;             // everything chosen so far is better than (last_v, last_t)
#pragma unroll 1
  for (int r = 0; r < TK; ++r) {
    float bv = -INFINITY; int bt = -1;
    for (int e = lane; e < nent; e += 32) {
      const float v = osc[e]; const int t = oid[e];
      if (t < 0) continue;
      const bool after_last = (last_t < 0) || v < last_v || (v == last_v && t > last_t);   // not chosen yet
      if (after_last && better(v, t, bv, bt)) { bv = v; bt = t; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int ot = __shfl_xor_sync(0xffffffffu, bt, o);
      if (better(ov, ot, bv, bt)) { bv = ov; bt = ot; }
    }
    tiles[r] = bt;
    if (bt >= 0) { last_v = bv; last_t = bt; }
  }
  __syncwarp();
  // ---- 2. exact scores of the candidate items; every lane keeps its own sorted top TK
  float ts[TK]; int ti[TK];
#pragma unroll
  for (int r = 0; r < TK; ++r) { ts[r] = -INFINITY; ti[r] = -1; }
#pragma unroll 1
  for (int r = 0; r < TK; ++r) {
    const int t = tiles[r];
    if (t < 0) continue;
    for (int j = lane; j < s.nt; j += 32) {
      const int row = s.row_lo + t * s.nt + j;
      if (row >= s.row_hi) continue;
      const uint4* e = reinterpret_cast<const uint4*>(s.table + (size_t)row * s.ld_table);
      float acc = 0.f;
      for (int sp = 0; sp < s.n_split; ++sp) {
        const uint4* f = reinterpret_cast<const uint4*>(s.feats + ((size_t)sp * s.u_pad + u) * s.ld_feats);
        float a = 0.f;
        for (int c = 0; c < s.D / 8; ++c) {
          const uint4 fv = __ldg(f + c), ev = __ldg(e + c);
          const uint32_t fw[4] = {fv.x, fv.y, fv.z, fv.w}, ew[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float2 x = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&fw[q]));
            const float2 y = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ew[q]));
            a = fmaf(x.x, y.x, a);
            a = fmaf(x.y, y.y, a);
          }
        }
        acc += a;
      }
      if (better(acc, row, ts[TK - 1], ti[TK - 1])) {
        ts[TK - 1] = acc; ti[TK - 1] = row;
#pragma unroll
        for (int k = TK - 1; k > 0; --k) {
          if (better(ts[k], ti[k], ts[k - 1], ti[k - 1])) {
            const float fs = ts[k]; ts[k] = ts[k - 1]; ts[k - 1] = fs;
            const int is = ti[k]; ti[k] = ti[k - 1]; ti[k - 1] = is;
          }
        }
      }
    }
  }
  // ---- 3. warp merge: TK rounds; the lane whose head wins pops it
  __syncwarp();
  for (int e = lane; e < nent; e += 32) oid[e] = -1;    // empty every slot (phase-1 entries are consumed)
  __syncwarp();
#pragma unroll 1
  for (int r = 0; r < TK; ++r) {
    float bv = ts[0]; int bi = ti[0]; int bl = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      const int ol = __shfl_xor_sync(0xffffffffu, bl, o);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; bl = ol; }
    }
    if (lane == 0) {
      const int gid = bi < 0 ? -1 : (int)(s.id_base + bi);
      osc[r] = bv; oid[r] = gid;
      if (s.packed) { s.packed[(size_t)u * 2 * TK + r] = bv; reinterpret_cast<int*>(s.packed)[(size_t)u * 2 * TK + TK + r] = gid; }
    }
    if (lane == bl && bi >= 0) {                        // pop my head
#pragma unroll
      for (int k = 0; k < TK - 1; ++k) { ts[k] = ts[k + 1]; ti[k] = ti[k + 1]; }
      ts[TK - 1] = -INFINITY; ti[TK - 1] = -1;
    }
  }
}

// Phase 2, fast form (D = 64, one split, table rows contiguous): same contract as catalogue_refine_kernel.
//   * A ranking unit is RU CONSECUTIVE table rows = RU * 128 contiguous bytes, so the warp reads it as RU / 4 fully
//     coalesced 512-byte requests (lane l, request i -> 16-byte piece i * 32 + l = row i * 4 + l / 8, features
//     8 (l % 8) .. + 8): every lane only ever needs ITS eighth of the user's features (4 registers), all RU / 4 loads of
//     a unit are in flight before the first is used, and a row's score is an 8-lane butterfly of 8-term partial sums.
//     The general kernel above walks one row per lane with two loads in flight (0.44 ms at 16 384 users: as long as
//     the whole streaming phase of a 125 k-row shard).
//   * Lane (l & ~7) + (i & 7) keeps row i * 4 + l / 8's score (static register index i >> 3), so the TK * RU exact scores
//     of a user sit in registers across the warp.
//   * Each of the TK units holds an item whose EXACT score is the unit's exact maximum, so the TK-th best exact score is
//     at least tau = min over units of that maximum: only scores >= tau survive (typically TK .. 2 TK of 560), they are
//     compacted into shared memory, and their order is found by counting (one pass for <= 32 survivors; the selection
//     rounds of step 1 otherwise -- dyadic test data with hundreds of exact ties takes that path).
template <int RU>
__global__ void __launch_bounds__(256, 2) catalogue_refine64_kernel(TopkShape s) {
  constexpr int NI = RU / 4;                          // 512-byte requests per unit
  constexpr int NK = (NI + 7) / 8;                    // scores a lane keeps per unit
  constexpr int CAP = TK * RU;                        // survivors per user, worst case
  static_assert(RU % 4 == 0 && NK <= 2, "refine64: ranking unit of 4 .. 64 rows in multiples of 4");
  __shared__ float sv_s[8][CAP];
  __shared__ int sv_i[8][CAP];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t u = (int64_t)blockIdx.x * 8 + wib;
  if (u >= s.U) return;
  float* osc = s.out_scores + (size_t)u * s.slots * TK;
  int* oid = s.out_ids + (size_t)u * s.slots * TK;
  const int nent = s.slots * TK;
  // this lane's eighth of the user's features
  float f[8];
  {
    const uint4 fv = __ldg(reinterpret_cast<const uint4*>(s.feats + (size_t)u * s.ld_feats) + (lane & 7));
    const uint32_t fw[4] = {fv.x, fv.y, fv.z, fv.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float2 x = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&fw[q]));
      f[2 * q] = x.x; f[2 * q + 1] = x.y;
    }
  }
  // ---- 1. the TK best units (max desc, unit asc): entries cached in registers (4 per lane covers 12 list slots)
  int tiles[TK];
  {
    float ev[4]; int et[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = lane + 32 * q;
      et[q] = e < nent ? oid[e] : -1;
      ev[q] = e < nent ? osc[e] : -INFINITY;
    }
    float last_v = INFINITY; int last_t = -1;
#pragma unroll 1
    for (int r = 0; r < TK; ++r) {
      float bv = -INFINITY; int bt = -1;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const bool after_last = (last_t < 0) || ev[q] < last_v || (ev[q] == last_v && et[q] > last_t);
        if (et[q] >= 0 && after_last && better(ev[q], et[q], bv, bt)) { bv = ev[q]; bt = et[q]; }
      }
      for (int e = lane + 128; e < nent; e += 32) {     // more than 12 slots: the rest straight from memory
        const float v = osc[e]; const int t = oid[e];
        if (t < 0) continue;
        const bool after_last = (last_t < 0) || v < last_v || (v == last_v && t > last_t);
        if (after_last && better(v, t, bv, bt)) { bv = v; bt = t; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int ot = __shfl_xor_sync(0xffffffffu, bt, o);
        if (better(ov, ot, bv, bt)) { bv = ov; bt = ot; }
      }
#pragma unroll
      for (int q = 0; q < TK; ++q) if (q == r) tiles[q] = bt;
      if (bt >= 0) { last_v = bv; last_t = bt; }
    }
  }
  __syncwarp();
  for (int e = lane; e < nent; e += 32) oid[e] = -1;    // empty every slot (phase-1 entries are consumed)
  // ---- 2. exact scores of the TK units
  float sc[TK][NK];
  float tau = INFINITY;
#pragma unroll
  for (int r = 0; r < TK; ++r) {
#pragma unroll
    for (int k = 0; k < NK; ++k) sc[r][k] = -INFINITY;
    const int t = tiles[r];
    if (t < 0) { tau = -INFINITY; continue; }           // warp-uniform
    const int row0 = s.row_lo + t * RU + (lane >> 3);
    const uint4* e0 = reinterpret_cast<const uint4*>(s.table + (size_t)row0 * 64) + (lane & 7);
    uint4 ev[NI];
#pragma unroll
    for (int i = 0; i < NI; ++i)
      ev[i] = (row0 + 4 * i < s.row_hi) ? __ldg(e0 + i * 32) : make_uint4(0, 0, 0, 0);
    float um = -INFINITY;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const uint32_t ew[4] = {ev[i].x, ev[i].y, ev[i].z, ev[i].w};
      float a = 0.f;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 y = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ew[q]));
        a = fmaf(f[2 * q], y.x, a);
        a = fmaf(f[2 * q + 1], y.y, a);
      }
      a += __shfl_xor_sync(0xffffffffu, a, 1);
      a += __shfl_xor_sync(0xffffffffu, a, 2);
      a += __shfl_xor_sync(0xffffffffu, a, 4);
      if (row0 + 4 * i >= s.row_hi) a = -INFINITY;       // past the table: not an item
      um = fmaxf(um, a);
      if ((i & 7) == (lane & 7)) sc[r][i >> 3] = a;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) um = fmaxf(um, __shfl_xor_sync(0xffffffffu, um, o));
    tau = fminf(tau, um);
  }
  // ---- 3. survivors (score >= tau) -> shared memory, in any order
  float* mv = sv_s[wib];
  int* mi = sv_i[wib];
  int ns = 0;
#pragma unroll
  for (int r = 0; r < TK; ++r) {
    if (tiles[r] < 0) continue;
#pragma unroll
    for (int k = 0; k < NK; ++k) {
      const float a = sc[r][k];
      const bool keep = a >= tau && a > -INFINITY;
      const uint32_t m = __ballot_sync(0xffffffffu, keep);
      if (keep) {
        const int i = k * 8 + (lane & 7);
        mv[ns + __popc(m & ((1u << lane) - 1))] = a;
        mi[ns + __popc(m & ((1u << lane) - 1))] = s.row_lo + tiles[r] * RU + 4 * i + (lane >> 3);
      }
      ns += __popc(m);
    }
  }
  __syncwarp();
  // ---- 4. order them: (score desc, row asc)
  float my_v = -INFINITY; int my_i = -1; int my_rank = TK;
  if (ns <= 32) {
    if (lane < ns) { my_v = mv[lane]; my_i = mi[lane]; }
    int rank = 0;
    for (int j = 0; j < ns; ++j) {
      const float ov = __shfl_sync(0xffffffffu, my_v, j);
      const int oi = __shfl_sync(0xffffffffu, my_i, j);
      rank += (ov > my_v || (ov == my_v && oi < my_i)) ? 1 : 0;
    }
    if (lane < ns) my_rank = rank;
    if (lane >= ns && lane < TK) my_rank = lane;         // fewer than TK candidates: the tail is empty (-inf, -1)
  } else {
    float last_v = INFINITY; int last_i = -1;
#pragma unroll 1
    for (int r = 0; r < TK; ++r) {
      float bv = -INFINITY; int bi = -1;
      for (int e = lane; e < ns; e += 32) {
        const float v = mv[e]; const int id = mi[e];
        const bool after_last = (last_i < 0) || v < last_v || (v == last_v && id > last_i);
        if (after_last && better(v, id, bv, bi)) { bv = v; bi = id; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      if (lane == r) { my_v = bv; my_i = bi; my_rank = r; }
      if (bi >= 0) { last_v = bv; last_i = bi; }
    }
  }
  if (my_rank < TK) {
    const int gid = my_i < 0 ? -1 : (int)(s.id_base + my_i);
    osc[my_rank] = my_v; oid[my_rank] = gid;
    if (s.packed) {
      s.packed[(size_t)u * 2 * TK + my_rank] = my_v;
      reinterpret_cast<int*>(s.packed)[(size_t)u * 2 * TK + TK + my_rank] = gid;
    }
  }
}

// Phase 2, k-list form (k = s.k in TK + 1 .. KMAX; unit form only, so a ranking unit is s.nt <= 56 rows).  One warp per
// user row, same contract as the two kernels above:
//   1. the k best units (max desc, unit asc): k rounds of warp arg-best over the row's (unsorted) per-piece lists;
//   2. the exact scores of their k x RU rows, same bf16 operands, fp32 accumulation, into this warp's shared memory.
//      RU = 56: the coalesced D = 64 form of catalogue_refine64_kernel (a unit is RU / 4 512-byte requests, a row's
//      score an 8-lane butterfly); RU = 0: one row per lane as in catalogue_refine_kernel (other widths and splits);
//   3. tau = the minimum exact unit maximum (-inf when the row has fewer than k units): the k-th best score is >= tau,
//      so only scores >= tau survive, typically k .. 2k of k x RU, compacted with (score, row);
//   4. order by counting: a survivor's rank is the number of survivors ahead of it in (score desc, row asc).  More than
//      KSCAP survivors (dyadic data with mass ties: every one of the k x RU scores can tie) take k selection rounds over
//      all k x RU scores instead;
//   5. slot 0 of the row's lists (and, when requested, the 8k-byte wire row) gets the k best, (-inf, -1) past the end.
static constexpr int KSCAP = 256;                     // survivors ordered by counting
static constexpr int KWARPS = 8;                      // warps (user rows) per block
__host__ __device__ constexpr size_t refine_k_warp_bytes(int k, int ru) {
  return (size_t)k * ru * 4 + (size_t)k * 4 + (size_t)KSCAP * 8;
}

template <int RU>
__global__ void __launch_bounds__(32 * KWARPS) catalogue_refine_k_kernel(TopkShape s) {
  static_assert(RU == 0 || RU == 56, "refine_k: RU 56 (D = 64) or 0 (general)");
  extern __shared__ uint8_t smem_raw[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t u = (int64_t)blockIdx.x * KWARPS + wib;
  if (u >= s.U) return;
  const int k = s.k, ru = RU ? RU : s.nt, ncand = k * ru;
  uint8_t* wsm = smem_raw + (size_t)wib * refine_k_warp_bytes(k, ru);
  float* sc = reinterpret_cast<float*>(wsm);                       // [k][ru] exact scores
  int* units = reinterpret_cast<int*>(sc + ncand);                 // [k] chosen units (-1: the row has fewer)
  float* sv = reinterpret_cast<float*>(units + k);                 // [KSCAP] survivors
  int* si = reinterpret_cast<int*>(sv + KSCAP);
  float* osc = s.out_scores + (size_t)u * s.slots * k;
  int* oid = s.out_ids + (size_t)u * s.slots * k;
  const int nent = s.slots * k;
  // ---- 1. the k best units
  {
    float last_v = INFINITY; int last_t = -1;
#pragma unroll 1
    for (int r = 0; r < k; ++r) {
      float bv = -INFINITY; int bt = -1;
      for (int e = lane; e < nent; e += 32) {
        const float v = osc[e]; const int t = oid[e];
        if (t < 0) continue;
        const bool after_last = (last_t < 0) || v < last_v || (v == last_v && t > last_t);
        if (after_last && better(v, t, bv, bt)) { bv = v; bt = t; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int ot = __shfl_xor_sync(0xffffffffu, bt, o);
        if (better(ov, ot, bv, bt)) { bv = ov; bt = ot; }
      }
      if (lane == 0) units[r] = bt;
      if (bt >= 0) { last_v = bv; last_t = bt; }
    }
  }
  __syncwarp();
  for (int e = lane; e < nent; e += 32) oid[e] = -1;    // empty every slot (phase-1 entries are consumed)
  // ---- 2. exact scores of the k units, tau
  float tau = INFINITY;
  if constexpr (RU != 0) {
    constexpr int NI = RU / 4;
    float f[8];                                         // this lane's eighth of the user's features
    {
      const uint4 fv = __ldg(reinterpret_cast<const uint4*>(s.feats + (size_t)u * s.ld_feats) + (lane & 7));
      const uint32_t fw[4] = {fv.x, fv.y, fv.z, fv.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float2 x = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&fw[q]));
        f[2 * q] = x.x; f[2 * q + 1] = x.y;
      }
    }
#pragma unroll 1
    for (int r = 0; r < k; ++r) {
      const int t = units[r];
      if (t < 0) { tau = -INFINITY; continue; }         // warp-uniform
      const int row0 = s.row_lo + t * RU + (lane >> 3);
      const uint4* e0 = reinterpret_cast<const uint4*>(s.table + (size_t)row0 * 64) + (lane & 7);
      uint4 ev[NI];
#pragma unroll
      for (int i = 0; i < NI; ++i)
        ev[i] = (row0 + 4 * i < s.row_hi) ? __ldg(e0 + i * 32) : make_uint4(0, 0, 0, 0);
      float um = -INFINITY;
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const uint32_t ew[4] = {ev[i].x, ev[i].y, ev[i].z, ev[i].w};
        float a = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float2 y = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ew[q]));
          a = fmaf(f[2 * q], y.x, a);
          a = fmaf(f[2 * q + 1], y.y, a);
        }
        a += __shfl_xor_sync(0xffffffffu, a, 1);
        a += __shfl_xor_sync(0xffffffffu, a, 2);
        a += __shfl_xor_sync(0xffffffffu, a, 4);
        if (row0 + 4 * i >= s.row_hi) a = -INFINITY;     // past the table: not an item
        um = fmaxf(um, a);
        if ((lane & 7) == 0) sc[r * RU + 4 * i + (lane >> 3)] = a;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) um = fmaxf(um, __shfl_xor_sync(0xffffffffu, um, o));
      tau = fminf(tau, um);
    }
  } else {
#pragma unroll 1
    for (int r = 0; r < k; ++r) {
      const int t = units[r];
      if (t < 0) { tau = -INFINITY; continue; }         // warp-uniform
      float um = -INFINITY;
      for (int j = lane; j < ru; j += 32) {
        const int row = s.row_lo + t * ru + j;
        float acc = -INFINITY;                          // past the table: not an item
        if (row < s.row_hi) {
          const uint4* e = reinterpret_cast<const uint4*>(s.table + (size_t)row * s.ld_table);
          acc = 0.f;
          for (int sp = 0; sp < s.n_split; ++sp) {
            const uint4* f = reinterpret_cast<const uint4*>(s.feats + ((size_t)sp * s.u_pad + u) * s.ld_feats);
            float a = 0.f;
            for (int c = 0; c < s.D / 8; ++c) {
              const uint4 fv = __ldg(f + c), ev = __ldg(e + c);
              const uint32_t fw[4] = {fv.x, fv.y, fv.z, fv.w}, ew[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float2 x = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&fw[q]));
                const float2 y = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ew[q]));
                a = fmaf(x.x, y.x, a);
                a = fmaf(x.y, y.y, a);
              }
            }
            acc += a;
          }
        }
        sc[r * ru + j] = acc;
        um = fmaxf(um, acc);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) um = fmaxf(um, __shfl_xor_sync(0xffffffffu, um, o));
      tau = fminf(tau, um);
    }
  }
  __syncwarp();
  // ---- 3. survivors (score >= tau) -> (sv, si), as many as fit; ns counts them all
  int ns = 0;
  for (int e0 = 0; e0 < ncand; e0 += 32) {
    const int e = e0 + lane;
    const int t = e < ncand ? units[e / ru] : -1;
    const float a = t >= 0 ? sc[e] : -INFINITY;
    const bool keep = a >= tau && a > -INFINITY;
    const uint32_t m = __ballot_sync(0xffffffffu, keep);
    const int at = ns + __popc(m & ((1u << lane) - 1));
    if (keep && at < KSCAP) { sv[at] = a; si[at] = s.row_lo + t * ru + e % ru; }
    ns += __popc(m);
  }
  __syncwarp();
  // ---- 4./5. order and write
  float* pk = s.packed ? s.packed + (size_t)u * 2 * k : nullptr;
  auto put = [&](int r, float v, int row) {
    const int gid = row < 0 ? -1 : (int)(s.id_base + row);
    osc[r] = v; oid[r] = gid;
    if (pk) { pk[r] = v; reinterpret_cast<int*>(pk)[k + r] = gid; }
  };
  if (ns <= KSCAP) {
    for (int e = lane; e < ns; e += 32) {
      const float v = sv[e]; const int row = si[e];
      int rank = 0;
      for (int j = 0; j < ns; ++j) rank += (sv[j] > v || (sv[j] == v && si[j] < row)) ? 1 : 0;
      if (rank < k) put(rank, v, row);
    }
    for (int r = ns + lane; r < k; r += 32) put(r, -INFINITY, -1);   // fewer than k items: the tail is empty
  } else {
    float last_v = INFINITY; int last_i = -1;
#pragma unroll 1
    for (int r = 0; r < k; ++r) {
      float bv = -INFINITY; int bi = -1;
      for (int e = lane; e < ncand; e += 32) {
        const int t = units[e / ru];
        if (t < 0) continue;
        const float v = sc[e]; const int id = s.row_lo + t * ru + e % ru;
        if (v == -INFINITY) continue;                   // past the table
        const bool after_last = (last_i < 0) || v < last_v || (v == last_v && id > last_i);
        if (after_last && better(v, id, bv, bi)) { bv = v; bi = id; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
      }
      if (lane == 0) put(r, bv, bi);
      if (bi >= 0) { last_v = bv; last_i = bi; }
    }
  }
}

// K9 for lists of L = k > TK entries, SORTED by (score desc, id asc) with empty entries (id < 0) only at the tail -- what
// phase 2 writes.  One warp per user.  The first k entries of every list are the only candidates; an entry's rank is its
// position in its own list plus, for every other list, the count of entries ahead of it (binary search: the lists are
// sorted).  Equal (score, id) in two lists are ordered by list index, so ranks are distinct and the result is the same
// on every rank that merges the same buffer.  List l of user u starts at word u * u_stride + l * l_stride of `sc` and
// of `ids`.
__global__ void __launch_bounds__(256) merge_topk_k_kernel(const float* sc, const int* ids, int64_t u_stride,
                                                           int64_t l_stride, int64_t U, int nlists, int k, float* out_sc,
                                                           int64_t* out_ids) {
  const int lane = threadIdx.x & 31;
  const int64_t u = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (u >= U) return;
  for (int r = lane; r < k; r += 32) { out_sc[u * k + r] = -INFINITY; out_ids[u * k + r] = -1; }
  __syncwarp();
  const float* s0 = sc + u * u_stride;
  const int* i0 = ids + u * u_stride;
  for (int e = lane; e < nlists * k; e += 32) {
    const int l = e / k, p = e % k;
    const float v = s0[l * l_stride + p]; const int id = i0[l * l_stride + p];
    if (id < 0) continue;
    int rank = p;
    for (int m = 0; m < nlists && rank < k; ++m) {
      if (m == l) continue;
      const float* sm = s0 + m * l_stride;
      const int* im = i0 + m * l_stride;
      int lo = 0, hi = k;                               // first entry of list m that is NOT ahead of (v, id, l)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const float y = sm[mid]; const int yi = im[mid];
        const bool ahead = yi >= 0 && (y > v || (y == v && (yi < id || (yi == id && m < l))));
        if (ahead) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) { out_sc[u * k + rank] = v; out_ids[u * k + rank] = id; }
  }
}

// K9: merge `nlists` candidate lists of length TK per user into the best k, order (score desc, id asc).
__global__ void merge_topk_kernel(const float* sc, const int* ids, int64_t U, int nlists, int k, float* out_sc,
                                  int64_t* out_ids) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= U) return;
  float ts[TK]; int ti[TK];
#pragma unroll
  for (int r = 0; r < TK; ++r) { ts[r] = -INFINITY; ti[r] = -1; }
  const float* s0 = sc + (size_t)u * nlists * TK;
  const int* i0 = ids + (size_t)u * nlists * TK;
  for (int n = 0; n < nlists * TK; ++n) {
    const float v = s0[n]; const int id = i0[n];
    if (id < 0) continue;
    const bool better = (ti[TK - 1] < 0) || v > ts[TK - 1] || (v == ts[TK - 1] && id < ti[TK - 1]);
    if (!better) continue;
    ts[TK - 1] = v; ti[TK - 1] = id;
#pragma unroll
    for (int r = TK - 1; r > 0; --r) {
      const bool up = (ti[r - 1] < 0) || ts[r] > ts[r - 1] || (ts[r] == ts[r - 1] && ti[r] < ti[r - 1]);
      if (up) {
        const float fs = ts[r]; ts[r] = ts[r - 1]; ts[r - 1] = fs;
        const int is = ti[r]; ti[r] = ti[r - 1]; ti[r - 1] = is;
      }
    }
  }
  for (int r = 0; r < k; ++r) {
    out_sc[u * k + r] = ts[r];
    out_ids[u * k + r] = ti[r];
  }
}

// K9 over the all-gathered send buffers: list l of user u is packed[(l * U + u) * 2 TK ...] = TK scores, TK int32 ids.
__global__ void merge_topk_packed_kernel(const float* packed, int64_t U, int nlists, int k, float* out_sc, int64_t* out_ids) {
  const int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= U) return;
  float ts[TK]; int ti[TK];
#pragma unroll
  for (int r = 0; r < TK; ++r) { ts[r] = -INFINITY; ti[r] = -1; }
  for (int l = 0; l < nlists; ++l) {
    const float* s0 = packed + ((size_t)l * U + u) * 2 * TK;
    const int* i0 = reinterpret_cast<const int*>(s0) + TK;
    for (int n = 0; n < TK; ++n) {
      const float v = s0[n]; const int id = i0[n];
      if (id < 0) continue;
      const bool better = (ti[TK - 1] < 0) || v > ts[TK - 1] || (v == ts[TK - 1] && id < ti[TK - 1]);
      if (!better) continue;
      ts[TK - 1] = v; ti[TK - 1] = id;
#pragma unroll
      for (int r = TK - 1; r > 0; --r) {
        const bool up = (ti[r - 1] < 0) || ts[r] > ts[r - 1] || (ts[r] == ts[r - 1] && ti[r] < ti[r - 1]);
        if (up) {
          const float fs = ts[r]; ts[r] = ts[r - 1]; ts[r - 1] = fs;
          const int is = ti[r]; ti[r] = ti[r - 1]; ti[r - 1] = is;
        }
      }
    }
  }
  for (int r = 0; r < k; ++r) {
    out_sc[u * k + r] = ts[r];
    out_ids[u * k + r] = ti[r];
  }
}

}  // namespace srfrd

using namespace srfrd;

// tile configuration: UBS user tiles x NT item columns x NACC accumulator stages;
// TMEM: NACC * UBS * NT accumulator + UBS * a_cols operand columns <= 512
struct TopkCfg { int ubs, nt, nacc, ru; };   // nt: item rows per MMA / smem tile; ru: rows per ranking unit (phase 2's "tile")
static TopkCfg pick_cfg(int D, int n_split) {
  const int a_cols = n_split * (D / 2);
  // unit form (catalogue_unitmax_kernel): 4 stages x MT columns + 2 user tiles x a_cols; SRFRD_TOPK_UNIT=0 keeps the
  // tile form for A/B timing
  static const bool unit_form = [] { const char* e = getenv("SRFRD_TOPK_UNIT"); return !(e && e[0] == '0'); }();
  const int mt = (512 - 2 * a_cols) / 4 / 16 * 16;
  if (unit_form && mt >= 64 && mt <= 112) return TopkCfg{2, mt, 4, mt / 2};
  const TopkCfg cands[] = {{2, 64, 3, 64}, {1, 64, 3, 64}, {1, 64, 2, 64}, {1, 32, 2, 32}};
  for (const TopkCfg& c : cands)
    if (c.nacc * c.ubs * c.nt + c.ubs * a_cols <= 512) return c;
  return TopkCfg{0, 0, 0, 0};
}

struct TopkPlan { int ugroups, tiles_total, grid, slots; int64_t share; };
static TopkPlan make_plan(const TopkCfg& c, int64_t U, int64_t n_rows, int64_t row_lo, int D) {
  TopkPlan p;
  const int64_t table_bytes = (n_rows - row_lo) * (int64_t)D * 2;
  // SRFRD_TOPK_ALIGN=0: the plain equal split (A/B timing)
  const char* align_env = getenv("SRFRD_TOPK_ALIGN");
  const bool aligned = !(align_env && align_env[0] == '0');
  p.tiles_total = (int)((n_rows - row_lo + c.nt - 1) / c.nt);
  p.ugroups = (int)((U + c.ubs * TILE_U - 1) / (c.ubs * TILE_U));
  const int64_t total = (int64_t)p.ugroups * p.tiles_total;
  int64_t grid = num_sms();
  if (grid > total) grid = total;
  // A piece restarts its lists cold (about 10 ln(n/10) insertions per row over n tiles): never cut a user group into
  // pieces shorter than 4096 items just to occupy more SMs.
  const int64_t min_tiles = 4096 / c.nt < 1 ? 1 : 4096 / c.nt;
  const int64_t min_share = p.tiles_total < min_tiles ? p.tiles_total : min_tiles;
  p.share = (total + grid - 1) / grid;
  if (p.share < min_share) p.share = min_share;
  // Time-aligned sweeps.  CTA i streams the item tiles [i * share, (i + 1) * share) mod tiles_total; CTAs run at the same
  // pace, so with share = (a / b) tiles_total there are only b distinct windows, each swept by grid / b CTAs TOGETHER (one
  // reads a tile from HBM, the others find it in L2) and the table crosses the HBM bus ~a times per pass.  The plain equal
  // split gives share = (37 / 16) tiles_total at 64 user groups on 148 SMs: 37 windows, 16 passes of a 128 MB table that
  // just misses L2 (ncu: 2.1 GB of DRAM reads for 0.13 GB of operands).  Taken when it costs at most 3 % of the SM time.
  if (table_bytes > (48ll << 20) && p.ugroups >= 2 && p.share > min_share) {
    int best_a = 1 << 30; int64_t best_share = 0;
    for (int b = 1; b <= 12; ++b) {
      int64_t a = ((int64_t)p.ugroups * b + grid - 1) / grid;
      const int64_t share = (a * p.tiles_total + b - 1) / b;
      if ((total + share - 1) / share > grid) continue;
      const double eff = (double)total / ((double)grid * (double)share);
      if (eff >= 0.97 && a < best_a) { best_a = (int)a; best_share = share; }
    }
    if (best_share > 0 && aligned) p.share = best_share;
  }
  p.grid = (int)((total + p.share - 1) / p.share);
  // a user group spans tiles_total consecutive indices; CTA boundaries fall on multiples of share
  const int64_t max_pieces = (p.tiles_total + p.share - 1) / p.share + 1;
  p.slots = (int)(2 * max_pieces);
  return p;
}

// Shared memory of the unit form (bytes, 227 KB a block): ring of `stages` k-blocks of MT item rows, the barrier area
// (2 * stages + 32 words), the k-list variant's 256 per-row lists of k (score, unit) pairs, alignment slack.
static constexpr int UNIT_SMEM_MAX = 227 * 1024;
static size_t unit_smem_bytes(int mt, int stages, int k) {
  return (size_t)stages * mt * KB * 2 + (size_t)(2 * stages + 32) * 8 + (k > TK ? (size_t)KL_ROWS * k * 8 : 0) + 2048;
}
// Ring length (k-blocks) of the unit form.  TK form: what 216 KB holds.  k-list variant: that, shortened to what its lists
// leave; a multiple of 2 * kblocks (each slot's parity belongs to two issuers) and at least 4 item tiles (tile n - 2's
// slot is refilled only after tile n's MMAs are issued); 0 = does not fit.
static int unit_stages(int mt, int kblocks, int k) {
  const int b_tile = mt * KB * 2, unit = 2 * kblocks;
  int stages = ((216 * 1024) / b_tile) / unit * unit;
  if (k <= TK) return stages;
  while (stages >= 2 * unit && unit_smem_bytes(mt, stages, k) > (size_t)UNIT_SMEM_MAX) stages -= unit;
  return stages >= 2 * unit ? stages : 0;
}
// Largest list length the plan serves for this width: TK for the tile form, else the largest k <= KMAX whose lists fit
// next to a 4-tile ring (D = 64: 64; D = 128, one split: 64; D = 256: 48).
static int topk_kmax(const TopkCfg& c, int D) {
  if (c.ubs == 0 || c.nacc != 4) return c.ubs ? TK : 0;
  int k = KMAX;
  while (k > TK && !unit_stages(c.nt, (D + KB - 1) / KB, k)) --k;
  return k;
}
static int check_k(const TopkCfg& c, int D, int n_split, int k) {
  SRFRD_REQUIRE(c.ubs > 0, "catalogue_topk: D=%d with n_split=%d does not fit tensor memory", D, n_split);
  SRFRD_REQUIRE(k >= 1 && k <= KMAX, "catalogue_topk: k must be in 1..%d (got %d)", KMAX, k);
  SRFRD_REQUIRE(k <= TK || c.nacc == 4, "catalogue_topk: k=%d > %d needs the unit form; D=%d with n_split=%d runs the tile "
                "form (n_split * D > 256), which keeps at most %d", k, TK, D, n_split, TK);
  const int kmax = topk_kmax(c, D);
  SRFRD_REQUIRE(k <= kmax, "catalogue_topk: k=%d exceeds the limit %d for D=%d with n_split=%d (the per-row lists must fit "
                "shared memory next to a 4-tile ring)", k, kmax, D, n_split);
  return 0;
}

extern "C" int srfrd_catalogue_topk_plan(int64_t U, int64_t n_rows, int64_t row_lo, int D, int n_split, int* chunks_out,
                                         int k) {
  SRFRD_REQUIRE(chunks_out, "catalogue_topk_plan: null output");
  const TopkCfg c = pick_cfg(D, n_split);
  if (int rc = check_k(c, D, n_split, k)) return rc;
  *chunks_out = make_plan(c, U, n_rows, row_lo, D).slots;
  return 0;
}

extern "C" int srfrd_catalogue_topk_kmax(int D, int n_split, int* kmax_out) {
  SRFRD_REQUIRE(kmax_out, "catalogue_topk_kmax: null output");
  const TopkCfg c = pick_cfg(D, n_split);
  SRFRD_REQUIRE(c.ubs > 0, "catalogue_topk: D=%d with n_split=%d does not fit tensor memory", D, n_split);
  *kmax_out = topk_kmax(c, D);
  return 0;
}

template <int UBS, int NT, int NACC>
static int launch_tilemax(const CUtensorMap& tmE, TopkShape& s, int grid, cudaStream_t stream) {
  const int b_tile = NT * KB * 2;
  const int nepi = 8 * UBS;
  const int list_bytes = (2 * TK + 1) * nepi * 32 * 4;
  const int unit = NACC * s.kblocks;                    // ring length must be a multiple of this (see kernel comment)
  s.stages = ((220 * 1024 - list_bytes) / b_tile) / unit * unit;
  if (s.stages > 8 * unit) s.stages = 8 * unit;
  SRFRD_REQUIRE(s.stages >= unit, "catalogue_topk: item tile ring does not fit shared memory");
  const size_t smem = (size_t)s.stages * b_tile + list_bytes + 1024 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    SRFRD_CUDA(cudaFuncSetAttribute(catalogue_tilemax_kernel<UBS, NT, NACC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  catalogue_tilemax_kernel<UBS, NT, NACC><<<grid, 32 * (nepi + 4), smem, stream>>>(tmE, s);
  SRFRD_LAUNCH_CHECK();
  return 0;
}

template <int MT>
static int launch_unitmax(const CUtensorMap& tmE, TopkShape& s, int grid, cudaStream_t stream) {
  const int unit = 2 * s.kblocks;                       // ring length: a multiple of 2 * kblocks (see kernel comment)
  s.stages = unit_stages(MT, s.kblocks, s.k);
  SRFRD_REQUIRE(s.stages >= unit, "catalogue_topk: item tile ring does not fit shared memory");
  const size_t smem = unit_smem_bytes(MT, s.stages, s.k);
  static bool attr_set = false;
  if (!attr_set) {
    SRFRD_CUDA(cudaFuncSetAttribute(catalogue_unitmax_kernel<MT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    SRFRD_CUDA(cudaFuncSetAttribute(catalogue_unitmax_kernel<MT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    SRFRD_CUDA(cudaFuncSetAttribute(catalogue_unitmax_kernel<MT, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  if (s.k > TK) catalogue_unitmax_kernel<MT, false, true><<<grid, 384, smem, stream>>>(tmE, s);
  else if (s.trace) catalogue_unitmax_kernel<MT, true><<<grid, 384, smem, stream>>>(tmE, s);
  else catalogue_unitmax_kernel<MT, false><<<grid, 384, smem, stream>>>(tmE, s);
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_catalogue_topk(const void* feats_bf16, int64_t U, int64_t u_pad, int n_split, const void* table_bf16,
                                    int64_t n_rows, int64_t row_lo, int64_t id_base, int D, int ld_feats, int ld_table,
                                    int chunks, float* part_scores, int* part_ids, float* packed_out, void* stream_, int k) {
  cudaStream_t stream = (cudaStream_t)stream_;
  SRFRD_REQUIRE(feats_bf16 && table_bf16 && part_scores && part_ids, "catalogue_topk: null pointer");
  SRFRD_REQUIRE(n_split >= 1 && n_split <= 3, "catalogue_topk: n_split must be 1..3");
  SRFRD_REQUIRE(D % 16 == 0 && ld_feats % 8 == 0 && ld_table % 8 == 0, "catalogue_topk: D %% 16 and ld %% 8 required (D=%d)", D);
  SRFRD_REQUIRE(((uintptr_t)feats_bf16 & 15) == 0 && ((uintptr_t)table_bf16 & 15) == 0, "catalogue_topk: operands must be 16-byte aligned");
  SRFRD_REQUIRE(U > 0 && n_rows > row_lo && row_lo >= 0, "catalogue_topk: empty problem");
  SRFRD_REQUIRE(n_rows < (1ll << 31) && id_base + n_rows < (1ll << 31), "catalogue_topk: ids must fit int32");
  const TopkCfg c = pick_cfg(D, n_split);
  if (int rc = check_k(c, D, n_split, k)) return rc;
  const int L = k > TK ? k : TK;                        // list length of every buffer
  const TopkPlan pl = make_plan(c, U, n_rows, row_lo, D);
  SRFRD_REQUIRE(chunks == pl.slots, "catalogue_topk: chunks must come from srfrd_catalogue_topk_plan");
  SRFRD_REQUIRE(u_pad >= U, "catalogue_topk: u_pad < U");
  TopkShape s;
  s.U = (int)U; s.D = D; s.n_split = n_split; s.u_pad = (int)u_pad;
  s.row_lo = (int)row_lo; s.row_hi = (int)n_rows; s.id_base = id_base;
  s.kblocks = (D + KB - 1) / KB;
  s.nt = c.ru;
  s.tiles_total = pl.tiles_total; s.ugroups = pl.ugroups; s.share = pl.share; s.slots = pl.slots;
  s.feats = (const bf16*)feats_bf16; s.ld_feats = ld_feats;
  s.table = (const bf16*)table_bf16; s.ld_table = ld_table;
  s.out_scores = part_scores; s.out_ids = part_ids; s.packed = packed_out;
  s.k = L;
  { const char* dbg = getenv("SRFRD_TOPK_DEBUG"); s.debug = dbg ? atoi(dbg) : 0; }
  s.trace = nullptr;
  const char* trace_path = getenv("SRFRD_TOPK_TRACE");
  const size_t trace_bytes = 512 * 12 * sizeof(long long);
  if (trace_path) {
    SRFRD_CUDA(cudaMalloc(&s.trace, trace_bytes));
    SRFRD_CUDA(cudaMemsetAsync(s.trace, 0, trace_bytes, stream));
  }
  // list slots a user group does not use stay empty (index -1)
  SRFRD_CUDA(cudaMemsetAsync(part_ids, 0xFF, (size_t)U * pl.slots * L * sizeof(int), stream));
  CUtensorMap tmE;
  if (int rc = make_tmap_bf16_2d(&tmE, table_bf16, n_rows, D, ld_table, c.nt, KB)) return rc;
  int rc;
  if (c.nacc == 4 && c.nt == 112) rc = launch_unitmax<112>(tmE, s, pl.grid, stream);
  else if (c.nacc == 4 && c.nt == 96) rc = launch_unitmax<96>(tmE, s, pl.grid, stream);
  else if (c.nacc == 4 && c.nt == 80) rc = launch_unitmax<80>(tmE, s, pl.grid, stream);
  else if (c.nacc == 4 && c.nt == 64) rc = launch_unitmax<64>(tmE, s, pl.grid, stream);
  else if (c.ubs == 2 && c.nt == 64 && c.nacc == 3) rc = launch_tilemax<2, 64, 3>(tmE, s, pl.grid, stream);
  else if (c.ubs == 1 && c.nt == 64 && c.nacc == 3) rc = launch_tilemax<1, 64, 3>(tmE, s, pl.grid, stream);
  else if (c.ubs == 1 && c.nt == 64 && c.nacc == 2) rc = launch_tilemax<1, 64, 2>(tmE, s, pl.grid, stream);
  else rc = launch_tilemax<1, 32, 2>(tmE, s, pl.grid, stream);
  if (rc) return rc;
  if (trace_path) {                                     // profiling only: synchronous dump of CTA 0's stamps
    static long long host_trace[512 * 12];
    SRFRD_CUDA(cudaMemcpyAsync(host_trace, s.trace, trace_bytes, cudaMemcpyDeviceToHost, stream));
    SRFRD_CUDA(cudaStreamSynchronize(stream));
    SRFRD_CUDA(cudaFree(s.trace));
    if (FILE* f = fopen(trace_path, "w")) {
      for (int q = 0; q < 512; ++q) {
        for (int j = 0; j < 12; ++j) fprintf(f, "%lld%c", host_trace[q * 12 + j], j == 11 ? '\n' : ' ');
      }
      fclose(f);
    }
  }
  if (s.debug == 2) return 0;                           // profiling: phase 1 only
  // SRFRD_TOPK_REFINE=0: the general one-row-per-lane kernel everywhere (A/B timing)
  const char* refine_env = getenv("SRFRD_TOPK_REFINE");
  const bool fast_refine = !(refine_env && refine_env[0] == '0');
  const bool fast = fast_refine && D == 64 && n_split == 1 && ld_table == 64;
  if (k > TK) {
    const size_t smem = KWARPS * refine_k_warp_bytes(L, c.ru);
    static bool attr_set = false;
    if (!attr_set) {
      SRFRD_CUDA(cudaFuncSetAttribute(catalogue_refine_k_kernel<56>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      SRFRD_CUDA(cudaFuncSetAttribute(catalogue_refine_k_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      attr_set = true;
    }
    const unsigned blocks = (unsigned)((U + KWARPS - 1) / KWARPS);
    if (fast && c.ru == 56) catalogue_refine_k_kernel<56><<<blocks, 32 * KWARPS, smem, stream>>>(s);
    else catalogue_refine_k_kernel<0><<<blocks, 32 * KWARPS, smem, stream>>>(s);
  } else if (fast && c.ru == 56) catalogue_refine64_kernel<56><<<(unsigned)((U + 7) / 8), 256, 0, stream>>>(s);
  else if (fast && c.ru == 64) catalogue_refine64_kernel<64><<<(unsigned)((U + 7) / 8), 256, 0, stream>>>(s);
  else catalogue_refine_kernel<<<(unsigned)((U + 7) / 8), 256, 0, stream>>>(s);
  SRFRD_LAUNCH_CHECK();
  return 0;
}

template <int MT>
static int launch_unitrank(const CUtensorMap& tmE, TopkShape& s, int grid, cudaStream_t stream) {
  s.stages = unit_stages(MT, s.kblocks, TK);            // no lists: the top-10 form's full ring
  SRFRD_REQUIRE(s.stages >= 2 * s.kblocks, "catalogue_rank: item tile ring does not fit shared memory");
  const size_t smem = unit_smem_bytes(MT, s.stages, TK);
  static bool attr_set = false;
  if (!attr_set) {
    SRFRD_CUDA(cudaFuncSetAttribute(catalogue_unitmax_kernel<MT, false, false, true>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  catalogue_unitmax_kernel<MT, false, false, true><<<grid, 384, smem, stream>>>(tmE, s);
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_catalogue_rank(const void* feats_bf16, int64_t U, int64_t u_pad, int n_split, const void* table_bf16,
                                    int64_t n_rows, int64_t row_lo, int64_t id_base, int D, int ld_feats, int ld_table,
                                    const void* target_rows_bf16, int ld_target, const int64_t* target_ids,
                                    float* target_scores, int* rank_out, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  SRFRD_REQUIRE(feats_bf16 && table_bf16 && target_rows_bf16 && target_ids && rank_out, "catalogue_rank: null pointer");
  SRFRD_REQUIRE(n_split >= 1 && n_split <= 3, "catalogue_rank: n_split must be 1..3");
  SRFRD_REQUIRE(D % 16 == 0 && ld_feats % 8 == 0 && ld_table % 8 == 0 && ld_target % 8 == 0 && ld_target >= D,
                "catalogue_rank: D %% 16 and ld %% 8 required (D=%d)", D);
  SRFRD_REQUIRE(((uintptr_t)feats_bf16 & 15) == 0 && ((uintptr_t)table_bf16 & 15) == 0 &&
                ((uintptr_t)target_rows_bf16 & 15) == 0, "catalogue_rank: operands must be 16-byte aligned");
  SRFRD_REQUIRE(U > 0 && n_rows > row_lo && row_lo >= 0, "catalogue_rank: empty problem");
  SRFRD_REQUIRE(n_rows < (1ll << 31) && id_base + n_rows < (1ll << 31), "catalogue_rank: ids must fit int32");
  SRFRD_REQUIRE(u_pad >= U, "catalogue_rank: u_pad < U");
  const TopkCfg c = pick_cfg(D, n_split);
  SRFRD_REQUIRE(c.ubs > 0 && c.nacc == 4, "catalogue_rank: needs the unit form (n_split * D <= 256); D=%d with n_split=%d "
                "runs the tile form", D, n_split);
  const TopkPlan pl = make_plan(c, U, n_rows, row_lo, D);
  TopkShape s = {};
  s.U = (int)U; s.D = D; s.n_split = n_split; s.u_pad = (int)u_pad;
  s.row_lo = (int)row_lo; s.row_hi = (int)n_rows; s.id_base = id_base;
  s.kblocks = (D + KB - 1) / KB;
  s.nt = c.ru;
  s.tiles_total = pl.tiles_total; s.ugroups = pl.ugroups; s.share = pl.share; s.slots = pl.slots;
  s.feats = (const bf16*)feats_bf16; s.ld_feats = ld_feats;
  s.table = (const bf16*)table_bf16; s.ld_table = ld_table;
  s.k = TK;
  s.target_rows = (const bf16*)target_rows_bf16; s.ld_target = ld_target;
  s.target_ids = target_ids; s.target_scores = target_scores; s.rank_out = rank_out;
  SRFRD_CUDA(cudaMemsetAsync(rank_out, 0, (size_t)U * sizeof(int), stream));
  CUtensorMap tmE;
  if (int rc = make_tmap_bf16_2d(&tmE, table_bf16, n_rows, D, ld_table, c.nt, KB)) return rc;
  if (c.nt == 112) return launch_unitrank<112>(tmE, s, pl.grid, stream);
  if (c.nt == 96) return launch_unitrank<96>(tmE, s, pl.grid, stream);
  if (c.nt == 80) return launch_unitrank<80>(tmE, s, pl.grid, stream);
  return launch_unitrank<64>(tmE, s, pl.grid, stream);
}

extern "C" int srfrd_merge_topk(const float* scores, const int* ids, int64_t U, int nlists, int k, float* out_scores,
                                int64_t* out_ids, void* stream) {
  SRFRD_REQUIRE(scores && ids && out_scores && out_ids, "merge_topk: null pointer");
  SRFRD_REQUIRE(k >= 1 && k <= KMAX, "merge_topk: k must be in 1..%d", KMAX);
  if (U == 0) return 0;
  if (k > TK)                                           // lists of k entries
    merge_topk_k_kernel<<<(unsigned)((U + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        scores, ids, (int64_t)nlists * k, k, U, nlists, k, out_scores, out_ids);
  else
    merge_topk_kernel<<<(unsigned)((U + 127) / 128), 128, 0, (cudaStream_t)stream>>>(scores, ids, U, nlists, k, out_scores, out_ids);
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_merge_topk_packed(const float* packed, int64_t U, int nlists, int k, float* out_scores,
                                       int64_t* out_ids, void* stream) {
  SRFRD_REQUIRE(packed && out_scores && out_ids, "merge_topk_packed: null pointer");
  SRFRD_REQUIRE(k >= 1 && k <= KMAX && nlists >= 1, "merge_topk_packed: k must be in 1..%d", KMAX);
  if (U == 0) return 0;
  if (k > TK)                                           // wire rows of k scores + k ids
    merge_topk_k_kernel<<<(unsigned)((U + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        packed, reinterpret_cast<const int*>(packed) + k, 2 * k, U * 2 * k, U, nlists, k, out_scores, out_ids);
  else
    merge_topk_packed_kernel<<<(unsigned)((U + 127) / 128), 128, 0, (cudaStream_t)stream>>>(packed, U, nlists, k, out_scores, out_ids);
  SRFRD_LAUNCH_CHECK();
  return 0;
}
