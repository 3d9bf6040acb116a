// Shared device/host helpers for the srfrd_b200 kernels (sm_100a only).
#pragma once
#include <stdlib.h>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "srfrd_b200 kernels are written for sm_100a (B200) only"
#endif

namespace srfrd {

typedef __nv_bfloat16 bf16;

// ---------------------------------------------------------------------------------------------
// host-side error reporting (api.cu owns the storage)
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define SRFRD_CUDA(expr)                                                           \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) return ::srfrd::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define SRFRD_REQUIRE(cond, ...)          \
  do {                                    \
    if (!(cond)) {                        \
      ::srfrd::set_error(__VA_ARGS__);    \
      return 2;                           \
    }                                     \
  } while (0)

#define SRFRD_LAUNCH_CHECK() SRFRD_CUDA(cudaGetLastError())

// Programmatic dependent launch: a kernel launched through launch_pdl may begin (prologue: barrier init, TMEM
// allocation, descriptor prefetch) while the previous kernel of the stream / graph is still draining; it must call
// pdl_prologue_done() before it touches anything an earlier kernel wrote.  Opt-in: SRFRD_PDL=1 (see api.cu).
bool pdl_enabled();
// Dynamic row count (srfrd_set_row_limit): device pointer the row-wise entry points read their row count from, or null.
const int* row_limit();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

inline int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
// wait until every earlier grid has completed and its writes are visible, then allow the next grid to start launching
__device__ __forceinline__ void pdl_prologue_done() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {   // SASS FMNMX3 (sm_100+)
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float bf2f(bf16 v) { return __bfloat162float(v); }
__device__ __forceinline__ bf16 f2bf(float v) { return __float2bfloat16_rn(v); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ void unpack_bf16x8(const uint4& u, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __nv_bfloat162 t = *reinterpret_cast<const __nv_bfloat162*>(&w[i]);
    f[2 * i] = __low2float(t);
    f[2 * i + 1] = __high2float(t);
  }
}

// LayerNorm of a result row in a GEMM epilogue (gemm_tn's LNF kernels, the attention kernel's fused out-projection): the
// statistics are those of the ROUNDED bf16 values (what a separate LayerNorm kernel would read back).  Each thread
// accumulates its own columns, the threads of a row then combine their partial (sum, sum of squares).
__device__ __forceinline__ void lnf_accum8(const uint4& pk, float& sum, float& sq) {
  const uint32_t pw[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float lo = __uint_as_float(pw[i] << 16), hi = __uint_as_float(pw[i] & 0xffff0000u);
    sum += lo + hi;
    sq = fmaf(lo, lo, fmaf(hi, hi, sq));
  }
}
// (own partial sums, the row partner's) -> mean, rstd and nb = -mean * rstd over n columns
__device__ __forceinline__ void lnf_stats(float sum, float sq, float osum, float osq, int n, float eps, float& mean,
                                          float& rstd, float& nb) {
  const float invn = 1.f / (float)n;
  mean = (sum + osum) * invn;
  const float var = fmaxf((sq + osq) * invn - mean * mean, 0.f);
  rstd = rsqrtf(var + eps);
  nb = -mean * rstd;
}
// 8 rounded values -> 8 normalised, scaled and shifted bf16 values (w, b: the LayerNorm weight / bias of these columns)
__device__ __forceinline__ uint4 lnf_apply8(const uint4& x, float rstd, float nb, const float* w, const float* b) {
  float f[8], y[8];
  unpack_bf16x8(x, f);
#pragma unroll
  for (int i = 0; i < 8; ++i) y[i] = fmaf(fmaf(f[i], rstd, nb), w[i], b[i]);
  return make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]), pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
}
__device__ __forceinline__ void red_add_f32(float* addr, float v) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Stateless counter-based RNG for dropout: the same (seed, stream, index) always gives the same
// bit, so backward regenerates the forward mask instead of storing it.
__device__ __forceinline__ uint32_t hash_u32(uint64_t seed, uint32_t stream, uint64_t idx) {
  // 32-bit arithmetic only: the mask of an attention tile is one hash per (query, key) pair, evaluated again in the backward
  // pass, and a splitmix64 finaliser (two 64-bit multiplies = ~25 instructions) made dropout double the attention kernels'
  // time (C2 at p = 0.5: forward 32 -> 58 us, backward 53 -> 105 us per step).  The seed / stream terms are loop invariant;
  // per element this is two multiplies for the fold and the lowbias32 finaliser (full avalanche on 32 bits).
  uint32_t x = (uint32_t)idx * 0x9E3779B1u ^ (uint32_t)(idx >> 32) * 0x85EBCA77u ^ (uint32_t)seed ^
               (uint32_t)(seed >> 32) * 0xC2B2AE3Du ^ stream * 0x27D4EB2Fu;
  x ^= x >> 16; x *= 0x7FEB352Du;
  x ^= x >> 15; x *= 0x846CA68Bu;
  x ^= x >> 16;
  return x;
}
__device__ __forceinline__ uint64_t mix_seed(uint64_t seed, const float* step) {
  return step ? seed ^ ((uint64_t)__float_as_uint(__ldg(step)) * 0xD6E8FEB86659FD93ull) : seed;
}
// keep-mask: true with probability 1-p; threshold = p * 2^32
__device__ __forceinline__ bool dropout_keep(uint64_t seed, uint32_t stream, uint64_t idx, uint32_t thresh) {
  return hash_u32(seed, stream, idx) >= thresh;
}

// ---------------------------------------------------------------------------------------------
// mbarrier / TMA / tcgen05 PTX wrappers
// ---------------------------------------------------------------------------------------------
// one lane of a converged warp (warp-uniform control flow around the single-thread tcgen05 / TMA issue)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Spin with a watchdog: a mis-programmed pipeline traps (-> launch error) instead of hanging the GPU.
// (A leaner spin -- try_wait + branch + counter with the clock behind an out-of-line call -- was tried in round 2: ncu's
//  source view shows the watchdog arithmetic below is evaluated on every failed test, 12 issue slots each.  It measured
//  WORSE in the catalogue kernel, 4.9 vs 3.0 ms: the extra instructions act as a back-off, and a tight try_wait loop in
//  13 waiting warps starves the warps that would complete the barriers.  Kept as it was.)
__device__ __forceinline__ bool mbar_try_wait_a(uint32_t bar_addr, uint32_t parity) {   // bar_addr: shared-space address
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar_addr), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar_addr, uint32_t parity) {
  if (mbar_try_wait_a(bar_addr, parity)) return;
  long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait_a(bar_addr, parity)) {
    if (((++spins) & 0x3ffu) == 0 && (clock64() - t0) > 4000000000ll) {
      printf("srfrd_b200: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait_a(smem_u32(bar), parity); }
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar_addr) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}

// Several barriers at once: an mbarrier test costs ~250 cycles even when the phase completed long ago (measured), so the
// tests are issued back to back and only then examined -- their latencies overlap instead of adding up.
__device__ __forceinline__ void mbar_wait2(uint64_t* a, uint32_t pa, uint64_t* b, uint32_t pb) {
  const bool oa = mbar_try_wait(a, pa), ob = mbar_try_wait(b, pb);
  if (!oa) mbar_wait(a, pa);
  if (!ob) mbar_wait(b, pb);
}
__device__ __forceinline__ void mbar_wait3(uint64_t* a, uint32_t pa, uint64_t* b, uint32_t pb, uint64_t* c, uint32_t pc) {
  const bool oa = mbar_try_wait(a, pa), ob = mbar_try_wait(b, pb), oc = mbar_try_wait(c, pc);
  if (!oa) mbar_wait(a, pa);
  if (!ob) mbar_wait(b, pb);
  if (!oc) mbar_wait(c, pc);
}

#define SRFRD_EVICT_NORMAL 0x1000000000000000ull
#define SRFRD_EVICT_FIRST 0x12F0000000000000ull
#define SRFRD_EVICT_LAST 0x14F0000000000000ull

// Ask the TMA unit to pull a box into L2 only (no shared memory, no barrier).  Issued one or more tiles ahead of the real
// load, whose latency then is the L2 -> SM leg instead of an HBM round trip under load (~3 700 cycles measured).
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* tmap, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(tmap), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1,
                                            uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], bf16 operands, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns (thread i <- lane base+i).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld1(uint32_t taddr, uint32_t& v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// UMMA descriptors (bit layouts per the PTX ISA "tcgen05 matrix/instruction descriptor" tables)
// ---------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, 128-byte swizzle, operand tiles written by TMA with
// CU_TENSOR_MAP_SWIZZLE_128B into 1024-byte-aligned smem.
//   [0,14)  start address >> 4      [16,30) leading byte offset >> 4   [32,46) stride byte offset >> 4
//   [46,48) version = 1 (sm_100)    [61,64) layout type: 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor for kind::f16 with BF16 A/B and FP32 accumulator.
//   [4,6) c_format = 1 (F32)  [7,10) a_format = 1 (BF16)  [10,13) b_format = 1 (BF16)
//   [15] a_major (0 = K-major, 1 = MN-major)  [16] b_major  [17,23) N >> 3  [24,29) M >> 4
__host__ __device__ __forceinline__ uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;
  d |= 1u << 7;
  d |= 1u << 10;
  d |= (uint32_t)(a_mn_major & 1) << 15;
  d |= (uint32_t)(b_mn_major & 1) << 16;
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

// ---------------------------------------------------------------------------------------------
// host: TMA descriptor construction (driver entry point fetched through the runtime, so the
// library does not link against libcuda)
// ---------------------------------------------------------------------------------------------
// 2-D bf16 row-major tensor [rows, cols] with row pitch ld (elements); box = [box_rows, box_cols];
// 128-byte swizzle (box_cols * 2 bytes must be <= 128); out-of-bounds elements read as zero.
int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_rows, uint32_t box_cols);

// ---- l2_emb regulariser: segment table of the flat parameter buffer (loss_scatter_adam.cu, dp_adam.cu)
static constexpr int L2_THREADS = 256;            // threads of srfrd_param_l2 = the most tensors it supports

// Segment lookup of the Adam variants that add the regulariser's gradient: s_off[t] = float4 index where tensor t starts.
// A thread's grid-stride indices only increase, so it finds its first segment by binary search and then walks forward.
struct L2Segments {
  const int64_t* seg;        // device {offset, numel} per tensor (offsets 4-aligned, increasing)
  int n_seg;
  const float* coef;         // l2 / ||p_t|| per tensor (srfrd_param_l2)
  const float* reg;          // l2 * sum_t ||p_t||, added to the published loss
};

// The tables live in a function-scope shared buffer, so a kernel's plain (l2-off) instantiation allocates none of it.
struct L2Smem { int64_t off[L2_THREADS]; float coef[L2_THREADS]; };
__device__ __forceinline__ L2Smem& l2_smem() { __shared__ L2Smem s; return s; }

__device__ __forceinline__ void l2_load_starts(const L2Segments& l2s, int64_t* s_off, float* s_coef) {
  for (int t = threadIdx.x; t < l2s.n_seg; t += blockDim.x) {
    s_off[t] = l2s.seg[2 * t] >> 2;
    s_coef[t] = l2s.coef[t];
  }
}

__device__ __forceinline__ int l2_find(const int64_t* s_off, int n_seg, int64_t i4) {
  int lo = 0, hi = n_seg - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (s_off[mid] <= i4) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__device__ __forceinline__ int l2_advance(const int64_t* s_off, int n_seg, int t, int64_t i4) {
  while (t + 1 < n_seg && s_off[t + 1] <= i4) ++t;
  return t;
}

}  // namespace srfrd
