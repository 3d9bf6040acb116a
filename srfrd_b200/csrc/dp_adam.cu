// Data-parallel gradient exchange fused with the optimizer, over NVLink peer memory (SURVEY.md 8e row "Training").
//
// The reference has no data parallelism; the obvious build -- NCCL all-reduce of the flat gradient bucket, then the same
// dense Adam on every rank -- leaves a ~55 us collective plus a 16 us optimizer at the end of a 0.48 ms step.  Here ONE
// kernel per rank does reduce-scatter -> Adam -> all-gather through peer pointers (torch symmetric memory; every rank's
// gradient bucket and parameter buffer are mapped into every process):
//   1. entry barrier: every rank's gradients are complete (release / acquire flags in each rank's signal words)
//   2. rank r owns elements [r n/G, (r+1) n/G): it sums that slice of ALL ranks' gradient buckets in rank order
//      (local + G-1 peer loads), applies torch.optim.Adam's arithmetic with ITS slice of the moments (no rank needs the
//      others' m, v), writes the new parameters into EVERY rank's parameter buffer and zeroes every rank's gradient slice
//      (each slice has exactly one reader, so zeroing right after the read is race-free)
//   3. rank 0 also reduces the two loss accumulators in the bucket's tail and writes the loss to every rank
//   4. exit barrier: all ranks have finished writing parameters everywhere
// Every element is computed by exactly one rank, so the replicas stay bit-identical.  NVLink traffic per rank:
// (G-1)/G of the bucket in, the same out -- half of an all-reduce -- and the optimizer's HBM traffic drops by G.
#include "common.cuh"
#include "srfrd_b200.h"

namespace srfrd {

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// bounded spin: a missing peer traps (launch error) instead of hanging the GPU until NCCL's watchdog fires
__device__ __forceinline__ void spin_until_sys(const uint32_t* p, uint32_t e) {
  long long t0 = clock64();
  while ((int)(ld_acquire_sys(p) - e) < 0) {
    if (clock64() - t0 > 20000000000ll) { printf("srfrd_b200: dp_adam peer barrier timed out\n"); __trap(); }
  }
}
__device__ __forceinline__ void spin_until_gpu(const uint32_t* p, uint32_t e) {
  long long t0 = clock64();
  while ((int)(ld_acquire_gpu(p) - e) < 0) {
    if (clock64() - t0 > 20000000000ll) { printf("srfrd_b200: dp_adam grid barrier timed out\n"); __trap(); }
  }
}

static constexpr int DP_MAX_WORLD = 16;
static constexpr int DP_THREADS = 512;

struct DpAdam {
  float* const* grad;        // device array [world]: every rank's gradient bucket (n + 4 floats; tail = loss accumulators)
  float* const* param;       // device array [world]: every rank's parameter buffer (n + 4 floats; tail[0] = loss)
  uint32_t* const* sig;      // device array [world]: every rank's signal words (>= world uint32)
  int rank, world;
  int64_t n;                 // parameters (multiple of 4)
  float* m; float* v;        // local moments (full length; only the owned slice is touched)
  float lr, beta1, beta2, eps;
  float* state;              // local Adam state8
  const float* norm;         // local (already all-reduced) weight sums
  uint32_t* local;           // local words: [0] epoch, [1] grid arrival counter, [2] exit flag, [3] entry flag
  L2Segments l2s;            // l2_emb regulariser (L2 instantiation only)
};

// L2: g += coef[tensor] * p on the reduced gradient (added once, after the sum over ranks) and rank 0 adds reg to the loss.
template <bool L2>
__global__ void __launch_bounds__(DP_THREADS, 1) dp_adam_kernel(DpAdam p) {
  __shared__ float s_bc[2];
  __shared__ uint32_t s_epoch;
  pdl_prologue_done();
  const int tid = threadIdx.x;
  int64_t* s_off = nullptr;
  float* s_coef = nullptr;
  if constexpr (L2) {
    s_off = l2_smem().off;
    s_coef = l2_smem().coef;
    l2_load_starts(p.l2s, s_off, s_coef);
  }
  if (tid == 0) {
    s_epoch = p.local[0];
    const float step = p.state[0] + 1.f;
    s_bc[0] = (float)(1.0 - pow((double)p.beta1, (double)step));
    s_bc[1] = (float)(1.0 - pow((double)p.beta2, (double)step));
  }
  __syncthreads();
  const uint32_t e = s_epoch + 1;
  // ---- 1. entry barrier across ranks (block 0), then across this rank's blocks
  if (blockIdx.x == 0) {
    if (tid < p.world) {
      __threadfence_system();
      st_release_sys(p.sig[tid] + p.rank, e);               // peer tid: my gradients are complete
      spin_until_sys(p.sig[p.rank] + tid, e);                // peer tid's gradients are complete
    }
    __syncthreads();
    if (tid == 0) st_release_gpu(p.local + 3, e);
  } else {
    if (tid == 0) spin_until_gpu(p.local + 3, e);
    __syncthreads();
  }
  // ---- 2. my slice: reduce, Adam, broadcast, zero
  const float step_size = p.lr / s_bc[0];
  const float inv_sqrt_bc2 = rsqrtf(s_bc[1]);
  const int64_t n4 = p.n >> 2;
  const int64_t per = (n4 + p.world - 1) / p.world;
  const int64_t lo = (int64_t)p.rank * per, hi = min(n4, lo + per);
  float4* gp[DP_MAX_WORLD]; float4* pp_[DP_MAX_WORLD];
#pragma unroll
  for (int r = 0; r < DP_MAX_WORLD; ++r) {
    gp[r] = r < p.world ? reinterpret_cast<float4*>(p.grad[r]) : nullptr;
    pp_[r] = r < p.world ? reinterpret_cast<float4*>(p.param[r]) : nullptr;
  }
  int sg = 0;
  if constexpr (L2) sg = l2_find(s_off, p.l2s.n_seg, lo + (int64_t)blockIdx.x * blockDim.x + tid);
  for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + tid; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < DP_MAX_WORLD; ++r)
      if (r < p.world) {
        const float4 t = __ldcg(gp[r] + i);
        g.x += t.x; g.y += t.y; g.z += t.z; g.w += t.w;
      }
    float4 w = pp_[p.rank][i];
    float4 mm = reinterpret_cast<float4*>(p.m)[i], vv = reinterpret_cast<float4*>(p.v)[i];
    float* wa = &w.x; float* ga = &g.x; float* ma = &mm.x; float* va = &vv.x;
    if constexpr (L2) {
      sg = l2_advance(s_off, p.l2s.n_seg, sg, i);
      const float c = s_coef[sg];
#pragma unroll
      for (int j = 0; j < 4; ++j) ga[j] += c * wa[j];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ma[j] = p.beta1 * ma[j] + (1.f - p.beta1) * ga[j];
      va[j] = p.beta2 * va[j] + (1.f - p.beta2) * ga[j] * ga[j];
      wa[j] -= step_size * ma[j] / (sqrtf(va[j]) * inv_sqrt_bc2 + p.eps);
    }
    reinterpret_cast<float4*>(p.m)[i] = mm;
    reinterpret_cast<float4*>(p.v)[i] = vv;
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < DP_MAX_WORLD; ++r)
      if (r < p.world) { pp_[r][i] = w; gp[r][i] = z; }
  }
  // ---- 3. loss (rank 0 owns the bucket's tail)
  if (p.rank == 0 && blockIdx.x == 0 && tid == 0) {
    float a = 0.f, b = 0.f;
    for (int r = 0; r < p.world; ++r) { a += __ldcg(p.grad[r] + p.n); b += __ldcg(p.grad[r] + p.n + 1); }
    float loss = (p.norm[0] > 0.f ? a / p.norm[0] : 0.f) + (p.norm[1] > 0.f ? b / p.norm[1] : 0.f);
    if constexpr (L2) loss = loss + p.l2s.reg[0];
    for (int r = 0; r < p.world; ++r) { p.param[r][p.n] = loss; p.grad[r][p.n] = 0.f; p.grad[r][p.n + 1] = 0.f; }
  }
  // ---- 4. all blocks of this rank done -> exit barrier across ranks -> release this rank's blocks
  __threadfence_system();
  __syncthreads();
  if (tid == 0) {
    if (atomicAdd(p.local + 1, 1u) == gridDim.x - 1) {
      p.local[1] = 0;
      __threadfence_system();
      for (int r = 0; r < p.world; ++r) st_release_sys(p.sig[r] + p.rank, e + 1);      // my writes to peer r are done
      for (int r = 0; r < p.world; ++r) spin_until_sys(p.sig[p.rank] + r, e + 1);        // peer r's writes to me are done
      p.state[0] = p.state[0] + 1.f;
      p.state[1] = s_bc[0];
      p.state[2] = s_bc[1];
      p.state[3] = __uint_as_float(__float_as_uint(p.state[3]) + 1u);
      p.local[0] = e + 1;
      __threadfence();
      st_release_gpu(p.local + 2, e + 1);
    } else {
      spin_until_gpu(p.local + 2, e + 1);
    }
  }
  __syncthreads();
}

}  // namespace srfrd

using namespace srfrd;

extern "C" int srfrd_dp_adam_step(float* const* grad_ptrs_dev, float* const* param_ptrs_dev, uint32_t* const* signal_ptrs_dev,
                                  int rank, int world, int64_t n, float* m, float* v, float lr, float beta1, float beta2,
                                  float eps, float* state8, const float* norm2, uint32_t* local4, void* stream,
                                  const int64_t* l2_seg, int l2_n_seg, const float* l2_coef, const float* l2_reg) {
  SRFRD_REQUIRE(grad_ptrs_dev && param_ptrs_dev && signal_ptrs_dev && m && v && state8 && norm2 && local4, "dp_adam_step: null pointer");
  const bool l2 = l2_seg != nullptr;
  SRFRD_REQUIRE(!l2 || (l2_coef && l2_reg && l2_n_seg >= 1 && l2_n_seg <= L2_THREADS),
                "dp_adam_step: the l2 term needs coef, reg and 1..%d segments", L2_THREADS);
  SRFRD_REQUIRE(world >= 1 && world <= DP_MAX_WORLD && rank >= 0 && rank < world, "dp_adam_step: bad rank %d / world %d", rank, world);
  SRFRD_REQUIRE(n > 0 && n % 4 == 0, "dp_adam_step: n must be a positive multiple of 4");
  DpAdam p;
  p.grad = grad_ptrs_dev; p.param = param_ptrs_dev; p.sig = signal_ptrs_dev; p.rank = rank; p.world = world; p.n = n;
  p.m = m; p.v = v; p.lr = lr; p.beta1 = beta1; p.beta2 = beta2; p.eps = eps; p.state = state8; p.norm = norm2; p.local = local4;
  p.l2s = L2Segments{l2_seg, l2_n_seg, l2_coef, l2_reg};
  const int64_t slice4 = (n / 4 + world - 1) / world;
  int64_t grid = (slice4 + DP_THREADS - 1) / DP_THREADS;
  if (grid < 1) grid = 1;
  if (grid > num_sms()) grid = num_sms();            // every block must be resident (in-kernel grid barrier)
  if (l2)
    SRFRD_CUDA(launch_pdl(dp_adam_kernel<true>, dim3((unsigned)grid), dim3(DP_THREADS), 0, (cudaStream_t)stream, p));
  else
    SRFRD_CUDA(launch_pdl(dp_adam_kernel<false>, dim3((unsigned)grid), dim3(DP_THREADS), 0, (cudaStream_t)stream, p));
  SRFRD_LAUNCH_CHECK();
  return 0;
}
