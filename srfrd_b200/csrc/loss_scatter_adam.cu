// HBM/atomic-bound kernels around the encoder:
//   K4  fused gather-dot scoring + discriminator-weighted BCE forward AND backward (SURVEY.md rows A6, A7, L)
//   K5  sparse embedding-gradient scatter-add for the input sequence (row A8, k7)
//   K7  flat fused Adam with device-resident step state (row A8, k8)
#include "common.cuh"
#include "srfrd_b200.h"

namespace srfrd {

static constexpr int MAXC = 16;

struct ScoreParams {
  const float* h; int ldh;              // (T, W) final hidden state, W = D (+F for SRFRN)
  const float* item_table;              // (n_rows, D)
  const float* fake_table;              // (3, F) or null (SRFRN only)
  const int64_t *pos, *neg, *prs, *nrs; // (T)
  const float *w_pos, *w_neg;           // (T) or null -> 1[pos != 0]
  const float* norm;                    // device [2]: sum(w_pos), sum(w_neg)    (fused mode)
  const float *dzp_in, *dzn_in;         // (T) upstream logit gradients          (bwd mode)
  float *zp, *zn;                       // (T) logits out or null
  float* loss_acc;                      // device [2] += sum w*softplus(-z+), sum w*softplus(z-)
  float* dh; int lddh;                  // (T, W) or null
  float* d_item; float* d_fake;         // gradient tables (red.add) or null
  int64_t T; int D, F;
  int mode;                             // 0 = logits only, 1 = fused loss fwd+bwd, 2 = bwd from dz
  const int* row_tok;                   // packed layout: h / dh row t belongs to dense token row_tok[t] (-1: no token); ids,
  const int* rows_dev;                  // weights and logits stay indexed by the dense token.  rows_dev: device row count
  int group;                            // rows a warp takes per pass: 32 (dense: ~4 of them are active), 8 (packed: nearly all are)
};

__device__ __forceinline__ float softplus(float x) { return fmaxf(x, 0.f) + log1pf(__expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoidf(float x) { return 1.f / (1.f + __expf(-x)); }

// A warp takes 32 consecutive tokens at a time: their ids / weights arrive in one coalesced load each, the hidden-state
// gradient rows of the inactive tokens (pad slots: 88 % of a C2 batch) are zeroed with 16-byte stores, and only the active
// tokens go through the gather-dot-scatter path below (one token per pass, lane c owns columns c, c+32, ...).
// Gradients of the 3-row fake table are kept in registers and flushed once per warp: every active token hits the same two
// rows, which made them the most contended addresses of the step.
template <int NC>
__global__ void __launch_bounds__(256, (NC <= 9 ? 2 : 1)) score_kernel(ScoreParams p) {
  __shared__ float red[2][8];
  pdl_prologue_done();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int64_t warp0 = (int64_t)blockIdx.x * nw + warp, nwarps = (int64_t)gridDim.x * nw;
  const int W = p.D + (p.fake_table ? p.F : 0);
  float lp_acc = 0.f, ln_acc = 0.f;
  float inv_np = 0.f, inv_nn = 0.f;
  if (p.mode == 1) {
    const float a = __ldg(p.norm), b = __ldg(p.norm + 1);
    inv_np = a > 0.f ? 1.f / a : 0.f;
    inv_nn = b > 0.f ? 1.f / b : 0.f;
  }
  float fk1[NC], fk2[NC];                    // d_fake rows 1 and 2, columns owned by this lane
#pragma unroll
  for (int i = 0; i < NC; ++i) fk1[i] = fk2[i] = 0.f;
  const bool dh_vec = p.dh && (p.lddh == W) && (W % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.dh) & 15) == 0);
  if (p.rows_dev) p.T = min(p.T, (int64_t)__ldg(p.rows_dev));
  const int G = p.group;
  for (int64_t t0 = warp0 * G; t0 < p.T; t0 += nwarps * G) {
    const int64_t tl = t0 + lane;
    bool in = lane < G && tl < p.T;
    int my_tok = 0;                           // packed layout: dense token whose ids / weights / logits this row uses
    if (p.row_tok && in) { my_tok = __ldg(p.row_tok + tl); in = my_tok >= 0; }
    const int64_t my_src = p.row_tok ? (int64_t)my_tok : tl;
    int64_t my_pid = 0, my_nid = 0, my_pf = 0, my_nf = 0;
    float my_a = 0.f, my_b = 0.f;             // mode 1: (w_pos, w_neg); mode 2: (dz+, dz-)
    bool my_active = false;
    if (in) {
      my_pid = __ldg(p.pos + my_src);
      my_nid = __ldg(p.neg + my_src);
      if (p.mode == 1) {
        my_a = p.w_pos ? __ldg(p.w_pos + my_src) : (my_pid != 0 ? 1.f : 0.f);
        my_b = p.w_neg ? __ldg(p.w_neg + my_src) : my_a;
        my_active = (my_a != 0.f) || (my_b != 0.f) || p.zp;
      } else if (p.mode == 2) {
        my_a = __ldg(p.dzp_in + my_src);
        my_b = __ldg(p.dzn_in + my_src);
        my_active = (my_a != 0.f) || (my_b != 0.f);
      } else {
        my_active = true;
      }
      if (p.fake_table && my_active) { my_pf = __ldg(p.prs + my_src); my_nf = __ldg(p.nrs + my_src); }
    }
    unsigned mask = __ballot_sync(0xffffffffu, my_active);
    if (p.dh) {                               // zero rows of the inactive tokens
      const int nrow = (int)min((int64_t)G, p.T - t0);
      if (dh_vec) {
        const int per_row = W >> 2, total = nrow * per_row;
        float4* base = reinterpret_cast<float4*>(p.dh + t0 * p.lddh);
        for (int i = lane; i < total; i += 32)
          if (!((mask >> (i / per_row)) & 1u)) base[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        for (int r = 0; r < nrow; ++r) {
          if ((mask >> r) & 1u) continue;
          for (int c = lane; c < W; c += 32) p.dh[(t0 + r) * p.lddh + c] = 0.f;
        }
      }
    }
    // One token per pass; for narrow rows (NC <= 4) the NEXT active token's three rows (h, E[pos], E[neg]) are fetched
    // before the current token's reductions and atomics, so two tokens' gathers are in flight per warp: at catalogue
    // scale the kernel is bound by memory-level parallelism (ncu: 37 % of HBM peak with one token in flight).
    struct Tok {
      int64_t t, tsrc, pid, nid; int pf, nf; float ta, tb;
      float hv[NC], ep[NC], en[NC];
    };
    auto fetch = [&](Tok& k, int r) {
      k.t = t0 + r;
      k.tsrc = p.row_tok ? (int64_t)__shfl_sync(0xffffffffu, my_tok, r) : k.t;
      k.pid = __shfl_sync(0xffffffffu, my_pid, r); k.nid = __shfl_sync(0xffffffffu, my_nid, r);
      k.pf = (int)__shfl_sync(0xffffffffu, (int)my_pf, r); k.nf = (int)__shfl_sync(0xffffffffu, (int)my_nf, r);
      k.ta = __shfl_sync(0xffffffffu, my_a, r); k.tb = __shfl_sync(0xffffffffu, my_b, r);
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const int c = lane + 32 * i;
        k.hv[i] = k.ep[i] = k.en[i] = 0.f;
        if (c < W) {
          k.hv[i] = p.h[k.t * p.ldh + c];
          if (c < p.D) {
            k.ep[i] = __ldg(p.item_table + k.pid * p.D + c);
            k.en[i] = __ldg(p.item_table + k.nid * p.D + c);
          } else {
            k.ep[i] = __ldg(p.fake_table + (int64_t)k.pf * p.F + (c - p.D));
            k.en[i] = __ldg(p.fake_table + (int64_t)k.nf * p.F + (c - p.D));
          }
        }
      }
    };
    auto finish = [&](const Tok& k) {
      float sp = 0.f, sn = 0.f;
#pragma unroll
      for (int i = 0; i < NC; ++i) { sp = fmaf(k.hv[i], k.ep[i], sp); sn = fmaf(k.hv[i], k.en[i], sn); }
      const float zp = warp_sum(sp), zn = warp_sum(sn);
      if (p.zp && lane == 0) { p.zp[k.tsrc] = zp; p.zn[k.tsrc] = zn; }
      if (p.mode == 0) return;
      float dzp = k.ta, dzn = k.tb;
      if (p.mode == 1) {
        lp_acc += k.ta * softplus(-zp);
        ln_acc += k.tb * softplus(zn);
        dzp = k.ta * (sigmoidf(zp) - 1.f) * inv_np;
        dzn = k.tb * sigmoidf(zn) * inv_nn;
      }
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const int c = lane + 32 * i;
        if (c < W) {
          if (p.dh) p.dh[k.t * p.lddh + c] = dzp * k.ep[i] + dzn * k.en[i];
          if (c < p.D) {
            // padding_idx = 0: the pad row never receives gradient (SRFR_model.py:10)
            if (p.d_item && k.pid != 0 && dzp != 0.f) red_add_f32(p.d_item + k.pid * p.D + c, dzp * k.hv[i]);
            if (p.d_item && k.nid != 0 && dzn != 0.f) red_add_f32(p.d_item + k.nid * p.D + c, dzn * k.hv[i]);
          } else {
            const float gp = dzp * k.hv[i], gn = dzn * k.hv[i];
            fk1[i] += (k.pf == 1 ? gp : 0.f) + (k.nf == 1 ? gn : 0.f);
            fk2[i] += (k.pf == 2 ? gp : 0.f) + (k.nf == 2 ? gn : 0.f);
          }
        }
      }
    };
    if (NC <= 4) {
      if (mask) {
        Tok cur, nxt;
        { const int r = __ffs(mask) - 1; mask &= mask - 1; fetch(cur, r); }
        while (true) {
          const bool more = mask != 0;
          if (more) { const int r = __ffs(mask) - 1; mask &= mask - 1; fetch(nxt, r); }
          finish(cur);
          if (!more) break;
          cur = nxt;
        }
      }
    } else {
      while (mask) {
        const int r = __ffs(mask) - 1;
        mask &= mask - 1;
        Tok cur;
        fetch(cur, r);
        finish(cur);
      }
    }
  }
  if (p.d_fake) {
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const int c = lane + 32 * i;
      if (c >= p.D && c < W) {
        if (fk1[i] != 0.f) red_add_f32(p.d_fake + 1 * p.F + (c - p.D), fk1[i]);
        if (fk2[i] != 0.f) red_add_f32(p.d_fake + 2 * p.F + (c - p.D), fk2[i]);
      }
    }
  }
  if (p.mode == 1 && p.loss_acc) {
    if (lane == 0) { red[0][warp] = lp_acc; red[1][warp] = ln_acc; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float a = 0.f, b = 0.f;
      for (int w = 0; w < nw; ++w) { a += red[0][w]; b += red[1][w]; }
      red_add_f32(p.loss_acc, a);
      red_add_f32(p.loss_acc + 1, b);
    }
  }
}

// out[0] = sum w_pos (or #pos != 0), out[1] = sum w_neg
__global__ void __launch_bounds__(256) weight_sums_kernel(const int64_t* pos, const float* w_pos, const float* w_neg,
                                                          int64_t T, float* out) {
  __shared__ float red[2][8];
  float a = 0.f, b = 0.f;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (int64_t)gridDim.x * blockDim.x) {
    const float wp = w_pos ? w_pos[t] : (pos[t] != 0 ? 1.f : 0.f);
    a += wp;
    b += w_neg ? w_neg[t] : wp;
  }
  a = warp_sum(a); b = warp_sum(b);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[0][warp] = a; red[1][warp] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    a = b = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { a += red[0][w]; b += red[1][w]; }
    red_add_f32(out, a);
    red_add_f32(out + 1, b);
  }
}

// The accumulators are CONSUMED (zeroed for the next step): no separate fill kernel in the step graph.
__global__ void loss_finalize_kernel(float* acc, const float* norm, float* loss) {
  pdl_prologue_done();
  const float a = norm[0] > 0.f ? acc[0] / norm[0] : 0.f;
  const float b = norm[1] > 0.f ? acc[1] / norm[1] : 0.f;
  loss[0] = a + b;
  acc[0] = 0.f; acc[1] = 0.f;
}

// ---------------------------------------------------------------------------------------------
// K5: gradient of the input-sequence lookups.  One CTA per sequence, one thread per feature column.
struct EmbedBwdParams {
  const bf16* dx0; int ldx;          // (T, ldx), already pad-masked
  const int64_t* seq;                // (B, L)
  const int64_t* aux_ids;            // mode 1: (B, L) fake ids or null; mode 2: (B,) labels
  int L, D, F, mode;
  float item_scale;
  float* d_item;                     // (n_rows, D)
  float* d_aux;                      // mode 1: (3, F); mode 2: (labels, D)
};

__global__ void embed_bwd_kernel(EmbedBwdParams p) {
  extern __shared__ int64_t ids[];   // [L] seq ids, [L] fake ids
  pdl_prologue_done();
  const int64_t b = blockIdx.x;
  const int c = threadIdx.x;
  const int H = p.D + (p.mode == 1 ? p.F : 0);
  for (int l = threadIdx.x; l < p.L; l += blockDim.x) {
    ids[l] = p.seq[b * p.L + l];
    ids[p.L + l] = (p.mode == 1 && p.aux_ids) ? p.aux_ids[b * p.L + l] : 0;
  }
  __syncthreads();
  if (c >= H) return;
  float acc1 = 0.f, acc2 = 0.f, accu = 0.f;
  for (int l = 0; l < p.L; ++l) {
    const int64_t id = ids[l];
    if (id == 0) continue;
    const float v = bf2f(p.dx0[(b * p.L + l) * p.ldx + c]);
    if (c < p.D) {
      red_add_f32(p.d_item + id * p.D + c, v * p.item_scale);
      accu += v;
    } else {
      const int64_t f = ids[p.L + l];
      if (f == 1) acc1 += v;
      else if (f == 2) acc2 += v;
    }
  }
  if (p.mode == 1 && c >= p.D && p.d_aux) {        // fake_embed padding_idx = 0: row 0 gets nothing
    if (acc1 != 0.f) red_add_f32(p.d_aux + 1 * p.F + (c - p.D), acc1);
    if (acc2 != 0.f) red_add_f32(p.d_aux + 2 * p.F + (c - p.D), acc2);
  }
  if (p.mode == 2 && c < p.D && p.d_aux && accu != 0.f)
    red_add_f32(p.d_aux + p.aux_ids[b] * p.D + c, accu);
}

// K5 on the packed layout, row-parallel: a block takes RPB packed rows per pass and a SLICE of up to 64 columns
// (blockIdx.y), thread (y, x) owns column slice*64 + x of row y.  A row with a dense token (row_tok >= 0) and a non-zero
// input id adds its dx0 row to the item table (red.add), to the positional table through a per-block shared accumulator
// [L][slice width] (shared-memory atomics, flushed once per block; the dense path takes this gradient from a column sum
// over the (B, L*H) view) and to the fake / user-label table.  Column slices keep the accumulator at L * 256 bytes, so
// several blocks fit an SM also at maxlen 200, D = 256 (one 200 KB accumulator per SM measured 0.52 ms at C4).
static constexpr int EB_SLICE = 64;
__global__ void __launch_bounds__(512) embed_bwd_packed_kernel(EmbedBwdParams p, const int* row_tok, const int* rows_dev, int64_t cap,
                                                              float* d_pos) {
  extern __shared__ float spos[];            // [L * EB_SLICE]
  pdl_prologue_done();
  const int x = threadIdx.x, y = threadIdx.y, RPB = blockDim.y;
  const int c = blockIdx.y * EB_SLICE + x;
  const int H = p.D + (p.mode == 1 ? p.F : 0);
  const int tid = y * blockDim.x + x, nthr = blockDim.x * blockDim.y;
  const bool pos_slice = blockIdx.y * EB_SLICE < p.D;
  if (pos_slice) for (int i = tid; i < p.L * EB_SLICE; i += nthr) spos[i] = 0.f;
  __syncthreads();
  const int64_t M = min(cap, (int64_t)__ldg(rows_dev));
  float acc1 = 0.f, acc2 = 0.f;
  for (int64_t r = (int64_t)blockIdx.x * RPB + y; r < M; r += (int64_t)gridDim.x * RPB) {
    const int tok = __ldg(row_tok + r);
    if (tok < 0 || c >= H) continue;
    const int64_t id = __ldg(p.seq + tok);
    if (id == 0) continue;                   // (a kept pad row has id 0: masked input, no gradient)
    const float v = bf2f(p.dx0[r * p.ldx + c]);
    if (c < p.D) {
      red_add_f32(p.d_item + id * p.D + c, v * p.item_scale);
      atomicAdd(&spos[(tok % p.L) * EB_SLICE + x], v);
      if (p.mode == 2 && p.d_aux) red_add_f32(p.d_aux + p.aux_ids[tok / p.L] * p.D + c, v);
    } else if (p.aux_ids) {
      const int64_t f = __ldg(p.aux_ids + tok);
      if (f == 1) acc1 += v;
      else if (f == 2) acc2 += v;
    }
  }
  if (p.mode == 1 && c >= p.D && c < H && p.d_aux) {        // fake_embed padding_idx = 0: row 0 gets nothing
    if (acc1 != 0.f) red_add_f32(p.d_aux + 1 * p.F + (c - p.D), acc1);
    if (acc2 != 0.f) red_add_f32(p.d_aux + 2 * p.F + (c - p.D), acc2);
  }
  __syncthreads();
  if (d_pos && pos_slice)
    for (int i = tid; i < p.L * EB_SLICE; i += nthr) {
      const int l = i / EB_SLICE, cc = blockIdx.y * EB_SLICE + i % EB_SLICE;
      if (cc < p.D && spos[i] != 0.f) red_add_f32(d_pos + l * p.D + cc, spos[i]);
    }
}

// out[(n / seg_in) * seg_out + n % seg_in] += in[n] where n % seg_in < seg_out
__global__ void add_segments_kernel(float* in, int64_t n, int seg_in, int seg_out, float* out) {
  pdl_prologue_done();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % seg_in);
  if (c < seg_out) out[(i / seg_in) * seg_out + c] += in[i];
  in[i] = 0.f;                           // consumed: the scratch accumulator is zero again for the next step
}

// ---------------------------------------------------------------------------------------------
// K7: Adam.  state = {step, 1 - beta1^step, 1 - beta2^step}; kept on device so a captured CUDA
// graph can replay the whole training step.
__global__ void adam_tick_kernel(float* state, float beta1, float beta2) {
  pdl_prologue_done();
  const float step = state[0] + 1.f;
  state[0] = step;
  state[1] = (float)(1.0 - pow((double)beta1, (double)step));
  state[2] = (float)(1.0 - pow((double)beta2, (double)step));
  // state[3]: the same counter as a 32-bit INTEGER bit pattern (the fp32 step stalls at 2^24); this word is what the
  // dropout masks and the on-device sampler mix into their seeds (mix_seed reads the raw bits)
  state[3] = __uint_as_float(__float_as_uint(state[3]) + 1u);
}

// ---------------------------------------------------------------------------------------------
// l2_emb regulariser (trainer.py:31-39: loss += l2 * torch.norm(p) for every parameter tensor p).  One launch computes,
// for each tensor t of the flat parameter buffer, coef[t] = l2 / ||p_t|| (0 when the norm is 0: torch's gradient of the
// norm of a zero tensor is 0) and reg = l2 * sum_t ||p_t||.  Deterministic: the buffer is cut into fixed chunks of
// L2_CHUNK floats that never cross a tensor boundary; each chunk's sum of squares is reduced in fp64 by one block in a
// fixed order, and the last block to finish sums the chunks of each tensor in chunk order.  No float atomics, so every
// data-parallel replica computes bit-identical coefficients from bit-identical parameters.
static constexpr int64_t L2_CHUNK = 8192;          // floats per chunk: 8 float4 per thread

// chunk starts of each segment (exclusive prefix of ceil(numel / L2_CHUNK)); s_c0[n_seg] = total
__device__ __forceinline__ void l2_chunk_prefix(const int64_t* seg, int n_seg, int64_t* s_c0) {
  const int t = threadIdx.x;
  s_c0[t + 1] = t < n_seg ? (seg[2 * t + 1] + L2_CHUNK - 1) / L2_CHUNK : 0;
  if (t == 0) s_c0[0] = 0;
  __syncthreads();
  for (int d = 1; d < L2_THREADS; d <<= 1) {            // Hillis-Steele inclusive scan over s_c0[1..]
    const int64_t a = t >= d ? s_c0[t + 1 - d] : 0;
    __syncthreads();
    s_c0[t + 1] += a;
    __syncthreads();
  }
}

__device__ __forceinline__ double block_sum_f64(double x, double* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = x;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < L2_THREADS / 32; ++w) s += s_red[w];
  __syncthreads();
  return s;                                             // valid in thread 0
}

// ws: [0] = uint32 blocks-done counter (zero between launches), [1 .. n_chunks] = fp64 chunk sums of squares
__global__ void __launch_bounds__(L2_THREADS) param_l2_kernel(const float* __restrict__ p, const int64_t* __restrict__ seg,
                                                               int n_seg, int64_t n_chunks, float l2, float* coef, float* reg,
                                                               double* ws) {
  __shared__ int64_t s_c0[L2_THREADS + 1];
  __shared__ double s_red[L2_THREADS / 32];
  __shared__ double s_norm[L2_THREADS];
  __shared__ bool s_last;
  pdl_prologue_done();
  l2_chunk_prefix(seg, n_seg, s_c0);
  double* part = ws + 1;
  for (int64_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    int lo = 0, hi = n_seg - 1;                         // segment t holding chunk c: s_c0[t] <= c < s_c0[t + 1]
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (s_c0[mid] <= c) lo = mid; else hi = mid - 1;
    }
    const int64_t off = seg[2 * lo], numel = seg[2 * lo + 1];
    const int64_t b = (c - s_c0[lo]) * L2_CHUNK;        // chunk start within the segment
    const int64_t e = min(numel, b + L2_CHUNK);
    const float4* p4 = reinterpret_cast<const float4*>(p + off);
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < (int)(L2_CHUNK / 4 / L2_THREADS); ++k) {
      const int64_t j = b + 4 * ((int64_t)k * L2_THREADS + threadIdx.x);   // first float of this float4
      if (j < e) {
        const float4 x = __ldcg(p4 + j / 4);
        const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (j + q < e) acc = fma((double)xs[q], (double)xs[q], acc);   // never reads the zero padding as data
      }
    }
    const double s = block_sum_f64(acc, s_red);
    if (threadIdx.x == 0) part[c] = s;
  }
  // ---- last block: per-segment sums in chunk order, then the fixed-order total
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(reinterpret_cast<unsigned*>(ws), 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = warp; t < n_seg; t += L2_THREADS / 32) {
    double s = 0.0;
    for (int64_t c = s_c0[t] + lane; c < s_c0[t + 1]; c += 32) s += __ldcg(part + c);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
      const double nrm = sqrt(s);
      s_norm[t] = nrm;
      coef[t] = nrm > 0.0 ? (float)((double)l2 / nrm) : 0.f;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int t = 0; t < n_seg; ++t) tot += s_norm[t];
    reg[0] = (float)((double)l2 * tot);
    *reinterpret_cast<unsigned*>(ws) = 0u;
  }
}

// One launch for the tail of a training step: Adam tick (step counters, bias corrections), the dense Adam update, and
// the loss read-out.  Every block derives the NEW step state from the old one (thread 0: two pow() per block), the last
// block to finish publishes it -- by then every block has read the old state -- and block 0 finalises the loss.
// state8 = {step, 1 - beta1^step, 1 - beta2^step, uint32 step bits, int blocks-done counter, -, -, -}.
// L2: g += coef[tensor] * p (the gradient of l2 * ||p_t||, from the parameters before this update) and loss += reg.
// ROWS (lazy item-table Adam, RowGate): the grid-stride loop skips the table's float4s, the non-table floats of a float4
// the table ends in are done one by one, and the table is walked row-parallel over its stamps: each warp loads 32 stamps,
// and every stamped row among them is updated by the whole warp.  Same per-element arithmetic as the dense loop, so a
// stamped row gets exactly the dense update; an unstamped row is not read (its gradient is zero: no kernel wrote it).
template <bool L2, bool ROWS>
__global__ void __launch_bounds__(256) adam_fused_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                                         float* __restrict__ v, int64_t n, float lr, float beta1, float beta2,
                                                         float eps, float* state, int zero_grad, float* acc, const float* norm,
                                                         float* loss, L2Segments l2s, RowGate rg) {
  __shared__ float s_bc[2];
  __shared__ uint32_t s_epoch;
  pdl_prologue_done();
  if (threadIdx.x == 0) {
    const float step = state[0] + 1.f;
    s_bc[0] = (float)(1.0 - pow((double)beta1, (double)step));
    s_bc[1] = (float)(1.0 - pow((double)beta2, (double)step));
    if constexpr (ROWS) s_epoch = __float_as_uint(state[3]) + 1u;
  }
  if (blockIdx.x == 0 && threadIdx.x == 32 && acc) {
    const float a = norm[0] > 0.f ? acc[0] / norm[0] : 0.f;
    const float b = norm[1] > 0.f ? acc[1] / norm[1] : 0.f;
    if constexpr (L2) loss[0] = a + b + l2s.reg[0];
    else loss[0] = a + b;
    acc[0] = 0.f; acc[1] = 0.f;
  }
  int64_t* s_off = nullptr;
  float* s_coef = nullptr;
  if constexpr (L2) {
    s_off = l2_smem().off;
    s_coef = l2_smem().coef;
    l2_load_starts(l2s, s_off, s_coef);
  }
  __syncthreads();
  const float step_size = lr / s_bc[0];
  const float inv_sqrt_bc2 = rsqrtf(s_bc[1]);
  const int64_t n4 = n >> 2;
  int t = 0;
  if constexpr (L2) t = l2_find(s_off, l2s.n_seg, (int64_t)blockIdx.x * blockDim.x + threadIdx.x);
  // ROWS: the table's float4s [t0, t1) are left to the row walk below; j counts the others
  int64_t t0 = 0, skip = 0;
  if constexpr (ROWS) {
    t0 = rg.off >> 2;
    skip = ((rg.off + rg.rows * rg.D + 3) >> 2) - t0;
  }
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n4 - skip; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = ROWS && j >= t0 ? j + skip : j;
    float4 pp = reinterpret_cast<float4*>(p)[i], gg = reinterpret_cast<float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    float* pa = &pp.x; float* ga = &gg.x; float* ma = &mm.x; float* va = &vv.x;
    if constexpr (L2) {
      t = l2_advance(s_off, l2s.n_seg, t, i);
      const float c = s_coef[t];
#pragma unroll
      for (int j = 0; j < 4; ++j) ga[j] += c * pa[j];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ma[j] = beta1 * ma[j] + (1.f - beta1) * ga[j];
      va[j] = beta2 * va[j] + (1.f - beta2) * ga[j] * ga[j];
      pa[j] -= step_size * ma[j] / (sqrtf(va[j]) * inv_sqrt_bc2 + eps);
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (zero_grad) reinterpret_cast<float4*>(g)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    m[i] = beta1 * m[i] + (1.f - beta1) * g[i];
    v[i] = beta2 * v[i] + (1.f - beta2) * g[i] * g[i];
    p[i] -= step_size * m[i] / (sqrtf(v[i]) * inv_sqrt_bc2 + eps);
    if (zero_grad) g[i] = 0.f;
  }
  if constexpr (ROWS) {
    const int64_t tend = rg.off + rg.rows * rg.D;
    // the float4 the table ends in: its floats past the table are dense
    if (blockIdx.x == 0 && threadIdx.x < ((4 - (tend & 3)) & 3)) {
      const int64_t i = tend + threadIdx.x;
      m[i] = beta1 * m[i] + (1.f - beta1) * g[i];
      v[i] = beta2 * v[i] + (1.f - beta2) * g[i] * g[i];
      p[i] -= step_size * m[i] / (sqrtf(v[i]) * inv_sqrt_bc2 + eps);
      if (zero_grad) g[i] = 0.f;
    }
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t epoch = s_epoch;
    for (int64_t r0 = warp * 32; r0 < rg.rows; r0 += n_warps * 32) {
      const int64_t r = r0 + lane;
      unsigned hit = __ballot_sync(0xffffffffu, r < rg.rows && __ldcg(rg.stamp + r) == epoch);
      while (hit) {
        const int64_t e0 = rg.off + (r0 + __ffs(hit) - 1) * rg.D;
        hit &= hit - 1;
        if ((rg.D & 3) == 0) {
          for (int64_t i = (e0 >> 2) + lane; i < ((e0 + rg.D) >> 2); i += 32) {
            float4 pp = reinterpret_cast<float4*>(p)[i], gg = reinterpret_cast<float4*>(g)[i];
            float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
            float* pa = &pp.x; float* ga = &gg.x; float* ma = &mm.x; float* va = &vv.x;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              ma[q] = beta1 * ma[q] + (1.f - beta1) * ga[q];
              va[q] = beta2 * va[q] + (1.f - beta2) * ga[q] * ga[q];
              pa[q] -= step_size * ma[q] / (sqrtf(va[q]) * inv_sqrt_bc2 + eps);
            }
            reinterpret_cast<float4*>(p)[i] = pp;
            reinterpret_cast<float4*>(m)[i] = mm;
            reinterpret_cast<float4*>(v)[i] = vv;
            if (zero_grad) reinterpret_cast<float4*>(g)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        } else {                                           // D % 4 != 0: rows straddle float4s, one float per lane
          for (int64_t i = e0 + lane; i < e0 + rg.D; i += 32) {
            m[i] = beta1 * m[i] + (1.f - beta1) * g[i];
            v[i] = beta2 * v[i] + (1.f - beta2) * g[i] * g[i];
            p[i] -= step_size * m[i] / (sqrtf(v[i]) * inv_sqrt_bc2 + eps);
            if (zero_grad) g[i] = 0.f;
          }
        }
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int* done = reinterpret_cast<int*>(state + 4);
    if (atomicAdd(done, 1) == (int)gridDim.x - 1) {        // last block: every block has read the old state
      *done = 0;
      state[0] = state[0] + 1.f;
      state[1] = s_bc[0];
      state[2] = s_bc[1];
      state[3] = __uint_as_float(__float_as_uint(state[3]) + 1u);
    }
  }
}

// Lazy item-table Adam, part 1: stamp[id] = epoch for every id in 1..n_items of the step's id arrays (a, b, c: n_tok ids
// each; list: n_list ids; null arrays are skipped).  epoch = the uint32 step bits + 1 = the value the next Adam launch
// compares with, so nothing is ever cleared and a replayed graph stamps a new epoch without the host.
__global__ void __launch_bounds__(256) touch_rows_kernel(const int64_t* __restrict__ a, const int64_t* __restrict__ b,
                                                         const int64_t* __restrict__ c, int64_t n_tok,
                                                         const int64_t* __restrict__ list, int64_t n_list, int64_t n_items,
                                                         uint32_t* __restrict__ stamp, const float* __restrict__ state) {
  pdl_prologue_done();
  const uint32_t epoch = __float_as_uint(state[3]) + 1u;
  const int64_t total = 3 * n_tok + n_list;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = i / n_tok < 3 && n_tok > 0 ? i / n_tok : 3;
    const int64_t* src = s == 0 ? a : s == 1 ? b : s == 2 ? c : list;
    if (!src) continue;
    const int64_t id = src[s < 3 ? i - s * n_tok : i - 3 * n_tok];
    if (id >= 1 && id <= n_items) stamp[id] = epoch;
  }
}

__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, int64_t n, float lr, float beta1, float beta2,
                                                   float eps, const float* __restrict__ state, int zero_grad) {
  pdl_prologue_done();
  // torch.optim.Adam (trainer.py:390): step_size = lr / bc1; denom = sqrt(v) / sqrt(bc2) + eps
  const float step_size = lr / state[1];
  const float inv_sqrt_bc2 = rsqrtf(state[2]);
  const int64_t n4 = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 pp = reinterpret_cast<float4*>(p)[i], gg = reinterpret_cast<float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    float* pa = &pp.x; float* ga = &gg.x; float* ma = &mm.x; float* va = &vv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ma[j] = beta1 * ma[j] + (1.f - beta1) * ga[j];
      va[j] = beta2 * va[j] + (1.f - beta2) * ga[j] * ga[j];
      pa[j] -= step_size * ma[j] / (sqrtf(va[j]) * inv_sqrt_bc2 + eps);
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (zero_grad) reinterpret_cast<float4*>(g)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    m[i] = beta1 * m[i] + (1.f - beta1) * g[i];
    v[i] = beta2 * v[i] + (1.f - beta2) * g[i] * g[i];
    p[i] -= step_size * m[i] / (sqrtf(v[i]) * inv_sqrt_bc2 + eps);
    if (zero_grad) g[i] = 0.f;
  }
}

}  // namespace srfrd

using namespace srfrd;

static int score_launch(ScoreParams& p, void* stream) {
  const int W = p.D + (p.fake_table ? p.F : 0);
  SRFRD_REQUIRE(W <= 32 * MAXC, "score: width %d unsupported", W);
  if (p.T == 0) return 0;
  if (p.group != 8) p.group = 32;
  int64_t blocks = (p.T + 8 * p.group - 1) / (8 * p.group);     // a warp takes `group` rows per pass
  const int64_t cap = (int64_t)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  const int nc = (W + 31) / 32;
#define SCORE_CALL(NC) SRFRD_CUDA(launch_pdl(score_kernel<NC>, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, p))
  if (nc <= 1) SCORE_CALL(1);
  else if (nc <= 2) SCORE_CALL(2);
  else if (nc <= 3) SCORE_CALL(3);
  else if (nc <= 4) SCORE_CALL(4);
  else if (nc <= 6) SCORE_CALL(6);
  else if (nc <= 9) SCORE_CALL(9);
  else SCORE_CALL(MAXC);
#undef SCORE_CALL
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_score_fwd(const float* h, int ldh, const float* item_table, const float* fake_table,
                               const int64_t* pos, const int64_t* neg, const int64_t* prs, const int64_t* nrs,
                               int64_t T, int D, int F, float* zp, float* zn, void* stream) {
  SRFRD_REQUIRE(h && item_table && pos && neg && zp && zn, "score_fwd: null pointer");
  SRFRD_REQUIRE(!fake_table || (prs && nrs), "score_fwd: fake ids required with a fake table");
  ScoreParams p = {};
  p.h = h; p.ldh = ldh; p.item_table = item_table; p.fake_table = fake_table; p.pos = pos; p.neg = neg; p.prs = prs;
  p.nrs = nrs; p.T = T; p.D = D; p.F = F; p.zp = zp; p.zn = zn; p.mode = 0;
  return score_launch(p, stream);
}

extern "C" int srfrd_score_bwd(const float* h, int ldh, const float* item_table, const float* fake_table,
                               const int64_t* pos, const int64_t* neg, const int64_t* prs, const int64_t* nrs,
                               const float* dzp, const float* dzn, int64_t T, int D, int F, float* dh, int lddh,
                               float* d_item, float* d_fake, void* stream) {
  SRFRD_REQUIRE(h && item_table && pos && neg && dzp && dzn && dh, "score_bwd: null pointer");
  SRFRD_REQUIRE(!fake_table || (prs && nrs), "score_bwd: fake ids required with a fake table");
  ScoreParams p = {};
  p.h = h; p.ldh = ldh; p.item_table = item_table; p.fake_table = fake_table; p.pos = pos; p.neg = neg; p.prs = prs;
  p.nrs = nrs; p.T = T; p.D = D; p.F = F; p.dzp_in = dzp; p.dzn_in = dzn; p.dh = dh; p.lddh = lddh; p.d_item = d_item;
  p.d_fake = d_fake; p.mode = 2;
  return score_launch(p, stream);
}

extern "C" int srfrd_score_loss_fused(const float* h, int ldh, const float* item_table, const float* fake_table,
                                      const int64_t* pos, const int64_t* neg, const int64_t* prs, const int64_t* nrs,
                                      const float* w_pos, const float* w_neg, const float* norm, int64_t T, int D,
                                      int F, float* zp, float* zn, float* loss_acc, float* dh, int lddh, float* d_item,
                                      float* d_fake, void* stream) {
  SRFRD_REQUIRE(h && item_table && pos && neg && norm && loss_acc, "score_loss_fused: null pointer");
  SRFRD_REQUIRE(!fake_table || (prs && nrs), "score_loss_fused: fake ids required with a fake table");
  SRFRD_REQUIRE((zp == nullptr) == (zn == nullptr), "score_loss_fused: pass both logit outputs or neither");
  ScoreParams p = {};
  p.h = h; p.ldh = ldh; p.item_table = item_table; p.fake_table = fake_table; p.pos = pos; p.neg = neg; p.prs = prs;
  p.nrs = nrs; p.w_pos = w_pos; p.w_neg = w_neg; p.norm = norm; p.T = T; p.D = D; p.F = F; p.zp = zp; p.zn = zn;
  p.loss_acc = loss_acc; p.dh = dh; p.lddh = lddh; p.d_item = d_item; p.d_fake = d_fake; p.mode = 1;
  return score_launch(p, stream);
}

extern "C" int srfrd_score_loss_fused_packed(const float* h, int ldh, const float* item_table, const float* fake_table,
                                             const int64_t* pos, const int64_t* neg, const int64_t* prs, const int64_t* nrs,
                                             const float* w_pos, const float* w_neg, const float* norm, int D, int F,
                                             float* loss_acc, float* dh, int lddh, float* d_item, float* d_fake,
                                             const int* row_tok, const int* rows_dev, int64_t cap_rows, void* stream) {
  SRFRD_REQUIRE(h && item_table && pos && neg && norm && loss_acc && row_tok && rows_dev, "score_loss_fused_packed: null pointer");
  SRFRD_REQUIRE(!fake_table || (prs && nrs), "score_loss_fused_packed: fake ids required with a fake table");
  ScoreParams p = {};
  p.h = h; p.ldh = ldh; p.item_table = item_table; p.fake_table = fake_table; p.pos = pos; p.neg = neg; p.prs = prs;
  p.nrs = nrs; p.w_pos = w_pos; p.w_neg = w_neg; p.norm = norm; p.T = cap_rows; p.D = D; p.F = F;
  p.loss_acc = loss_acc; p.dh = dh; p.lddh = lddh; p.d_item = d_item; p.d_fake = d_fake; p.mode = 1;
  p.row_tok = row_tok; p.rows_dev = rows_dev; p.group = 8;
  return score_launch(p, stream);
}

extern "C" int srfrd_weight_sums(const int64_t* pos, const float* w_pos, const float* w_neg, int64_t T, float* out2,
                                 void* stream) {
  SRFRD_REQUIRE(pos && out2, "weight_sums: null pointer");
  SRFRD_CUDA(cudaMemsetAsync(out2, 0, 2 * sizeof(float), (cudaStream_t)stream));
  if (T == 0) return 0;
  int64_t blocks = (T + 2047) / 2048;
  if (blocks > num_sms() * 2) blocks = num_sms() * 2;
  weight_sums_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(pos, w_pos, w_neg, T, out2);
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_loss_finalize(float* acc2, const float* norm2, float* loss, void* stream) {
  SRFRD_REQUIRE(acc2 && norm2 && loss, "loss_finalize: null pointer");
  SRFRD_CUDA(launch_pdl(loss_finalize_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, acc2, norm2, loss));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_embed_bwd(const void* dx0, int ldx, const int64_t* seq, const int64_t* aux_ids, int64_t B, int L,
                               int D, int F, int mode, float item_scale, float* d_item, float* d_aux, void* stream) {
  SRFRD_REQUIRE(dx0 && seq && d_item, "embed_bwd: null pointer");
  SRFRD_REQUIRE(mode >= 0 && mode <= 2, "embed_bwd: bad mode");
  SRFRD_REQUIRE(mode != 2 || aux_ids, "embed_bwd: labels required for mode 2");
  const int H = D + (mode == 1 ? F : 0);
  SRFRD_REQUIRE(H <= 1024, "embed_bwd: width %d unsupported", H);
  if (B == 0) return 0;
  EmbedBwdParams p;
  p.dx0 = (const bf16*)dx0; p.ldx = ldx; p.seq = seq; p.aux_ids = aux_ids; p.L = L; p.D = D; p.F = F; p.mode = mode;
  p.item_scale = item_scale; p.d_item = d_item; p.d_aux = d_aux;
  const int threads = (H + 31) & ~31;
  SRFRD_CUDA(launch_pdl(embed_bwd_kernel, dim3((unsigned)B), dim3(threads), 2 * L * sizeof(int64_t), (cudaStream_t)stream, p));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_embed_bwd_packed(const void* dx0, int ldx, const int64_t* seq, const int64_t* aux_ids,
                                      const int* row_tok, const int* rows_dev, int64_t cap_rows, int L, int D, int F,
                                      int mode, float item_scale, float* d_item, float* d_aux, float* d_pos, void* stream) {
  SRFRD_REQUIRE(dx0 && seq && d_item && row_tok && rows_dev, "embed_bwd_packed: null pointer");
  SRFRD_REQUIRE(mode >= 0 && mode <= 2, "embed_bwd_packed: bad mode");
  SRFRD_REQUIRE(mode != 2 || aux_ids, "embed_bwd_packed: labels required for mode 2");
  const int H = D + (mode == 1 ? F : 0);
  SRFRD_REQUIRE(H <= 512, "embed_bwd_packed: width %d unsupported", H);
  if (cap_rows == 0) return 0;
  EmbedBwdParams p;
  p.dx0 = (const bf16*)dx0; p.ldx = ldx; p.seq = seq; p.aux_ids = aux_ids; p.L = L; p.D = D; p.F = F; p.mode = mode;
  p.item_scale = item_scale; p.d_item = d_item; p.d_aux = d_aux;
  const int slices = (H + EB_SLICE - 1) / EB_SLICE;
  const int tx = EB_SLICE, ty = 8;
  const size_t smem = (size_t)L * EB_SLICE * sizeof(float);
  SRFRD_REQUIRE(smem <= 200 * 1024, "embed_bwd_packed: L = %d too long for the shared positional accumulator", L);
  static bool attr = false;
  if (!attr) {
    SRFRD_CUDA(cudaFuncSetAttribute(embed_bwd_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = true;
  }
  int per_sm = (int)((200 * 1024) / (smem + 1024));
  if (per_sm > 4) per_sm = 4;
  if (per_sm < 1) per_sm = 1;
  int64_t gx = ((int64_t)num_sms() * per_sm + slices - 1) / slices;
  const int64_t need = (cap_rows + ty - 1) / ty;
  if (gx > need) gx = need;
  if (gx < 1) gx = 1;
  const dim3 grid((unsigned)gx, (unsigned)slices);
  SRFRD_CUDA(launch_pdl(embed_bwd_packed_kernel, grid, dim3(tx, ty), smem, (cudaStream_t)stream, p, row_tok, rows_dev, cap_rows,
                        d_pos));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_add_segments(float* in, int64_t n, int seg_in, int seg_out, float* out, void* stream) {
  SRFRD_REQUIRE(in && out && seg_in > 0 && seg_out <= seg_in, "add_segments: bad arguments");
  if (n == 0) return 0;
  SRFRD_CUDA(launch_pdl(add_segments_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, (cudaStream_t)stream, in, n, seg_in,
                        seg_out, out));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_adam_tick(float* state3, float beta1, float beta2, void* stream) {
  SRFRD_REQUIRE(state3, "adam_tick: null state");
  SRFRD_CUDA(launch_pdl(adam_tick_kernel, dim3(1), dim3(1), 0, (cudaStream_t)stream, state3, beta1, beta2));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_adam_step(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                               float eps, const float* state3, int zero_grad, void* stream) {
  SRFRD_REQUIRE(p && g && m && v && state3, "adam_step: null pointer");
  SRFRD_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0, "adam_step: buffers must be 16-byte aligned");
  if (n == 0) return 0;
  int64_t blocks = (n / 4 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  SRFRD_CUDA(launch_pdl(adam_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, p, g, m, v, n, lr, beta1, beta2,
                        eps, state3, zero_grad));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_adam_step_fused(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                                     float eps, float* state8, int zero_grad, float* acc2, const float* norm2, float* loss,
                                     void* stream, const int64_t* l2_seg, int l2_n_seg, const float* l2_coef,
                                     const float* l2_reg) {
  SRFRD_REQUIRE(p && g && m && v && state8, "adam_step_fused: null pointer");
  SRFRD_REQUIRE(!acc2 || (norm2 && loss), "adam_step_fused: the loss read-out needs norm and loss");
  SRFRD_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0, "adam_step_fused: buffers must be 16-byte aligned");
  const bool l2 = l2_seg != nullptr;
  SRFRD_REQUIRE(!l2 || (l2_coef && l2_reg && acc2), "adam_step_fused: the l2 term needs coef, reg and the loss read-out");
  SRFRD_REQUIRE(!l2 || (l2_n_seg >= 1 && l2_n_seg <= L2_THREADS && n % 4 == 0),
                "adam_step_fused: l2 needs 1..%d segments and n a multiple of 4", L2_THREADS);
  int64_t blocks = (n / 4 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  const L2Segments l2s{l2_seg, l2_n_seg, l2_coef, l2_reg};
  if (l2)
    SRFRD_CUDA(launch_pdl(adam_fused_kernel<true, false>, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, p, g, m,
                          v, n, lr, beta1, beta2, eps, state8, zero_grad, acc2, norm2, loss, l2s, RowGate{}));
  else
    SRFRD_CUDA(launch_pdl(adam_fused_kernel<false, false>, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, p, g, m,
                          v, n, lr, beta1, beta2, eps, state8, zero_grad, acc2, norm2, loss, l2s, RowGate{}));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_touch_rows(const int64_t* a, const int64_t* b, const int64_t* c, int64_t n_tok, const int64_t* list,
                                int64_t n_list, int64_t n_items, uint32_t* stamp, const float* state8, void* stream) {
  SRFRD_REQUIRE(stamp && state8, "touch_rows: null pointer");
  SRFRD_REQUIRE(n_tok >= 0 && n_list >= 0 && n_items >= 0, "touch_rows: negative count");
  SRFRD_REQUIRE(n_list == 0 || list, "touch_rows: n_list > 0 needs the list");
  const int64_t total = 3 * n_tok + n_list;
  if (total == 0) return 0;
  int64_t blocks = (total + 255) / 256;
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  SRFRD_CUDA(launch_pdl(touch_rows_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, a, b, c, n_tok, list,
                        n_list, n_items, stamp, state8));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_adam_step_fused_rows(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1,
                                          float beta2, float eps, float* state8, int zero_grad, float* acc2,
                                          const float* norm2, float* loss, int64_t table_off, int64_t table_rows, int D,
                                          const uint32_t* stamp, void* stream) {
  SRFRD_REQUIRE(p && g && m && v && state8 && stamp, "adam_step_fused_rows: null pointer");
  SRFRD_REQUIRE(!acc2 || (norm2 && loss), "adam_step_fused_rows: the loss read-out needs norm and loss");
  SRFRD_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0,
                "adam_step_fused_rows: buffers must be 16-byte aligned");
  SRFRD_REQUIRE(n % 4 == 0 && table_off % 4 == 0 && table_off >= 0 && table_rows >= 0 && D >= 1 &&
                table_off + table_rows * D <= n,
                "adam_step_fused_rows: the table (offset %lld, %lld x %d) must start 4-aligned inside n = %lld (a multiple of 4)",
                (long long)table_off, (long long)table_rows, D, (long long)n);
  const int64_t dense4 = n / 4 - (((table_off + table_rows * D + 3) >> 2) - (table_off >> 2));
  int64_t blocks = (dense4 > table_rows ? dense4 : table_rows) / 256 + 1;
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  SRFRD_CUDA(launch_pdl(adam_fused_kernel<false, true>, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, p, g, m, v,
                        n, lr, beta1, beta2, eps, state8, zero_grad, acc2, norm2, loss, L2Segments{},
                        RowGate{table_off, table_rows, D, stamp}));
  SRFRD_LAUNCH_CHECK();
  return 0;
}

extern "C" int srfrd_param_l2_plan(const int64_t* seg_host, int n_seg, int64_t* n_chunks) {
  SRFRD_REQUIRE(seg_host && n_chunks, "param_l2_plan: null pointer");
  SRFRD_REQUIRE(n_seg >= 1 && n_seg <= L2_THREADS, "param_l2_plan: %d segments (1..%d supported)", n_seg, L2_THREADS);
  int64_t c = 0, end = 0;
  for (int t = 0; t < n_seg; ++t) {
    const int64_t off = seg_host[2 * t], numel = seg_host[2 * t + 1];
    SRFRD_REQUIRE(off % 4 == 0 && off >= end && numel >= 0, "param_l2_plan: segment %d must start 4-aligned after the last", t);
    end = off + numel;
    c += (numel + L2_CHUNK - 1) / L2_CHUNK;
  }
  *n_chunks = c;
  return 0;
}

extern "C" int srfrd_param_l2(const float* p, const int64_t* seg, int n_seg, int64_t n_chunks, float l2, float* coef,
                              float* reg, double* ws, void* stream) {
  SRFRD_REQUIRE(p && seg && coef && reg && ws, "param_l2: null pointer");
  SRFRD_REQUIRE(((uintptr_t)p & 15) == 0, "param_l2: the parameter buffer must be 16-byte aligned");
  SRFRD_REQUIRE(n_seg >= 1 && n_seg <= L2_THREADS && n_chunks >= 0, "param_l2: bad segment / chunk count");
  int64_t grid = n_chunks < 1 ? 1 : n_chunks;
  if (grid > num_sms() * 8) grid = num_sms() * 8;
  SRFRD_CUDA(launch_pdl(param_l2_kernel, dim3((unsigned)grid), dim3(L2_THREADS), 0, (cudaStream_t)stream, p, seg, n_seg,
                        n_chunks, l2, coef, reg, ws));
  SRFRD_LAUNCH_CHECK();
  return 0;
}
