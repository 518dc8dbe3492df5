// LayerNorm forward / backward for the decoder (ln_1, ln_2, ln_f; trajectory_gpt2.py:323,353,779).
//
// Forward reads the fp32 residual stream and emits the bf16 GEMM operand plus per-row mean / rstd.
// Backward fuses the residual-gradient add: dx_resid += LN'(dy), optionally emitting the bf16 copy
// the next dgrad/wgrad GEMM consumes.  HBM-bound; one warp per row, 128-bit accesses, row kept in
// registers (d <= 2048).
#include <stdlib.h>
#include "common.cuh"
#include "dropout.cuh"

namespace neko {

constexpr int LN_MAX_D = 2048;  // NV (float4 per lane) is a template parameter: 1,2,4,6,8,16

template <int LN_MAX_VEC>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, uint16_t* __restrict__ y,
                                                            uint16_t* __restrict__ y2, float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                            int N, int d, float eps, int out_f16) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= N) return;
  const int nv = d >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x + (size_t)row * d);
  float4 v[LN_MAX_VEC];
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < LN_MAX_VEC; ++k) {
    const int i = lane + k * 32;
    if (i < nv) {
      v[k] = x4[i];
      sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
  }
  const float mean = warp_sum(sum) / (float)d;
  float sq = 0.f;
#pragma unroll
  for (int k = 0; k < LN_MAX_VEC; ++k) {
    const int i = lane + k * 32;
    if (i < nv) {
      const float a = v[k].x - mean, b = v[k].y - mean, c = v[k].z - mean, e = v[k].w - mean;
      sq += (a * a + b * b) + (c * c + e * e);
    }
  }
  const float rstd = rsqrtf(warp_sum(sq) / (float)d + eps);
  if (lane == 0) {
    mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
  const float4* g4 = reinterpret_cast<const float4*>(gamma);
  const float4* b4 = reinterpret_cast<const float4*>(beta);
  uint2* yv = reinterpret_cast<uint2*>(y + (size_t)row * d);
  uint2* yv2 = y2 ? reinterpret_cast<uint2*>(y2 + (size_t)row * d) : nullptr;
#pragma unroll
  for (int k = 0; k < LN_MAX_VEC; ++k) {
    const int i = lane + k * 32;
    if (i < nv) {
      const float4 g = __ldg(g4 + i), bb = __ldg(b4 + i);
      const float o0 = (v[k].x - mean) * rstd * g.x + bb.x, o1 = (v[k].y - mean) * rstd * g.y + bb.y;
      const float o2 = (v[k].z - mean) * rstd * g.z + bb.z, o3 = (v[k].w - mean) * rstd * g.w + bb.w;
      yv[i] = make_uint2(pack_16x2(o0, o1, out_f16 != 0), pack_16x2(o2, o3, out_f16 != 0));
      if (yv2) yv2[i] = make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
    }
  }
}

// Backward.  Threads own COLUMNS (one float4 = 4 columns each, blockDim = d/4 rounded up to a warp), a CTA walks
// its rows four at a time: 12 independent 128/64-bit loads per thread are in flight before the first use, the
// 8 row statistics are block-reduced with shuffles + one __syncthreads, and the column sums dgamma / dbeta / colsum
// live in 12 registers per thread for the whole kernel (one global atomicAdd per column per CTA at the end).
constexpr int LNB_ROWS = 4;

__global__ void __launch_bounds__(512) layernorm_bwd_kernel(const bf16* __restrict__ dy, const float* __restrict__ x,
                                                            const float* __restrict__ gamma, const float* __restrict__ mean,
                                                            const float* __restrict__ rstd, float* __restrict__ dx_resid,
                                                            bf16* __restrict__ dx_bf16, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, float* __restrict__ dx_colsum, int N, int d,
                                                            int rows_per_cta, DropCfg drop) {
  __shared__ float red[2][16][2 * LNB_ROWS];  // [parity][warp][s1 x4, s2 x4]
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int c4 = threadIdx.x;            // this thread's float4 column group
  const bool act = c4 < (d >> 2);
  const float4 g = act ? __ldg(reinterpret_cast<const float4*>(gamma) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag, ac = ag;
  const int row0 = blockIdx.x * rows_per_cta;
  const int row1 = min(N, row0 + rows_per_cta);
  const float inv_d = 1.0f / (float)d;
  const uint32_t dkey = drop.seed ? drop_key(drop) : 0u;
  int parity = 0;
  for (int rb = row0; rb < row1; rb += LNB_ROWS, parity ^= 1) {
    float4 xv[LNB_ROWS], rv[LNB_ROWS];
    uint2 dv[LNB_ROWS];
    float mu[LNB_ROWS], rs[LNB_ROWS];
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const int row = rb + r;
      const bool ok = act && row < row1;
      const size_t off = (size_t)(ok ? row : row0) * d;
      xv[r] = ok ? reinterpret_cast<const float4*>(x + off)[c4] : make_float4(0.f, 0.f, 0.f, 0.f);
      dv[r] = ok ? reinterpret_cast<const uint2*>(dy + off)[c4] : make_uint2(0u, 0u);
      rv[r] = ok ? reinterpret_cast<const float4*>(dx_resid + off)[c4] : make_float4(0.f, 0.f, 0.f, 0.f);
      mu[r] = (row < row1) ? __ldg(mean + row) : 0.f;
      rs[r] = (row < row1) ? __ldg(rstd + row) : 0.f;
    }
    float s[2 * LNB_ROWS];
    float4 gy[LNB_ROWS], xh[LNB_ROWS];
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const float2 d01 = unpack_bf16x2(dv[r].x), d23 = unpack_bf16x2(dv[r].y);
      xh[r] = make_float4((xv[r].x - mu[r]) * rs[r], (xv[r].y - mu[r]) * rs[r], (xv[r].z - mu[r]) * rs[r], (xv[r].w - mu[r]) * rs[r]);
      gy[r] = make_float4(d01.x * g.x, d01.y * g.y, d23.x * g.z, d23.y * g.w);
      s[r] = (gy[r].x + gy[r].y) + (gy[r].z + gy[r].w);
      s[LNB_ROWS + r] = (gy[r].x * xh[r].x + gy[r].y * xh[r].y) + (gy[r].z * xh[r].z + gy[r].w * xh[r].w);
      // column sums of dy and dy * xhat
      ab.x += d01.x; ab.y += d01.y; ab.z += d23.x; ab.w += d23.y;
      ag.x += d01.x * xh[r].x; ag.y += d01.y * xh[r].y; ag.z += d23.x * xh[r].z; ag.w += d23.y * xh[r].w;
    }
#pragma unroll
    for (int i = 0; i < 2 * LNB_ROWS; ++i) s[i] = warp_sum(s[i]);
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < 2 * LNB_ROWS; ++i) red[parity][wid][i] = s[i];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 2 * LNB_ROWS; ++i) {
      float t = 0.f;
      for (int w = 0; w < nwarps; ++w) t += red[parity][w][i];
      s[i] = t * inv_d;
    }
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const int row = rb + r;
      if (act && row < row1) {
        const float m1 = s[r], m2 = s[LNB_ROWS + r];
        float4 o = rv[r];
        o.x += rs[r] * (gy[r].x - m1 - xh[r].x * m2);
        o.y += rs[r] * (gy[r].y - m1 - xh[r].y * m2);
        o.z += rs[r] * (gy[r].z - m1 - xh[r].z * m2);
        o.w += rs[r] * (gy[r].w - m1 - xh[r].w * m2);
        const size_t off = (size_t)row * d;
        reinterpret_cast<float4*>(dx_resid + off)[c4] = o;
        if (drop.seed) {  // gradient entering the dropped-out residual branch: mask * scale * dx
          const uint32_t rk = drop_rowkey(dkey, (uint32_t)row);
          float m0, m1, m2_, m3;
          drop_pair(rk, 2u * c4, drop.thr16, drop.scale, m0, m1);
          drop_pair(rk, 2u * c4 + 1u, drop.thr16, drop.scale, m2_, m3);
          o.x *= m0; o.y *= m1; o.z *= m2_; o.w *= m3;
        }
        if (dx_bf16) reinterpret_cast<uint2*>(dx_bf16 + off)[c4] = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
        ac.x += o.x; ac.y += o.y; ac.z += o.z; ac.w += o.w;
      }
    }
  }
  if (act) {
    float* pg = dgamma + 4 * c4;
    float* pb = dbeta + 4 * c4;
    atomicAdd(pg, ag.x); atomicAdd(pg + 1, ag.y); atomicAdd(pg + 2, ag.z); atomicAdd(pg + 3, ag.w);
    atomicAdd(pb, ab.x); atomicAdd(pb + 1, ab.y); atomicAdd(pb + 2, ab.z); atomicAdd(pb + 3, ab.w);
    if (dx_colsum) {
      float* pc = dx_colsum + 4 * c4;
      atomicAdd(pc, ac.x); atomicAdd(pc + 1, ac.y); atomicAdd(pc + 2, ac.z); atomicAdd(pc + 3, ac.w);
    }
  }
}


// ---------------------------------------------------------------------------------------------
// Backward, staged variant (the default).  Same column-owner arithmetic as above, but the three row streams (x fp32,
// dy bf16, dx fp32) of the next row blocks are fetched by 1-D bulk async copies (cp.async.bulk, completion on an
// mbarrier) into a shared-memory ring while the current block is reduced: the memory pipeline stays LNS_STAGES row
// blocks deep instead of draining at every block-wide reduction (the register variant measured 37 us / launch at
// N=7680, d=768 with 16 % of the warps active and 'long scoreboard' as top stall, profiles/r01_ncu_ln_attn.txt).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ln_smem_u32(const void* q) { return (uint32_t)__cvta_generic_to_shared(q); }
__device__ __forceinline__ void ln_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nLNW:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra LND;\nbra LNW;\nLND:\n}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void ln_bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}

__global__ void __launch_bounds__(512) layernorm_bwd_staged_kernel(const bf16* __restrict__ dy, const float* __restrict__ x,
                                                                   const float* __restrict__ gamma, const float* __restrict__ mean,
                                                                   const float* __restrict__ rstd, float* __restrict__ dx_resid,
                                                                   bf16* __restrict__ dx_bf16, float* __restrict__ dgamma,
                                                                   float* __restrict__ dbeta, float* __restrict__ dx_colsum, int N, int d,
                                                                   int rows_per_cta, int stages, DropCfg drop) {
  extern __shared__ __align__(128) uint8_t ln_raw[];
  __shared__ float red[2][16][2 * LNB_ROWS];
  __shared__ __align__(8) uint64_t full[4];
  pdl_launch_dependents();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int c4 = threadIdx.x;
  const bool act = c4 < (d >> 2);
  const uint32_t xb = (uint32_t)LNB_ROWS * d * 4, yb = (uint32_t)LNB_ROWS * d * 2;   // bytes of one row block of x / dx, dy
  const uint32_t stage_bytes = 2 * xb + yb;
  const int row0 = blockIdx.x * rows_per_cta;
  const int row1 = min(N, row0 + rows_per_cta);
  const int n_iter = (row1 - row0 + LNB_ROWS - 1) / LNB_ROWS;
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ln_smem_u32(&full[s])));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();
  auto issue = [&](int it) {   // thread 0: fetch row block `it` into its ring slot
    const int s = it % stages;
    const int rb = row0 + it * LNB_ROWS;
    const uint32_t nr = (uint32_t)min(LNB_ROWS, row1 - rb);
    const uint32_t bar = ln_smem_u32(&full[s]);
    const uint32_t base = ln_smem_u32(ln_raw) + (uint32_t)s * stage_bytes;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(nr * (uint32_t)d * 10u) : "memory");
    ln_bulk_load(base, x + (size_t)rb * d, nr * d * 4, bar);
    ln_bulk_load(base + xb, dx_resid + (size_t)rb * d, nr * d * 4, bar);
    ln_bulk_load(base + 2 * xb, dy + (size_t)rb * d, nr * d * 2, bar);
  };
  if (threadIdx.x == 0)
    for (int it = 0; it < min(stages, n_iter); ++it) issue(it);

  const float4 g = act ? __ldg(reinterpret_cast<const float4*>(gamma) + c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  float4 ag = make_float4(0.f, 0.f, 0.f, 0.f), ab = ag, ac = ag;
  const float inv_d = 1.0f / (float)d;
  const uint32_t dkey = drop.seed ? drop_key(drop) : 0u;
  int parity = 0;
  for (int it = 0; it < n_iter; ++it, parity ^= 1) {
    const int rb = row0 + it * LNB_ROWS;
    const int s = it % stages;
    float mu[LNB_ROWS], rs[LNB_ROWS];
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const int row = rb + r;
      mu[r] = (row < row1) ? __ldg(mean + row) : 0.f;
      rs[r] = (row < row1) ? __ldg(rstd + row) : 0.f;
    }
    ln_mbar_wait(ln_smem_u32(&full[s]), (uint32_t)((it / stages) & 1));
    const uint8_t* sb = ln_raw + (size_t)s * stage_bytes;
    float4 xv[LNB_ROWS], rv[LNB_ROWS];
    uint2 dv[LNB_ROWS];
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const bool ok = act && (rb + r) < row1;
      xv[r] = ok ? reinterpret_cast<const float4*>(sb + (size_t)r * d * 4)[c4] : make_float4(0.f, 0.f, 0.f, 0.f);
      rv[r] = ok ? reinterpret_cast<const float4*>(sb + xb + (size_t)r * d * 4)[c4] : make_float4(0.f, 0.f, 0.f, 0.f);
      dv[r] = ok ? reinterpret_cast<const uint2*>(sb + 2 * xb + (size_t)r * d * 2)[c4] : make_uint2(0u, 0u);
    }
    float sred[2 * LNB_ROWS];
    float4 gy[LNB_ROWS], xh[LNB_ROWS];
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const float2 d01 = unpack_bf16x2(dv[r].x), d23 = unpack_bf16x2(dv[r].y);
      xh[r] = make_float4((xv[r].x - mu[r]) * rs[r], (xv[r].y - mu[r]) * rs[r], (xv[r].z - mu[r]) * rs[r], (xv[r].w - mu[r]) * rs[r]);
      gy[r] = make_float4(d01.x * g.x, d01.y * g.y, d23.x * g.z, d23.y * g.w);
      sred[r] = (gy[r].x + gy[r].y) + (gy[r].z + gy[r].w);
      sred[LNB_ROWS + r] = (gy[r].x * xh[r].x + gy[r].y * xh[r].y) + (gy[r].z * xh[r].z + gy[r].w * xh[r].w);
      ab.x += d01.x; ab.y += d01.y; ab.z += d23.x; ab.w += d23.y;
      ag.x += d01.x * xh[r].x; ag.y += d01.y * xh[r].y; ag.z += d23.x * xh[r].z; ag.w += d23.y * xh[r].w;
    }
#pragma unroll
    for (int i = 0; i < 2 * LNB_ROWS; ++i) sred[i] = warp_sum(sred[i]);
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < 2 * LNB_ROWS; ++i) red[parity][wid][i] = sred[i];
    }
    __syncthreads();   // every thread has read its slice of ring slot s: the slot may be refilled
    if (threadIdx.x == 0 && it + stages < n_iter) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(it + stages);
    }
#pragma unroll
    for (int i = 0; i < 2 * LNB_ROWS; ++i) {
      float t = 0.f;
      for (int w = 0; w < nwarps; ++w) t += red[parity][w][i];
      sred[i] = t * inv_d;
    }
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const int row = rb + r;
      if (act && row < row1) {
        const float m1 = sred[r], m2 = sred[LNB_ROWS + r];
        float4 o = rv[r];
        o.x += rs[r] * (gy[r].x - m1 - xh[r].x * m2);
        o.y += rs[r] * (gy[r].y - m1 - xh[r].y * m2);
        o.z += rs[r] * (gy[r].z - m1 - xh[r].z * m2);
        o.w += rs[r] * (gy[r].w - m1 - xh[r].w * m2);
        const size_t off = (size_t)row * d;
        reinterpret_cast<float4*>(dx_resid + off)[c4] = o;
        if (drop.seed) {
          const uint32_t rk = drop_rowkey(dkey, (uint32_t)row);
          float m0, m1_, m2_, m3;
          drop_pair(rk, 2u * c4, drop.thr16, drop.scale, m0, m1_);
          drop_pair(rk, 2u * c4 + 1u, drop.thr16, drop.scale, m2_, m3);
          o.x *= m0; o.y *= m1_; o.z *= m2_; o.w *= m3;
        }
        if (dx_bf16) reinterpret_cast<uint2*>(dx_bf16 + off)[c4] = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
        ac.x += o.x; ac.y += o.y; ac.z += o.z; ac.w += o.w;
      }
    }
  }
  if (act) {
    float* pg = dgamma + 4 * c4;
    float* pb = dbeta + 4 * c4;
    atomicAdd(pg, ag.x); atomicAdd(pg + 1, ag.y); atomicAdd(pg + 2, ag.z); atomicAdd(pg + 3, ag.w);
    atomicAdd(pb, ab.x); atomicAdd(pb + 1, ab.y); atomicAdd(pb + 2, ab.z); atomicAdd(pb + 3, ab.w);
    if (dx_colsum) {
      float* pc = dx_colsum + 4 * c4;
      atomicAdd(pc, ac.x); atomicAdd(pc + 1, ac.y); atomicAdd(pc + 2, ac.z); atomicAdd(pc + 3, ac.w);
    }
  }
}


// ---------------------------------------------------------------------------------------------
// Backward, warp-per-row variant (default for d = 128 * NV, NV <= 8).  A warp owns whole rows: the two row statistics
// need one shuffle reduction per ROW (the column-owner kernels above pay a block-wide reduction per 4 rows: ~1200
// warp-instructions per row, issue-bound at 25 % -- profiles/r01_ncu_ln_bwd.txt), every lane keeps its 4*NV columns of
// dgamma / dbeta / colsum in registers across all rows of the warp, and the CTA folds its warps' partials through shared
// memory (warp after warp, no atomics) before ONE global atomicAdd per column.  ~200 warp-instructions per row.
// ---------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256, 2) layernorm_bwd_rows_kernel(const bf16* __restrict__ dy, const float* __restrict__ x,
                                                                    const float* __restrict__ gamma, const float* __restrict__ mean,
                                                                    const float* __restrict__ rstd, float* __restrict__ dx_resid,
                                                                    bf16* __restrict__ dx_bf16, float* __restrict__ dgamma,
                                                                    float* __restrict__ dbeta, float* __restrict__ dx_colsum, int N, int d,
                                                                    DropCfg drop) {
  // shared memory: gamma [d] | per-warp column accumulators [nwarps][3][d] (dgamma, dbeta, colsum).  Keeping the
  // accumulators out of the register file (72 registers at d = 768) lets two CTAs share an SM: twice the rows in flight.
  extern __shared__ __align__(16) float lnr_s[];
  float* sg = lnr_s;
  pdl_launch_dependents();
  pdl_wait();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  float* wacc = lnr_s + d + (size_t)wid * 3 * d;
  for (int i = threadIdx.x; i < d; i += blockDim.x) sg[i] = gamma[i];
  for (int i = lane; i < 3 * d; i += 32) wacc[i] = 0.f;
  __syncthreads();
  const float inv_d = 1.0f / (float)d;
  const uint32_t dkey = drop.seed ? drop_key(drop) : 0u;
  const int gw = blockIdx.x * nwarps + wid, tw = gridDim.x * nwarps;
  for (int row = gw; row < N; row += tw) {
    const size_t off = (size_t)row * d;
    const float4* x4 = reinterpret_cast<const float4*>(x + off);
    const uint2* d2 = reinterpret_cast<const uint2*>(dy + off);
    float4* r4 = reinterpret_cast<float4*>(dx_resid + off);
    float4 xv[NV], rv[NV];
    uint2 dv[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) { xv[k] = x4[lane + 32 * k]; dv[k] = d2[lane + 32 * k]; rv[k] = r4[lane + 32 * k]; }
    const float mu = __ldg(mean + row), rs = __ldg(rstd + row);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int c4 = lane + 32 * k;
      const float4 g = *reinterpret_cast<const float4*>(sg + 4 * c4);
      const float2 d01 = unpack_bf16x2(dv[k].x), d23 = unpack_bf16x2(dv[k].y);
      xv[k] = make_float4((xv[k].x - mu) * rs, (xv[k].y - mu) * rs, (xv[k].z - mu) * rs, (xv[k].w - mu) * rs);   // xhat
      const float g0 = d01.x * g.x, g1 = d01.y * g.y, g2 = d23.x * g.z, g3 = d23.y * g.w;
      s1 += (g0 + g1) + (g2 + g3);
      s2 += (g0 * xv[k].x + g1 * xv[k].y) + (g2 * xv[k].z + g3 * xv[k].w);
      float4* ag = reinterpret_cast<float4*>(wacc + 4 * c4);
      float4* ab = reinterpret_cast<float4*>(wacc + d + 4 * c4);
      float4 t = *ag;
      t.x += d01.x * xv[k].x; t.y += d01.y * xv[k].y; t.z += d23.x * xv[k].z; t.w += d23.y * xv[k].w;
      *ag = t;
      t = *ab;
      t.x += d01.x; t.y += d01.y; t.z += d23.x; t.w += d23.y;
      *ab = t;
    }
    const float m1 = warp_sum(s1) * inv_d, m2 = warp_sum(s2) * inv_d;
    uint32_t rk = 0u;
    if (drop.seed) rk = drop_rowkey(dkey, (uint32_t)row);
    uint2* b2 = dx_bf16 ? reinterpret_cast<uint2*>(dx_bf16 + off) : nullptr;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int c4 = lane + 32 * k;
      const float4 g = *reinterpret_cast<const float4*>(sg + 4 * c4);
      const float2 d01 = unpack_bf16x2(dv[k].x), d23 = unpack_bf16x2(dv[k].y);
      float4 o = rv[k];
      o.x += rs * (d01.x * g.x - m1 - xv[k].x * m2);
      o.y += rs * (d01.y * g.y - m1 - xv[k].y * m2);
      o.z += rs * (d23.x * g.z - m1 - xv[k].z * m2);
      o.w += rs * (d23.y * g.w - m1 - xv[k].w * m2);
      r4[c4] = o;
      if (drop.seed) {  // gradient entering the dropped-out residual branch: mask * scale * dx
        float m0, m1_, m2_, m3;
        drop_pair(rk, 2u * c4, drop.thr16, drop.scale, m0, m1_);
        drop_pair(rk, 2u * c4 + 1u, drop.thr16, drop.scale, m2_, m3);
        o.x *= m0; o.y *= m1_; o.z *= m2_; o.w *= m3;
      }
      if (b2) b2[c4] = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
      if (dx_colsum) {
        float4* ac = reinterpret_cast<float4*>(wacc + 2 * d + 4 * c4);
        float4 t = *ac;
        t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
        *ac = t;
      }
    }
  }
  __syncthreads();
  // fold the warps' slices: one thread per column, one global atomic per column and CTA
  for (int i = threadIdx.x; i < d; i += blockDim.x) {
    float a = 0.f, b = 0.f, c = 0.f;
    for (int w = 0; w < nwarps; ++w) {
      const float* s = lnr_s + d + (size_t)w * 3 * d;
      a += s[i]; b += s[d + i]; c += s[2 * d + i];
    }
    atomicAdd(dgamma + i, a);
    atomicAdd(dbeta + i, b);
    if (dx_colsum) atomicAdd(dx_colsum + i, c);
  }
}

}  // namespace neko

namespace neko {

static bool ln_al(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

// Argument checks and kernel choice of neko_layernorm_bwd, shared with neko_layernorm_bwd_path so that the query reports
// exactly what a launch runs.  Touches no device state beyond sm_count().
struct LnBwdPlan {
  int kernel;          // 0 warp-per-row, 1 staged, 2 register (column-owner kernels)
  int grid, threads, rows_per_cta, stages;
  size_t smem;
};

static int ln_bwd_plan(const uint16_t* dy_bf16, const float* x, const float* gamma, const float* mean, const float* rstd,
                       const float* dx_resid, const uint16_t* dx_bf16, const float* dgamma, const float* dbeta, int N, int d,
                       LnBwdPlan& p) {
  NEKO_REQUIRE(dy_bf16 && x && gamma && mean && rstd && dx_resid && dgamma && dbeta, "layernorm_bwd: null pointer");
  NEKO_REQUIRE(N > 0 && d > 0 && d % 4 == 0 && d <= LN_MAX_D, "layernorm_bwd: need d %% 4 == 0 and d <= %d (got %d)", LN_MAX_D, d);
  NEKO_REQUIRE(ln_al(x, 16) && ln_al(dx_resid, 16) && ln_al(gamma, 16) && ln_al(dy_bf16, 8) && ln_al(dx_bf16, 8),
               "layernorm_bwd: x, dx_resid and gamma must be 16-byte aligned, dy and dx_bf16 8-byte aligned");
  // warp-per-row variant (default): d = 128 * NV with NV <= 8
  static const bool force_cols = getenv("NEKO_LN_BWD_COLUMNS") != nullptr;
  if (!force_cols && d % 128 == 0 && d <= 1024) {
    int grid = 2 * sm_count();                                       // two CTAs per SM
    const int rows_per_grid = grid * 8;
    if (N < rows_per_grid) grid = (N + 7) / 8;
    p = LnBwdPlan{0, grid, 256, 0, 0, (size_t)(1 + 8 * 3) * d * sizeof(float)};   // gamma + 8 warps x 3 accumulator rows
    return NEKO_OK;
  }
  // column-owner kernels: one float4 column group per thread, a CTA owns rows_per_cta consecutive rows.
  // ~2 CTAs per SM: enough loads in flight (12 per thread), few enough CTAs that the final atomics stay cheap
  int ctas = sm_count() * 2;
  if (const char* e = getenv("NEKO_LN_CTAS")) {   // values below 1 (or not a number) keep the default
    const int v = atoi(e);
    if (v >= 1) ctas = v;
  }
  int rows_per_cta = (N + ctas - 1) / ctas;
  rows_per_cta = ((rows_per_cta + LNB_ROWS - 1) / LNB_ROWS) * LNB_ROWS;
  ctas = (N + rows_per_cta - 1) / rows_per_cta;
  const int threads = ((d / 4 + 31) / 32) * 32;
  // staged variant: ring of `stages` row blocks (40 d bytes each) in shared memory, two CTAs per SM
  const size_t stage_bytes = (size_t)LNB_ROWS * d * 10;
  int stages = (int)((100 * 1024) / stage_bytes);
  if (stages > 4) stages = 4;
  static const bool force_reg = getenv("NEKO_LN_BWD_REGISTER") != nullptr;
  if (stages >= 2 && d % 8 == 0 && ln_al(dy_bf16, 16) && !force_reg) {
    p = LnBwdPlan{1, ctas, threads, rows_per_cta, stages, stage_bytes * stages};
    return NEKO_OK;
  }
  p = LnBwdPlan{2, ctas, threads, rows_per_cta, 0, 0};
  return NEKO_OK;
}

}  // namespace neko

extern "C" {

int neko_layernorm_fwd(const float* x, const float* gamma, const float* beta, uint16_t* y_bf16, uint16_t* y2_bf16, float* mean,
                       float* rstd, int N, int d, float eps, int out_f16, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(x && gamma && beta && y_bf16 && mean && rstd, "layernorm_fwd: null pointer");
  NEKO_REQUIRE(N > 0 && d > 0 && d % 4 == 0 && d <= LN_MAX_D, "layernorm_fwd: need d %% 4 == 0 and d <= %d (got %d)", LN_MAX_D, d);
  NEKO_REQUIRE(ln_al(x, 16) && ln_al(gamma, 16) && ln_al(beta, 16) && ln_al(y_bf16, 8) && ln_al(y2_bf16, 8),
               "layernorm_fwd: x, gamma and beta must be 16-byte aligned, y and y2 8-byte aligned");
  const int threads = 256;
  const long long blocks = ((long long)N * 32 + threads - 1) / threads;
#define NEKO_LN_FWD(NV) launch_pdl(layernorm_fwd_kernel<NV>, dim3((unsigned)blocks), dim3(threads), 0, as_stream(stream), x, gamma, beta, y_bf16, y2_bf16, mean, rstd, N, d, eps, out_f16)
  const int need = (d / 4 + 31) / 32;
  if (need <= 1) NEKO_LN_FWD(1); else if (need <= 2) NEKO_LN_FWD(2); else if (need <= 4) NEKO_LN_FWD(4);
  else if (need <= 6) NEKO_LN_FWD(6); else if (need <= 8) NEKO_LN_FWD(8); else NEKO_LN_FWD(16);
#undef NEKO_LN_FWD
  NEKO_LAUNCH_CHECK("layernorm_fwd_kernel");
  return NEKO_OK;
}

int neko_layernorm_bwd_path(const uint16_t* dy_bf16, const float* x, const float* gamma, const float* mean, const float* rstd,
                            const float* dx_resid, const uint16_t* dx_bf16, const float* dgamma, const float* dbeta,
                            const float* dx_colsum, int N, int d, const neko_dropout* branch_drop, neko_layernorm_bwd_path_info* out) {
  using namespace neko;
  (void)dx_colsum;
  (void)branch_drop;
  LnBwdPlan p;
  const int rc = ln_bwd_plan(dy_bf16, x, gamma, mean, rstd, dx_resid, dx_bf16, dgamma, dbeta, N, d, p);
  if (rc != NEKO_OK) return rc;
  if (out) {
    out->grid = p.grid;
    out->rows_per_cta = p.rows_per_cta;
    out->stages = p.stages;
  }
  return p.kernel;
}

int neko_layernorm_bwd(const uint16_t* dy_bf16, const float* x, const float* gamma, const float* mean, const float* rstd,
                       float* dx_resid, uint16_t* dx_bf16, float* dgamma, float* dbeta, float* dx_colsum, int N, int d,
                       const neko_dropout* branch_drop, void* stream) {
  using namespace neko;
  LnBwdPlan p;
  const int rc = ln_bwd_plan(dy_bf16, x, gamma, mean, rstd, dx_resid, dx_bf16, dgamma, dbeta, N, d, p);
  if (rc != NEKO_OK) return rc;
  const DropCfg dc = drop_cfg(branch_drop);
  if (p.kernel == 0) {
    const int nv = d / 128;
#define NEKO_LNB_ROWS(NV_) { static bool attr_##NV_ = false;                                                                      \
      if (!attr_##NV_) {                                                                                                          \
        cudaError_t e_ = cudaFuncSetAttribute(layernorm_bwd_rows_kernel<NV_>, cudaFuncAttributeMaxDynamicSharedMemorySize, 104 * 1024); \
        if (e_ != cudaSuccess) return check_cuda(e_, "cudaFuncSetAttribute(layernorm_bwd_rows)");                                    \
        attr_##NV_ = true; } }                                                                                                      \
    launch_pdl(layernorm_bwd_rows_kernel<NV_>, dim3(p.grid), dim3(p.threads), p.smem, as_stream(stream), \
                                      reinterpret_cast<const bf16*>(dy_bf16), x, gamma, mean, rstd, dx_resid, reinterpret_cast<bf16*>(dx_bf16), \
                                      dgamma, dbeta, dx_colsum, N, d, dc)
    switch (nv) {
      case 1: NEKO_LNB_ROWS(1); break;
      case 2: NEKO_LNB_ROWS(2); break;
      case 3: NEKO_LNB_ROWS(3); break;
      case 4: NEKO_LNB_ROWS(4); break;
      case 5: NEKO_LNB_ROWS(5); break;
      case 6: NEKO_LNB_ROWS(6); break;
      case 7: NEKO_LNB_ROWS(7); break;
      default: NEKO_LNB_ROWS(8); break;
    }
#undef NEKO_LNB_ROWS
    NEKO_LAUNCH_CHECK("layernorm_bwd_rows_kernel");
    return NEKO_OK;
  }
  if (p.kernel == 1) {
    static size_t attr_smem = 0;
    if (p.smem > attr_smem) {
      cudaError_t e = cudaFuncSetAttribute(layernorm_bwd_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem);
      if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(layernorm_bwd_staged)");
      attr_smem = p.smem;
    }
    launch_pdl(layernorm_bwd_staged_kernel, dim3(p.grid), dim3(p.threads), p.smem, as_stream(stream), reinterpret_cast<const bf16*>(dy_bf16), x,
               gamma, mean, rstd, dx_resid, reinterpret_cast<bf16*>(dx_bf16), dgamma, dbeta, dx_colsum, N, d, p.rows_per_cta, p.stages, dc);
    NEKO_LAUNCH_CHECK("layernorm_bwd_staged_kernel");
    return NEKO_OK;
  }
  launch_pdl(layernorm_bwd_kernel, dim3(p.grid), dim3(p.threads), 0, as_stream(stream), reinterpret_cast<const bf16*>(dy_bf16), x, gamma, mean, rstd,
             dx_resid, reinterpret_cast<bf16*>(dx_bf16), dgamma, dbeta, dx_colsum, N, d, p.rows_per_cta, dc);
  NEKO_LAUNCH_CHECK("layernorm_bwd_kernel");
  return NEKO_OK;
}

}  // extern "C"
