// LayerNorm forward / backward for the decoder (ln_1, ln_2, ln_f; trajectory_gpt2.py:323,353,779).
//
// Forward reads the fp32 residual stream and emits the bf16 GEMM operand plus per-row mean / rstd.
// Backward fuses the residual-gradient add: dx_resid += LN'(dy), optionally emitting the bf16 copy
// the next dgrad/wgrad GEMM consumes.  HBM-bound; one warp per row, 128-bit accesses, row kept in
// registers (d <= 2048).
#include <stdlib.h>
#include "common.cuh"
#include "dropout.cuh"
#include "ordered.cuh"

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

// the column-owner kernels' final flush: one atomicAdd per column and CTA
__device__ __forceinline__ void ln_cols_flush(int c4, const float4& ag, const float4& ab, const float4& ac, float* dgamma, float* dbeta,
                                              float* dx_colsum) {
  float* pg = dgamma + 4 * c4;
  float* pb = dbeta + 4 * c4;
  atomicAdd(pg, ag.x); atomicAdd(pg + 1, ag.y); atomicAdd(pg + 2, ag.z); atomicAdd(pg + 3, ag.w);
  atomicAdd(pb, ab.x); atomicAdd(pb + 1, ab.y); atomicAdd(pb + 2, ab.z); atomicAdd(pb + 3, ab.w);
  if (dx_colsum) {
    float* pc = dx_colsum + 4 * c4;
    atomicAdd(pc, ac.x); atomicAdd(pc + 1, ac.y); atomicAdd(pc + 2, ac.z); atomicAdd(pc + 3, ac.w);
  }
}

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
#define LN_COLS_STAGED 0
#include "ln_bwd_cols.cuh"
#undef LN_COLS_STAGED
  }
  if (act) ln_cols_flush(c4, ag, ab, ac, dgamma, dbeta, dx_colsum);
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
#define LN_COLS_STAGED 1
#include "ln_bwd_cols.cuh"
#undef LN_COLS_STAGED
  }
  if (act) ln_cols_flush(c4, ag, ab, ac, dgamma, dbeta, dx_colsum);
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
  for (int row = gw; row < N; row += tw)
#define LN_ROW_GUARD 0
#define LN_ROW_COLSUM dx_colsum
#include "ln_bwd_row.cuh"
#undef LN_ROW_GUARD
#undef LN_ROW_COLSUM
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


// ---------------------------------------------------------------------------------------------
// Backward, ordered (deterministic mode): the warp-per-row math for any d % 4 == 0, d <= 2048.  Block `blk` = rows
// [64 blk, 64 blk + 64): warp w takes rows 64 blk + w, + 8, ... in ascending order into its own shared accumulators, the warps
// are folded in order 0..7 and the block's dgamma | dbeta | colsum partials go to workspace row blk.
// ---------------------------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(256) layernorm_bwd_ordered_kernel(const bf16* __restrict__ dy, const float* __restrict__ x,
                                                                    const float* __restrict__ gamma, const float* __restrict__ mean,
                                                                    const float* __restrict__ rstd, float* __restrict__ dx_resid,
                                                                    bf16* __restrict__ dx_bf16, float* __restrict__ ws, int N, int d,
                                                                    int n_blocks, int with_colsum, DropCfg drop) {
  extern __shared__ __align__(16) float lno_s[];   // gamma [d] | per-warp accumulators [8][3][d]
  float* sg = lno_s;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* wacc = lno_s + d + (size_t)wid * 3 * d;
  for (int i = threadIdx.x; i < d; i += blockDim.x) sg[i] = gamma[i];
  const int nv4 = d >> 2;
  const float inv_d = 1.0f / (float)d;
  const uint32_t dkey = drop.seed ? drop_key(drop) : 0u;
  for (int blk = blockIdx.x; blk < n_blocks; blk += gridDim.x) {
    for (int i = lane; i < 3 * d; i += 32) wacc[i] = 0.f;
    __syncthreads();
    const int r_end = min(N, (blk + 1) * ORD_ROWS);
    for (int row = blk * ORD_ROWS + wid; row < r_end; row += 8)
#define LN_ROW_GUARD 1
#define LN_ROW_COLSUM with_colsum
#include "ln_bwd_row.cuh"
#undef LN_ROW_GUARD
#undef LN_ROW_COLSUM
    __syncthreads();
    float* out = ws + (size_t)blk * 3 * d;
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
      float a = 0.f, b = 0.f, c = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const float* s = lno_s + d + (size_t)w * 3 * d;
        a += s[i]; b += s[d + i]; c += s[2 * d + i];
      }
      out[i] = a;
      out[d + i] = b;
      if (with_colsum) out[2 * d + i] = c;
    }
    __syncthreads();   // the next block re-zeroes the accumulators just read
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

int64_t neko_layernorm_bwd_ordered_workspace_bytes(int N, int d) {
  using namespace neko;
  NEKO_REQUIRE(N > 0 && d > 0 && d % 4 == 0 && d <= LN_MAX_D, "layernorm_bwd_ordered: need N > 0, d %% 4 == 0 and d <= %d", LN_MAX_D);
  return (int64_t)((N + ORD_ROWS - 1) / ORD_ROWS) * 3 * d * (int64_t)sizeof(float);
}

int neko_layernorm_bwd_ordered(const uint16_t* dy_bf16, const float* x, const float* gamma, const float* mean, const float* rstd,
                               float* dx_resid, uint16_t* dx_bf16, float* dgamma, float* dbeta, float* dx_colsum, int N, int d,
                               const neko_dropout* branch_drop, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(dy_bf16 && x && gamma && mean && rstd && dx_resid && dgamma && dbeta && workspace, "layernorm_bwd_ordered: null pointer");
  const int64_t need = neko_layernorm_bwd_ordered_workspace_bytes(N, d);
  if (need < 0) return (int)need;
  NEKO_REQUIRE(workspace_bytes >= need, "layernorm_bwd_ordered: workspace of %lld bytes, need %lld", (long long)workspace_bytes, (long long)need);
  NEKO_REQUIRE(ln_al(x, 16) && ln_al(dx_resid, 16) && ln_al(gamma, 16) && ln_al(dy_bf16, 8) && ln_al(dx_bf16, 8) && ln_al(workspace, 16),
               "layernorm_bwd_ordered: x, dx_resid, gamma and the workspace must be 16-byte aligned, dy and dx_bf16 8-byte aligned");
  const int n_blocks = (N + ORD_ROWS - 1) / ORD_ROWS;
  const int need_v = (d / 4 + 31) / 32;
  const size_t smem = (size_t)(1 + 8 * 3) * d * sizeof(float);
  float* ws = static_cast<float*>(workspace);
  const DropCfg dc = drop_cfg(branch_drop);
  const int grid = ordered_grid(n_blocks);
#define NEKO_LN_ORD(NV_) {                                                                                                          \
    static bool attr_ = false;                                                                                                      \
    if (!attr_) {                                                                                                                   \
      cudaError_t e_ = cudaFuncSetAttribute(layernorm_bwd_ordered_kernel<NV_>, cudaFuncAttributeMaxDynamicSharedMemorySize,           \
                                            (int)((1 + 8 * 3) * LN_MAX_D * sizeof(float)));                                        \
      if (e_ != cudaSuccess) return check_cuda(e_, "cudaFuncSetAttribute(layernorm_bwd_ordered)");                                  \
      attr_ = true;                                                                                                                 \
    }                                                                                                                               \
    layernorm_bwd_ordered_kernel<NV_><<<grid, 256, smem, as_stream(stream)>>>(                                                      \
        reinterpret_cast<const bf16*>(dy_bf16), x, gamma, mean, rstd, dx_resid, reinterpret_cast<bf16*>(dx_bf16), ws, N, d,        \
        n_blocks, dx_colsum != nullptr, dc); }
  if (need_v <= 1) NEKO_LN_ORD(1) else if (need_v <= 2) NEKO_LN_ORD(2) else if (need_v <= 3) NEKO_LN_ORD(3)
  else if (need_v <= 4) NEKO_LN_ORD(4) else if (need_v <= 6) NEKO_LN_ORD(6) else if (need_v <= 8) NEKO_LN_ORD(8)
  else if (need_v <= 12) NEKO_LN_ORD(12) else NEKO_LN_ORD(16)
#undef NEKO_LN_ORD
  NEKO_LAUNCH_CHECK("layernorm_bwd_ordered_kernel");
  OrdDst dst{};
  dst.p[0] = dgamma; dst.p[1] = dbeta; dst.p[2] = dx_colsum;
  dst.off[0] = 0; dst.off[1] = d; dst.off[2] = 2 * d;
  dst.n = dx_colsum ? 3 : 2;
  for (int i = dst.n; i < 7; ++i) dst.off[i] = i == dst.n ? dst.n * d : 0x7fffffff;
  return ordered_colreduce(ws, 3LL * d, n_blocks, dst.n * d, dst, 1, as_stream(stream));
}

}  // extern "C"
