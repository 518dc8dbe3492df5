#include <algorithm>
// Memory-bound helpers around the GEMMs: dtype cast, bias-gradient column sums, row gather/scatter.
#include "common.cuh"
#include "dropout.cuh"

namespace neko {

__global__ void __launch_bounds__(256) cast_f32_16_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, long long n, int f16) {
  const long long nv = n >> 2;
  const float4* s4 = reinterpret_cast<const float4*>(src);
  uint2* d2 = reinterpret_cast<uint2*>(dst);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
    const float4 v = __ldg(s4 + i);
    d2[i] = make_uint2(pack_16x2(v.x, v.y, f16 != 0), pack_16x2(v.z, v.w, f16 != 0));
  }
  for (long long i = (nv << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = cvt_16(src[i], f16 != 0);
}

// out[n] += sum over a row chunk of X[m, n].  Block = 32 x 8 threads, each thread owns 2 adjacent columns.
__global__ void __launch_bounds__(256) cast_f32_dual_kernel(const float* __restrict__ src, uint16_t* __restrict__ d16, uint16_t* __restrict__ dbf, long long n) {
  const long long nv = n >> 2;
  const float4* s4 = reinterpret_cast<const float4*>(src);
  uint2* a2 = reinterpret_cast<uint2*>(d16);
  uint2* b2 = reinterpret_cast<uint2*>(dbf);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
    const float4 v = __ldg(s4 + i);
    a2[i] = make_uint2(pack_f16x2(v.x, v.y), pack_f16x2(v.z, v.w));
    b2[i] = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
  }
  for (long long i = (nv << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    d16[i] = cvt_16(src[i], true);
    dbf[i] = cvt_16(src[i], false);
  }
}

__global__ void __launch_bounds__(256) colsum_bf16_kernel(const bf16* __restrict__ X, long long ld, int M, int N, int rows_per_cta,
                                                          float* __restrict__ out) {
  __shared__ float red[8][64];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 64 + tx * 2;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(M, r0 + rows_per_cta);
  float a0 = 0.f, a1 = 0.f;
  if (col + 1 < N) {
    for (int r = r0 + ty; r < r1; r += 8) {
      const float2 v = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(X + (size_t)r * ld + col));
      a0 += v.x; a1 += v.y;
    }
  } else if (col < N) {
    for (int r = r0 + ty; r < r1; r += 8) a0 += __bfloat162float(X[(size_t)r * ld + col]);
  }
  red[ty][tx * 2] = a0;
  red[ty][tx * 2 + 1] = a1;
  __syncthreads();
  if (threadIdx.x < 64) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][threadIdx.x];
    const int c = blockIdx.x * 64 + threadIdx.x;
    if (c < N) atomicAdd(out + c, s);
  }
}

// wide variant: 16-byte loads (8 columns per thread), four rows in flight per thread
__global__ void __launch_bounds__(256) colsum_bf16_wide_kernel(const bf16* __restrict__ X, long long ld, int M, int N, int rows_per_cta,
                                                               float* __restrict__ out) {
  __shared__ float red[8][256];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int col = blockIdx.x * 256 + tx * 8;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(M, r0 + rows_per_cta);
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 0.f;
  if (col < N) {   // N % 8 == 0: a column group is either fully inside or fully outside
    const bf16* base = X + col;
    int r = r0 + ty;
    for (; r + 24 < r1; r += 32) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const uint4*>(base + (size_t)(r + 8 * u) * ld);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) { const float2 f = unpack_bf16x2(w[j]); a[2 * j] += f.x; a[2 * j + 1] += f.y; }
      }
    }
    for (; r < r1; r += 8) {
      const uint4 v = *reinterpret_cast<const uint4*>(base + (size_t)r * ld);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) { const float2 f = unpack_bf16x2(w[j]); a[2 * j] += f.x; a[2 * j + 1] += f.y; }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[ty][tx * 8 + i] = a[i];
  __syncthreads();
  {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][threadIdx.x];
    const int c = blockIdx.x * 256 + threadIdx.x;
    if (c < N) atomicAdd(out + c, s);
  }
}

__global__ void __launch_bounds__(256) gather_rows_bf16_kernel(const bf16* __restrict__ src, long long ld_src, const int32_t* __restrict__ rows,
                                                               int n_rows, int n, bf16* __restrict__ dst, long long ld_dst) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n_rows) return;
  const bf16* s = src + (size_t)rows[w] * ld_src;
  bf16* d = dst + (size_t)w * ld_dst;
  if ((n & 7) == 0 && (ld_src & 7) == 0 && (ld_dst & 7) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(s);
    uint4* d4 = reinterpret_cast<uint4*>(d);
    for (int i = lane; i < (n >> 3); i += 32) d4[i] = __ldg(s4 + i);
  } else {
    for (int i = lane; i < n; i += 32) d[i] = s[i];
  }
}

__global__ void __launch_bounds__(256) scatter_rows_bf16_kernel(const bf16* __restrict__ src, long long ld_src, const int32_t* __restrict__ rows,
                                                                int n_rows, int n, bf16* __restrict__ dst, long long ld_dst) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n_rows) return;
  const bf16* s = src + (size_t)w * ld_src;
  bf16* d = dst + (size_t)rows[w] * ld_dst;
  if ((n & 7) == 0 && (ld_src & 7) == 0 && (ld_dst & 7) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(s);
    uint4* d4 = reinterpret_cast<uint4*>(d);
    for (int i = lane; i < (n >> 3); i += 32) d4[i] = __ldg(s4 + i);
  } else {
    for (int i = lane; i < n; i += 32) d[i] = s[i];
  }
}

__global__ void __launch_bounds__(256) scatter_rows_add_kernel(const bf16* __restrict__ src, long long ld_src, const int32_t* __restrict__ rows,
                                                               int n_rows, int n, float* __restrict__ dst, long long ld_dst) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n_rows) return;
  const bf16* s = src + (size_t)w * ld_src;
  float* d = dst + (size_t)rows[w] * ld_dst;  // rows are unique: plain read-modify-write
  for (int i = lane; i < n; i += 32) d[i] += __bfloat162float(s[i]);
}

// ---- GEGLU gate (MLP.forward with gate, trajectory_gpt2.py:267-276): h = gelu(c_fc(x)) * gated_layer(x) ----
// forward: act (16-bit, format of the GELU output) * gate (bf16) -> product in the forward operand format (+ bf16 copy)
__global__ void __launch_bounds__(256) geglu_fwd_kernel(const uint16_t* __restrict__ act, const bf16* __restrict__ gate,
                                                        uint16_t* __restrict__ out, uint16_t* __restrict__ out_bf, long long n8,
                                                        int act_f16, int out_f16) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 a = reinterpret_cast<const uint4*>(act)[i];
    const uint4 g = reinterpret_cast<const uint4*>(gate)[i];
    const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, gw[4] = {g.x, g.y, g.z, g.w};
    uint32_t o[4], ob[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 av = act_f16 ? unpack_f16x2(aw[j]) : unpack_bf16x2(aw[j]);
      const float2 gv = unpack_bf16x2(gw[j]);
      o[j] = pack_16x2(av.x * gv.x, av.y * gv.y, out_f16 != 0);
      ob[j] = pack_bf16x2(av.x * gv.x, av.y * gv.y);
    }
    reinterpret_cast<uint4*>(out)[i] = make_uint4(o[0], o[1], o[2], o[3]);
    if (out_bf) reinterpret_cast<uint4*>(out_bf)[i] = make_uint4(ob[0], ob[1], ob[2], ob[3]);
  }
}
// backward: dh (bf16) -> d_gate = dh * gelu(pre), d_pre = dh * gate * gelu'(pre)
__global__ void __launch_bounds__(256) geglu_bwd_kernel(const bf16* __restrict__ dh, const bf16* __restrict__ pre,
                                                        const bf16* __restrict__ gate, bf16* __restrict__ d_gate,
                                                        bf16* __restrict__ d_pre, long long n8) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 dv = reinterpret_cast<const uint4*>(dh)[i];
    const uint4 pv = reinterpret_cast<const uint4*>(pre)[i];
    const uint4 gv = reinterpret_cast<const uint4*>(gate)[i];
    const uint32_t dw[4] = {dv.x, dv.y, dv.z, dv.w}, pw[4] = {pv.x, pv.y, pv.z, pv.w}, gw[4] = {gv.x, gv.y, gv.z, gv.w};
    uint32_t og[4], op[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 d2 = unpack_bf16x2(dw[j]), p2 = unpack_bf16x2(pw[j]), g2 = unpack_bf16x2(gw[j]);
      float y0, y1, s0, s1;
      gelu_erf_both(p2.x, y0, s0);
      gelu_erf_both(p2.y, y1, s1);
      og[j] = pack_bf16x2(d2.x * y0, d2.y * y1);
      op[j] = pack_bf16x2(d2.x * g2.x * s0, d2.y * g2.y * s1);
    }
    reinterpret_cast<uint4*>(d_gate)[i] = make_uint4(og[0], og[1], og[2], og[3]);
    reinterpret_cast<uint4*>(d_pre)[i] = make_uint4(op[0], op[1], op[2], op[3]);
  }
}

// ---- dropout on an fp32 [rows, cols] tensor in place (embd dropout and its backward), and the mask itself ----
__global__ void __launch_bounds__(256) dropout_apply_kernel(float* __restrict__ x, long long ld, int rows, int cols, DropCfg drop) {
  const uint32_t key = drop_key(drop);
  const int pairs = (cols + 1) >> 1;
  const long long total = (long long)rows * pairs;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(i / pairs), pr = (int)(i - (long long)row * pairs);
    float m0, m1;
    drop_pair(drop_rowkey(key, (uint32_t)row), (uint32_t)pr, drop.thr16, drop.scale, m0, m1);
    float* q = x + (long long)row * ld + 2 * pr;
    q[0] *= m0;
    if (2 * pr + 1 < cols) q[1] *= m1;
  }
}
__global__ void __launch_bounds__(256) dropout_mask_kernel(uint8_t* __restrict__ keep, int rows, int cols, DropCfg drop) {
  const uint32_t key = drop_key(drop);
  const int pairs = (cols + 1) >> 1;
  const long long total = (long long)rows * pairs;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int row = (int)(i / pairs), pr = (int)(i - (long long)row * pairs);
    float m0, m1;
    drop_pair(drop_rowkey(key, (uint32_t)row), (uint32_t)pr, drop.thr16, 1.0f, m0, m1);
    uint8_t* q = keep + (long long)row * cols + 2 * pr;
    q[0] = m0 != 0.f;
    if (2 * pr + 1 < cols) q[1] = m1 != 0.f;
  }
}

}  // namespace neko

extern "C" {

static int cast_impl(const float* src, uint16_t* dst, int64_t n, int f16, void* stream) {
  using namespace neko;
  if (n == 0) return NEKO_OK;   // an empty tensor may have no storage (null pointers): nothing to do
  NEKO_REQUIRE(src && dst && n > 0, "cast: bad arguments");
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0, "cast: misaligned buffers");
  long long blocks = (n / 4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  cast_f32_16_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(src, dst, n, f16);
  NEKO_LAUNCH_CHECK("cast_f32_16_kernel");
  return NEKO_OK;
}

int neko_cast_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, void* stream) { return cast_impl(src, dst, n, 0, stream); }
int neko_cast_f32_to_f16(const float* src, uint16_t* dst, int64_t n, void* stream) { return cast_impl(src, dst, n, 1, stream); }

int neko_cast_f32_to_f16_bf16(const float* src, uint16_t* dst_f16, uint16_t* dst_bf16, int64_t n, void* stream) {
  using namespace neko;
  if (n == 0) return NEKO_OK;
  NEKO_REQUIRE(src && dst_f16 && dst_bf16 && n > 0, "cast: bad arguments");
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst_f16) & 7) == 0 &&
               (reinterpret_cast<uintptr_t>(dst_bf16) & 7) == 0, "cast: misaligned buffers");
  long long blocks = (n / 4 + 255) / 256;
  const long long cap = (long long)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  cast_f32_dual_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(src, dst_f16, dst_bf16, n);
  NEKO_LAUNCH_CHECK("cast_f32_dual_kernel");
  return NEKO_OK;
}

int neko_colsum_bf16(const uint16_t* X, int64_t ld, int M, int N, float* out, int accumulate, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(X && out && M > 0 && N > 0 && ld >= N, "colsum: bad arguments");
  NEKO_REQUIRE(ld % 2 == 0 && (reinterpret_cast<uintptr_t>(X) & 3) == 0, "colsum: X must be 4-byte aligned with an even pitch");
  if (!accumulate) {
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)N, as_stream(stream));
    if (e != cudaSuccess) return check_cuda(e, "cudaMemsetAsync(colsum)");
  }
  if (N % 8 == 0 && ld % 8 == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0) {
    const int cb = (N + 255) / 256;
    int chunks = (sm_count() * 8 + cb - 1) / cb;     // ~8 resident CTAs per SM (32 registers, 8 KB shared memory each)
    if (chunks > (M + 31) / 32) chunks = (M + 31) / 32;
    if (chunks < 1) chunks = 1;
    const int rpc = (M + chunks - 1) / chunks;
    dim3 grid(cb, (M + rpc - 1) / rpc);
    colsum_bf16_wide_kernel<<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const bf16*>(X), ld, M, N, rpc, out);
    NEKO_LAUNCH_CHECK("colsum_bf16_wide_kernel");
    return NEKO_OK;
  }
  const int col_blocks = (N + 63) / 64;
  int row_chunks = (sm_count() * 4 + col_blocks - 1) / col_blocks;
  if (row_chunks > (M + 63) / 64) row_chunks = (M + 63) / 64;
  if (row_chunks < 1) row_chunks = 1;
  const int rows_per_cta = (M + row_chunks - 1) / row_chunks;
  dim3 grid(col_blocks, (M + rows_per_cta - 1) / rows_per_cta);
  colsum_bf16_kernel<<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const bf16*>(X), ld, M, N, rows_per_cta, out);
  NEKO_LAUNCH_CHECK("colsum_bf16_kernel");
  return NEKO_OK;
}

int neko_gather_rows_bf16(const uint16_t* src, int64_t ld_src, const int32_t* rows, int n_rows, int n, uint16_t* dst,
                          int64_t ld_dst, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(src && rows && dst && n > 0 && n_rows >= 0, "gather_rows: bad arguments");
  if (n_rows == 0) return NEKO_OK;
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0, "gather_rows: misaligned");
  const long long blocks = ((long long)n_rows * 32 + 255) / 256;
  gather_rows_bf16_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const bf16*>(src), ld_src, rows, n_rows, n,
                                                                            reinterpret_cast<bf16*>(dst), ld_dst);
  NEKO_LAUNCH_CHECK("gather_rows_bf16_kernel");
  return NEKO_OK;
}

int neko_scatter_rows_bf16(const uint16_t* src, int64_t ld_src, const int32_t* rows, int n_rows, int n, uint16_t* dst,
                           int64_t ld_dst, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(src && rows && dst && n > 0 && n_rows >= 0, "scatter_rows: bad arguments");
  if (n_rows == 0) return NEKO_OK;
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0, "scatter_rows: misaligned");
  const long long blocks = ((long long)n_rows * 32 + 255) / 256;
  scatter_rows_bf16_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const bf16*>(src), ld_src, rows, n_rows, n,
                                                                             reinterpret_cast<bf16*>(dst), ld_dst);
  NEKO_LAUNCH_CHECK("scatter_rows_bf16_kernel");
  return NEKO_OK;
}

int neko_scatter_rows_add_f32(const uint16_t* src_bf16, int64_t ld_src, const int32_t* rows, int n_rows, int n, float* dst,
                              int64_t ld_dst, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(src_bf16 && rows && dst && n > 0 && n_rows >= 0, "scatter_rows_add: bad arguments");
  if (n_rows == 0) return NEKO_OK;
  const long long blocks = ((long long)n_rows * 32 + 255) / 256;
  scatter_rows_add_kernel<<<(unsigned)blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const bf16*>(src_bf16), ld_src, rows, n_rows, n, dst, ld_dst);
  NEKO_LAUNCH_CHECK("scatter_rows_add_kernel");
  return NEKO_OK;
}

int neko_dropout_apply(float* x, int64_t ld, int rows, int cols, const neko_dropout* drop, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(x && rows > 0 && cols > 0 && ld >= cols, "dropout_apply: bad arguments");
  const DropCfg c = drop_cfg(drop);
  if (!c.seed) return NEKO_OK;
  const long long total = (long long)rows * ((cols + 1) / 2);
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)sm_count() * 16);
  dropout_apply_kernel<<<blocks, 256, 0, as_stream(stream)>>>(x, ld, rows, cols, c);
  NEKO_LAUNCH_CHECK("dropout_apply_kernel");
  return NEKO_OK;
}

int neko_dropout_mask(uint8_t* keep, int rows, int cols, const neko_dropout* drop, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(keep && rows > 0 && cols > 0 && drop && drop->seed, "dropout_mask: bad arguments");
  DropCfg c{drop->seed, drop->stream, drop->thr16, 1.0f};
  const long long total = (long long)rows * ((cols + 1) / 2);
  const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)sm_count() * 16);
  dropout_mask_kernel<<<blocks, 256, 0, as_stream(stream)>>>(keep, rows, cols, c);
  NEKO_LAUNCH_CHECK("dropout_mask_kernel");
  return NEKO_OK;
}

int neko_geglu_fwd(const uint16_t* act, const uint16_t* gate_bf16, uint16_t* out, uint16_t* out_bf16, int64_t n, int act_f16,
                   int out_f16, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(act && gate_bf16 && out && n > 0 && n % 8 == 0, "geglu_fwd: bad arguments (n must be a multiple of 8)");
  NEKO_REQUIRE(((reinterpret_cast<uintptr_t>(act) | reinterpret_cast<uintptr_t>(gate_bf16) | reinterpret_cast<uintptr_t>(out) |
                 reinterpret_cast<uintptr_t>(out_bf16)) & 15) == 0, "geglu_fwd: misaligned buffers");
  const long long n8 = n / 8;
  const int blocks = (int)std::min<long long>((n8 + 255) / 256, (long long)sm_count() * 16);
  geglu_fwd_kernel<<<blocks, 256, 0, as_stream(stream)>>>(act, reinterpret_cast<const bf16*>(gate_bf16), out, out_bf16, n8, act_f16, out_f16);
  NEKO_LAUNCH_CHECK("geglu_fwd_kernel");
  return NEKO_OK;
}

int neko_geglu_bwd(const uint16_t* dh_bf16, const uint16_t* pre_bf16, const uint16_t* gate_bf16, uint16_t* d_gate_bf16,
                   uint16_t* d_pre_bf16, int64_t n, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(dh_bf16 && pre_bf16 && gate_bf16 && d_gate_bf16 && d_pre_bf16 && n > 0 && n % 8 == 0, "geglu_bwd: bad arguments");
  NEKO_REQUIRE(((reinterpret_cast<uintptr_t>(dh_bf16) | reinterpret_cast<uintptr_t>(pre_bf16) | reinterpret_cast<uintptr_t>(gate_bf16) |
                 reinterpret_cast<uintptr_t>(d_gate_bf16) | reinterpret_cast<uintptr_t>(d_pre_bf16)) & 15) == 0, "geglu_bwd: misaligned buffers");
  const long long n8 = n / 8;
  const int blocks = (int)std::min<long long>((n8 + 255) / 256, (long long)sm_count() * 16);
  geglu_bwd_kernel<<<blocks, 256, 0, as_stream(stream)>>>(reinterpret_cast<const bf16*>(dh_bf16), reinterpret_cast<const bf16*>(pre_bf16),
                                                          reinterpret_cast<const bf16*>(gate_bf16), reinterpret_cast<bf16*>(d_gate_bf16),
                                                          reinterpret_cast<bf16*>(d_pre_bf16), n8);
  NEKO_LAUNCH_CHECK("geglu_bwd_kernel");
  return NEKO_OK;
}

}  // extern "C"
