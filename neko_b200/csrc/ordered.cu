// Ordered (deterministic) reductions for the deterministic training mode (DESIGN.md "Deterministic training mode").
//
// The default backward sums floats with atomics in whatever order the CTAs arrive.  The kernels here give every sum a fixed
// order that depends on the problem shape only -- not on the grid, the SM count or timing:
//   - column sums (LayerNorm dgamma / dbeta / dx_colsum, whose kernel is in layernorm.cu; bias gradients): rows are cut into
//     fixed blocks of ORD_ROWS rows; each block writes its column partials to a workspace row, and ordered_colreduce_kernel
//     folds the rows in a fixed order with one writer per output element;
//   - scatter-adds into tables (embedding / position-table gradients): (table row, source row) pairs are sorted with a
//     stable radix sort and every table row is summed by one warp in ascending source-row order;
//   - the gradient sum of squares: fixed 8192-element block partials, then one CTA folds them in a fixed order.
// Every launch goes to the caller's stream, allocates nothing and synchronises nothing (CUDA-graph capturable); scratch memory
// comes from a caller-provided workspace with a *_workspace_bytes query.
#include <stdlib.h>

#include <cub/device/device_radix_sort.cuh>

#include "ordered.cuh"

namespace neko {

constexpr int SSQ_CHUNK = 8192;       // elements per fixed block of the sum of squares

int ordered_grid(long long units) {
  long long g = units;
  if (const char* e = getenv("NEKO_ORDERED_CTAS")) {
    const long long c = atoll(e);
    if (c > 0 && c < g) g = c;
  }
  if (g > (1LL << 30)) g = 1LL << 30;
  return g < 1 ? 1 : (int)g;
}

// ---------------------------------------------------------------------------------------------
// column fold: one warp-column of 32 outputs per CTA step; warp w sums workspace rows w, w + 8, ... in ascending order,
// then warp 0 adds the eight warp partials in order 0..7.  The order is a function of n_blocks alone.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ordered_colreduce_kernel(const float* __restrict__ ws, long long ld, int n_blocks, int ncols,
                                                                OrdDst dst, int accumulate) {
  __shared__ float red[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int n_groups = (ncols + 31) / 32;
  for (int gi = blockIdx.x; gi < n_groups; gi += gridDim.x) {
    const int c = gi * 32 + lane;
    float s = 0.f;
    if (c < ncols) {
#pragma unroll 4
      for (int b = w; b < n_blocks; b += 8) s += ws[(size_t)b * ld + c];
    }
    red[w][lane] = s;
    __syncthreads();
    if (w == 0 && c < ncols) {
      float t = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) t += red[k][lane];
      int r = 0;
      while (c >= dst.off[r + 1]) ++r;
      float* q = dst.p[r] + (c - dst.off[r]);
      *q = accumulate ? *q + t : t;
    }
    __syncthreads();
  }
}

int ordered_colreduce(const float* ws, long long ld, int n_blocks, int ncols, const OrdDst& dst, int accumulate, cudaStream_t st) {
  ordered_colreduce_kernel<<<ordered_grid((ncols + 31) / 32), 256, 0, st>>>(ws, ld, n_blocks, ncols, dst, accumulate);
  NEKO_LAUNCH_CHECK("ordered_colreduce_kernel");
  return NEKO_OK;
}

// ---------------------------------------------------------------------------------------------
// bias-gradient column sums of a bf16 matrix: unit (row block rb, 64-column group cb); thread row ty takes rows
// 64 rb + ty, + 8, ... in ascending order, the eight thread rows are folded in order.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) colsum_bf16_ordered_kernel(const bf16* __restrict__ X, long long ld, int M, int N, int n_rb,
                                                                  int n_cb, float* __restrict__ ws) {
  __shared__ float red[8][64];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const long long units = (long long)n_rb * n_cb;
  for (long long u = blockIdx.x; u < units; u += gridDim.x) {
    const int rb = (int)(u / n_cb), cb = (int)(u - (long long)rb * n_cb);
    const int col = cb * 64 + tx * 2;
    const int r0 = rb * ORD_ROWS, r1 = min(M, r0 + ORD_ROWS);
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
      const int c = cb * 64 + threadIdx.x;
      if (c < N) ws[(size_t)rb * N + c] = s;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// sorted scatter-add: keys sorted ascending (stable, so equal keys keep ascending source rows).  Unit = (sorted index i,
// 128-column chunk); the unit at the first index of a key's segment sums the segment's source rows in order and adds the
// total to the key's table row: one writer per element.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ordered_segsum_kernel(const unsigned* __restrict__ keys, const int* __restrict__ vals, long long n,
                                                             const float* __restrict__ src, int d, SegDst dst) {
  const int lane = threadIdx.x & 31;
  const int nv4 = d >> 2, nch = (nv4 + 31) / 32;
  const long long units = n * nch;
  for (long long u = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); u < units; u += (long long)gridDim.x * 8) {
    const long long i = u / nch;
    const int c4 = (int)(u - i * nch) * 32 + lane;
    const unsigned k = keys[i];
    if (k >= (unsigned)dst.off[3] || (i > 0 && keys[i - 1] == k) || c4 >= nv4) continue;
    long long lo = i + 1, hi = n;   // segment end: first index holding a larger key
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (keys[mid] == k) lo = mid + 1; else hi = mid;
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (long long j = i; j < lo; ++j) {
      const float4 v = reinterpret_cast<const float4*>(src + (size_t)vals[j] * d)[c4];
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    int r = 0;
    while (k >= (unsigned)dst.off[r + 1]) ++r;
    float4* o = reinterpret_cast<float4*>(dst.p[r] + (size_t)(k - (unsigned)dst.off[r]) * d) + c4;
    float4 t = *o;
    t.x += acc.x; t.y += acc.y; t.z += acc.z; t.w += acc.w;
    *o = t;
  }
}

int key_bits(unsigned max_key) {
  int b = 1;
  while (b < 32 && (max_key >> b) != 0u) ++b;
  return b;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

int sort_ws_layout(long long n, int end_bit, void* base, SortWs& s) {
  memset(&s, 0, sizeof(s));
  size_t temp = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, temp, (const unsigned*)nullptr, (unsigned*)nullptr, (const int*)nullptr,
                                                  (int*)nullptr, n, 0, end_bit);
  if (e != cudaSuccess) return check_cuda(e, "cub::DeviceRadixSort::SortPairs (size query)");
  const size_t kb = align256((size_t)n * 4);
  char* p = static_cast<char*>(base);
  s.kin = reinterpret_cast<unsigned*>(p);
  s.vin = reinterpret_cast<int*>(p + kb);
  s.kout = reinterpret_cast<unsigned*>(p + 2 * kb);
  s.vout = reinterpret_cast<int*>(p + 3 * kb);
  s.temp = p + 4 * kb;
  s.temp_bytes = temp;
  s.total = 4 * kb + align256(temp);
  return NEKO_OK;
}

int sort_and_segsum(SortWs& s, long long n, int end_bit, const float* src, int d, const SegDst& dst, cudaStream_t st) {
  size_t temp = s.temp_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(s.temp, temp, s.kin, s.kout, s.vin, s.vout, n, 0, end_bit, st);
  if (e != cudaSuccess) return check_cuda(e, "cub::DeviceRadixSort::SortPairs");
  const long long warps = n * (((d >> 2) + 31) / 32);
  ordered_segsum_kernel<<<ordered_grid((warps + 7) / 8), 256, 0, st>>>(s.kout, s.vout, n, src, d, dst);
  NEKO_LAUNCH_CHECK("ordered_segsum_kernel");
  return NEKO_OK;
}

// ---------------------------------------------------------------------------------------------
// sum of squares: block b = elements [8192 b, 8192 b + 8192); thread t takes float4 t, t + 256, ... in order; warp butterfly;
// warps folded in order.  One CTA then folds the block partials (thread t: partials t, t + 1024, ...; fixed tree).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sumsq_ordered_kernel(const float* __restrict__ x, long long n, long long n_blocks,
                                                            float* __restrict__ part) {
  __shared__ float red[8];
  for (long long b = blockIdx.x; b < n_blocks; b += gridDim.x) {
    float acc = 0.f;
    const long long base = b * SSQ_CHUNK;
#pragma unroll
    for (int k = 0; k < SSQ_CHUNK / 1024; ++k) {
      const long long i = base + (long long)(k * 256 + threadIdx.x) * 4;
      if (i + 4 <= n) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(x + i));
        acc += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
      } else {
        for (long long e = i; e < n && e < i + 4; ++e) acc += x[e] * x[e];
      }
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int w = 0; w < 8; ++w) t += red[w];
      part[b] = t;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(1024) sumsq_ordered_final_kernel(const float* __restrict__ part, long long n_blocks, float* __restrict__ out) {
  __shared__ float red[32];
  float acc = 0.f;
  for (long long b = threadIdx.x; b < n_blocks; b += 1024) acc += part[b];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 32; ++w) t += red[w];
    *out += t;
  }
}

static bool al(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

}  // namespace neko

extern "C" {

int64_t neko_colsum_bf16_ordered_workspace_bytes(int M, int N) {
  using namespace neko;
  NEKO_REQUIRE(M > 0 && N > 0, "colsum_ordered: bad shape %d x %d", M, N);
  return (int64_t)((M + ORD_ROWS - 1) / ORD_ROWS) * N * (int64_t)sizeof(float);
}

int neko_colsum_bf16_ordered(const uint16_t* X, int64_t ld, int M, int N, float* out, int accumulate, void* workspace,
                             int64_t workspace_bytes, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(X && out && workspace && ld >= N, "colsum_ordered: bad arguments");
  const int64_t need = neko_colsum_bf16_ordered_workspace_bytes(M, N);
  if (need < 0) return (int)need;
  NEKO_REQUIRE(workspace_bytes >= need, "colsum_ordered: workspace of %lld bytes, need %lld", (long long)workspace_bytes, (long long)need);
  NEKO_REQUIRE(ld % 2 == 0 && al(X, 4) && al(workspace, 4), "colsum_ordered: X must be 4-byte aligned with an even pitch");
  const int n_rb = (M + ORD_ROWS - 1) / ORD_ROWS, n_cb = (N + 63) / 64;
  float* ws = static_cast<float*>(workspace);
  colsum_bf16_ordered_kernel<<<ordered_grid((long long)n_rb * n_cb), 256, 0, as_stream(stream)>>>(reinterpret_cast<const bf16*>(X), ld,
                                                                                                   M, N, n_rb, n_cb, ws);
  NEKO_LAUNCH_CHECK("colsum_bf16_ordered_kernel");
  OrdDst dst{};
  dst.p[0] = out; dst.off[0] = 0; dst.off[1] = N; dst.n = 1;
  for (int i = 2; i < 7; ++i) dst.off[i] = 0x7fffffff;
  return ordered_colreduce(ws, N, n_rb, N, dst, accumulate, as_stream(stream));
}

int64_t neko_sumsq_f32_ordered_workspace_bytes(int64_t n) {
  using namespace neko;
  NEKO_REQUIRE(n >= 0, "sumsq_ordered: negative length");
  return ((n + SSQ_CHUNK - 1) / SSQ_CHUNK) * (int64_t)sizeof(float);
}

int neko_sumsq_f32_ordered(const float* x, int64_t n, float* out_accum, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(x && out_accum && n >= 0, "sumsq_ordered: bad arguments");
  if (n == 0) return NEKO_OK;
  const int64_t need = neko_sumsq_f32_ordered_workspace_bytes(n);
  NEKO_REQUIRE(workspace && workspace_bytes >= need, "sumsq_ordered: workspace of %lld bytes, need %lld", (long long)workspace_bytes, (long long)need);
  NEKO_REQUIRE(al(x, 16) && al(workspace, 4), "sumsq_ordered: misaligned");
  const long long n_blocks = (n + SSQ_CHUNK - 1) / SSQ_CHUNK;
  float* part = static_cast<float*>(workspace);
  sumsq_ordered_kernel<<<ordered_grid(n_blocks), 256, 0, as_stream(stream)>>>(x, n, n_blocks, part);
  NEKO_LAUNCH_CHECK("sumsq_ordered_kernel");
  sumsq_ordered_final_kernel<<<1, 1024, 0, as_stream(stream)>>>(part, n_blocks, out_accum);
  NEKO_LAUNCH_CHECK("sumsq_ordered_final_kernel");
  return NEKO_OK;
}

int64_t neko_patch_pos_bwd_ordered_workspace_bytes(int P, int n_row_bins, int n_col_bins) {
  using namespace neko;
  NEKO_REQUIRE(P > 0 && n_row_bins > 0 && n_col_bins > 0, "patch_pos_bwd_ordered: bad sizes");
  SortWs s;
  const int rc = sort_ws_layout(2LL * P, key_bits((unsigned)(n_row_bins + n_col_bins)), nullptr, s);
  if (rc != NEKO_OK) return rc;
  return (int64_t)s.total;
}

}  // extern "C"

namespace neko {

// keys: [0, P) row-table bins, [P, 2P) n_row + column-table bins; out-of-range bins get the sentinel n_row + n_col (skipped)
__global__ void __launch_bounds__(256) patch_pos_keys_kernel(const int32_t* __restrict__ row_bin, const int32_t* __restrict__ col_bin, int P,
                                                             int n_row, int n_col, unsigned* __restrict__ keys, int* __restrict__ vals) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  const unsigned sentinel = (unsigned)(n_row + n_col);
  const int rb = row_bin[p], cb = col_bin[p];
  keys[p] = (rb >= 0 && rb < n_row) ? (unsigned)rb : sentinel;
  keys[P + p] = (cb >= 0 && cb < n_col) ? (unsigned)(n_row + cb) : sentinel;
  vals[p] = p;
  vals[P + p] = p;
}

}  // namespace neko

extern "C" {

int neko_patch_pos_bwd_ordered(const float* dx, int P, int d, const int32_t* row_bin, const int32_t* col_bin, float* d_row_tab,
                               int n_row_bins, float* d_col_tab, int n_col_bins, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(dx && row_bin && col_bin && d_row_tab && d_col_tab && workspace, "patch_pos_bwd_ordered: null pointer");
  NEKO_REQUIRE(P > 0 && d > 0 && d % 4 == 0 && n_row_bins > 0 && n_col_bins > 0, "patch_pos_bwd_ordered: bad sizes");
  NEKO_REQUIRE(al(dx, 16) && al(d_row_tab, 16) && al(d_col_tab, 16) && al(workspace, 256),
               "patch_pos_bwd_ordered: dx and the tables must be 16-byte aligned, the workspace 256-byte aligned");
  const int end_bit = key_bits((unsigned)(n_row_bins + n_col_bins));
  SortWs s;
  int rc = sort_ws_layout(2LL * P, end_bit, workspace, s);
  if (rc != NEKO_OK) return rc;
  NEKO_REQUIRE(workspace_bytes >= (int64_t)s.total, "patch_pos_bwd_ordered: workspace of %lld bytes, need %lld", (long long)workspace_bytes,
               (long long)s.total);
  patch_pos_keys_kernel<<<(P + 255) / 256, 256, 0, as_stream(stream)>>>(row_bin, col_bin, P, n_row_bins, n_col_bins, s.kin, s.vin);
  NEKO_LAUNCH_CHECK("patch_pos_keys_kernel");
  SegDst dst{};
  dst.p[0] = d_row_tab; dst.p[1] = d_col_tab; dst.p[2] = nullptr;
  dst.off[0] = 0; dst.off[1] = n_row_bins; dst.off[2] = n_row_bins + n_col_bins; dst.off[3] = n_row_bins + n_col_bins;
  return sort_and_segsum(s, 2LL * P, end_bit, dx, d, dst, as_stream(stream));
}

}  // extern "C"
