// Causal self-attention with left padding, forward and backward (flash style: the S x S score matrix of
// Attention._attn, trajectory_gpt2.py:163-188, is never materialised).
//
// Reference semantics: w = q k^T / sqrt(dh); w = where(tril, w, -1e4); w += (1 - token_mask) * -1e4;
// softmax; w v.  For a valid query row the -1e4 terms underflow to exactly 0 probability in fp32, so the
// row attends keys in [first_valid[b], query].  Padded query rows (left pad, or the right pad of --pad_seq)
// are never read by the loss (gato_policy.py:177-180) nor by valid rows; they are written as zeros.
//
// Tensor-core path: warp-level mma.sync m16n8k16 bf16 with fp32 accumulation.  Tiles (64 rows x dh) are
// brought in with cp.async into a double-buffered shared-memory ring (the next K/V -- or Q/dO -- tile is in
// flight while the current one is consumed) and fragments come from ldmatrix / ldmatrix.trans, so no
// transposed copies are ever built.  dh = 32 (24 heads x 32 at d=768) makes this op latency/exp-bound rather
// than MMA-bound (SURVEY.md section 7); it is <3% of the step FLOPs.
#include "common.cuh"
#include "dropout.cuh"

namespace neko {

constexpr int ATT_BLK = 64;       // queries per CTA = keys per tile
constexpr int ATT_THREADS = 128;  // 4 warps x 16 rows

__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  const int n = valid ? 16 : 0;  // src-size 0 => zero fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Shared-memory tile: 64 rows x DH bf16, row pitch DH + 8 elements (16-byte chunks of 8 consecutive rows fall
// into distinct banks: conflict-free ldmatrix and cp.async).
template <int DH>
struct Tile {
  static constexpr int PITCH = DH + 8;
  static constexpr int BYTES = ATT_BLK * PITCH * 2;
  uint32_t base;  // shared-space address
  __device__ __forceinline__ uint32_t addr(int r, int c) const { return base + (uint32_t)(r * PITCH + c) * 2u; }
};

// rows [r0, r0+64) x DH of one head, 16 bytes per cp.async; rows >= r_end are zero-filled
template <int DH>
__device__ __forceinline__ void load_tile_async(const Tile<DH>& dst, const bf16* __restrict__ src, long long row_pitch, int r0, int r_end) {
  constexpr int VPR = DH / 8;
  for (int i = threadIdx.x; i < ATT_BLK * VPR; i += ATT_THREADS) {
    const int r = i / VPR, v = i % VPR;
    const bool ok = (r0 + r) < r_end;
    const bf16* p = src + (long long)(ok ? (r0 + r) : 0) * row_pitch + v * 8;
    cp_async16(dst.addr(r, v * 8), p, ok);
  }
}

// A fragment: rows row0..row0+15, k columns k0..k0+15 of a [row][k] tile
template <int DH>
__device__ __forceinline__ void frag_a(const Tile<DH>& t, int row0, int k0, int lane, uint32_t (&a)[4]) {
  ldsm_x4(t.addr(row0 + (lane & 15), k0 + ((lane >> 4) << 3)), a[0], a[1], a[2], a[3]);
}
// B fragments of two adjacent n-tiles (n0..n0+15) for k0..k0+15 from a tile stored [n][k]
template <int DH>
__device__ __forceinline__ void frag_b_nk(const Tile<DH>& t, int n0, int k0, int lane, uint32_t (&b)[4]) {
  ldsm_x4(t.addr(n0 + (lane & 7) + ((lane >> 4) << 3), k0 + (((lane >> 3) & 1) << 3)), b[0], b[1], b[2], b[3]);
}
// B fragments of two adjacent n-tiles (n0..n0+15) for k0..k0+15 from a tile stored [k][n]
template <int DH>
__device__ __forceinline__ void frag_b_kn(const Tile<DH>& t, int k0, int n0, int lane, uint32_t (&b)[4]) {
  ldsm_x4_t(t.addr(k0 + (lane & 7) + (((lane >> 3) & 1) << 3), n0 + ((lane >> 4) << 3)), b[0], b[1], b[2], b[3]);
}

// Where one (sample, head) lives.  Padded layout: sample b is rows [b*S, (b+1)*S) of qkv / out / dout, keys and queries
// from first_valid[b] up to S_valid, statistics (lse, delta) at [b, h, :] of [B, H, S].  VARLEN (packed layout, no
// padding rows): sample b is rows [cu[b], cu[b+1]) with keys and queries from 0, statistics at [h, cu[b]:] of [H, T].
// The dropout coordinates stay those of the padded layout: row (b*H + h)*S + first_valid[b] + query, column
// first_valid[b] + key, with S the padded width -- the masks are the padded kernels' bit for bit.
struct AttnSeq {
  long long row0;   // first row of the sample
  long long stat0;  // first lse / delta element of this (sample, head)
  int lo;           // first valid key / query
  int valid;        // queries and keys in [lo, valid) are live
  int end;          // rows [0, end) exist: tile loads zero-fill past it, write-out stops there
  int doff;         // dropout row / column offset
};
template <bool VARLEN>
__device__ __forceinline__ AttnSeq attn_seq(int b, int h, int H, int S, int S_valid, int T, const int32_t* __restrict__ first_valid,
                                            const int32_t* __restrict__ cu_seqlens) {
  AttnSeq r;
  if (VARLEN) {
    const int c0 = cu_seqlens[b];
    r.row0 = c0; r.stat0 = (long long)h * T + c0; r.lo = 0; r.valid = r.end = cu_seqlens[b + 1] - c0; r.doff = first_valid[b];
  } else {
    r.row0 = (long long)b * S; r.stat0 = ((long long)b * H + h) * S; r.lo = first_valid[b]; r.valid = S_valid; r.end = S; r.doff = 0;
  }
  return r;
}
// multipliers of keys (col, col + 1) for any column parity (VARLEN: the column offset first_valid[b] may be odd)
__device__ __forceinline__ void drop_cols(uint32_t rowkey, int col, uint32_t thr16, float scale, float& m0, float& m1) {
  const uint32_t b0 = drop_bits(rowkey, (uint32_t)col >> 1);
  if ((col & 1) == 0) {
    m0 = (b0 & 0xffffu) >= thr16 ? scale : 0.f;
    m1 = (b0 >> 16) >= thr16 ? scale : 0.f;
  } else {
    m0 = (b0 >> 16) >= thr16 ? scale : 0.f;
    m1 = (drop_bits(rowkey, ((uint32_t)col >> 1) + 1u) & 0xffffu) >= thr16 ? scale : 0.f;
  }
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// DROP: attn_dropout (trajectory_gpt2.py:179) on the softmax weights: the row sum (normaliser) uses the undropped
// probabilities, the P V product the masked and rescaled ones; mask element = (row (b*H + h)*S + query, column key).
template <int DH, bool DROP, bool VARLEN>
__global__ void __launch_bounds__(ATT_THREADS) attn_fwd_kernel(const bf16* __restrict__ qkv, const int32_t* __restrict__ first_valid,
                                                               bf16* __restrict__ out, bf16* __restrict__ out2, float* __restrict__ lse, int S,
                                                               int S_valid, int H, float scale_log2, int out_f16, DropCfg drop,
                                                               const int32_t* __restrict__ cu_seqlens, int T) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  pdl_launch_dependents();
  pdl_wait();
  const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
  const Tile<DH> sQ{s0};
  auto sK = [&](int bi) { return Tile<DH>{s0 + (1 + bi) * Tile<DH>::BYTES}; };  // double-buffered K / V tiles
  auto sV = [&](int bi) { return Tile<DH>{s0 + (3 + bi) * Tile<DH>::BYTES}; };

  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * ATT_BLK;
  AttnSeq sq{};
  if (VARLEN) {
    sq = attn_seq<VARLEN>(b, h, H, S, S_valid, T, first_valid, cu_seqlens);
    if (q0 >= sq.end) return;
  }
  // the padded instantiations take every bound from the kernel arguments, as they always have (same code, same registers)
  const int r_end = VARLEN ? sq.end : S, s_valid = VARLEN ? sq.valid : S_valid, doff = VARLEN ? sq.doff : 0;
  const int d = H * DH;
  const long long pitch = 3LL * d;
  const bf16* base = qkv + (VARLEN ? sq.row0 : (long long)b * S) * pitch;
  const int lo = VARLEN ? sq.lo : first_valid[b];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int row_a = q0 + warp * 16 + g, row_b = row_a + 8;
  const int q_hi = min(q0 + ATT_BLK, s_valid);  // queries in [max(q0,lo), q_hi) are live

  float o[DH / 8][4];
#pragma unroll
  for (int n = 0; n < DH / 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;
  float m_a = -INFINITY, m_b = -INFINITY, l_a = 0.f, l_b = 0.f;
  uint32_t rk_a = 0u, rk_b = 0u;
  if (DROP) {
    const uint32_t dkey = drop_key(drop);
    rk_a = drop_rowkey(dkey, (uint32_t)((b * H + h) * S + doff + row_a));
    rk_b = drop_rowkey(dkey, (uint32_t)((b * H + h) * S + doff + row_b));
  }

  if (q_hi > lo && q_hi > q0) {
    const int j_begin = (lo / ATT_BLK) * ATT_BLK;
    load_tile_async<DH>(sQ, base + h * DH, pitch, q0, r_end);
    load_tile_async<DH>(sK(0), base + d + h * DH, pitch, j_begin, r_end);
    load_tile_async<DH>(sV(0), base + 2 * d + h * DH, pitch, j_begin, r_end);
    cp_async_commit();
    uint32_t qa[DH / 16][4];
    int buf = 0;
    for (int j0 = j_begin; j0 < q_hi; j0 += ATT_BLK, buf ^= 1) {
      const bool more = (j0 + ATT_BLK) < q_hi;
      if (more) {  // prefetch the next K/V tile into the other buffer
        load_tile_async<DH>(sK(buf ^ 1), base + d + h * DH, pitch, j0 + ATT_BLK, r_end);
        load_tile_async<DH>(sV(buf ^ 1), base + 2 * d + h * DH, pitch, j0 + ATT_BLK, r_end);
        cp_async_commit();
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
      if (j0 == j_begin) {
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) frag_a<DH>(sQ, warp * 16, k * 16, lane, qa[k]);
      }
      float s[ATT_BLK / 8][4];
#pragma unroll
      for (int n2 = 0; n2 < ATT_BLK / 16; ++n2) {
        s[2 * n2][0] = s[2 * n2][1] = s[2 * n2][2] = s[2 * n2][3] = 0.f;
        s[2 * n2 + 1][0] = s[2 * n2 + 1][1] = s[2 * n2 + 1][2] = s[2 * n2 + 1][3] = 0.f;
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) {
          uint32_t kb[4];
          frag_b_nk<DH>(sK(buf), n2 * 16, k * 16, lane, kb);
          mma_bf16(s[2 * n2], qa[k], kb[0], kb[1]);
          mma_bf16(s[2 * n2 + 1], qa[k], kb[2], kb[3]);
        }
      }
      // mask + online softmax (rows row_a, row_b; this thread holds keys j0 + n*8 + 2q, +1)
      float mx_a = -INFINITY, mx_b = -INFINITY;
      // rows beyond S_valid (right padding) are not masked here: they run on finite garbage and are zeroed at write-out
      const bool need_mask = (j0 < lo) || (j0 + ATT_BLK > q0);
      if (need_mask) {
#pragma unroll
        for (int n = 0; n < ATT_BLK / 8; ++n) {
          const int key = j0 + n * 8 + 2 * q;
          if (key < lo || key > row_a || row_a >= s_valid) s[n][0] = -INFINITY;
          if (key + 1 < lo || key + 1 > row_a || row_a >= s_valid) s[n][1] = -INFINITY;
          if (key < lo || key > row_b || row_b >= s_valid) s[n][2] = -INFINITY;
          if (key + 1 < lo || key + 1 > row_b || row_b >= s_valid) s[n][3] = -INFINITY;
        }
      }
#pragma unroll
      for (int n = 0; n < ATT_BLK / 8; ++n) {
        mx_a = fmaxf(mx_a, fmaxf(s[n][0], s[n][1]));
        mx_b = fmaxf(mx_b, fmaxf(s[n][2], s[n][3]));
      }
      mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 1));
      mx_a = fmaxf(mx_a, __shfl_xor_sync(0xffffffffu, mx_a, 2));
      mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 1));
      mx_b = fmaxf(mx_b, __shfl_xor_sync(0xffffffffu, mx_b, 2));
      const float mn_a = fmaxf(m_a, mx_a), mn_b = fmaxf(m_b, mx_b);
      const float ref_a = (mn_a == -INFINITY) ? 0.f : mn_a * scale_log2;
      const float ref_b = (mn_b == -INFINITY) ? 0.f : mn_b * scale_log2;
      const float corr_a = ex2_ftz(m_a * scale_log2 - ref_a), corr_b = ex2_ftz(m_b * scale_log2 - ref_b);
      m_a = mn_a; m_b = mn_b;
      float sum_a = 0.f, sum_b = 0.f;
#pragma unroll
      for (int n = 0; n < ATT_BLK / 8; ++n) {
        s[n][0] = ex2_ftz(fmaf(s[n][0], scale_log2, -ref_a));
        s[n][1] = ex2_ftz(fmaf(s[n][1], scale_log2, -ref_a));
        s[n][2] = ex2_ftz(fmaf(s[n][2], scale_log2, -ref_b));
        s[n][3] = ex2_ftz(fmaf(s[n][3], scale_log2, -ref_b));
        sum_a += s[n][0] + s[n][1];
        sum_b += s[n][2] + s[n][3];
      }
      l_a = l_a * corr_a + sum_a;
      l_b = l_b * corr_b + sum_b;
      if (DROP) {
#pragma unroll
        for (int n = 0; n < ATT_BLK / 8; ++n) {
          float m0, m1;
          if (VARLEN) {
            const int col = doff + j0 + n * 8 + 2 * q;
            drop_cols(rk_a, col, drop.thr16, drop.scale, m0, m1);
            s[n][0] *= m0; s[n][1] *= m1;
            drop_cols(rk_b, col, drop.thr16, drop.scale, m0, m1);
            s[n][2] *= m0; s[n][3] *= m1;
          } else {
            const uint32_t pr = (uint32_t)((j0 + n * 8) >> 1) + q;
            drop_pair(rk_a, pr, drop.thr16, drop.scale, m0, m1);
            s[n][0] *= m0; s[n][1] *= m1;
            drop_pair(rk_b, pr, drop.thr16, drop.scale, m0, m1);
            s[n][2] *= m0; s[n][3] *= m1;
          }
        }
      }
#pragma unroll
      for (int n = 0; n < DH / 8; ++n) {
        o[n][0] *= corr_a; o[n][1] *= corr_a; o[n][2] *= corr_b; o[n][3] *= corr_b;
      }
      // O += P V  (P from the score accumulators; V tile is [key][dh] -> transposed ldmatrix)
#pragma unroll
      for (int kk = 0; kk < ATT_BLK / 16; ++kk) {
        uint32_t pa[4];
        pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
        pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
        pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int n2 = 0; n2 < DH / 16; ++n2) {
          uint32_t vb[4];
          frag_b_kn<DH>(sV(buf), kk * 16, n2 * 16, lane, vb);
          mma_bf16(o[2 * n2], pa, vb[0], vb[1]);
          mma_bf16(o[2 * n2 + 1], pa, vb[2], vb[3]);
        }
      }
      __syncthreads();  // everyone is done with this buffer before the prefetch two iterations ahead reuses it
    }
    l_a += __shfl_xor_sync(0xffffffffu, l_a, 1);
    l_a += __shfl_xor_sync(0xffffffffu, l_a, 2);
    l_b += __shfl_xor_sync(0xffffffffu, l_b, 1);
    l_b += __shfl_xor_sync(0xffffffffu, l_b, 2);
  }
  // write-out: dead rows (padding) -> zeros, lse = +inf so that backward sees p = 0
  if (row_a < lo || row_a >= s_valid) l_a = 0.f;   // padding rows
  if (row_b < lo || row_b >= s_valid) l_b = 0.f;
  const float inv_a = (l_a > 0.f) ? 1.f / l_a : 0.f, inv_b = (l_b > 0.f) ? 1.f / l_b : 0.f;
  const float kLn2 = 0.6931471805599453f;
  bf16* ob = out + (VARLEN ? sq.row0 : (long long)b * S) * d + h * DH;
  bf16* ob2 = out2 ? out2 + (VARLEN ? sq.row0 : (long long)b * S) * d + h * DH : nullptr;
  if (row_a < r_end) {
#pragma unroll
    for (int n = 0; n < DH / 8; ++n) {
      *reinterpret_cast<uint32_t*>(ob + (long long)row_a * d + n * 8 + 2 * q) = pack_16x2(o[n][0] * inv_a, o[n][1] * inv_a, out_f16 != 0);
      if (ob2) *reinterpret_cast<uint32_t*>(ob2 + (long long)row_a * d + n * 8 + 2 * q) = pack_bf16x2(o[n][0] * inv_a, o[n][1] * inv_a);
    }
    if (q == 0) lse[(VARLEN ? sq.stat0 : ((long long)b * H + h) * S) + row_a] = (l_a > 0.f) ? (m_a * scale_log2 + log2f(l_a)) * kLn2 : INFINITY;
  }
  if (row_b < r_end) {
#pragma unroll
    for (int n = 0; n < DH / 8; ++n) {
      *reinterpret_cast<uint32_t*>(ob + (long long)row_b * d + n * 8 + 2 * q) = pack_16x2(o[n][2] * inv_b, o[n][3] * inv_b, out_f16 != 0);
      if (ob2) *reinterpret_cast<uint32_t*>(ob2 + (long long)row_b * d + n * 8 + 2 * q) = pack_bf16x2(o[n][2] * inv_b, o[n][3] * inv_b);
    }
    if (q == 0) lse[(VARLEN ? sq.stat0 : ((long long)b * H + h) * S) + row_b] = (l_b > 0.f) ? (m_b * scale_log2 + log2f(l_b)) * kLn2 : INFINITY;
  }
}

// ---------------------------------------------------------------------------------------------
// backward.  dQ kernel first (it also produces delta[b,h,i] = sum_c dO[i,c] O[i,c] from the tiles it holds),
// then the dK/dV kernel.  No atomics: each kernel owns its output rows and recomputes P.
// ---------------------------------------------------------------------------------------------
// With dropout:  O = (P o M) V  (M = mask * 1/(1-p)),  dP = (dO V^T) o M,  dS = P o (dP - delta),  delta = rowsum(dO o O).
template <int DH, bool DROP, bool VARLEN>
__global__ void __launch_bounds__(ATT_THREADS) attn_bwd_dq_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ out,
                                                                  const bf16* __restrict__ dout, const float* __restrict__ lse,
                                                                  float* __restrict__ delta, const int32_t* __restrict__ first_valid,
                                                                  const int32_t* __restrict__ cu_seqlens, bf16* __restrict__ dqkv, int S,
                                                                  int S_valid, int T, int H, float scale, float scale_log2, int out_f16,
                                                                  DropCfg drop) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  pdl_launch_dependents();
  pdl_wait();
  const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
  const Tile<DH> sQ{s0};
  const Tile<DH> sdO{s0 + Tile<DH>::BYTES};
  const Tile<DH> sO{s0 + 2 * Tile<DH>::BYTES};
  auto sK = [&](int bi) { return Tile<DH>{s0 + (3 + bi) * Tile<DH>::BYTES}; };
  auto sV = [&](int bi) { return Tile<DH>{s0 + (5 + bi) * Tile<DH>::BYTES}; };
  float* s_delta = reinterpret_cast<float*>(smem_raw + 7 * Tile<DH>::BYTES);

  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * ATT_BLK;
  const AttnSeq sq = attn_seq<VARLEN>(b, h, H, S, S_valid, T, first_valid, cu_seqlens);
  if (VARLEN && q0 >= sq.end) return;
  const int d = H * DH;
  const long long pitch = 3LL * d;
  const bf16* base = qkv + sq.row0 * pitch;
  const bf16* dob = dout + sq.row0 * d + h * DH;
  const bf16* ob = out + sq.row0 * d + h * DH;
  const int lo = sq.lo;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int row_a = q0 + warp * 16 + g, row_b = row_a + 8;
  const int q_hi = min(q0 + ATT_BLK, sq.valid);
  const float kLog2e = 1.4426950408889634f;
  float* delta_b = delta + sq.stat0;

  float dq[DH / 8][4];
#pragma unroll
  for (int n = 0; n < DH / 8; ++n) dq[n][0] = dq[n][1] = dq[n][2] = dq[n][3] = 0.f;

  uint32_t rk_a = 0u, rk_b = 0u;
  if (DROP) {
    const uint32_t dkey = drop_key(drop);
    rk_a = drop_rowkey(dkey, (uint32_t)((b * H + h) * S + sq.doff + row_a));
    rk_b = drop_rowkey(dkey, (uint32_t)((b * H + h) * S + sq.doff + row_b));
  }
  const bool live = (q_hi > lo) && (q_hi > q0);
  if (!live) {
    // delta of dead rows is never read with a non-zero P, but keep the buffer defined
    if (threadIdx.x < ATT_BLK && q0 + threadIdx.x < sq.end) delta_b[q0 + threadIdx.x] = 0.f;
  } else {
    const float* lse_b = lse + sq.stat0;
    const int j_begin = (lo / ATT_BLK) * ATT_BLK;
    load_tile_async<DH>(sQ, base + h * DH, pitch, q0, sq.end);
    load_tile_async<DH>(sdO, dob, d, q0, sq.end);
    load_tile_async<DH>(sO, ob, d, q0, sq.end);
    load_tile_async<DH>(sK(0), base + d + h * DH, pitch, j_begin, sq.end);
    load_tile_async<DH>(sV(0), base + 2 * d + h * DH, pitch, j_begin, sq.end);
    cp_async_commit();
    const float lse_a = (row_a < sq.end) ? lse_b[row_a] * kLog2e : INFINITY, lse_bb = (row_b < sq.end) ? lse_b[row_b] * kLog2e : INFINITY;
    uint32_t qa[DH / 16][4], doa[DH / 16][4];
    float del_a = 0.f, del_b = 0.f;
    int buf = 0;
    for (int j0 = j_begin; j0 < q_hi; j0 += ATT_BLK, buf ^= 1) {
      const bool more = (j0 + ATT_BLK) < q_hi;
      if (more) {
        load_tile_async<DH>(sK(buf ^ 1), base + d + h * DH, pitch, j0 + ATT_BLK, sq.end);
        load_tile_async<DH>(sV(buf ^ 1), base + 2 * d + h * DH, pitch, j0 + ATT_BLK, sq.end);
        cp_async_commit();
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
      if (j0 == j_begin) {
        // delta = rowsum(dO * O): two threads per row, then published through shared memory
        {
          const int r = threadIdx.x >> 1, half = threadIdx.x & 1;
          const bf16* po = reinterpret_cast<const bf16*>(smem_raw + 2 * Tile<DH>::BYTES) + r * Tile<DH>::PITCH + half * (DH / 2);
          const bf16* pg = reinterpret_cast<const bf16*>(smem_raw + 1 * Tile<DH>::BYTES) + r * Tile<DH>::PITCH + half * (DH / 2);
          float acc = 0.f;
#pragma unroll
          for (int c = 0; c < DH / 2; c += 2) {
            const uint32_t ou = *reinterpret_cast<const uint32_t*>(po + c);
            const float2 a = out_f16 ? unpack_f16x2(ou) : unpack_bf16x2(ou);
            const float2 bb = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(pg + c));
            acc += a.x * bb.x + a.y * bb.y;
          }
          acc += __shfl_xor_sync(0xffffffffu, acc, 1);
          if (half == 0) {
            s_delta[r] = acc;
            if (q0 + r < sq.end) delta_b[q0 + r] = acc;
          }
        }
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) {
          frag_a<DH>(sQ, warp * 16, k * 16, lane, qa[k]);
          frag_a<DH>(sdO, warp * 16, k * 16, lane, doa[k]);
        }
        __syncthreads();
        del_a = s_delta[warp * 16 + g];
        del_b = s_delta[warp * 16 + g + 8];
      }
      float s[ATT_BLK / 8][4], dp[ATT_BLK / 8][4];
#pragma unroll
      for (int n2 = 0; n2 < ATT_BLK / 16; ++n2) {
#pragma unroll
        for (int e = 0; e < 4; ++e) { s[2 * n2][e] = s[2 * n2 + 1][e] = 0.f; dp[2 * n2][e] = dp[2 * n2 + 1][e] = 0.f; }
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) {
          uint32_t kb[4], vb[4];
          frag_b_nk<DH>(sK(buf), n2 * 16, k * 16, lane, kb);
          frag_b_nk<DH>(sV(buf), n2 * 16, k * 16, lane, vb);
          mma_bf16(s[2 * n2], qa[k], kb[0], kb[1]);
          mma_bf16(s[2 * n2 + 1], qa[k], kb[2], kb[3]);
          mma_bf16(dp[2 * n2], doa[k], vb[0], vb[1]);
          mma_bf16(dp[2 * n2 + 1], doa[k], vb[2], vb[3]);
        }
      }
      // interior tiles (all keys valid and strictly below every query of the tile) need no per-element predicate
      // (rows beyond S_valid carry lse = +inf from the forward: their p is 0 without a predicate)
      const bool need_mask = (j0 < lo) || (j0 + ATT_BLK > q0);
#pragma unroll
      for (int n = 0; n < ATT_BLK / 8; ++n) {
        float p0 = ex2_ftz(fmaf(s[n][0], scale_log2, -lse_a)), p1 = ex2_ftz(fmaf(s[n][1], scale_log2, -lse_a));
        float p2 = ex2_ftz(fmaf(s[n][2], scale_log2, -lse_bb)), p3 = ex2_ftz(fmaf(s[n][3], scale_log2, -lse_bb));
        if (need_mask) {
          const int key = j0 + n * 8 + 2 * q;
          const bool va = row_a < sq.valid, vb = row_b < sq.valid;
          if (!(va && key >= lo && key <= row_a)) p0 = 0.f;
          if (!(va && key + 1 >= lo && key + 1 <= row_a)) p1 = 0.f;
          if (!(vb && key >= lo && key <= row_b)) p2 = 0.f;
          if (!(vb && key + 1 >= lo && key + 1 <= row_b)) p3 = 0.f;
        }
        if (DROP) {
          float m0, m1;
          if (VARLEN) {
            const int col = sq.doff + j0 + n * 8 + 2 * q;
            drop_cols(rk_a, col, drop.thr16, drop.scale, m0, m1);
            dp[n][0] *= m0; dp[n][1] *= m1;
            drop_cols(rk_b, col, drop.thr16, drop.scale, m0, m1);
            dp[n][2] *= m0; dp[n][3] *= m1;
          } else {
            const uint32_t pr = (uint32_t)((j0 + n * 8) >> 1) + q;
            drop_pair(rk_a, pr, drop.thr16, drop.scale, m0, m1);
            dp[n][0] *= m0; dp[n][1] *= m1;
            drop_pair(rk_b, pr, drop.thr16, drop.scale, m0, m1);
            dp[n][2] *= m0; dp[n][3] *= m1;
          }
        }
        s[n][0] = p0 * (dp[n][0] - del_a) * scale;
        s[n][1] = p1 * (dp[n][1] - del_a) * scale;
        s[n][2] = p2 * (dp[n][2] - del_b) * scale;
        s[n][3] = p3 * (dp[n][3] - del_b) * scale;
      }
      // dQ += dS K   (K tile is [key][dh]: k index = key -> transposed ldmatrix)
#pragma unroll
      for (int kk = 0; kk < ATT_BLK / 16; ++kk) {
        uint32_t sa[4];
        sa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
        sa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
        sa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        sa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int n2 = 0; n2 < DH / 16; ++n2) {
          uint32_t kb[4];
          frag_b_kn<DH>(sK(buf), kk * 16, n2 * 16, lane, kb);
          mma_bf16(dq[2 * n2], sa, kb[0], kb[1]);
          mma_bf16(dq[2 * n2 + 1], sa, kb[2], kb[3]);
        }
      }
      __syncthreads();
    }
  }
  bf16* dqb = dqkv + sq.row0 * pitch + h * DH;
  if (row_a < sq.end) {
#pragma unroll
    for (int n = 0; n < DH / 8; ++n)
      *reinterpret_cast<uint32_t*>(dqb + (long long)row_a * pitch + n * 8 + 2 * q) = pack_bf16x2(dq[n][0], dq[n][1]);
  }
  if (row_b < sq.end) {
#pragma unroll
    for (int n = 0; n < DH / 8; ++n)
      *reinterpret_cast<uint32_t*>(dqb + (long long)row_b * pitch + n * 8 + 2 * q) = pack_bf16x2(dq[n][2], dq[n][3]);
  }
}

// dK, dV: one CTA owns 64 keys (4 warps x 16) of one head and sweeps the query tiles at or below it.
template <int DH, bool DROP, bool VARLEN>
__global__ void __launch_bounds__(ATT_THREADS) attn_bwd_dkv_kernel(const bf16* __restrict__ qkv, const bf16* __restrict__ dout,
                                                                   const float* __restrict__ lse, const float* __restrict__ delta,
                                                                   const int32_t* __restrict__ first_valid,
                                                                   const int32_t* __restrict__ cu_seqlens, bf16* __restrict__ dqkv, int S,
                                                                   int S_valid, int T, int H, float scale, float scale_log2, DropCfg drop) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  pdl_launch_dependents();
  pdl_wait();
  const uint32_t s0 = (uint32_t)__cvta_generic_to_shared(smem_raw);
  const Tile<DH> sK{s0};
  const Tile<DH> sV{s0 + Tile<DH>::BYTES};
  auto sQ = [&](int bi) { return Tile<DH>{s0 + (2 + bi) * Tile<DH>::BYTES}; };
  auto sdO = [&](int bi) { return Tile<DH>{s0 + (4 + bi) * Tile<DH>::BYTES}; };
  float* s_lse = reinterpret_cast<float*>(smem_raw + 6 * Tile<DH>::BYTES);  // [2][64]
  float* s_delta = s_lse + 2 * ATT_BLK;                                      // [2][64]
  uint32_t* s_rk = reinterpret_cast<uint32_t*>(s_delta + 2 * ATT_BLK);       // [2][64] dropout row keys of the query tile

  const int b = blockIdx.z, h = blockIdx.y, j0 = blockIdx.x * ATT_BLK;
  const AttnSeq sq = attn_seq<VARLEN>(b, h, H, S, S_valid, T, first_valid, cu_seqlens);
  if (VARLEN && j0 >= sq.end) return;
  const int d = H * DH;
  const long long pitch = 3LL * d;
  const bf16* base = qkv + sq.row0 * pitch;
  const bf16* dob = dout + sq.row0 * d + h * DH;
  const float* lse_b = lse + sq.stat0;
  const float* delta_b = delta + sq.stat0;
  const int lo = sq.lo;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int key_a = j0 + warp * 16 + g, key_b = key_a + 8;
  const float kLog2e = 1.4426950408889634f;

  float dk[DH / 8][4], dv[DH / 8][4];
#pragma unroll
  for (int n = 0; n < DH / 8; ++n) {
    dk[n][0] = dk[n][1] = dk[n][2] = dk[n][3] = 0.f;
    dv[n][0] = dv[n][1] = dv[n][2] = dv[n][3] = 0.f;
  }
  const bool live = (j0 + ATT_BLK > lo) && (j0 < sq.valid);
  const uint32_t dkey = DROP ? drop_key(drop) : 0u;
  if (live) {
    auto load_q_tile = [&](int bufi, int i0) {
      load_tile_async<DH>(sQ(bufi), base + h * DH, pitch, i0, sq.end);
      load_tile_async<DH>(sdO(bufi), dob, d, i0, sq.end);
      if (threadIdx.x < ATT_BLK) {
        const int i = i0 + threadIdx.x;
        s_lse[bufi * ATT_BLK + threadIdx.x] = (i < sq.end) ? lse_b[i] * kLog2e : INFINITY;
        s_delta[bufi * ATT_BLK + threadIdx.x] = (i < sq.end) ? delta_b[i] : 0.f;
        if (DROP) s_rk[bufi * ATT_BLK + threadIdx.x] = drop_rowkey(dkey, (uint32_t)((b * H + h) * S + sq.doff + i));
      }
    };
    load_tile_async<DH>(sK, base + d + h * DH, pitch, j0, sq.end);
    load_tile_async<DH>(sV, base + 2 * d + h * DH, pitch, j0, sq.end);
    load_q_tile(0, j0);
    cp_async_commit();
    uint32_t ka[DH / 16][4], va[DH / 16][4];
    int buf = 0;
    for (int i0 = j0; i0 < sq.valid; i0 += ATT_BLK, buf ^= 1) {
      const bool more = (i0 + ATT_BLK) < sq.valid;
      if (more) {
        load_q_tile(buf ^ 1, i0 + ATT_BLK);
        cp_async_commit();
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
      if (i0 == j0) {
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) {
          frag_a<DH>(sK, warp * 16, k * 16, lane, ka[k]);
          frag_a<DH>(sV, warp * 16, k * 16, lane, va[k]);
        }
      }
      // S^T = K Q^T and dP^T = V dO^T   (rows = this warp's 16 keys, cols = 64 queries)
      float st[ATT_BLK / 8][4], dpt[ATT_BLK / 8][4];
#pragma unroll
      for (int n2 = 0; n2 < ATT_BLK / 16; ++n2) {
#pragma unroll
        for (int e = 0; e < 4; ++e) { st[2 * n2][e] = st[2 * n2 + 1][e] = 0.f; dpt[2 * n2][e] = dpt[2 * n2 + 1][e] = 0.f; }
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) {
          uint32_t qb[4], gb[4];
          frag_b_nk<DH>(sQ(buf), n2 * 16, k * 16, lane, qb);
          frag_b_nk<DH>(sdO(buf), n2 * 16, k * 16, lane, gb);
          mma_bf16(st[2 * n2], ka[k], qb[0], qb[1]);
          mma_bf16(st[2 * n2 + 1], ka[k], qb[2], qb[3]);
          mma_bf16(dpt[2 * n2], va[k], gb[0], gb[1]);
          mma_bf16(dpt[2 * n2 + 1], va[k], gb[2], gb[3]);
        }
      }
      // P^T = exp(S^T * scale - lse[query]); dS^T = P^T * (dP^T - delta[query]) * scale
      const bool need_mask = (j0 < lo) || (i0 < j0 + ATT_BLK);   // queries beyond S_valid have lse = +inf -> p = 0
      const float* lsp = s_lse + buf * ATT_BLK;
      const float* dlp = s_delta + buf * ATT_BLK;
#pragma unroll
      for (int n = 0; n < ATT_BLK / 8; ++n) {
        const int c0 = n * 8 + 2 * q;  // local query column
        const int qi0 = i0 + c0, qi1 = qi0 + 1;
        const float l0 = lsp[c0], l1 = lsp[c0 + 1];
        float p00 = ex2_ftz(fmaf(st[n][0], scale_log2, -l0)), p01 = ex2_ftz(fmaf(st[n][1], scale_log2, -l1));
        float p10 = ex2_ftz(fmaf(st[n][2], scale_log2, -l0)), p11 = ex2_ftz(fmaf(st[n][3], scale_log2, -l1));
        if (need_mask) {   // diagonal tile, left padding inside the key tile, or right padding inside the query tile
          if (!((key_a >= lo) && (key_a <= qi0) && (qi0 < sq.valid))) p00 = 0.f;
          if (!((key_a >= lo) && (key_a <= qi1) && (qi1 < sq.valid))) p01 = 0.f;
          if (!((key_b >= lo) && (key_b <= qi0) && (qi0 < sq.valid))) p10 = 0.f;
          if (!((key_b >= lo) && (key_b <= qi1) && (qi1 < sq.valid))) p11 = 0.f;
        }
        const float d0 = dlp[c0], d1 = dlp[c0 + 1];
        float m00 = 1.f, m01 = 1.f, m10 = 1.f, m11 = 1.f;
        if (DROP) {  // element (query, key): bits of column pair (col >> 1), half-word col & 1
          const uint32_t r0 = s_rk[buf * ATT_BLK + c0], r1 = s_rk[buf * ATT_BLK + c0 + 1];
          const int col_a = sq.doff + key_a, col_b = col_a + 8;
          const uint32_t sh = (uint32_t)(col_a & 1) << 4;   // col_b = col_a + 8 has the same parity
          const uint32_t pa_ = (uint32_t)col_a >> 1, pb_ = (uint32_t)col_b >> 1;
          m00 = ((drop_bits(r0, pa_) >> sh) & 0xffffu) >= drop.thr16 ? drop.scale : 0.f;
          m01 = ((drop_bits(r1, pa_) >> sh) & 0xffffu) >= drop.thr16 ? drop.scale : 0.f;
          m10 = ((drop_bits(r0, pb_) >> sh) & 0xffffu) >= drop.thr16 ? drop.scale : 0.f;
          m11 = ((drop_bits(r1, pb_) >> sh) & 0xffffu) >= drop.thr16 ? drop.scale : 0.f;
        }
        dpt[n][0] = p00 * (dpt[n][0] * m00 - d0) * scale;
        dpt[n][1] = p01 * (dpt[n][1] * m01 - d1) * scale;
        dpt[n][2] = p10 * (dpt[n][2] * m10 - d0) * scale;
        dpt[n][3] = p11 * (dpt[n][3] * m11 - d1) * scale;
        st[n][0] = p00 * m00; st[n][1] = p01 * m01; st[n][2] = p10 * m10; st[n][3] = p11 * m11;
      }
      // dV += P^T dO ; dK += dS^T Q   (k index = query: tiles are [query][dh] -> transposed ldmatrix)
#pragma unroll
      for (int kk = 0; kk < ATT_BLK / 16; ++kk) {
        uint32_t pa[4], sa[4];
        pa[0] = pack_bf16x2(st[2 * kk][0], st[2 * kk][1]);
        pa[1] = pack_bf16x2(st[2 * kk][2], st[2 * kk][3]);
        pa[2] = pack_bf16x2(st[2 * kk + 1][0], st[2 * kk + 1][1]);
        pa[3] = pack_bf16x2(st[2 * kk + 1][2], st[2 * kk + 1][3]);
        sa[0] = pack_bf16x2(dpt[2 * kk][0], dpt[2 * kk][1]);
        sa[1] = pack_bf16x2(dpt[2 * kk][2], dpt[2 * kk][3]);
        sa[2] = pack_bf16x2(dpt[2 * kk + 1][0], dpt[2 * kk + 1][1]);
        sa[3] = pack_bf16x2(dpt[2 * kk + 1][2], dpt[2 * kk + 1][3]);
#pragma unroll
        for (int n2 = 0; n2 < DH / 16; ++n2) {
          uint32_t gb[4], qb[4];
          frag_b_kn<DH>(sdO(buf), kk * 16, n2 * 16, lane, gb);
          frag_b_kn<DH>(sQ(buf), kk * 16, n2 * 16, lane, qb);
          mma_bf16(dv[2 * n2], pa, gb[0], gb[1]);
          mma_bf16(dv[2 * n2 + 1], pa, gb[2], gb[3]);
          mma_bf16(dk[2 * n2], sa, qb[0], qb[1]);
          mma_bf16(dk[2 * n2 + 1], sa, qb[2], qb[3]);
        }
      }
      __syncthreads();
    }
  }
  bf16* dkb = dqkv + sq.row0 * pitch + d + h * DH;
  bf16* dvb = dqkv + sq.row0 * pitch + 2 * d + h * DH;
  if (key_a < sq.end) {
#pragma unroll
    for (int n = 0; n < DH / 8; ++n) {
      *reinterpret_cast<uint32_t*>(dkb + (long long)key_a * pitch + n * 8 + 2 * q) = pack_bf16x2(dk[n][0], dk[n][1]);
      *reinterpret_cast<uint32_t*>(dvb + (long long)key_a * pitch + n * 8 + 2 * q) = pack_bf16x2(dv[n][0], dv[n][1]);
    }
  }
  if (key_b < sq.end) {
#pragma unroll
    for (int n = 0; n < DH / 8; ++n) {
      *reinterpret_cast<uint32_t*>(dkb + (long long)key_b * pitch + n * 8 + 2 * q) = pack_bf16x2(dk[n][2], dk[n][3]);
      *reinterpret_cast<uint32_t*>(dvb + (long long)key_b * pitch + n * 8 + 2 * q) = pack_bf16x2(dv[n][2], dv[n][3]);
    }
  }
}

template <int DH>
static size_t fwd_smem() { return 5 * (size_t)Tile<DH>::BYTES; }
template <int DH>
static size_t dq_smem() { return 7 * (size_t)Tile<DH>::BYTES + ATT_BLK * sizeof(float); }
template <int DH>
static size_t dkv_smem() { return 6 * (size_t)Tile<DH>::BYTES + 6 * ATT_BLK * sizeof(float); }

// VARLEN: S = the padded width (dropout coordinates), S_grid = the longest sample, T = packed rows; padded: S_grid = S, T unused
template <int DH, bool DROP, bool VARLEN>
static int launch_fwd(const bf16* qkv, const int32_t* fv, const int32_t* cu, bf16* out, bf16* out2, float* lse, int B, int S, int S_valid,
                      int S_grid, int T, int H, int out_f16, DropCfg drop, cudaStream_t st) {
  const size_t smem = fwd_smem<DH>();
  cudaError_t e = cudaFuncSetAttribute(attn_fwd_kernel<DH, DROP, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(attn_fwd)");
  const float scale_log2 = 1.4426950408889634f / sqrtf((float)DH);
  dim3 grid((S_grid + ATT_BLK - 1) / ATT_BLK, H, B);
  launch_pdl(attn_fwd_kernel<DH, DROP, VARLEN>, grid, dim3(ATT_THREADS), smem, st, qkv, fv, out, out2, lse, S, S_valid, H, scale_log2, out_f16,
             drop, cu, T);
  NEKO_LAUNCH_CHECK("attn_fwd_kernel");
  return NEKO_OK;
}

template <int DH, bool DROP, bool VARLEN>
static int launch_bwd(const bf16* qkv, const bf16* out, const bf16* dout, const float* lse, float* delta, const int32_t* fv, const int32_t* cu,
                      bf16* dqkv, int B, int S, int S_valid, int S_grid, int T, int H, int out_f16, DropCfg drop, cudaStream_t st) {
  const size_t s1 = dq_smem<DH>(), s2 = dkv_smem<DH>();
  cudaError_t e = cudaFuncSetAttribute(attn_bwd_dq_kernel<DH, DROP, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(attn_bwd_dq)");
  e = cudaFuncSetAttribute(attn_bwd_dkv_kernel<DH, DROP, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(attn_bwd_dkv)");
  const float scale = 1.0f / sqrtf((float)DH);
  const float scale_log2 = 1.4426950408889634f * scale;
  dim3 grid((S_grid + ATT_BLK - 1) / ATT_BLK, H, B);
  launch_pdl(attn_bwd_dq_kernel<DH, DROP, VARLEN>, grid, dim3(ATT_THREADS), s1, st, qkv, out, dout, lse, delta, fv, cu, dqkv, S, S_valid, T, H,
             scale, scale_log2, out_f16, drop);
  NEKO_LAUNCH_CHECK("attn_bwd_dq_kernel");
  launch_pdl(attn_bwd_dkv_kernel<DH, DROP, VARLEN>, grid, dim3(ATT_THREADS), s2, st, qkv, dout, lse, delta, fv, cu, dqkv, S, S_valid, T, H,
             scale, scale_log2, drop);
  NEKO_LAUNCH_CHECK("attn_bwd_dkv_kernel");
  return NEKO_OK;
}

// ---------------------------------------------------------------------------------------------
// Single-query attention against a key/value cache (KV-cached decode of the predict_* loops, gato_policy.py:452-476):
// one CTA per head; scores of all cached keys in shared memory, fp32 softmax, weighted sum of V.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) attn_decode_kernel(const bf16* __restrict__ q, const bf16* __restrict__ kc, const bf16* __restrict__ vc,
                                                          int len, int d, int dh, float scale, uint16_t* __restrict__ out, int out_f16) {
  extern __shared__ float dec_s[];          // [len] scores, then [128] reduction scratch
  float* red = dec_s + len;
  const int h = blockIdx.x, tid = threadIdx.x;
  const bf16* qh = q + h * dh;
  // scores
  float lmax = -INFINITY;
  for (int j = tid; j < len; j += 128) {
    const bf16* kr = kc + (size_t)j * d + h * dh;
    float acc = 0.f;
    for (int c = 0; c < dh; c += 2) {
      const float2 a = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(qh + c));
      const float2 b = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(kr + c));
      acc = fmaf(a.x, b.x, fmaf(a.y, b.y, acc));
    }
    acc *= scale;
    dec_s[j] = acc;
    lmax = fmaxf(lmax, acc);
  }
  lmax = warp_max(lmax);
  if ((tid & 31) == 0) red[tid >> 5] = lmax;
  __syncthreads();
  const float mx = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
  __syncthreads();
  float lsum = 0.f;
  for (int j = tid; j < len; j += 128) {
    const float p = __expf(dec_s[j] - mx);
    dec_s[j] = p;
    lsum += p;
  }
  lsum = warp_sum(lsum);
  if ((tid & 31) == 0) red[tid >> 5] = lsum;
  __syncthreads();
  const float inv = 1.0f / (red[0] + red[1] + red[2] + red[3]);
  __syncthreads();
  // out[c] = sum_j p_j v[j][c]: thread = (dimension c, key slice)
  const int slices = 128 / dh > 0 ? 128 / dh : 1;
  const int c = tid % dh, sl = tid / dh;
  float acc = 0.f;
  if (sl < slices)
    for (int j = sl; j < len; j += slices) acc = fmaf(dec_s[j], __bfloat162float(vc[(size_t)j * d + h * dh + c]), acc);
  red[tid] = (sl < slices) ? acc : 0.f;
  __syncthreads();
  if (tid < dh) {
    float t = 0.f;
    for (int s2 = 0; s2 < slices; ++s2) t += red[s2 * dh + tid];
    out[h * dh + tid] = cvt_16(t * inv, out_f16 != 0);
  }
}

// tcgen05 forward (attention_tc.cu): 0 = ran, 1 = shape not covered, < 0 = error
bool attention_fwd_tc_eligible(const void* qkv, const void* out, const void* out2, int H, int dh);
int attention_fwd_tc(const bf16* qkv, const int32_t* fv, bf16* out, bf16* out2, float* lse, int B, int S, int S_valid, int H, int dh, int out_f16,
                     DropCfg drop, cudaStream_t st);

// argument checks of neko_attention_fwd, shared with neko_attention_fwd_path
static int attention_fwd_args(const uint16_t* qkv, const int32_t* first_valid, const uint16_t* out, const float* lse, int B, int S,
                              int S_valid, int H, int dh) {
  NEKO_REQUIRE(qkv && first_valid && out && lse, "attention_fwd: null pointer");
  NEKO_REQUIRE(B > 0 && S > 0 && H > 0 && S_valid > 0 && S_valid <= S, "attention_fwd: bad sizes");
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "attention_fwd: misaligned");
  NEKO_REQUIRE((long long)B * H * S < (1LL << 32), "attention_fwd: B*H*S exceeds the dropout row-id range");
  NEKO_REQUIRE(dh == 16 || dh == 32 || dh == 64 || dh == 128, "attention: head dim %d not supported (16, 32, 64, 128)", dh);
  return NEKO_OK;
}

}  // namespace neko

extern "C" {

int neko_attention_fwd(const uint16_t* qkv, const int32_t* first_valid, uint16_t* out, uint16_t* out2_bf16, float* lse, int B, int S,
                       int S_valid, int H, int dh, int out_f16, const neko_dropout* drop, void* stream) {
  using namespace neko;
  const int rc = attention_fwd_args(qkv, first_valid, out, lse, B, S, S_valid, H, dh);
  if (rc != NEKO_OK) return rc;
  const bf16* x = reinterpret_cast<const bf16*>(qkv);
  bf16* o = reinterpret_cast<bf16*>(out);
  bf16* o2 = reinterpret_cast<bf16*>(out2_bf16);
  cudaStream_t st = as_stream(stream);
  const DropCfg dc = drop_cfg(drop);
  {  // tensor-core (tcgen05 / TMEM / TMA) path for head dims 32 and 64; the mma.sync kernels below are the fallback
    const int rc_tc = attention_fwd_tc(x, first_valid, o, o2, lse, B, S, S_valid, H, dh, out_f16, dc, st);
    if (rc_tc <= 0) return rc_tc;
  }
#define NEKO_ATT_FWD(DH_) (dc.seed ? launch_fwd<DH_, true, false>(x, first_valid, nullptr, o, o2, lse, B, S, S_valid, S, 0, H, out_f16, dc, st) \
                                   : launch_fwd<DH_, false, false>(x, first_valid, nullptr, o, o2, lse, B, S, S_valid, S, 0, H, out_f16, dc, st))
  switch (dh) {
    case 16: return NEKO_ATT_FWD(16);
    case 32: return NEKO_ATT_FWD(32);
    case 64: return NEKO_ATT_FWD(64);
    case 128: return NEKO_ATT_FWD(128);
    default: set_error("attention: head dim %d not supported (16, 32, 64, 128)", dh); return NEKO_EINVAL;
  }
#undef NEKO_ATT_FWD
}

int neko_attention_fwd_path(const uint16_t* qkv, const int32_t* first_valid, const uint16_t* out, const uint16_t* out2_bf16, const float* lse,
                            int B, int S, int S_valid, int H, int dh, int out_f16, const neko_dropout* drop) {
  using namespace neko;
  (void)out_f16;
  (void)drop;
  const int rc = attention_fwd_args(qkv, first_valid, out, lse, B, S, S_valid, H, dh);
  if (rc != NEKO_OK) return rc;
  return attention_fwd_tc_eligible(qkv, out, out2_bf16, H, dh) ? 1 : 0;
}

int neko_attention_decode(const uint16_t* q, const uint16_t* k_cache, const uint16_t* v_cache, int len, int H, int dh, uint16_t* out,
                          int out_f16, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(q && k_cache && v_cache && out, "attention_decode: null pointer");
  NEKO_REQUIRE(len > 0 && len <= 8192 && H > 0 && dh > 0 && dh <= 128 && dh % 2 == 0 && 128 % dh == 0, "attention_decode: bad sizes (len=%d dh=%d)", len, dh);
  // q and the key rows are read as pairs of bf16 (32-bit loads)
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(q) & 3) == 0 && (reinterpret_cast<uintptr_t>(k_cache) & 3) == 0, "attention_decode: misaligned");
  const size_t smem = (size_t)(len + 128) * sizeof(float);
  attn_decode_kernel<<<H, 128, smem, as_stream(stream)>>>(reinterpret_cast<const bf16*>(q), reinterpret_cast<const bf16*>(k_cache),
                                                         reinterpret_cast<const bf16*>(v_cache), len, H * dh, dh, 1.0f / sqrtf((float)dh), out,
                                                         out_f16);
  NEKO_LAUNCH_CHECK("attn_decode_kernel");
  return NEKO_OK;
}

int neko_attention_bwd(const uint16_t* qkv, const uint16_t* out, const uint16_t* dout, const float* lse, const int32_t* first_valid,
                       uint16_t* dqkv, float* delta, int B, int S, int S_valid, int H, int dh, int out_f16, const neko_dropout* drop,
                       void* stream) {
  using namespace neko;
  NEKO_REQUIRE(qkv && out && dout && lse && first_valid && dqkv && delta, "attention_bwd: null pointer");
  NEKO_REQUIRE(B > 0 && S > 0 && H > 0 && S_valid > 0 && S_valid <= S, "attention_bwd: bad sizes");
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(dout) & 15) == 0, "attention_bwd: misaligned");
  NEKO_REQUIRE((long long)B * H * S < (1LL << 32), "attention_bwd: B*H*S exceeds the dropout row-id range");
  cudaStream_t st = as_stream(stream);
  const bf16* x = reinterpret_cast<const bf16*>(qkv);
  const bf16* o = reinterpret_cast<const bf16*>(out);
  const bf16* g = reinterpret_cast<const bf16*>(dout);
  bf16* dx = reinterpret_cast<bf16*>(dqkv);
  const DropCfg dc = drop_cfg(drop);
#define NEKO_ATT_BWD(DH_) (dc.seed ? launch_bwd<DH_, true, false>(x, o, g, lse, delta, first_valid, nullptr, dx, B, S, S_valid, S, 0, H, out_f16, dc, st) \
                                   : launch_bwd<DH_, false, false>(x, o, g, lse, delta, first_valid, nullptr, dx, B, S, S_valid, S, 0, H, out_f16, dc, st))
  switch (dh) {
    case 16: return NEKO_ATT_BWD(16);
    case 32: return NEKO_ATT_BWD(32);
    case 64: return NEKO_ATT_BWD(64);
    case 128: return NEKO_ATT_BWD(128);
    default: set_error("attention: head dim %d not supported (16, 32, 64, 128)", dh); return NEKO_EINVAL;
  }
#undef NEKO_ATT_BWD
}

int neko_attention_varlen_fwd(const uint16_t* qkv, const int32_t* cu_seqlens, const int32_t* first_valid, uint16_t* out, uint16_t* out2_bf16,
                              float* lse, int B, int T, int S_max, int S_width, int H, int dh, int out_f16, const neko_dropout* drop,
                              void* stream) {
  using namespace neko;
  NEKO_REQUIRE(qkv && cu_seqlens && first_valid && out && lse, "attention_varlen_fwd: null pointer");
  NEKO_REQUIRE(B > 0 && T > 0 && H > 0 && S_max > 0 && S_max <= S_width, "attention_varlen_fwd: bad sizes");
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "attention_varlen_fwd: misaligned");
  NEKO_REQUIRE((long long)B * H * S_width < (1LL << 32), "attention_varlen_fwd: B*H*S_width exceeds the dropout row-id range");
  const bf16* x = reinterpret_cast<const bf16*>(qkv);
  bf16* o = reinterpret_cast<bf16*>(out);
  bf16* o2 = reinterpret_cast<bf16*>(out2_bf16);
  cudaStream_t st = as_stream(stream);
  const DropCfg dc = drop_cfg(drop);
#define NEKO_ATT_FWD(DH_) (dc.seed ? launch_fwd<DH_, true, true>(x, first_valid, cu_seqlens, o, o2, lse, B, S_width, S_max, S_max, T, H, out_f16, dc, st) \
                                   : launch_fwd<DH_, false, true>(x, first_valid, cu_seqlens, o, o2, lse, B, S_width, S_max, S_max, T, H, out_f16, dc, st))
  switch (dh) {
    case 16: return NEKO_ATT_FWD(16);
    case 32: return NEKO_ATT_FWD(32);
    case 64: return NEKO_ATT_FWD(64);
    case 128: return NEKO_ATT_FWD(128);
    default: set_error("attention: head dim %d not supported (16, 32, 64, 128)", dh); return NEKO_EINVAL;
  }
#undef NEKO_ATT_FWD
}

int neko_attention_varlen_bwd(const uint16_t* qkv, const uint16_t* out, const uint16_t* dout, const float* lse, const int32_t* cu_seqlens,
                              const int32_t* first_valid, uint16_t* dqkv, float* delta, int B, int T, int S_max, int S_width, int H, int dh,
                              int out_f16, const neko_dropout* drop, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(qkv && out && dout && lse && cu_seqlens && first_valid && dqkv && delta, "attention_varlen_bwd: null pointer");
  NEKO_REQUIRE(B > 0 && T > 0 && H > 0 && S_max > 0 && S_max <= S_width, "attention_varlen_bwd: bad sizes");
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(dout) & 15) == 0, "attention_varlen_bwd: misaligned");
  NEKO_REQUIRE((long long)B * H * S_width < (1LL << 32), "attention_varlen_bwd: B*H*S_width exceeds the dropout row-id range");
  cudaStream_t st = as_stream(stream);
  const bf16* x = reinterpret_cast<const bf16*>(qkv);
  const bf16* o = reinterpret_cast<const bf16*>(out);
  const bf16* g = reinterpret_cast<const bf16*>(dout);
  bf16* dx = reinterpret_cast<bf16*>(dqkv);
  const DropCfg dc = drop_cfg(drop);
#define NEKO_ATT_BWD(DH_) (dc.seed ? launch_bwd<DH_, true, true>(x, o, g, lse, delta, first_valid, cu_seqlens, dx, B, S_width, S_max, S_max, T, H, out_f16, dc, st) \
                                   : launch_bwd<DH_, false, true>(x, o, g, lse, delta, first_valid, cu_seqlens, dx, B, S_width, S_max, S_max, T, H, out_f16, dc, st))
  switch (dh) {
    case 16: return NEKO_ATT_BWD(16);
    case 32: return NEKO_ATT_BWD(32);
    case 64: return NEKO_ATT_BWD(64);
    case 128: return NEKO_ATT_BWD(128);
    default: set_error("attention: head dim %d not supported (16, 32, 64, 128)", dh); return NEKO_EINVAL;
  }
#undef NEKO_ATT_BWD
}

}  // extern "C"
