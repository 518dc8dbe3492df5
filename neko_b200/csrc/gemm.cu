// Dense bf16 GEMM on the 5th-generation tensor cores: C[M,N] = epilogue(sum_k A[m,k] * B[n,k]).
//
// Replaces every dense contraction of the decoder and its autograd: HF Conv1D addmm
// (trajectory_gpt2.py:222,253,274,277), predict_token (gato_policy.py:172),
// post_embedding_projection (embeddings.py:53), plus dgrad / wgrad of each.
//
// Structure (persistent, warp-specialised, one CTA per SM):
//   warp 0      TMA producer: cp.async.bulk.tensor 128B-swizzled boxes of A and B into a
//               STAGES-deep shared-memory ring, completion on mbarriers (full[]).
//   warp 1      MMA issuer: one elected lane issues tcgen05.mma (M=128, N=BN, K=16 per instruction)
//               with the fp32 accumulator in TMEM; tcgen05.commit releases ring slots (empty[]) and
//               publishes finished accumulators (tmem_full[]).  Two accumulator stages in TMEM so the
//               epilogue of tile i overlaps the main loop of tile i+1.
//   warps 2..5  epilogue: tcgen05.ld 32 columns at a time (each warp owns its 32-lane TMEM quarter),
//               fused bias / GELU / residual / GELU' and 128-bit global stores.
// Operands may be K-major or MN-major (UMMA descriptor major bits), so forward (x @ W[in,out]), dgrad and
// wgrad all run from the tensors as they lie in HBM -- no transposed copies.
#include <cuda.h>

#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <type_traits>
#include <unordered_map>

#include "common.cuh"
#include "dropout.cuh"
#include "tcgen05.cuh"

namespace neko {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 bytes = one swizzle row
// epilogue warps per CTA (template parameter EW): 8 = two per TMEM lane quarter, each owning half of the tile's columns (168
// registers per thread), or 16 = four per quarter, a quarter of the columns each (<= 112 registers): twice the warps to hide the
// tcgen05.ld -> math -> staging -> TMA-store chain of the epilogue-heavy launches behind
constexpr int GEMM_EPI_WARPS_MAX = 16;
constexpr int SMEM_BUDGET = 227 * 1024;
constexpr int STAGING_BYTES = 65536;    // per warp 8 KB (EW = 8: ring of 2 fp32 boxes of 32 rows x 128 B, or 4 16-bit boxes of 32 rows x 64 B) or 4 KB (EW = 16)

struct GemmParams {
  int M, N, K;
  int BN;          // 128 or 256
  int stages;
  int a_mn, b_mn;  // operand majors
  int epi;
  int accumulate;
  void* C;
  long long ldc;
  void* C2;
  long long ldc2;
  void* C3;
  long long ldc3;
  const float* bias;
  const void* aux;
  long long ld_aux;
  int vec_ok;      // all epilogue pointers / leading dimensions allow 16-byte accesses
  int flags;       // NEKO_GEMM_*_F16
  int splits;      // split-K factor (fp32 reduction into C when > 1)
  int n_fast;      // tile rasterisation: consecutive work units walk N first (else M first)
  int pair;        // 1: cta_group::2 CTA pairs (256 x BN tile per pair)
  int tma_store;   // outputs leave through shared-memory staging + cp.async.bulk.tensor stores
  int tma_aux;     // RESID_F32 / DGELU: the auxiliary operand arrives as TMA boxes in the staging ring (prefetched, coalesced)
  int streamk;     // 1: the (tile, k-block) space is cut into one contiguous range per worker (see WorkIter)
  float* sk_acc;   // stream-K: partial accumulators, [workers][TM][BN] fp32
  unsigned* sk_flags;  // stream-K: [workers] arrival counters, then [workers] consumer counters (zero between launches)
  int kb_per_split;
  DropCfg drop;    // RESID epilogues: C = aux + dropout(acc + bias)
};

// ---------------------------------------------------------------------------------------------
// epilogue on one 32-column chunk held by one thread (row = its TMEM lane)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, uint32_t (&v)[32], long long row, int col0) {
  const int ncols = min(32, p.N - col0);
  float f[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
  if (p.bias) {
    if (ncols == 32 && p.vec_ok) {
      const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b = __ldg(b4 + i);
        f[4 * i] += b.x; f[4 * i + 1] += b.y; f[4 * i + 2] += b.z; f[4 * i + 3] += b.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (i < ncols) f[i] += __ldg(p.bias + col0 + i);
    }
  }
  const bool fast = (ncols == 32) && p.vec_ok;
  const bool c_f16 = (p.flags & NEKO_GEMM_C_F16) != 0, c2_f16 = (p.flags & NEKO_GEMM_C2_F16) != 0;
  const bool gtanh = (p.flags & NEKO_GEMM_GELU_TANH) != 0;
  switch (p.epi) {
    case NEKO_EPI_BF16:
    case NEKO_EPI_GELU_BF16:
    case NEKO_EPI_DGELU_BF16: {
      uint16_t* c = reinterpret_cast<uint16_t*>(p.C) + row * p.ldc + col0;
      if (p.epi == NEKO_EPI_DGELU_BF16) {
        const bf16* a = reinterpret_cast<const bf16*>(p.aux) + row * p.ld_aux + col0;
        if (fast) {
          const uint4* a4 = reinterpret_cast<const uint4*>(a);
          auto body = [&](auto tag) {
            constexpr bool T = decltype(tag)::value;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint4 u = a4[i];
              const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 pre = unpack_bf16x2(w[j]);
                f[8 * i + 2 * j] *= gelu_grad_sel<T>(pre.x);
                f[8 * i + 2 * j + 1] *= gelu_grad_sel<T>(pre.y);
              }
            }
          };
          if (gtanh) body(std::true_type{}); else body(std::false_type{});
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < ncols) f[i] *= gtanh ? gelu_tanh_grad(__bfloat162float(a[i])) : gelu_erf_grad(__bfloat162float(a[i]));
        }
      }
      if (fast) {
        uint4* c4 = reinterpret_cast<uint4*>(c);
#pragma unroll
        for (int i = 0; i < 4; ++i)
          c4[i] = make_uint4(pack_16x2(f[8 * i], f[8 * i + 1], c_f16), pack_16x2(f[8 * i + 2], f[8 * i + 3], c_f16),
                             pack_16x2(f[8 * i + 4], f[8 * i + 5], c_f16), pack_16x2(f[8 * i + 6], f[8 * i + 7], c_f16));
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < ncols) c[i] = cvt_16(f[i], c_f16);
      }
      if (p.epi == NEKO_EPI_GELU_BF16) {
        uint16_t* c2 = reinterpret_cast<uint16_t*>(p.C2) + row * p.ldc2 + col0;
#pragma unroll
        if (gtanh) {
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = gelu_tanh(f[i]);
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = gelu_erf(f[i]);
        }
        if (fast) {
          uint4* c4 = reinterpret_cast<uint4*>(c2);
#pragma unroll
          for (int i = 0; i < 4; ++i)
            c4[i] = make_uint4(pack_16x2(f[8 * i], f[8 * i + 1], c2_f16), pack_16x2(f[8 * i + 2], f[8 * i + 3], c2_f16),
                               pack_16x2(f[8 * i + 4], f[8 * i + 5], c2_f16), pack_16x2(f[8 * i + 6], f[8 * i + 7], c2_f16));
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < ncols) c2[i] = cvt_16(f[i], c2_f16);
        }
        if (p.C3) {
          uint16_t* c3 = reinterpret_cast<uint16_t*>(p.C3) + row * p.ldc3 + col0;
          if (fast) {
            uint4* c4 = reinterpret_cast<uint4*>(c3);
#pragma unroll
            for (int i = 0; i < 4; ++i)
              c4[i] = make_uint4(pack_bf16x2(f[8 * i], f[8 * i + 1]), pack_bf16x2(f[8 * i + 2], f[8 * i + 3]),
                                 pack_bf16x2(f[8 * i + 4], f[8 * i + 5]), pack_bf16x2(f[8 * i + 6], f[8 * i + 7]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (i < ncols) c3[i] = cvt_16(f[i], false);
          }
        }
      }
      break;
    }
    default: {  // fp32 outputs
      float* c = reinterpret_cast<float*>(p.C) + row * p.ldc + col0;
      if (p.drop.seed && (p.epi == NEKO_EPI_RESID_F32 || p.epi == NEKO_EPI_RESID_F32_BF16)) {
        const uint32_t rk = drop_rowkey(drop_key(p.drop), (uint32_t)row);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float m0, m1;
          drop_pair(rk, (uint32_t)((col0 >> 1) + i), p.drop.thr16, p.drop.scale, m0, m1);
          f[2 * i] *= m0; f[2 * i + 1] *= m1;
        }
      }
      const float* add = nullptr;
      if (p.epi == NEKO_EPI_RESID_F32 || p.epi == NEKO_EPI_RESID_F32_BF16)
        add = reinterpret_cast<const float*>(p.aux) + row * p.ld_aux + col0;
      else if (p.accumulate && p.splits == 1)
        add = c;
      if (add) {  // read everything before the (possibly aliasing) stores below
        if (fast) {
          const float4* a4 = reinterpret_cast<const float4*>(add);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 a = a4[i];
            f[4 * i] += a.x; f[4 * i + 1] += a.y; f[4 * i + 2] += a.z; f[4 * i + 3] += a.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < ncols) f[i] += add[i];
        }
      }
      if (p.splits > 1) {  // split-K partial: reduce into C (pre-initialised by the host) with fp32 RED
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < ncols) atomicAdd(c + i, f[i]);
      } else if (fast) {
        float4* c4 = reinterpret_cast<float4*>(c);
#pragma unroll
        for (int i = 0; i < 8; ++i) c4[i] = make_float4(f[4 * i], f[4 * i + 1], f[4 * i + 2], f[4 * i + 3]);
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < ncols) c[i] = f[i];
      }
      if (p.epi == NEKO_EPI_RESID_F32_BF16) {
        uint16_t* c2 = reinterpret_cast<uint16_t*>(p.C2) + row * p.ldc2 + col0;
        if (fast) {
          uint4* c4 = reinterpret_cast<uint4*>(c2);
#pragma unroll
          for (int i = 0; i < 4; ++i)
            c4[i] = make_uint4(pack_16x2(f[8 * i], f[8 * i + 1], c2_f16), pack_16x2(f[8 * i + 2], f[8 * i + 3], c2_f16),
                               pack_16x2(f[8 * i + 4], f[8 * i + 5], c2_f16), pack_16x2(f[8 * i + 6], f[8 * i + 7], c2_f16));
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < ncols) c2[i] = cvt_16(f[i], c2_f16);
        }
      }
      break;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// staged epilogue: registers -> swizzled shared-memory box (32 rows x 32 columns) -> one bulk tensor store.
// Every global write is a full, coalesced box (TMA clips the M / N tails); accumulate and split-K use the
// reduce-add form, so C is never read back.
// ---------------------------------------------------------------------------------------------
struct Stager {
  uint8_t* base;     // this warp's staging ring (1024-byte aligned)
  int lane;
  int slot;          // next ring slot
  int wide;          // 1: 4 KB slots (some output of this epilogue is fp32), 0: 2 KB slots (all outputs 16-bit)
};

template <int EW>
__device__ __forceinline__ void stage_and_store(Stager& s, const CUtensorMap* map, const float (&f)[32], int kind /*0 f32, 1 bf16, 2 f16*/,
                                                bool reduce, int col0, int row0) {
  // ring of staging slots: before overwriting a slot, the bulk store that last used it must have read it out,
  // i.e. at most (slots - 1) younger stores may still be pending
  constexpr int WIDE_SLOTS = (STAGING_BYTES / EW) / 4096, NARROW_SLOTS = (STAGING_BYTES / EW) / 2048;
  uint8_t* b;
  if (s.wide) {
    b = s.base + (s.slot << 12);
    s.slot = (s.slot + 1) & (WIDE_SLOTS - 1);
    if (s.lane == 0) tma_store_wait_read<WIDE_SLOTS - 1>();
  } else {
    b = s.base + (s.slot << 11);
    s.slot = (s.slot + 1) & (NARROW_SLOTS - 1);
    if (s.lane == 0) tma_store_wait_read<NARROW_SLOTS - 1>();
  }
  __syncwarp();
  const int r = s.lane;
  if (kind == 0) {
#pragma unroll
    for (int c = 0; c < 8; ++c)
      *reinterpret_cast<float4*>(b + r * 128 + ((c ^ (r & 7)) << 4)) = make_float4(f[4 * c], f[4 * c + 1], f[4 * c + 2], f[4 * c + 3]);
  } else {
    const bool h = kind == 2;
#pragma unroll
    for (int c = 0; c < 4; ++c)
      *reinterpret_cast<uint4*>(b + r * 64 + ((c ^ ((r >> 1) & 3)) << 4)) =
          make_uint4(pack_16x2(f[8 * c], f[8 * c + 1], h), pack_16x2(f[8 * c + 2], f[8 * c + 3], h),
                     pack_16x2(f[8 * c + 4], f[8 * c + 5], h), pack_16x2(f[8 * c + 6], f[8 * c + 7], h));
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();
  if (s.lane == 0) {
    if (reduce) tma_reduce_add_2d(map, smem_u32(b), col0, row0);
    else        tma_store_2d(map, smem_u32(b), col0, row0);
    tma_store_commit();
  }
}

template <int EW>
__device__ __forceinline__ void epilogue_chunk_staged(const GemmParams& p, Stager& s, const CUtensorMap* mc, const CUtensorMap* mc2,
                                                      const CUtensorMap* mc3, uint32_t (&v)[32], long long row, int row0, int col0,
                                                      bool split_first) {
  const int ncols = min(32, p.N - col0);
  const bool in_rows = row < p.M;
  const bool fast = (ncols == 32) && p.vec_ok;
  float f[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
  if (p.bias && split_first) {
    if (fast) {
      const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 b = __ldg(b4 + i);
        f[4 * i] += b.x; f[4 * i + 1] += b.y; f[4 * i + 2] += b.z; f[4 * i + 3] += b.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (i < ncols) f[i] += __ldg(p.bias + col0 + i);
    }
  }
  const bool c_f16 = (p.flags & NEKO_GEMM_C_F16) != 0, c2_f16 = (p.flags & NEKO_GEMM_C2_F16) != 0;
  const bool gtanh = (p.flags & NEKO_GEMM_GELU_TANH) != 0;
  switch (p.epi) {
    case NEKO_EPI_BF16:
      stage_and_store<EW>(s, mc, f, c_f16 ? 2 : 1, false, col0, row0);
      break;
    case NEKO_EPI_GELU_BF16:
      stage_and_store<EW>(s, mc, f, c_f16 ? 2 : 1, false, col0, row0);
      if (gtanh) {
#pragma unroll
        for (int i = 0; i < 32; ++i) f[i] = gelu_tanh(f[i]);
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) f[i] = gelu_erf(f[i]);
      }
      stage_and_store<EW>(s, mc2, f, c2_f16 ? 2 : 1, false, col0, row0);
      if (p.C3) stage_and_store<EW>(s, mc3, f, 1, false, col0, row0);
      break;
    case NEKO_EPI_DGELU_BF16: {
      if (in_rows) {
        const bf16* a = reinterpret_cast<const bf16*>(p.aux) + row * p.ld_aux + col0;
        if (fast) {
          const uint4* a4 = reinterpret_cast<const uint4*>(a);
          auto body = [&](auto tag) {
            constexpr bool T = decltype(tag)::value;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint4 u = a4[i];
              const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float2 pre = unpack_bf16x2(w[j]);
                f[8 * i + 2 * j] *= gelu_grad_sel<T>(pre.x);
                f[8 * i + 2 * j + 1] *= gelu_grad_sel<T>(pre.y);
              }
            }
          };
          if (gtanh) body(std::true_type{}); else body(std::false_type{});
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < ncols) f[i] *= gtanh ? gelu_tanh_grad(__bfloat162float(a[i])) : gelu_erf_grad(__bfloat162float(a[i]));
        }
      }
      stage_and_store<EW>(s, mc, f, c_f16 ? 2 : 1, false, col0, row0);
      break;
    }
    case NEKO_EPI_F32:
      stage_and_store<EW>(s, mc, f, 0, p.accumulate || p.splits > 1, col0, row0);
      break;
    default: {  // NEKO_EPI_RESID_F32 / NEKO_EPI_RESID_F32_BF16
      if (p.drop.seed) {  // resid_dropout on the branch output, before the residual add
        const uint32_t rk = drop_rowkey(drop_key(p.drop), (uint32_t)row);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float m0, m1;
          drop_pair(rk, (uint32_t)((col0 >> 1) + i), p.drop.thr16, p.drop.scale, m0, m1);
          f[2 * i] *= m0; f[2 * i + 1] *= m1;
        }
      }
      if (in_rows) {
        const float* add = reinterpret_cast<const float*>(p.aux) + row * p.ld_aux + col0;
        if (fast) {
          const float4* a4 = reinterpret_cast<const float4*>(add);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 a = a4[i];
            f[4 * i] += a.x; f[4 * i + 1] += a.y; f[4 * i + 2] += a.z; f[4 * i + 3] += a.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (i < ncols) f[i] += add[i];
        }
      }
      stage_and_store<EW>(s, mc, f, 0, false, col0, row0);
      if (p.epi == NEKO_EPI_RESID_F32_BF16) stage_and_store<EW>(s, mc2, f, c2_f16 ? 2 : 1, false, col0, row0);
      break;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Epilogue of one tile for the two epilogues that read an auxiliary operand (RESID_F32: C = aux + dropout(acc + bias), fp32;
// DGELU: C = acc * gelu'(aux), 16-bit).  The aux box of a 32 x 32 chunk is brought into this warp's staging slot by TMA
// (issued one chunk ahead, the first two before the accumulator is even complete), combined in place and stored from the
// same slot: the aux read is asynchronous and coalesced instead of 32 row-strided 16-byte loads per warp instruction.
// ---------------------------------------------------------------------------------------------
template <bool F32>
__device__ __forceinline__ void aux_issue(uint8_t* slot, const CUtensorMap* map_aux, uint32_t bar, int lane, int col0, int row0) {
  if (lane == 0) {
    mbar_expect_tx(bar, F32 ? 4096u : 2048u);
    tma_load_2d(smem_u32(slot), map_aux, bar, col0, row0);
  }
}

template <bool F32>
__device__ __forceinline__ void aux_combine_store(const GemmParams& p, uint8_t* b, const CUtensorMap* mc, uint32_t (&v)[32], int lane,
                                                  long long row, int row0, int col0) {
  const int ncols = min(32, p.N - col0);
  float f[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
  const int r = lane;
  if (F32) {
    if (p.bias) {
      if (ncols == 32) {
        const float4* b4 = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 bb = __ldg(b4 + i);
          f[4 * i] += bb.x; f[4 * i + 1] += bb.y; f[4 * i + 2] += bb.z; f[4 * i + 3] += bb.w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < ncols) f[i] += __ldg(p.bias + col0 + i);
      }
    }
    if (p.drop.seed) {  // resid_dropout on the branch output, before the residual add
      const uint32_t rk = drop_rowkey(drop_key(p.drop), (uint32_t)row);
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        float m0, m1;
        drop_pair(rk, (uint32_t)((col0 >> 1) + i), p.drop.thr16, p.drop.scale, m0, m1);
        f[2 * i] *= m0; f[2 * i + 1] *= m1;
      }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float4* q = reinterpret_cast<float4*>(b + r * 128 + ((c ^ (r & 7)) << 4));
      const float4 a = *q;
      *q = make_float4(f[4 * c] + a.x, f[4 * c + 1] + a.y, f[4 * c + 2] + a.z, f[4 * c + 3] + a.w);
    }
  } else {
    const bool h = (p.flags & NEKO_GEMM_C_F16) != 0;
    const bool gtanh = (p.flags & NEKO_GEMM_GELU_TANH) != 0;
    auto body = [&](auto tag) {
      constexpr bool T = decltype(tag)::value;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        uint4* q = reinterpret_cast<uint4*>(b + r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
        const uint4 u = *q;
        const uint32_t w[4] = {u.x, u.y, u.z, u.w};
        float g[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 pre = unpack_bf16x2(w[j]);
          g[2 * j] = f[8 * c + 2 * j] * gelu_grad_sel<T>(pre.x);
          g[2 * j + 1] = f[8 * c + 2 * j + 1] * gelu_grad_sel<T>(pre.y);
        }
        *q = make_uint4(pack_16x2(g[0], g[1], h), pack_16x2(g[2], g[3], h), pack_16x2(g[4], g[5], h), pack_16x2(g[6], g[7], h));
      }
    };
    if (gtanh) body(std::true_type{}); else body(std::false_type{});
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncwarp();
  if (lane == 0) {
    tma_store_2d(mc, smem_u32(b), col0, row0);
    tma_store_commit();
  }
}

// ---------------------------------------------------------------------------------------------
// kernel
// ---------------------------------------------------------------------------------------------
// PAIR = true: the two CTAs of a cluster (one TPC) form a cta_group::2 pair that computes one 256 x BN tile.  Each CTA
// stages its own 128 rows of A and HALF of the B tile; the leader (cluster rank 0) issues M=256 MMAs that read both
// shared memories and write both tensor memories, so every operand byte crosses L2 -> SM once per PAIR instead of
// once per CTA (the single-CTA kernel is bound by that traffic, profiles/r01_ncu_gemm_full.md).
// stream-K owner: add the helper's partial accumulator (this thread's row, 32 columns from `col`) to the freshly loaded chunk
__device__ __forceinline__ void sk_add_partial(uint32_t (&v)[32], const float* sk_row, int col) {
  const float4* p4 = reinterpret_cast<const float4*>(sk_row + col);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 a = __ldcg(p4 + j);   // written by another SM during this launch: L2, never a stale L1 line
    v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + a.x);
    v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + a.y);
    v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + a.z);
    v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + a.w);
  }
}

// ---------------------------------------------------------------------------------------------
// Work distribution.  Classic: worker w takes units w, w + W, ... of the (tile, k-split) list.  Stream-K (p.streamk): the
// linearised (tile, k-block) space is cut into W contiguous ranges of (almost) equal length, so a launch whose tile count is
// 1.2 x the worker count costs 1.2 rounds of main loop instead of 2.  The host enables it only when every range is at least one
// tile long; a tile is then shared by at most two workers: worker w ENDS with the head k-blocks of a tile (kind 2: it owns the
// tile and runs the epilogue) and worker w + 1 STARTS with its tail k-blocks (kind 1: it stores the raw partial accumulator into
// workspace slot w + 1 and signals).  The helper does its part first and the owner last, so the owner practically never waits.
// ---------------------------------------------------------------------------------------------
struct Work {
  long long tile;
  int kb0, kb1;
  int kind;          // 0 whole tile / k-split unit, 1 helper (partial -> workspace), 2 owner (adds the next worker's partial)
  bool split_first;
};
struct WorkIter {
  long long u, u_step, units;      // classic
  int splits, kb_per_split, k_blocks;
  long long lin, end;              // stream-K
  int streamk;
  __device__ __forceinline__ WorkIter(const GemmParams& p, long long worker, long long workers, long long tiles, int kblocks)
      : u(worker), u_step(workers), units(tiles * p.splits), splits(p.splits), kb_per_split(p.kb_per_split), k_blocks(kblocks),
        lin(0), end(0), streamk(p.streamk) {
    if (streamk) {
      const long long total = tiles * (long long)kblocks;
      lin = worker * total / workers;
      end = (worker + 1) * total / workers;
    }
  }
  __device__ __forceinline__ bool next(Work& w) {
    if (!streamk) {
      if (u >= units) return false;
      w.tile = u / splits;
      const int ks = (int)(u - w.tile * splits);
      w.kb0 = ks * kb_per_split;
      w.kb1 = min(k_blocks, w.kb0 + kb_per_split);
      w.kind = 0;
      w.split_first = ks == 0;
      u += u_step;
      return true;
    }
    if (lin >= end) return false;
    w.tile = lin / k_blocks;
    w.kb0 = (int)(lin - w.tile * k_blocks);
    w.kb1 = (int)min((long long)k_blocks, (long long)w.kb0 + (end - lin));
    w.kind = (w.kb0 > 0) ? 1 : (w.kb1 < k_blocks ? 2 : 0);
    w.split_first = true;
    lin += w.kb1 - w.kb0;
    return true;
  }
};

template <bool PAIR, int EW>
__global__ void __launch_bounds__(64 + 32 * EW, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_c, const __grid_constant__ CUtensorMap map_c2,
                    const __grid_constant__ CUtensorMap map_c3, const __grid_constant__ CUtensorMap map_aux,
                    const __grid_constant__ CUtensorMap map_ws, const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment for the 128B swizzle atoms
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int BN = p.BN;
  const int stages = p.stages;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;  // position inside the CTA pair
  const int BNL = PAIR ? BN / 2 : BN;                    // rows of the B tile staged by THIS CTA
  const uint32_t a_bytes = BM * BK * 2;
  const uint32_t b_bytes = (uint32_t)BNL * BK * 2;
  const uint32_t stage_bytes = a_bytes + b_bytes;
  uint8_t* staging = smem + (size_t)stages * stage_bytes;  // 1024-byte aligned: stage_bytes is a multiple of 1024
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + STAGING_BYTES);
  // barrier layout: full[stages], empty[stages], tmem_full[2], tmem_empty[2], then the TMEM base address
  const uint32_t bar0 = smem_u32(bars);
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (stages + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * stages + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * stages + 2 + a); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * stages + 4);
  auto aux_bar = [&](int e, int slot) { return bar0 + 8u * (2 * stages + 5 + 2 * e + slot); };   // per epilogue warp, per staging slot

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t tmem_cols = (2u * BN <= 256u) ? 256u : 512u;  // two accumulator stages of BN columns, rounded to a power of two
  pdl_launch_dependents();             // the next kernel of the stream may start its own prologue as SMs free up

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
    for (int s = 0; s < stages; ++s) {
      mbar_init(full_bar(s), PAIR ? 2 : 1);   // pair: one expect_tx arrival per CTA, both on the leader's barrier
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), PAIR ? 2 * EW : EW);  // pair: both CTAs' epilogues release the leader
    }
    for (int e = 0; e < EW; ++e) {
      mbar_init(aux_bar(e, 0), 1);
      mbar_init(aux_bar(e, 1), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();   // barriers of BOTH CTAs are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  pdl_wait();                          // everything above overlapped the previous kernel's tail; its outputs are visible from here

  constexpr int TM = PAIR ? 2 * BM : BM;  // rows of C per work unit
  const int m_blocks = (p.M + TM - 1) / TM;
  const int n_blocks = (p.N + BN - 1) / BN;
  const int k_blocks = (p.K + BK - 1) / BK;
  const long long tiles = (long long)m_blocks * n_blocks;
  const long long units = tiles * p.splits;  // work unit = (tile, k-split)
  const long long u_first = PAIR ? (blockIdx.x >> 1) : blockIdx.x;   // both CTAs of a pair walk the same units
  const long long u_step = PAIR ? (gridDim.x >> 1) : gridDim.x;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      WorkIter it(p, u_first, u_step, tiles, k_blocks);
      Work w;
      while (it.next(w)) {
        const long long t = w.tile;
        const int m0 = (int)(p.n_fast ? (t / n_blocks) : (t % m_blocks)) * TM + (int)rank * BM;   // this CTA's 128 rows
        const int n0 = (int)(p.n_fast ? (t % n_blocks) : (t / m_blocks)) * BN + (int)rank * BNL;  // this CTA's slice of B
        const int kb0 = w.kb0, kb1 = w.kb1;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
          const uint32_t sb = sa + a_bytes;
          const int k0 = kb * BK;
          if (PAIR) {
            // both CTAs post their bytes on the LEADER's full barrier; the loads land in the local shared memory
            const uint32_t fb = mapa_shared(full_bar(stage), 0);
            mbar_expect_tx_cluster(fb, stage_bytes);
            if (!p.a_mn) {
              tma_load_2d_pair(sa, &map_a, fb, k0, m0);
            } else {
              for (int g = 0; g < BM / 64; ++g) tma_load_2d_pair(sa + g * (BK * 128), &map_a, fb, m0 + g * 64, k0);
            }
            if (!p.b_mn) {
              tma_load_2d_pair(sb, &map_b, fb, k0, n0);
            } else {
              for (int g = 0; g < BNL / 64; ++g) tma_load_2d_pair(sb + g * (BK * 128), &map_b, fb, n0 + g * 64, k0);
            }
          } else {
            mbar_expect_tx(full_bar(stage), stage_bytes);
            if (!p.a_mn) {
              tma_load_2d(sa, &map_a, full_bar(stage), k0, m0);  // box {64 k, 128 m}
            } else {
              for (int g = 0; g < BM / 64; ++g)                  // boxes {64 m, 64 k}
                tma_load_2d(sa + g * (BK * 128), &map_a, full_bar(stage), m0 + g * 64, k0);
            }
            if (!p.b_mn) {
              tma_load_2d(sb, &map_b, full_bar(stage), k0, n0);  // box {64 k, BN n}
            } else {
              for (int g = 0; g < BN / 64; ++g)
                tma_load_2d(sb + g * (BK * 128), &map_b, full_bar(stage), n0 + g * 64, k0);
            }
          }
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && rank == 0) {  // pair: only the leader CTA issues
      // instruction descriptor: fp32 accumulate, {f16|bf16} x {f16|bf16}, M=128 (256 per pair), N=BN, operand majors
      const uint32_t a_fmt = (p.flags & NEKO_GEMM_A_F16) ? 0u : 1u, b_fmt = (p.flags & NEKO_GEMM_B_F16) ? 0u : 1u;  // F16 = 0, BF16 = 1
      const uint32_t idesc = (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | ((uint32_t)(p.a_mn ? 1 : 0) << 15) |
                             ((uint32_t)(p.b_mn ? 1 : 0) << 16) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      WorkIter it(p, u_first, u_step, tiles, k_blocks);
      Work w;
      while (it.next(w)) {
        const int kb0 = w.kb0, kb1 = w.kb1;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);  // epilogue drained this accumulator
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
          const uint32_t sb = sa + a_bytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // K-major: step 16 elements = 32 bytes inside the 128-byte swizzle row.
            // MN-major: step 16 k-rows = two 8-row swizzle atoms = 2048 bytes.
            const uint64_t da = p.a_mn ? make_smem_desc(sa + k * 2048, BK * 128, 1024) : make_smem_desc(sa + k * 32, 16, 1024);
            const uint64_t db = p.b_mn ? make_smem_desc(sb + k * 2048, BK * 128, 1024) : make_smem_desc(sb + k * 32, 16, 1024);
            if (PAIR) tc_mma_bf16_pair(d_tmem, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            else      tc_mma_bf16(d_tmem, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          if (PAIR) tc_commit_pair(empty_bar(stage)); else tc_commit(empty_bar(stage));  // ring slot free (in both CTAs)
          if (++stage == stages) { stage = 0; phase ^= 1u; }
        }
        if (PAIR) tc_commit_pair(tfull_bar(acc)); else tc_commit(tfull_bar(acc));      // accumulator complete
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    // ===================== epilogue warps =====================
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    Stager stg;
    const int e = warp - 2;            // 0..EW-1
    const int half = e >> 2;           // which part (half for EW = 8, quarter for EW = 16) of the tile's columns
    constexpr int PARTS = EW / 4;      // column parts per TMEM lane quarter
    stg.base = staging + (size_t)e * (STAGING_BYTES / EW);
    stg.lane = lane;
    stg.slot = 0;
    stg.wide = (p.epi == NEKO_EPI_F32 || p.epi == NEKO_EPI_RESID_F32 || p.epi == NEKO_EPI_RESID_F32_BF16) ? 1 : 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    uint32_t aux_phase[2] = {0u, 0u};
    const bool aux_f32 = (p.epi == NEKO_EPI_RESID_F32);
    const int aux_slot_bytes = aux_f32 ? 4096 : 2048;
    const int aux_slots = min(2, (STAGING_BYTES / EW) / aux_slot_bytes);   // 1 when a 4 KB warp region holds fp32 boxes
    WorkIter it(p, u_first, u_step, tiles, k_blocks);
    Work w;
    const unsigned sk_total = (unsigned)(EW * (PAIR ? 2 : 1));     // epilogue warps that store / consume one partial tile
    while (it.next(w)) {
      const long long t = w.tile;
      const bool split_first = w.split_first;
      const int m0 = (int)(p.n_fast ? (t / n_blocks) : (t % m_blocks)) * TM + (int)rank * BM;
      const int n0 = (int)(p.n_fast ? (t % n_blocks) : (t / m_blocks)) * BN;
      const long long row = (long long)m0 + q * 32 + lane;
      const uint32_t taddr = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(q * 32) << 16);
      // stream-K: rows of this thread / warp inside workspace slot `sk_slot` ([TM][BN] fp32 per slot)
      const long long sk_slot = (w.kind == 1) ? u_first : u_first + 1;
      const float* sk_row = (w.kind == 2) ? p.sk_acc + ((sk_slot * TM + (long long)rank * BM + q * 32 + lane) * BN) : nullptr;
      if (w.kind == 1) {
        // helper: the raw accumulator of this k-range goes to the workspace as fp32 boxes, then one arrival per warp
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        if (lane == 0) tma_store_wait_read<0>();        // nothing of an earlier epilogue may still read the staging region
        __syncwarp();
        const int nchh = (BN / 32 + PARTS - 1) / PARTS;
        for (int cc = 0; cc < nchh; ++cc) {
          const int c = half * nchh + cc;
          if (c * 32 >= BN) break;
          uint32_t v[32];
          tc_ld32(taddr + (uint32_t)(c * 32), v);
          uint8_t* b = stg.base;                        // one 4 KB fp32 box at a time
          if (lane == 0) tma_store_wait_read<0>();
          __syncwarp();
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(b + lane * 128 + ((j ^ (lane & 7)) << 4)) =
                make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&map_ws, smem_u32(b), c * 32, (int)(sk_slot * TM) + (int)rank * BM + q * 32);
            tma_store_commit();
          }
        }
        if (lane == 0) {
          asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // the partial is in global memory ...
          __threadfence();
          atomicAdd(p.sk_flags + sk_slot, 1u);                         // ... before the owner is told
        }
        __syncwarp();
      } else if (p.tma_aux) {
        // chunks of this warp: c = half * nch + cc.  The aux boxes of the first two are requested before the accumulator
        // is complete (the main loop of this tile is still running), later ones one chunk ahead.
        const int nch = BN / (32 * PARTS);
        const int c_first = half * nch;
        int n_live = 0;
        for (int cc = 0; cc < nch; ++cc) n_live += (n0 + (c_first + cc) * 32 < p.N) ? 1 : 0;
        const int row0 = m0 + q * 32;
        if (lane == 0) tma_store_wait_read<0>();     // the previous tile's stores have read both slots
        __syncwarp();
        for (int cc = 0; cc < aux_slots && cc < n_live; ++cc) {
          if (aux_f32) aux_issue<true>(stg.base + cc * aux_slot_bytes, &map_aux, aux_bar(e, cc), lane, n0 + (c_first + cc) * 32, row0);
          else         aux_issue<false>(stg.base + cc * aux_slot_bytes, &map_aux, aux_bar(e, cc), lane, n0 + (c_first + cc) * 32, row0);
        }
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        if (w.kind == 2) {      // owner: the helper's partial must have landed
          if (lane == 0) {
            while (*reinterpret_cast<volatile unsigned*>(p.sk_flags + sk_slot) < sk_total) __nanosleep(32);
            __threadfence();
          }
          __syncwarp();
        }
        for (int cc = 0; cc < n_live; ++cc) {
          const int slot = cc & (aux_slots - 1);
          const int col0 = n0 + (c_first + cc) * 32;
          uint32_t v[32];
          tc_ld32(taddr + (uint32_t)((c_first + cc) * 32), v);
          if (sk_row) sk_add_partial(v, sk_row, (c_first + cc) * 32);
          mbar_wait(aux_bar(e, slot), aux_phase[slot]);
          aux_phase[slot] ^= 1u;
          uint8_t* b = stg.base + slot * aux_slot_bytes;
          if (aux_f32) aux_combine_store<true>(p, b, &map_c, v, lane, row, row0, col0);
          else         aux_combine_store<false>(p, b, &map_c, v, lane, row, row0, col0);
          if (cc + aux_slots < n_live) {     // refill this slot with the aux box of a later chunk once its store has read it out
            if (lane == 0) tma_store_wait_read<0>();
            __syncwarp();
            if (aux_f32) aux_issue<true>(b, &map_aux, aux_bar(e, slot), lane, n0 + (c_first + cc + aux_slots) * 32, row0);
            else         aux_issue<false>(b, &map_aux, aux_bar(e, slot), lane, n0 + (c_first + cc + aux_slots) * 32, row0);
          }
        }
      } else {
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        if (w.kind == 2) {      // owner: the helper's partial must have landed
          if (lane == 0) {
            while (*reinterpret_cast<volatile unsigned*>(p.sk_flags + sk_slot) < sk_total) __nanosleep(32);
            __threadfence();
          }
          __syncwarp();
        }
        const int nch = (BN / 32 + PARTS - 1) / PARTS;      // BN = 192 is launched with EW = 8 only (6 chunks / 2 parts)
        for (int cc = 0; cc < nch; ++cc) {
          const int c = half * nch + cc;
          const int col0 = n0 + c * 32;
          if (c * 32 >= BN || col0 >= p.N) break;  // warp-uniform
          uint32_t v[32];
          tc_ld32(taddr + (uint32_t)(c * 32), v);
          if (sk_row) sk_add_partial(v, sk_row, c * 32);
          if (p.tma_store) epilogue_chunk_staged<EW>(p, stg, &map_c, &map_c2, &map_c3, v, row, m0 + q * 32, col0, split_first);
          else if (row < p.M) epilogue_chunk(p, v, row, col0);
        }
      }
      if (w.kind == 2) {        // the last consumer of a partial tile re-arms its counters for the next launch
        __syncwarp();
        if (lane == 0) {
          const unsigned prev = atomicAdd(p.sk_flags + u_step + sk_slot, 1u);
          if (prev == sk_total - 1u) {
            p.sk_flags[u_step + sk_slot] = 0u;
            p.sk_flags[sk_slot] = 0u;
            __threadfence();
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(mapa_shared(tempty_bar(acc), 0)); else mbar_arrive(tempty_bar(acc));
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
    if (p.tma_store && lane == 0) tma_store_wait_read<0>();  // staging buffers must outlive their bulk reads
  }

  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();  // pair: the peer may still read this CTA's shared memory / arrive on its barriers
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    else      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// host side: tensor maps (driver entry point fetched at run time -- no link-time libcuda dependency)
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

struct MapKey {
  const void* ptr;
  unsigned long long inner, outer, ld;
  unsigned box_inner, box_outer;
  int f16;  // 0 bf16, 1 f16 (operands, 128B swizzle); 2 f32 output box (128B swizzle); 3 / 4 bf16 / f16 output box (64B swizzle)
  bool operator==(const MapKey& o) const {
    return ptr == o.ptr && inner == o.inner && outer == o.outer && ld == o.ld && box_inner == o.box_inner && box_outer == o.box_outer && f16 == o.f16;
  }
};
struct MapKeyHash {
  size_t operator()(const MapKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h = h * 1000003u ^ k.inner; h = h * 1000003u ^ k.outer; h = h * 1000003u ^ k.ld;
    h = h * 1000003u ^ k.box_inner; h = h * 1000003u ^ k.box_outer; h = h * 1000003u ^ (size_t)k.f16;
    return h;
  }
};

// 2-D bf16 tensor [outer, inner] (inner contiguous, row pitch ld elements), box {box_inner, box_outer}.
int make_map(CUtensorMap* out, const void* ptr, unsigned long long inner, unsigned long long outer, unsigned long long ld,
                    unsigned box_inner, unsigned box_outer, int f16) {
  static std::mutex mu;
  static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
  const MapKey key{ptr, inner, outer, ld, box_inner, box_outer, f16};
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return NEKO_OK; }
  }
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_error("cuTensorMapEncodeTiled not available from the driver"); return NEKO_ECUDA; }
  const cuuint64_t dims[2] = {inner, outer};
  const unsigned long long esz = (f16 == 2) ? 4ull : 2ull;
  const cuuint64_t strides[1] = {ld * esz};
  const cuuint32_t box[2] = {box_inner, box_outer};
  const cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = (f16 == 2) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : ((f16 == 1 || f16 == 4) ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16);
  const CUtensorMapSwizzle sw = (f16 >= 3) ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B;
  const CUresult r = enc(out, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): ptr=%p inner=%llu outer=%llu ld=%llu box=%ux%u", (int)r, ptr, inner, outer, ld, box_inner, box_outer);
    return NEKO_ECUDA;
  }
  {
    std::lock_guard<std::mutex> g(mu);
    if (cache.size() > 4096) cache.clear();
    cache.emplace(key, *out);
  }
  return NEKO_OK;
}

}  // namespace neko

extern "C" int64_t neko_gemm_workspace_bytes(void) {
  // 148 workers x (128 x 256 fp32) = 74 pair tiles of 256 x 256: partial accumulators, then 2 x 148 counters, rounded up
  return (int64_t)neko::sm_count() * 128 * 256 * 4 + 4096;
}

namespace neko {

// Everything neko_gemm decides before it launches: the kernel parameters (minus the tensor-map-backed pointers that only the
// launch needs) and the host-side choices.  neko_gemm_plan reports it without launching.
struct GemmPlan {
  GemmParams p;
  int epi16;         // 16 epilogue warps (else 8)
  long long mb;      // row blocks of the chosen tile height (128, or 256 for a pair)
  int stage_bytes;   // one ring stage: A box + this CTA's B box
  int sms;           // persistent grid cap
};

// Argument checks and schedule selection of one neko_gemm call.  Launches nothing, touches no device memory.
static int plan_gemm(const neko_gemm_desc* gd, GemmPlan& pl) {
  NEKO_REQUIRE(gd != nullptr, "gemm: null descriptor");
  const int M = gd->M, N = gd->N, K = gd->K, a_mn = gd->a_mn, b_mn = gd->b_mn, epilogue = gd->epilogue;
  const int accumulate = gd->accumulate, flags = gd->flags;
  const void *A = gd->A, *B = gd->B, *aux = gd->aux;
  void *C = gd->C, *C2 = gd->C2, *C3 = gd->C3;
  const long long lda = gd->lda, ldb = gd->ldb, ldc = gd->ldc, ldc2 = gd->ldc2, ldc3 = gd->ldc3, ld_aux = gd->ld_aux;
  const float* bias = gd->bias;
  NEKO_REQUIRE(M > 0 && N > 0 && K > 0, "gemm: empty problem %dx%dx%d", M, N, K);
  NEKO_REQUIRE(A && B && C, "gemm: null operand");
  NEKO_REQUIRE(epilogue >= NEKO_EPI_BF16 && epilogue <= NEKO_EPI_RESID_F32_BF16, "gemm: unknown epilogue %d", epilogue);
  NEKO_REQUIRE(((flags & NEKO_GEMM_A_F16) != 0) == ((flags & NEKO_GEMM_B_F16) != 0), "gemm: A and B must have the same 16-bit format (tcgen05 kind::f16 traps on mixed f16/bf16)");
  NEKO_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0, "gemm: operands must be 16-byte aligned");
  NEKO_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "gemm: leading dimensions must be multiples of 8 elements (TMA 16-byte pitch), got %lld %lld", lda, ldb);
  NEKO_REQUIRE(lda >= (a_mn ? M : K) && ldb >= (b_mn ? N : K), "gemm: leading dimension smaller than the row length");
  if (epilogue == NEKO_EPI_GELU_BF16 || epilogue == NEKO_EPI_RESID_F32_BF16) NEKO_REQUIRE(C2 != nullptr, "gemm: epilogue %d needs C2", epilogue);
  if (epilogue == NEKO_EPI_RESID_F32 || epilogue == NEKO_EPI_RESID_F32_BF16 || epilogue == NEKO_EPI_DGELU_BF16)
    NEKO_REQUIRE(aux != nullptr, "gemm: epilogue %d needs aux", epilogue);
  NEKO_REQUIRE(!accumulate || epilogue == NEKO_EPI_F32, "gemm: accumulate is only defined for NEKO_EPI_F32");
  NEKO_REQUIRE(C3 == nullptr || epilogue == NEKO_EPI_GELU_BF16, "gemm: C3 is only defined for NEKO_EPI_GELU_BF16");
  // C = acc * gelu'(aux): the TMA-aux epilogue has no bias term, the per-thread ones would add it before the multiply
  NEKO_REQUIRE(bias == nullptr || epilogue != NEKO_EPI_DGELU_BF16, "gemm: NEKO_EPI_DGELU_BF16 takes no bias");

  GemmParams& p = pl.p;
  memset(&p, 0, sizeof(p));
  p.M = M; p.N = N; p.K = K;
  p.a_mn = a_mn ? 1 : 0; p.b_mn = b_mn ? 1 : 0;
  p.epi = epilogue; p.accumulate = accumulate; p.flags = flags;
  p.C = C; p.ldc = ldc; p.C2 = C2; p.ldc2 = ldc2; p.C3 = C3; p.ldc3 = ldc3; p.bias = bias; p.aux = aux; p.ld_aux = ld_aux;
  p.drop = drop_cfg(&gd->drop);
  NEKO_REQUIRE(!p.drop.seed || epilogue == NEKO_EPI_RESID_F32 || epilogue == NEKO_EPI_RESID_F32_BF16, "gemm: dropout is only defined for the residual epilogues");
  // tile shape, CTA pairing and split-K factor: minimise  waves x (main loop + epilogue)  in units of one k-block of a
  // 128 x 128 tile.  Per-k-block costs reflect the measured operand-traffic bound (profiles/): a single CTA moves
  // 32 KB (BN=128) or 48 KB (BN=256) per k-block, a CTA of a pair 24 KB / 32 KB for the same MMA work.  Split-K
  // (fp32 reduce-add into C) is only used for plain fp32 outputs: the weight gradients, whose M x N is a handful
  // of tiles while K is the whole token axis.
  // NEKO_GEMM_SMS caps the persistent grid (data-parallel runs leave a few SMs to the NCCL kernels that overlap backward:
  // a 227 KB CTA queued behind a long-running communication CTA would stall its whole statically partitioned share of tiles)
  static const int sms_cap = getenv("NEKO_GEMM_SMS") ? atoi(getenv("NEKO_GEMM_SMS")) : 0;
  const int sms = (sms_cap > 1 && sms_cap < sm_count()) ? (sms_cap & ~1) : sm_count();
  pl.sms = sms;
  const int kblocks = (K + BK - 1) / BK;
  // NEKO_GEMM_DETERMINISTIC: every output element is summed by one CTA in k order, whatever the tile shape (no split-K, no
  // stream-K; the NEKO_GEMM_SPLITS / NEKO_GEMM_STREAMK forcing is ignored).
  const bool deterministic = (flags & NEKO_GEMM_DETERMINISTIC) != 0;
  const bool can_split = (epilogue == NEKO_EPI_F32) && (bias == nullptr) && !deterministic;
  // CTA pairs pay off where the main loop dominates (measured per shape, profiles/r01_gemm_shapes.md): plain fp32
  // outputs (LM head, weight gradients) and wide 16-bit outputs; narrow-N and epilogue-heavy launches stay single-CTA.
  // (tools/gemm_sweep.py: at K >= 2048 the 256 x 256 pair tile also wins for N = 768 despite filling only 1.2 waves.)
  const bool plain16 = (epilogue == NEKO_EPI_BF16), resid = (epilogue == NEKO_EPI_RESID_F32 || epilogue == NEKO_EPI_RESID_F32_BF16);
  const bool gelu_wide = (epilogue == NEKO_EPI_GELU_BF16 && N >= 2048);   // 57.4 vs 59.4 us at M=7680, 104 vs 113 us at M=15808
  int pair_lo = 0, pair_hi = (epilogue == NEKO_EPI_F32 || (plain16 && (N >= 2048 || K >= 2048)) || (resid && K >= 2048) || gelu_wide) ? 1 : 0;
  if (const char* force = getenv("NEKO_GEMM_PAIR")) { pair_lo = pair_hi = atoi(force) ? 1 : 0; }
  double best = 1e30;
  // BN = 192 is implemented and tested (NEKO_GEMM_BN=192) but not chosen automatically: at the N = 768 shapes it measured
  // within +-2 us of the 128 / 256 choices (the main loop is bound by operand traffic, not by wave count)
  static const bool no192 = getenv("NEKO_GEMM_AUTO192") == nullptr;
  p.BN = 128; p.splits = 1; p.pair = 0;
  for (int pr = pair_lo; pr <= pair_hi; ++pr) {
    const long long mb_ = (M + (pr ? 2 * BM : BM) - 1) / (pr ? 2 * BM : BM);
    const int workers = pr ? sms / 2 : sms;
    for (int bn = 128; bn <= 256; bn += 64) {
      if (bn > 128 && N <= 128) break;
      // BN = 192 (4 x 192 = 768: fewer, fuller waves at the N = 768 shapes); a CTA of a pair would stage 96 rows of B, which
      // the 64-wide boxes of an MN-major operand cannot express
      if (bn == 192 && ((pr && b_mn) || no192)) continue;
      const double kb_cost = pr ? (bn == 128 ? 1.15 : (bn == 192 ? 1.27 : 1.4))
                                : (bn == 128 ? 1.15 : (bn == 192 ? 1.38 : 1.6));   // fitted to tools/gemm_sweep.py
      const long long tiles_ = mb_ * ((N + bn - 1) / bn);
      for (int sp = 1; sp <= (can_split ? 16 : 1); ++sp) {
        if (sp > 1 && kblocks / sp < 8) break;
        const long long units_ = tiles_ * sp;
        const double per_unit = ((kblocks + sp - 1) / sp) * kb_cost + 3.0 * (bn / 128.0) * (sp > 1 ? 1.5 : 1.0);
        const double cost = (double)((units_ + workers - 1) / workers) * per_unit;
        if (cost < best - 1e-9) { best = cost; p.BN = bn; p.splits = sp; p.pair = pr; }
      }
    }
  }
  const long long mb_ = (M + (p.pair ? 2 * BM : BM) - 1) / (p.pair ? 2 * BM : BM);
  pl.mb = mb_;
  if (const char* force = getenv("NEKO_GEMM_BN")) {
    const int v = atoi(force);
    if (v == 128 || v == 256 || (v == 192 && !(p.pair && b_mn))) p.BN = v;
  }
  if (const char* force = getenv("NEKO_GEMM_SPLITS")) { const int v = atoi(force); if (v >= 1 && can_split) p.splits = v; }
  // rasterisation: the operand that is re-read across the concurrently running tiles should be the small one --
  // walk the shorter block dimension fastest so one wave covers a squarish patch of C and the long operand streams
  // from HBM exactly once (head dgrad / wgrad: 800 MB of dlogits)
  p.n_fast = (((N + p.BN - 1) / p.BN) < mb_) ? 1 : 0;
  if (const char* force = getenv("NEKO_GEMM_NFAST")) p.n_fast = atoi(force) ? 1 : 0;
  p.kb_per_split = (kblocks + p.splits - 1) / p.splits;
  p.splits = (kblocks + p.kb_per_split - 1) / p.kb_per_split;  // no empty split
  const int bnl = p.pair ? p.BN / 2 : p.BN;  // B rows staged per CTA
  pl.stage_bytes = BM * BK * 2 + bnl * BK * 2;
  p.stages = (SMEM_BUDGET - 1024 - 512 - STAGING_BYTES) / pl.stage_bytes;
  if (p.stages > 8) p.stages = 8;
  const bool out_bf16 = (epilogue == NEKO_EPI_BF16 || epilogue == NEKO_EPI_GELU_BF16 || epilogue == NEKO_EPI_DGELU_BF16);
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  bool vec = al16(C) && (ldc % (out_bf16 ? 8 : 4) == 0);
  if (C2) vec = vec && al16(C2) && (ldc2 % 8 == 0);
  if (C3) vec = vec && al16(C3) && (ldc3 % 8 == 0);
  if (bias) vec = vec && al16(bias);
  if (aux) vec = vec && al16(aux) && (ld_aux % (epilogue == NEKO_EPI_DGELU_BF16 ? 8 : 4) == 0);
  p.vec_ok = vec ? 1 : 0;

  // outputs through TMA when every output tensor is 16-byte aligned with a 16-byte-multiple pitch
  auto tma_ok = [&](const void* q, long long ld, int esz) { return q == nullptr || (al16(q) && (ld * esz) % 16 == 0); };
  const int c_esz = out_bf16 ? 2 : 4;
  p.tma_store = (tma_ok(C, ldc, c_esz) && tma_ok(C2, ldc2, 2) && tma_ok(C3, ldc3, 2)) ? 1 : 0;
  if (getenv("NEKO_GEMM_DIRECT_STORE")) p.tma_store = 0;
  // the auxiliary operand of the residual / GELU' epilogues through TMA boxes (same staging slots as the output)
  static const bool no_tma_aux = getenv("NEKO_GEMM_NO_TMA_AUX") != nullptr;
  p.tma_aux = 0;
  if (p.tma_store && !no_tma_aux && p.splits == 1 && (epilogue == NEKO_EPI_RESID_F32 || epilogue == NEKO_EPI_DGELU_BF16)) {
    const int aesz = (epilogue == NEKO_EPI_RESID_F32) ? 4 : 2;
    if (tma_ok(aux, ld_aux, aesz) && (bias == nullptr || al16(bias))) p.tma_aux = 1;
  }
  // stream-K (see WorkIter): worth it when the tile count is a poor multiple of the worker count -- the N = 768 projections and
  // dgrads at the cfg2 token count run 90 pair tiles on 74 pairs, i.e. two rounds for 1.2 rounds of work
  p.streamk = 0; p.sk_acc = nullptr; p.sk_flags = nullptr;
  {
    const long long workers = p.pair ? sms / 2 : sms;
    const long long tiles_sk = mb_ * ((N + p.BN - 1) / p.BN);
    const long long tm = p.pair ? 2 * BM : BM;
    const long long rounds = (tiles_sk + workers - 1) / workers;
    const long long acc_bytes = workers * tm * p.BN * 4;
    const long long need = acc_bytes + 2 * workers * 4;
    const int sk_env = getenv("NEKO_GEMM_STREAMK") ? atoi(getenv("NEKO_GEMM_STREAMK")) : -1;
    bool want = p.splits == 1 && p.tma_store && epilogue != NEKO_EPI_F32 && p.BN != 192 && tiles_sk >= workers && kblocks >= 8 &&
                tiles_sk % workers != 0 && (double)(rounds * workers) >= 1.12 * (double)tiles_sk && rounds <= 4;
    if (sk_env == 0) want = false;
    if (sk_env < 0) want = false;          // default off until measured (NEKO_GEMM_STREAMK=1 enables)
    if (deterministic) want = false;
    if (want && gd->workspace && gd->workspace_bytes >= need && (reinterpret_cast<uintptr_t>(gd->workspace) & 127) == 0) {
      p.sk_acc = static_cast<float*>(gd->workspace);
      p.sk_flags = reinterpret_cast<unsigned*>(static_cast<char*>(gd->workspace) + acc_bytes);
      p.streamk = 1;
    }
  }
  // epilogue warps: 16 where the epilogue, not the main loop, bounds the launch (NEKO_GEMM_EPI16=0/1 forces; BN = 192 has no
  // 4-way column split)
  const int epi16_env = getenv("NEKO_GEMM_EPI16") ? atoi(getenv("NEKO_GEMM_EPI16")) : -1;   // read per call: tools/gemm_sweep.py flips it
  bool epi16 = (epilogue == NEKO_EPI_GELU_BF16);   // measured (profiles/r02_gemm_epi16_sweep.txt): 58 -> 54 us for c_fc, neutral or worse elsewhere
  if (epi16_env >= 0) epi16 = epi16_env != 0;
  if (p.BN == 192) epi16 = false;
  pl.epi16 = epi16 ? 1 : 0;
  return NEKO_OK;
}

}  // namespace neko

extern "C" int neko_gemm_plan(const neko_gemm_desc* gd, neko_gemm_plan_info* out) {
  using namespace neko;
  NEKO_REQUIRE(out != nullptr, "gemm_plan: null output");
  GemmPlan pl;
  const int rc = plan_gemm(gd, pl);
  if (rc != NEKO_OK) return rc;
  out->BN = pl.p.BN;
  out->pair = pl.p.pair;
  out->splits = pl.p.splits;
  out->epi_warps = pl.epi16 ? 16 : 8;
  out->streamk = pl.p.streamk;
  out->tma_store = pl.p.tma_store;
  out->tma_aux = pl.p.tma_aux;
  out->vec_ok = pl.p.vec_ok;
  out->n_fast = pl.p.n_fast;
  out->stages = pl.p.stages;
  return NEKO_OK;
}

extern "C" int neko_gemm(const neko_gemm_desc* gd, void* stream) {
  using namespace neko;
  GemmPlan pl;
  int rc = plan_gemm(gd, pl);
  if (rc != NEKO_OK) return rc;
  GemmParams& p = pl.p;
  const int M = p.M, N = p.N, K = p.K, flags = p.flags;
  const bool out_bf16 = (p.epi == NEKO_EPI_BF16 || p.epi == NEKO_EPI_GELU_BF16 || p.epi == NEKO_EPI_DGELU_BF16);
  if (p.splits > 1 && !p.accumulate) {  // (also correct for the reduce-add TMA path)
    // partial sums are RED-added: start from zero
    cudaError_t e = cudaMemset2DAsync(p.C, (size_t)p.ldc * sizeof(float), 0, (size_t)N * sizeof(float), (size_t)M, as_stream(stream));
    if (e != cudaSuccess) return check_cuda(e, "cudaMemset2DAsync(gemm split-K)");
  }
  CUtensorMap ma, mb, mc, mc2, mc3, maux;
  memset(&mc, 0, sizeof(mc)); memset(&mc2, 0, sizeof(mc2)); memset(&mc3, 0, sizeof(mc3)); memset(&maux, 0, sizeof(maux));
  if (p.tma_aux) {
    rc = make_map(&maux, p.aux, (unsigned long long)N, (unsigned long long)M, (unsigned long long)p.ld_aux, 32, 32, p.epi == NEKO_EPI_RESID_F32 ? 2 : 3);
    if (rc != NEKO_OK) return rc;
  }
  if (p.tma_store) {
    const int ckind = out_bf16 ? ((flags & NEKO_GEMM_C_F16) ? 4 : 3) : 2;
    rc = make_map(&mc, p.C, (unsigned long long)N, (unsigned long long)M, (unsigned long long)p.ldc, 32, 32, ckind);
    if (rc != NEKO_OK) return rc;
    if (p.C2) {
      rc = make_map(&mc2, p.C2, (unsigned long long)N, (unsigned long long)M, (unsigned long long)p.ldc2, 32, 32, (flags & NEKO_GEMM_C2_F16) ? 4 : 3);
      if (rc != NEKO_OK) return rc;
    }
    if (p.C3) {
      rc = make_map(&mc3, p.C3, (unsigned long long)N, (unsigned long long)M, (unsigned long long)p.ldc3, 32, 32, 3);
      if (rc != NEKO_OK) return rc;
    }
  }
  CUtensorMap mws;
  memset(&mws, 0, sizeof(mws));
  if (p.streamk) {
    const long long workers = p.pair ? pl.sms / 2 : pl.sms, tm = p.pair ? 2 * BM : BM;
    rc = make_map(&mws, p.sk_acc, (unsigned long long)p.BN, (unsigned long long)(workers * tm), (unsigned long long)p.BN, 32, 32, 2);
    if (rc != NEKO_OK) return rc;
  }
  const int bnl = p.pair ? p.BN / 2 : p.BN;  // B rows staged per CTA
  if (!p.a_mn) rc = make_map(&ma, gd->A, (unsigned long long)K, (unsigned long long)M, (unsigned long long)gd->lda, BK, BM, (flags & NEKO_GEMM_A_F16) ? 1 : 0);
  else         rc = make_map(&ma, gd->A, (unsigned long long)M, (unsigned long long)K, (unsigned long long)gd->lda, 64, BK, (flags & NEKO_GEMM_A_F16) ? 1 : 0);
  if (rc != NEKO_OK) return rc;
  if (!p.b_mn) rc = make_map(&mb, gd->B, (unsigned long long)K, (unsigned long long)N, (unsigned long long)gd->ldb, BK, (unsigned)bnl, (flags & NEKO_GEMM_B_F16) ? 1 : 0);
  else         rc = make_map(&mb, gd->B, (unsigned long long)N, (unsigned long long)K, (unsigned long long)gd->ldb, 64, BK, (flags & NEKO_GEMM_B_F16) ? 1 : 0);
  if (rc != NEKO_OK) return rc;

  const size_t smem = (size_t)p.stages * pl.stage_bytes + STAGING_BYTES + 1024 /*alignment slack*/ + 512 /*barriers*/;
  static std::once_flag attr_once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once, [] {
    const void* fns[] = {(const void*)gemm_tcgen05_kernel<false, 8>, (const void*)gemm_tcgen05_kernel<true, 8>,
                         (const void*)gemm_tcgen05_kernel<false, 16>, (const void*)gemm_tcgen05_kernel<true, 16>};
    for (const void* f : fns)
      if (attr_err == cudaSuccess) attr_err = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BUDGET);
  });
  if (attr_err != cudaSuccess) return check_cuda(attr_err, "cudaFuncSetAttribute(gemm)");
  const bool epi16 = pl.epi16 != 0;
  const int sms = pl.sms;
  const int threads = 64 + 32 * (epi16 ? 16 : 8);
  const long long units = pl.mb * ((N + p.BN - 1) / p.BN) * p.splits;   // stream-K: tiles >= workers, so the grid below is the full one
  if (p.pair) {
    const int pairs = sms / 2;
    const int grid = 2 * (int)(units < pairs ? units : pairs);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = as_stream(stream);
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 2 : 1;
    cudaError_t e = epi16 ? cudaLaunchKernelEx(&cfg, gemm_tcgen05_kernel<true, 16>, ma, mb, mc, mc2, mc3, maux, mws, p)
                          : cudaLaunchKernelEx(&cfg, gemm_tcgen05_kernel<true, 8>, ma, mb, mc, mc2, mc3, maux, mws, p);
    if (e != cudaSuccess) return check_cuda(e, "cudaLaunchKernelEx(gemm pair)");
  } else {
    const int grid = (int)(units < sms ? units : sms);
    cudaError_t e = epi16 ? launch_pdl(gemm_tcgen05_kernel<false, 16>, dim3(grid), dim3(threads), smem, as_stream(stream), ma, mb, mc, mc2, mc3, maux, mws, p)
                          : launch_pdl(gemm_tcgen05_kernel<false, 8>, dim3(grid), dim3(threads), smem, as_stream(stream), ma, mb, mc, mc2, mc3, maux, mws, p);
    if (e != cudaSuccess) return check_cuda(e, "cudaLaunchKernelEx(gemm)");
  }
  NEKO_LAUNCH_CHECK("gemm_tcgen05_kernel");
  return NEKO_OK;
}
