// Causal self-attention forward on the 5th-generation tensor cores (tcgen05 + TMEM + TMA) for head dims 32 and 64.
//
// Same contract as attn_fwd_kernel in attention.cu (Attention._attn, trajectory_gpt2.py:163-188: keys in
// [first_valid[b], query], padded rows written as zeros, lse per row); this is the path neko_attention_fwd takes when the
// shape allows it, the mma.sync kernel stays as the fallback (head dims 16 / 128, odd head counts at dh = 32).
//
// One CTA owns 128 queries of 64 feature columns of qkv: ONE head at dh = 64, a PAIR of heads at dh = 32 -- a 64-column
// TMA box is exactly one 128-byte swizzle row, and the two heads are addressed inside it by advancing the UMMA
// descriptor start by 64 bytes, the same mechanism as a K step.  Per 128-key tile and head:
//     S = Q K^T          tcgen05.mma  M=128 N=128 K=dh      (Q, K tiles K-major in shared memory, S in TMEM)
//     softmax            one THREAD per query row: tcgen05.ld of its TMEM lane, max / exp2 / sum in registers, no shuffles
//     P -> smem          bf16, written directly in the K-major 128B-swizzled UMMA layout
//     O_tile = P V       tcgen05.mma  M=128 N=dh K=128      (V tile MN-major as it lies in qkv), O_tile in TMEM
//     o = o * corr + O_tile   in registers (dh floats per thread): exact online-softmax rescaling
// Warp roles: 4 softmax warps per head (one per TMEM lane quarter), one TMA producer warp (double-buffered K/V), one MMA
// issuer warp.  While one head of the pair runs its softmax, the tensor pipe works on the other.
#include <stdlib.h>

#include "common.cuh"
#include "dropout.cuh"
#include "tcgen05.cuh"

namespace neko {

constexpr int ATC_BLK = 128;                       // queries per work item = keys per tile
constexpr int ATC_TILE = ATC_BLK * 128;            // bytes of one [128 rows x 64 bf16] operand tile
constexpr int ATC_NST = 3;                         // K/V ring depth

// Persistent: one CTA per SM walks work items (query tile, batch, head group), heaviest (latest) query tiles first.  The TMA
// producer runs ahead through a double-buffered Q slot and a 3-deep K/V ring, so the loads of the next item are in
// flight while the current one is in its softmax; TMEM, barriers and the tensor map are set up once per CTA.
template <int DH, bool DROP>
__global__ void __launch_bounds__(128 * (64 / DH) + 64, 1)
attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap map_qkv, const int32_t* __restrict__ first_valid, bf16* __restrict__ out,
                   bf16* __restrict__ out2, float* __restrict__ lse, int B, int S, int S_valid, int H, float scale_log2, int out_f16,
                   DropCfg drop) {
  constexpr int HEADS = 64 / DH;                   // heads per work item
  constexpr int NSW = 4 * HEADS;                   // softmax warps
  constexpr uint32_t TMEM_COLS = (HEADS * (128 + DH) > 256) ? 512u : 256u;
  extern __shared__ __align__(1024) uint8_t atc_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(atc_raw) + 1023) & ~(uintptr_t)1023);
  // tiles: Q[2] | K[NST] | V[NST] | P[HEADS][2]
  const uint32_t sQ0 = smem_u32(smem);
  const uint32_t sK0 = sQ0 + 2 * ATC_TILE, sV0 = sK0 + ATC_NST * ATC_TILE, sP0 = sV0 + ATC_NST * ATC_TILE;
  constexpr int P_TILE0 = 2 + 2 * ATC_NST;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (P_TILE0 + 2 * HEADS) * ATC_TILE);
  const uint32_t bar0 = smem_u32(bars);
  auto q_full = [&](int s) { return bar0 + 8u * s; };
  auto q_empty = [&](int s) { return bar0 + 8u * (2 + s); };
  auto kv_full = [&](int s) { return bar0 + 8u * (4 + s); };
  auto kv_empty = [&](int s) { return bar0 + 8u * (4 + ATC_NST + s); };
  auto s_full = [&](int h) { return bar0 + 8u * (4 + 2 * ATC_NST + h); };
  auto p_full = [&](int h) { return bar0 + 8u * (6 + 2 * ATC_NST + h); };
  auto o_full = [&](int h) { return bar0 + 8u * (8 + 2 * ATC_NST + h); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 10 + 2 * ATC_NST);

  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = H * DH;
  const int HP = H / HEADS;                        // head groups
  const int nq = (S + ATC_BLK - 1) / ATC_BLK;
  const int per_q = B * HP;
  const int n_items = nq * per_q;

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_qkv) : "memory");
    for (int s = 0; s < 2; ++s) { mbar_init(q_full(s), 1); mbar_init(q_empty(s), 1); }
    for (int s = 0; s < ATC_NST; ++s) { mbar_init(kv_full(s), 1); mbar_init(kv_empty(s), 1); }
    for (int h = 0; h < HEADS; ++h) { mbar_init(s_full(h), 1); mbar_init(p_full(h), 4); mbar_init(o_full(h), 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == NSW + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  pdl_wait();

  // work item -> (query tile, batch, head group); every role evaluates the same pure function
  struct Item { int b, hp, q0, lo, j_begin, nj; };
  auto item_at = [&](int id) {
    Item it;
    const int qt = nq - 1 - id / per_q;            // latest (heaviest) query tiles first
    const int r = id % per_q;
    it.b = r / HP; it.hp = r - it.b * HP;
    it.q0 = qt * ATC_BLK;
    it.lo = __ldg(first_valid + it.b);
    const int q_hi = min(it.q0 + ATC_BLK, S_valid);
    const bool live = (q_hi > it.lo) && (q_hi > it.q0);
    it.j_begin = (it.lo / ATC_BLK) * ATC_BLK;
    it.nj = live ? (q_hi - it.j_begin + ATC_BLK - 1) / ATC_BLK : 0;
    return it;
  };

  if (warp == NSW) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int qi = 0, t = 0;                           // live items / key tiles handled so far by this CTA
      for (int id = blockIdx.x; id < n_items; id += gridDim.x) {
        const Item it = item_at(id);
        if (it.nj == 0) continue;
        const int row_base = it.b * S, c0 = it.hp * 64;
        mbar_wait(q_empty(qi & 1), (uint32_t)(((qi >> 1) & 1) ^ 1));
        mbar_expect_tx(q_full(qi & 1), ATC_TILE);
        tma_load_2d(sQ0 + (qi & 1) * ATC_TILE, &map_qkv, q_full(qi & 1), c0, row_base + it.q0);
        ++qi;
        for (int jj = 0; jj < it.nj; ++jj, ++t) {
          const int st = t % ATC_NST;
          mbar_wait(kv_empty(st), (uint32_t)(((t / ATC_NST) & 1) ^ 1));
          mbar_expect_tx(kv_full(st), 2 * ATC_TILE);
          tma_load_2d(sK0 + st * ATC_TILE, &map_qkv, kv_full(st), d + c0, row_base + it.j_begin + jj * ATC_BLK);
          tma_load_2d(sV0 + st * ATC_TILE, &map_qkv, kv_full(st), 2 * d + c0, row_base + it.j_begin + jj * ATC_BLK);
        }
      }
    }
  } else if (warp == NSW + 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      // fp32 accumulate, bf16 x bf16; S: both operands K-major, N = 128; PV: B (= V) MN-major, N = DH
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      const uint32_t idesc_o = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(DH >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      auto issue_s = [&](uint32_t sq, int st, int h) {
        const uint32_t sk = sK0 + st * ATC_TILE;
#pragma unroll
        for (int ks = 0; ks < DH / 16; ++ks) {
          const uint32_t off = (uint32_t)(h * DH * 2 + ks * 32);   // inside the 128-byte swizzle row
          tc_mma_bf16(tmem_base + (uint32_t)(h * 128), make_smem_desc(sq + off, 16, 1024), make_smem_desc(sk + off, 16, 1024), idesc_s,
                      ks > 0 ? 1u : 0u);
        }
        tc_commit(s_full(h));
      };
      auto issue_pv = [&](int st, int h) {
        const uint32_t sv = sV0 + st * ATC_TILE;
        const uint32_t sp = sP0 + (uint32_t)h * 2 * ATC_TILE;
#pragma unroll
        for (int ks = 0; ks < ATC_BLK / 16; ++ks) {
          const uint64_t da = make_smem_desc(sp + (uint32_t)(ks >> 2) * ATC_TILE + (uint32_t)(ks & 3) * 32, 16, 1024);
          const uint64_t db = make_smem_desc(sv + (uint32_t)ks * 2048 + (uint32_t)(h * DH * 2), 64 * 128, 1024);
          tc_mma_bf16(tmem_base + (uint32_t)(HEADS * 128 + h * DH), da, db, idesc_o, ks > 0 ? 1u : 0u);
        }
        tc_commit(o_full(h));
      };
      int qi = 0, t = 0;
      for (int id = blockIdx.x; id < n_items; id += gridDim.x) {
        const Item it = item_at(id);
        if (it.nj == 0) continue;
        const uint32_t sq = sQ0 + (qi & 1) * ATC_TILE;
        mbar_wait(q_full(qi & 1), (uint32_t)((qi >> 1) & 1));
        mbar_wait(kv_full(t % ATC_NST), (uint32_t)((t / ATC_NST) & 1));
        tc_fence_after();
        for (int h = 0; h < HEADS; ++h) issue_s(sq, t % ATC_NST, h);
        for (int jj = 0; jj < it.nj; ++jj, ++t) {
          const bool more = jj + 1 < it.nj;
          if (more) {
            mbar_wait(kv_full((t + 1) % ATC_NST), (uint32_t)(((t + 1) / ATC_NST) & 1));
            tc_fence_after();
          }
          for (int h = 0; h < HEADS; ++h) {
            mbar_wait(p_full(h), (uint32_t)(t & 1));    // P of this tile is in shared memory; S and the previous O_tile were read out
            tc_fence_after();
            issue_pv(t % ATC_NST, h);
            if (more) issue_s(sq, (t + 1) % ATC_NST, h);
          }
          tc_commit(kv_empty(t % ATC_NST));             // fires when every MMA issued so far (all readers of this stage) has completed
        }
        tc_commit(q_empty(qi & 1));
        ++qi;
      }
    }
  } else {
    // ===================== softmax warps: one thread per query row =====================
    const int h = warp >> 2, quarter = warp & 3;
    const int rl = quarter * 32 + lane;               // row inside the tile = TMEM lane
    const uint32_t t_s = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(h * 128);
    const uint32_t t_o = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(HEADS * 128 + h * DH);
    uint8_t* p_row = smem + (P_TILE0 + 2 * h) * ATC_TILE + rl * 128;
    const uint32_t dkey = DROP ? drop_key(drop) : 0u;
    int t = 0;
    for (int id = blockIdx.x; id < n_items; id += gridDim.x) {
      const Item it = item_at(id);
      const int row = it.q0 + rl;
      const int head = it.hp * HEADS + h;
      float o[DH];
#pragma unroll
      for (int i = 0; i < DH; ++i) o[i] = 0.f;
      float m = -INFINITY, l = 0.f;
      uint32_t rk = 0u;
      if (DROP) rk = drop_rowkey(dkey, (uint32_t)((it.b * H + head) * S + row));
      const int lo = it.lo;
      const bool row_dead = (row < lo) || (row >= S_valid);   // padding rows: computed on garbage, written as zeros
      for (int jj = 0; jj < it.nj; ++jj, ++t) {
        const int j0 = it.j_begin + jj * ATC_BLK;
        if (jj > 0) {   // fold the previous tile's P V (relative to the running max m) into the register accumulator
          mbar_wait(o_full(h), (uint32_t)((t - 1) & 1));
          tc_fence_after();
#pragma unroll
          for (int c = 0; c < DH / 32; ++c) {
            uint32_t v[32];
            tc_ld32(t_o + (uint32_t)(c * 32), v);
#pragma unroll
            for (int i = 0; i < 32; ++i) o[c * 32 + i] += __uint_as_float(v[i]);
          }
        }
        mbar_wait(s_full(h), (uint32_t)(t & 1));
        tc_fence_after();
        // Masking is decided per (tile, warp, 32-key chunk), warp-uniformly:
        //   general   the tile contains left padding (j0 < lo): per-element key >= lo && key <= row
        //   diagonal  j0 == q0: this warp's rows are 32*quarter + lane, so chunks c < quarter are fully visible,
        //             c == quarter is triangular (column i visible iff i <= lane), c > quarter are invisible and SKIPPED
        //   interior  no mask.  Dead rows (left padding / beyond S_valid) are not masked here: they compute on finite
        //             garbage and are zeroed at write-out.
        const bool general = j0 < lo;
        const bool diag = (j0 + ATC_BLK > it.q0);
        const int cmin = lo - j0, cmax = row - j0;        // general mode: visible columns of this row are [cmin, cmax]
        const int c_end = (diag && !general) ? quarter + 1 : 4;
        // pass 1: row maximum over the visible keys of this tile
        float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};   // independent chains: the row is up to 128 values long
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c < c_end) {
            uint32_t v[32];
            tc_ld32(t_s + (uint32_t)(c * 32), v);
            if (general) {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (c * 32 + i >= cmin && c * 32 + i <= cmax) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(v[i]));
            } else if (diag && c == quarter) {
#pragma unroll
              for (int i = 0; i < 32; ++i)
                if (i <= lane) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(v[i]));
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(v[i]));
            }
          }
        }
        const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
        const float mn = fmaxf(m, mx);
        const float ref = (mn == -INFINITY) ? 0.f : mn * scale_log2;
        const float corr = ex2_ftz(m * scale_log2 - ref);   // m = -inf -> 0
        m = mn;
        // pass 2: probabilities -> row sum, bf16 P in the UMMA K-major swizzled layout
        float sum4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint8_t* dst = p_row + (c >> 1) * ATC_TILE;   // 64 keys per swizzle atom
          if (c < c_end) {
            uint32_t v[32];
            tc_ld32(t_s + (uint32_t)(c * 32), v);
            const bool tri = diag && !general && c == quarter;
#pragma unroll
            for (int k8 = 0; k8 < 4; ++k8) {
              float p[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                p[i] = ex2_ftz(fmaf(__uint_as_float(v[8 * k8 + i]), scale_log2, -ref));
                if (general) {
                  if (!(c * 32 + 8 * k8 + i >= cmin && c * 32 + 8 * k8 + i <= cmax)) p[i] = 0.f;
                } else if (tri) {
                  if (8 * k8 + i > lane) p[i] = 0.f;
                }
                sum4[i & 3] += p[i];
              }
              if (DROP) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  float m0, m1;
                  drop_pair(rk, (uint32_t)((j0 + c * 32 + 8 * k8) >> 1) + i, drop.thr16, drop.scale, m0, m1);
                  p[2 * i] *= m0; p[2 * i + 1] *= m1;
                }
              }
              const int chunk = (c & 1) * 4 + k8;         // 16-byte chunk inside the 128-byte row
              *reinterpret_cast<uint4*>(dst + ((chunk ^ (rl & 7)) << 4)) =
                  make_uint4(pack_bf16x2(p[0], p[1]), pack_bf16x2(p[2], p[3]), pack_bf16x2(p[4], p[5]), pack_bf16x2(p[6], p[7]));
            }
          } else {   // invisible chunk above the diagonal: P = 0
#pragma unroll
            for (int k8 = 0; k8 < 4; ++k8)
              *reinterpret_cast<uint4*>(dst + ((((c & 1) * 4 + k8) ^ (rl & 7)) << 4)) = make_uint4(0u, 0u, 0u, 0u);
          }
        }
        l = l * corr + ((sum4[0] + sum4[1]) + (sum4[2] + sum4[3]));
#pragma unroll
        for (int i = 0; i < DH; ++i) o[i] *= corr;
        tc_fence_before();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // P is read by the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive(p_full(h));
      }
      if (it.nj > 0) {
        mbar_wait(o_full(h), (uint32_t)((t - 1) & 1));
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < DH / 32; ++c) {
          uint32_t v[32];
          tc_ld32(t_o + (uint32_t)(c * 32), v);
#pragma unroll
          for (int i = 0; i < 32; ++i) o[c * 32 + i] += __uint_as_float(v[i]);
        }
      }
      // write-out: dead rows (padding) -> zeros, lse = +inf so that backward sees p = 0
      if (row < S) {
        if (row_dead) l = 0.f;
        const float inv = (l > 0.f) ? 1.f / l : 0.f;
        const long long off = ((long long)it.b * S + row) * d + head * DH;
        uint4* ob = reinterpret_cast<uint4*>(out + off);
#pragma unroll
        for (int k8 = 0; k8 < DH / 8; ++k8)
          ob[k8] = make_uint4(pack_16x2(o[8 * k8] * inv, o[8 * k8 + 1] * inv, out_f16 != 0), pack_16x2(o[8 * k8 + 2] * inv, o[8 * k8 + 3] * inv, out_f16 != 0),
                              pack_16x2(o[8 * k8 + 4] * inv, o[8 * k8 + 5] * inv, out_f16 != 0), pack_16x2(o[8 * k8 + 6] * inv, o[8 * k8 + 7] * inv, out_f16 != 0));
        if (out2) {
          uint4* ob2 = reinterpret_cast<uint4*>(out2 + off);
#pragma unroll
          for (int k8 = 0; k8 < DH / 8; ++k8)
            ob2[k8] = make_uint4(pack_bf16x2(o[8 * k8] * inv, o[8 * k8 + 1] * inv), pack_bf16x2(o[8 * k8 + 2] * inv, o[8 * k8 + 3] * inv),
                                 pack_bf16x2(o[8 * k8 + 4] * inv, o[8 * k8 + 5] * inv), pack_bf16x2(o[8 * k8 + 6] * inv, o[8 * k8 + 7] * inv));
        }
        lse[((long long)it.b * H + head) * S + row] = (l > 0.f) ? (m * scale_log2 + log2f(l)) * 0.6931471805599453f : INFINITY;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == NSW + 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

template <int DH, bool DROP>
static int launch_fwd_tc(const CUtensorMap& map, const int32_t* fv, bf16* out, bf16* out2, float* lse, int B, int S, int S_valid, int H,
                         int out_f16, DropCfg drop, cudaStream_t st) {
  constexpr int HEADS = 64 / DH;
  const size_t smem = (size_t)(2 + 2 * ATC_NST + 2 * HEADS) * ATC_TILE + 256 + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_fwd_tc_kernel<DH, DROP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(attn_fwd_tc)");
    attr_set = true;
  }
  const float scale_log2 = 1.4426950408889634f / sqrtf((float)DH);
  const long long items = (long long)((S + ATC_BLK - 1) / ATC_BLK) * B * (H / HEADS);
  const int grid = (int)(items < sm_count() ? items : sm_count());
  cudaError_t e = launch_pdl(attn_fwd_tc_kernel<DH, DROP>, dim3(grid), dim3(128 * HEADS + 64), smem, st, map, fv, out, out2, lse, B, S, S_valid, H,
                             scale_log2, out_f16, drop);
  if (e != cudaSuccess) return check_cuda(e, "cudaLaunchKernelEx(attn_fwd_tc)");
  NEKO_LAUNCH_CHECK("attn_fwd_tc_kernel");
  return NEKO_OK;
}

// true when neko_attention_fwd takes the tcgen05 path for these arguments (host only, launches nothing)
bool attention_fwd_tc_eligible(const void* qkv, const void* out, const void* out2, int H, int dh) {
  // Opt-in (NEKO_ATTN_TC=1, read per call so tests can toggle it): at the BASELINE head dim 32 the op is bound by exp /
  // barrier latency, not by the tensor pipe, and the mma.sync kernel with 4-6 resident CTAs per SM is faster
  // (41 us vs 57 us per launch at cfg2, profiles/r01_ncu_attn_tc.txt; DESIGN.md section 4).
  const char* on = getenv("NEKO_ATTN_TC");
  if (!(on && atoi(on) != 0)) return false;
  if (!(dh == 64 || (dh == 32 && H % 2 == 0))) return false;
  const int d = H * dh;
  return !((reinterpret_cast<uintptr_t>(qkv) & 15) || (reinterpret_cast<uintptr_t>(out) & 15) || (out2 && (reinterpret_cast<uintptr_t>(out2) & 15)) ||
           d % 8);
}

// returns NEKO_OK when the tensor-core path ran, 1 when the shape is not covered (caller falls back), < 0 on error
int attention_fwd_tc(const bf16* qkv, const int32_t* fv, bf16* out, bf16* out2, float* lse, int B, int S, int S_valid, int H, int dh, int out_f16,
                     DropCfg drop, cudaStream_t st) {
  if (!attention_fwd_tc_eligible(qkv, out, out2, H, dh)) return 1;
  const int d = H * dh;
  CUtensorMap map;
  int rc = make_map(&map, qkv, 3ull * d, (unsigned long long)B * S, 3ull * d, 64, ATC_BLK, 0);
  if (rc != NEKO_OK) return rc;
  if (dh == 32) return drop.seed ? launch_fwd_tc<32, true>(map, fv, out, out2, lse, B, S, S_valid, H, out_f16, drop, st)
                                 : launch_fwd_tc<32, false>(map, fv, out, out2, lse, B, S, S_valid, H, out_f16, drop, st);
  return drop.seed ? launch_fwd_tc<64, true>(map, fv, out, out2, lse, B, S, S_valid, H, out_f16, drop, st)
                   : launch_fwd_tc<64, false>(map, fv, out, out2, lse, B, S, S_valid, H, out_f16, drop, st);
}

}  // namespace neko
