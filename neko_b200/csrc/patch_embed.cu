// Image patch embedding: ImageEmbedding.forward / ResidualBlock_V2 (embeddings.py:28-61,111-131).
//
//   x = (img/255*2 - 1)/sqrt(p)  ->  patchify 16x16  ->  h = conv1(GELU(x)) 3->C, 3x3, per-patch zero pad
//   -> GroupNorm(groups) -> GELU -> conv2 C->3 -> x + .   -> flatten (c p1 p2) -> 16-bit row of the projection GEMM
//
// One CTA (8 warps) processes one patch at a time in a persistent loop with the weights resident in shared memory; the
// C x 256 intermediate never leaves the SM (the unfused torch path writes / re-reads 131 KB per patch four times).
// Both convolutions and all their gradients are small GEMMs on the tensor cores (mma.sync m16n8k16 bf16, fp32
// accumulate) over im2col operands built in shared memory:
//   conv1      H[px][c]      = colX[px][n] . W1[c][n]            n = (ci,ky,kx) + a ones column that carries the bias
//   conv2      out[px][co]  += h2pad[px+tap][c] . W2[co][c][tap] nine shifted GEMMs over a zero-bordered pixel grid
//   d conv2    dh2[px][c]    = colY[px][n] . W2r[c][n]           n = (co,tap), colY = im2col of dY
//   wgrads     dW2r[n][c]   += colY^T . h2      dW1[c][n] += dh^T . colX     (K = 256 pixels; ones column => db1)
// GroupNorm statistics / affine gradients are reduced with warp shuffles and per-warp shared-memory slots.
#include "common.cuh"
#include "ordered.cuh"

namespace neko {

constexpr int PE_P = 16;            // patch edge
constexpr int PE_PX = 256;          // pixels per patch
constexpr int PE_C = 128;           // mid channels (train.py always passes 128)
constexpr int PE_THREADS = 256;     // 8 warps: warp w owns pixels [32w, 32w+32) = image rows 2w, 2w+1
constexpr int PE_PAD = 18;          // padded edge
constexpr int PE_KP = 40;           // pitch of the K=32 im2col / weight tiles (80 bytes: conflict-free ldmatrix)
constexpr int PE_CP = PE_C + 8;     // pitch of 128-channel tiles
constexpr int PE_HP2 = 64 + 8;      // pitch of half-channel tiles (backward)

// gradient outputs of the backward
struct PatchGrads {
  float *dw1, *db1, *dgw, *dgb, *dw2, *db2;
};

struct PatchArgs {
  const void* images;
  int is_u8, n_img, Himg, Wimg, n_h, n_w, groups;
  const float *w1, *b1, *gw, *gb, *w2, *b2;
  uint16_t* out;        // fwd: [P,768] fp16
  uint16_t* out_bf;     // fwd: optional bf16 copy (wgrad operand)
  float* stats;         // [P, groups, 2]
  // backward only
  const bf16* dout;     // [P,768]
  PatchGrads grad;
};

// F16: the forward runs its operands in fp16 (values are O(1), 3 more mantissa bits); the backward, whose dY operand needs
// bf16's range, runs everything in bf16.
template <bool F16 = false>
__device__ __forceinline__ void pe_mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (F16)
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  else
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void pe_ldsm4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void pe_ldsm4t(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void pe_ldsm2(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}

// bf16 tile in shared memory with a run-time pitch (elements)
struct STile {
  uint32_t base;
  int pitch;
  __device__ __forceinline__ uint32_t addr(int r, int c) const { return base + (uint32_t)(r * pitch + c) * 2u; }
};
// A fragment (16 x 16) of a tile stored [m][k]
__device__ __forceinline__ void fa_mk(const STile& t, int m0, int k0, int lane, uint32_t (&a)[4]) {
  pe_ldsm4(t.addr(m0 + (lane & 15), k0 + ((lane >> 4) << 3)), a);
}
// A fragment of a tile stored [k][m] (transposed load)
__device__ __forceinline__ void fa_km(const STile& t, int k0, int m0, int lane, uint32_t (&a)[4]) {
  pe_ldsm4t(t.addr(k0 + (lane & 7) + (((lane >> 4) & 1) << 3), m0 + (((lane >> 3) & 1) << 3)), a);
}
// B fragments of two adjacent n-tiles from a tile stored [n][k]
__device__ __forceinline__ void fb_nk(const STile& t, int n0, int k0, int lane, uint32_t (&b)[4]) {
  pe_ldsm4(t.addr(n0 + (lane & 7) + ((lane >> 4) << 3), k0 + (((lane >> 3) & 1) << 3)), b);
}
// B fragments of two adjacent n-tiles from a tile stored [k][n] (transposed load)
__device__ __forceinline__ void fb_kn(const STile& t, int k0, int n0, int lane, uint32_t (&b)[4]) {
  pe_ldsm4t(t.addr(k0 + (lane & 7) + (((lane >> 3) & 1) << 3), n0 + ((lane >> 4) << 3)), b);
}

// ---- shared staging common to forward and backward -------------------------------------------------
// load + normalise one patch: xin (fp32, standard pixel order) and gx = gelu(x) on a zero-bordered 18x18 grid
__device__ __forceinline__ void pe_load_patch(const PatchArgs& a, float* gx, float* xin, int patch) {
  const int npp = a.n_h * a.n_w;
  const int n = patch / npp, r = patch - n * npp;
  const int ph = r / a.n_w, pw = r - ph * a.n_w;
  const int t = threadIdx.x, y = t >> 4, x = t & 15;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const size_t idx = (((size_t)n * 3 + c) * a.Himg + (size_t)ph * PE_P + y) * a.Wimg + (size_t)pw * PE_P + x;
    float v = a.is_u8 ? (float)reinterpret_cast<const uint8_t*>(a.images)[idx] : reinterpret_cast<const float*>(a.images)[idx];
    v = v / 255.0f * 2.0f - 1.0f;   // embeddings.py:40
    v = v / 4.0f;                   // / sqrt(patch_size), :41
    if (xin) xin[c * PE_PX + t] = v;
    gx[(c * PE_PAD + y + 1) * PE_PAD + x + 1] = gelu_erf(v);
  }
}
// im2col row of this thread's pixel: col[px][n] = grid[c3][y + dy(tap)][x + dx(tap)], n = c3*9 + tap; entry 27 = `one`
template <bool FLIP, bool F16 = false>
__device__ __forceinline__ void pe_im2col_row(const float* grid, bf16* col, float one) {
  const int t = threadIdx.x, y = t >> 4, x = t & 15;
  uint32_t w[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    float v[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int n = 2 * i + h;
      if (n < 27) {
        const int c3 = n / 9, tap = n - c3 * 9, ky = tap / 3, kx = tap - ky * 3;
        // forward conv reads in[y+ky-1][x+kx-1]; its transpose reads dY[y-ky+1][x-kx+1]   (grid has a 1-pixel border)
        v[h] = FLIP ? grid[(c3 * PE_PAD + y - ky + 2) * PE_PAD + x - kx + 2] : grid[(c3 * PE_PAD + y + ky) * PE_PAD + x + kx];
      } else {
        v[h] = (n == 27) ? one : 0.f;
      }
    }
    w[i] = F16 ? pack_f16x2(v[0], v[1]) : pack_bf16x2(v[0], v[1]);
  }
  uint4* dst = reinterpret_cast<uint4*>(col + t * PE_KP);
#pragma unroll
  for (int i = 0; i < 4; ++i) dst[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
}

// GroupNorm group of accumulator column (n-tile nt, lane quad index q): columns nt*8 + 2q, +1 -> group (nt*8 + 2q) / gs
// (gs = 4 channels per group with the reference's 32 groups over 128 channels; any gs that is a multiple of 2 works)

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
// Two CTAs per SM.  conv1 is cheap (K = 32), so it runs twice instead of holding the 256 x 128 tile in registers:
// pass A accumulates the GroupNorm sums, pass B recomputes 16 channels at a time, normalises, applies GELU and feeds
// the result -- already in the A-fragment layout -- straight into  Z[px][(co,tap)] += h2[px][c] W2[(co,tap)][c].
// conv2's output is then a 9-tap shifted gather of Z through shared memory.
constexpr int PE_ZP = 260;          // pitch (floats) of the transposed Z tile: conflict-free fragment stores and row reads

__global__ void __launch_bounds__(PE_THREADS, 2) patch_resblock_fwd_kernel(PatchArgs a) {
  extern __shared__ __align__(16) uint8_t pe_raw[];
  bf16* colX = reinterpret_cast<bf16*>(pe_raw);                       // [256][40]  (all forward tiles hold fp16 bit patterns)
  bf16* W1s = colX + PE_PX * PE_KP;                                    // [128][40]  (n = 27 column holds the bias)
  bf16* W2n = W1s + PE_C * PE_KP;                                      // [32][136]  W2n[co*9+tap][c], rows >= 27 zero
  float* Zs = reinterpret_cast<float*>(W2n + 32 * PE_CP);              // [32][260]  Z transposed: [(co,tap)][px]
  float* gx = Zs + 32 * PE_ZP;                                         // [3][18][18]
  float* xin = gx + 3 * PE_PAD * PE_PAD;                               // [3][256]
  float* gpart = xin + 3 * PE_PX;                                      // [8 warps][64 groups][2]
  float* gstat = gpart + 8 * 64 * 2;                                   // [64 groups][2] mean, rstd
  float* gws = gstat + 128;                                            // [128]
  float* gbs = gws + PE_C;                                             // [128]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
  const int P = a.n_img * a.n_h * a.n_w;
  const int gs = PE_C / a.groups, gshift = 31 - __clz(gs);             // channels per group: a power of two in [2, 64]
  const STile tX{(uint32_t)__cvta_generic_to_shared(colX), PE_KP}, tW1{(uint32_t)__cvta_generic_to_shared(W1s), PE_KP};
  const STile tW2{(uint32_t)__cvta_generic_to_shared(W2n), PE_CP};

  for (int i = tid; i < PE_C * PE_KP; i += PE_THREADS) {
    const int c = i / PE_KP, n = i - c * PE_KP;
    reinterpret_cast<__half*>(W1s)[i] = __float2half_rn(n < 27 ? a.w1[c * 27 + n] : (n == 27 ? a.b1[c] : 0.f));
  }
  for (int i = tid; i < 32 * PE_CP; i += PE_THREADS) {
    const int n = i / PE_CP, c = i - n * PE_CP;
    float v = 0.f;
    if (n < 27 && c < PE_C) { const int co = n / 9, tap = n - co * 9; v = a.w2[(co * PE_C + c) * 9 + tap]; }
    reinterpret_cast<__half*>(W2n)[i] = __float2half_rn(v);
  }
  for (int i = tid; i < 3 * PE_PAD * PE_PAD; i += PE_THREADS) gx[i] = 0.f;
  for (int i = tid; i < PE_C; i += PE_THREADS) { gws[i] = a.gw[i]; gbs[i] = a.gb[i]; }
  const float b2r[3] = {a.b2[0], a.b2[1], a.b2[2]};
  __syncthreads();

  for (int patch = blockIdx.x; patch < P; patch += gridDim.x) {
    pe_load_patch(a, gx, xin, patch);
    __syncthreads();
    pe_im2col_row<false, true>(gx, colX, 1.0f);
    __syncthreads();
    uint32_t ax[2][2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int k = 0; k < 2; ++k) fa_mk(tX, warp * 32 + mt * 16, k * 16, lane, ax[mt][k]);

    // conv1 (+bias) of this warp's 32 pixels for channels [16 n2, 16 n2 + 16)
    auto conv1 = [&](int n2, float (&h)[2][2][4]) {
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 4; ++e) h[mt][j][e] = 0.f;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        uint32_t b[4];
        fb_nk(tW1, n2 * 16, k * 16, lane, b);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          pe_mma<true>(h[mt][0], ax[mt][k], b[0], b[1]);
          pe_mma<true>(h[mt][1], ax[mt][k], b[2], b[3]);
        }
      }
    };

    // ---- pass A: GroupNorm sums.  Columns nt*8 + 2q, +1 of this thread belong to group (nt*8 + 2q) >> gshift ----
#pragma unroll 2
    for (int n2 = 0; n2 < 8; ++n2) {
      float h[2][2][4];
      conv1(n2, h);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int nt = 2 * n2 + j;
        float s = 0.f, ss = 0.f;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int e = 0; e < 4; ++e) { const float v = h[mt][j][e]; s += v; ss = fmaf(v, v, ss); }
        s += __shfl_xor_sync(0xffffffffu, s, 4); ss += __shfl_xor_sync(0xffffffffu, ss, 4);
        s += __shfl_xor_sync(0xffffffffu, s, 8); ss += __shfl_xor_sync(0xffffffffu, ss, 8);
        s += __shfl_xor_sync(0xffffffffu, s, 16); ss += __shfl_xor_sync(0xffffffffu, ss, 16);
        if (gs >= 4) { s += __shfl_xor_sync(0xffffffffu, s, 1); ss += __shfl_xor_sync(0xffffffffu, ss, 1); }
        if (gs >= 8) { s += __shfl_xor_sync(0xffffffffu, s, 2); ss += __shfl_xor_sync(0xffffffffu, ss, 2); }
        if (g == 0 && ((2 * q) & (min(gs, 8) - 1)) == 0) {   // one owner lane per (n-tile, group)
          float* slot = gpart + (warp * 64 + ((nt * 8 + 2 * q) >> gshift)) * 2;
          if ((nt * 8) & (gs - 1)) { slot[0] += s; slot[1] += ss; } else { slot[0] = s; slot[1] = ss; }   // gs > 8: several n-tiles per group
        }
      }
    }
    __syncthreads();
    if (tid < a.groups) {
      float s = 0.f, ss = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) { s += gpart[(w * 64 + tid) * 2]; ss += gpart[(w * 64 + tid) * 2 + 1]; }
      const float inv_n = 1.0f / (float)(gs * PE_PX);
      const float mean = s * inv_n;
      const float var = fmaxf(ss * inv_n - mean * mean, 0.f);
      const float rstd = rsqrtf(var + 1e-5f);
      gstat[2 * tid] = mean; gstat[2 * tid + 1] = rstd;
      a.stats[((size_t)patch * a.groups + tid) * 2] = mean;
      a.stats[((size_t)patch * a.groups + tid) * 2 + 1] = rstd;
    }
    __syncthreads();

    // ---- pass B: recompute 16 channels, normalise + GELU, Z += h2 . W2n^T ----
    float z[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int n = 0; n < 4; ++n)
#pragma unroll
        for (int e = 0; e < 4; ++e) z[mt][n][e] = 0.f;
#pragma unroll 2
    for (int kt = 0; kt < 8; ++kt) {
      float h[2][2][4];
      conv1(kt, h);
      uint32_t af[2][4];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int c0 = kt * 16 + j * 8 + 2 * q;
        const int grp = c0 >> gshift;
        const float mean = gstat[2 * grp], rstd = gstat[2 * grp + 1];
        const float w0 = gws[c0] * rstd, w1 = gws[c0 + 1] * rstd;
        const float o0 = fmaf(-mean, w0, gbs[c0]), o1 = fmaf(-mean, w1, gbs[c0 + 1]);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          // C fragment (rows g / g+8, columns 2q, 2q+1 of n-tile j)  ==  A fragment registers 2j (row g), 2j+1 (row g+8)
          af[mt][2 * j] = pack_f16x2(gelu_erf(fmaf(h[mt][j][0], w0, o0)), gelu_erf(fmaf(h[mt][j][1], w1, o1)));
          af[mt][2 * j + 1] = pack_f16x2(gelu_erf(fmaf(h[mt][j][2], w0, o0)), gelu_erf(fmaf(h[mt][j][3], w1, o1)));
        }
      }
#pragma unroll
      for (int n2 = 0; n2 < 2; ++n2) {
        uint32_t b[4];
        fb_nk(tW2, n2 * 16, kt * 16, lane, b);
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          pe_mma<true>(z[mt][2 * n2], af[mt], b[0], b[1]);
          pe_mma<true>(z[mt][2 * n2 + 1], af[mt], b[2], b[3]);
        }
      }
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int n = 0; n < 4; ++n)
#pragma unroll
        for (int e = 0; e < 4; ++e)
          Zs[(n * 8 + 2 * q + (e & 1)) * PE_ZP + warp * 32 + mt * 16 + g + (e >> 1) * 8] = z[mt][n][e];
    __syncthreads();
    // ---- conv2 = 9-tap shifted gather of Z, + residual + bias; thread = pixel, coalesced (c p1 p2) rows ----
    {
      const int y = tid >> 4, x = tid & 15;
      float o[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int dy = tap / 3 - 1, dx = tap % 3 - 1;
        if ((unsigned)(y + dy) < 16u && (unsigned)(x + dx) < 16u) {
#pragma unroll
          for (int co = 0; co < 3; ++co) o[co] += Zs[(co * 9 + tap) * PE_ZP + tid + dy * 16 + dx];
        }
      }
      uint16_t* orow = a.out + (size_t)patch * (3 * PE_PX);
      uint16_t* orow_b = a.out_bf ? a.out_bf + (size_t)patch * (3 * PE_PX) : nullptr;
#pragma unroll
      for (int co = 0; co < 3; ++co) {
        const float v = xin[co * PE_PX + tid] + b2r[co] + o[co];
        orow[co * PE_PX + tid] = cvt_16(v, true);
        if (orow_b) orow_b[co * PE_PX + tid] = cvt_16(v, false);
      }
    }
    // (the next iteration's writes to gx / xin / colX / gpart / Zs are each separated from this iteration's last
    //  read of the same buffer by at least one of the barriers above)
  }
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
// Slot layout of the ordered kernel's workspace (floats): dw1 [128][27] | db1 [128] | dgamma [128] | dbeta [128] | dw2 [3][128][9] | db2 [3].
constexpr int PS_DW1 = 0, PS_DB1 = PS_DW1 + PE_C * 27, PS_DGW = PS_DB1 + PE_C, PS_DGB = PS_DGW + PE_C, PS_DW2 = PS_DGB + PE_C,
              PS_DB2 = PS_DW2 + 3 * PE_C * 9, PS_SLOT = PS_DB2 + 3;
constexpr int PE_CHUNK = 8;         // patches per fixed chunk of the ordered kernel

__global__ void __launch_bounds__(PE_THREADS, 1) patch_resblock_bwd_kernel(PatchArgs a) {
#define PE_BWD_ORDERED 0
#include "patch_bwd_body.cuh"
#undef PE_BWD_ORDERED
}

// deterministic mode: see patch_bwd_body.cuh
__global__ void __launch_bounds__(PE_THREADS, 1) patch_resblock_bwd_ordered_kernel(PatchArgs a, float* ws, int n_chunks) {
#define PE_BWD_ORDERED 1
#include "patch_bwd_body.cuh"
#undef PE_BWD_ORDERED
}

static size_t patch_smem_bytes(bool bwd) {
  if (!bwd)
    return (size_t)(PE_PX * PE_KP + PE_C * PE_KP + 32 * PE_CP) * 2 +
           (size_t)(32 * PE_ZP + 3 * PE_PAD * PE_PAD + 3 * PE_PX + 8 * 64 * 2 + 128 + 2 * PE_C) * 4;
  return (size_t)(2 * PE_PX * PE_KP + 2 * PE_C * PE_KP + 2 * PE_PX * PE_HP2) * 2 +
         (size_t)(2 * 3 * PE_PAD * PE_PAD + 8 * 64 * 2 + 128 + 128 + 2 * PE_C + 8 * PE_C * 2 + 32) * 4;
}

// ---------------------------------------------------------------------------------------------
// patch position encodings
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) patch_pos_add_kernel(float* __restrict__ x, int P, int d, const int32_t* __restrict__ row_bin,
                                                            const int32_t* __restrict__ col_bin, const float* __restrict__ row_tab,
                                                            const float* __restrict__ col_tab) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= P) return;
  float4* x4 = reinterpret_cast<float4*>(x + (size_t)w * d);
  const float4* r4 = reinterpret_cast<const float4*>(row_tab + (size_t)row_bin[w] * d);
  const float4* c4 = reinterpret_cast<const float4*>(col_tab + (size_t)col_bin[w] * d);
  for (int i = lane; i < (d >> 2); i += 32) {
    float4 v = x4[i];
    const float4 r = __ldg(r4 + i), c = __ldg(c4 + i);
    v.x += r.x + c.x; v.y += r.y + c.y; v.z += r.z + c.z; v.w += r.w + c.w;
    x4[i] = v;
  }
}

__global__ void __launch_bounds__(256) patch_pos_bwd_kernel(const float* __restrict__ dx, int P, int d, const int32_t* __restrict__ row_bin,
                                                            const int32_t* __restrict__ col_bin, float* __restrict__ d_row_tab,
                                                            float* __restrict__ d_col_tab) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= P) return;
  const float* g = dx + (size_t)w * d;
  float* r = d_row_tab + (size_t)row_bin[w] * d;
  float* c = d_col_tab + (size_t)col_bin[w] * d;
  for (int i = lane; i < d; i += 32) {
    const float v = g[i];
    atomicAdd(r + i, v);
    atomicAdd(c + i, v);
  }
}

static int check_patch_args(int n_img, int Himg, int Wimg, int patch, int C, int groups) {
  NEKO_REQUIRE(patch == PE_P, "patch_resblock: only patch_size 16 is implemented (got %d)", patch);
  NEKO_REQUIRE(C == PE_C, "patch_resblock: only resid_mid_channels 128 is implemented (got %d)", C);
  NEKO_REQUIRE(groups > 0 && groups <= 64 && C % groups == 0 && (C / groups) % 2 == 0 && 64 % (C / groups) == 0 && ((C / groups) & (C / groups - 1)) == 0,
               "patch_resblock: unsupported num_groups %d", groups);
  NEKO_REQUIRE(n_img > 0 && Himg > 0 && Wimg > 0 && Himg % patch == 0 && Wimg % patch == 0, "Image dimensions must be divisible by patch size");
  return NEKO_OK;
}

// argument checks and PatchArgs of both backward entry points (who: the entry point the error names)
static int patch_bwd_args(PatchArgs& a, const char* who, const void* images, int is_u8, int n_img, int Himg, int Wimg, int patch, int C,
                          int groups, const float* conv1_w, const float* conv1_b, const float* gn_w, const float* gn_b, const float* conv2_w,
                          const float* gn_stats, const uint16_t* d_patches_bf16, float* d_conv1_w, float* d_conv1_b, float* d_gn_w,
                          float* d_gn_b, float* d_conv2_w, float* d_conv2_b) {
  NEKO_REQUIRE(images && conv1_w && conv1_b && gn_w && gn_b && conv2_w && gn_stats && d_patches_bf16 && d_conv1_w && d_conv1_b && d_gn_w &&
               d_gn_b && d_conv2_w && d_conv2_b, "%s: null pointer", who);
  const int rc = check_patch_args(n_img, Himg, Wimg, patch, C, groups);
  if (rc != NEKO_OK) return rc;
  a = PatchArgs{};
  a.images = images; a.is_u8 = is_u8; a.n_img = n_img; a.Himg = Himg; a.Wimg = Wimg; a.n_h = Himg / patch; a.n_w = Wimg / patch;
  a.groups = groups; a.w1 = conv1_w; a.b1 = conv1_b; a.gw = gn_w; a.gb = gn_b; a.w2 = conv2_w; a.b2 = nullptr;
  a.stats = const_cast<float*>(gn_stats); a.dout = reinterpret_cast<const bf16*>(d_patches_bf16);
  a.grad = PatchGrads{d_conv1_w, d_conv1_b, d_gn_w, d_gn_b, d_conv2_w, d_conv2_b};
  return NEKO_OK;
}

}  // namespace neko

extern "C" {

int neko_patch_resblock_fwd(const void* images, int is_u8, int n_img, int Himg, int Wimg, int patch, int C, int groups,
                            const float* conv1_w, const float* conv1_b, const float* gn_w, const float* gn_b, const float* conv2_w,
                            const float* conv2_b, uint16_t* patches_out, uint16_t* patches_out_bf16, float* gn_stats, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(images && conv1_w && conv1_b && gn_w && gn_b && conv2_w && conv2_b && patches_out && gn_stats, "patch_resblock_fwd: null pointer");
  int rc = check_patch_args(n_img, Himg, Wimg, patch, C, groups);
  if (rc != NEKO_OK) return rc;
  PatchArgs a{};
  a.images = images; a.is_u8 = is_u8; a.n_img = n_img; a.Himg = Himg; a.Wimg = Wimg; a.n_h = Himg / patch; a.n_w = Wimg / patch;
  a.groups = groups; a.w1 = conv1_w; a.b1 = conv1_b; a.gw = gn_w; a.gb = gn_b; a.w2 = conv2_w; a.b2 = conv2_b;
  a.out = patches_out; a.out_bf = patches_out_bf16; a.stats = gn_stats;
  const size_t smem = patch_smem_bytes(false);
  cudaError_t e = cudaFuncSetAttribute(patch_resblock_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(patch_fwd)");
  const int P = n_img * a.n_h * a.n_w;
  const int grid = P < 2 * sm_count() ? P : 2 * sm_count();   // two resident CTAs per SM
  patch_resblock_fwd_kernel<<<grid, PE_THREADS, smem, as_stream(stream)>>>(a);
  NEKO_LAUNCH_CHECK("patch_resblock_fwd_kernel");
  return NEKO_OK;
}

int neko_patch_resblock_bwd(const void* images, int is_u8, int n_img, int Himg, int Wimg, int patch, int C, int groups,
                            const float* conv1_w, const float* conv1_b, const float* gn_w, const float* gn_b, const float* conv2_w,
                            const float* gn_stats, const uint16_t* d_patches_bf16, float* d_conv1_w, float* d_conv1_b, float* d_gn_w,
                            float* d_gn_b, float* d_conv2_w, float* d_conv2_b, void* stream) {
  using namespace neko;
  PatchArgs a;
  const int rc = patch_bwd_args(a, "patch_resblock_bwd", images, is_u8, n_img, Himg, Wimg, patch, C, groups, conv1_w, conv1_b, gn_w, gn_b,
                                conv2_w, gn_stats, d_patches_bf16, d_conv1_w, d_conv1_b, d_gn_w, d_gn_b, d_conv2_w, d_conv2_b);
  if (rc != NEKO_OK) return rc;
  const size_t smem = patch_smem_bytes(true);
  cudaError_t e = cudaFuncSetAttribute(patch_resblock_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(patch_bwd)");
  const int P = n_img * a.n_h * a.n_w;
  const int grid = P < sm_count() ? P : sm_count();
  patch_resblock_bwd_kernel<<<grid, PE_THREADS, smem, as_stream(stream)>>>(a);
  NEKO_LAUNCH_CHECK("patch_resblock_bwd_kernel");
  return NEKO_OK;
}

int64_t neko_patch_resblock_bwd_ordered_workspace_bytes(int n_img, int Himg, int Wimg, int patch) {
  using namespace neko;
  NEKO_REQUIRE(patch == PE_P && n_img > 0 && Himg > 0 && Wimg > 0 && Himg % patch == 0 && Wimg % patch == 0,
               "patch_resblock_bwd_ordered: need patch 16 and image dimensions divisible by it");
  const long long P = (long long)n_img * (Himg / patch) * (Wimg / patch);
  NEKO_REQUIRE(P < (1LL << 30), "patch_resblock_bwd_ordered: too many patches");
  return (int64_t)((P + PE_CHUNK - 1) / PE_CHUNK) * PS_SLOT * (int64_t)sizeof(float);
}

int neko_patch_resblock_bwd_ordered(const void* images, int is_u8, int n_img, int Himg, int Wimg, int patch, int C, int groups,
                                    const float* conv1_w, const float* conv1_b, const float* gn_w, const float* gn_b, const float* conv2_w,
                                    const float* gn_stats, const uint16_t* d_patches_bf16, float* d_conv1_w, float* d_conv1_b,
                                    float* d_gn_w, float* d_gn_b, float* d_conv2_w, float* d_conv2_b, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(workspace, "patch_resblock_bwd_ordered: null pointer");
  PatchArgs a;
  const int rc = patch_bwd_args(a, "patch_resblock_bwd_ordered", images, is_u8, n_img, Himg, Wimg, patch, C, groups, conv1_w, conv1_b, gn_w,
                                gn_b, conv2_w, gn_stats, d_patches_bf16, d_conv1_w, d_conv1_b, d_gn_w, d_gn_b, d_conv2_w, d_conv2_b);
  if (rc != NEKO_OK) return rc;
  const int64_t need = neko_patch_resblock_bwd_ordered_workspace_bytes(n_img, Himg, Wimg, patch);
  if (need < 0) return (int)need;
  NEKO_REQUIRE(workspace_bytes >= need && (reinterpret_cast<uintptr_t>(workspace) & 3) == 0,
               "patch_resblock_bwd_ordered: workspace of %lld bytes, need %lld (4-byte aligned)", (long long)workspace_bytes, (long long)need);
  const size_t smem = patch_smem_bytes(true);
  cudaError_t e = cudaFuncSetAttribute(patch_resblock_bwd_ordered_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(patch_bwd_ordered)");
  const int P = n_img * a.n_h * a.n_w;
  const int n_chunks = (P + PE_CHUNK - 1) / PE_CHUNK;
  float* ws = static_cast<float*>(workspace);
  patch_resblock_bwd_ordered_kernel<<<ordered_grid(n_chunks), PE_THREADS, smem, as_stream(stream)>>>(a, ws, n_chunks);
  NEKO_LAUNCH_CHECK("patch_resblock_bwd_ordered_kernel");
  OrdDst dst{};
  dst.p[0] = d_conv1_w; dst.p[1] = d_conv1_b; dst.p[2] = d_gn_w; dst.p[3] = d_gn_b; dst.p[4] = d_conv2_w; dst.p[5] = d_conv2_b;
  dst.off[0] = PS_DW1; dst.off[1] = PS_DB1; dst.off[2] = PS_DGW; dst.off[3] = PS_DGB; dst.off[4] = PS_DW2; dst.off[5] = PS_DB2;
  dst.off[6] = PS_SLOT; dst.n = 6;
  return ordered_colreduce(ws, PS_SLOT, n_chunks, PS_SLOT, dst, 1, as_stream(stream));
}

int neko_patch_pos_add(float* x, int P, int d, const int32_t* row_bin, const int32_t* col_bin, const float* row_tab,
                       const float* col_tab, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(x && row_bin && col_bin && row_tab && col_tab && P > 0 && d > 0 && d % 4 == 0, "patch_pos_add: bad arguments");
  patch_pos_add_kernel<<<(unsigned)(((long long)P * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(x, P, d, row_bin, col_bin, row_tab, col_tab);
  NEKO_LAUNCH_CHECK("patch_pos_add_kernel");
  return NEKO_OK;
}

int neko_patch_pos_bwd(const float* dx, int P, int d, const int32_t* row_bin, const int32_t* col_bin, float* d_row_tab,
                       float* d_col_tab, void* stream) {
  using namespace neko;
  NEKO_REQUIRE(dx && row_bin && col_bin && d_row_tab && d_col_tab && P > 0 && d > 0, "patch_pos_bwd: bad arguments");
  patch_pos_bwd_kernel<<<(unsigned)(((long long)P * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(dx, P, d, row_bin, col_bin, d_row_tab, d_col_tab);
  NEKO_LAUNCH_CHECK("patch_pos_bwd_kernel");
  return NEKO_OK;
}

}  // extern "C"
