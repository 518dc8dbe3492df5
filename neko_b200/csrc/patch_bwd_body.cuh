// Body of the two patch ResNet backward kernels in patch_embed.cu, included into each of them.  PE_BWD_ORDERED selects where
// they differ:
//   0  patch_resblock_bwd_kernel(PatchArgs a): patches blockIdx.x, + gridDim.x, ...; the partials are reset once and leave by
//      atomicAdd into a.grad;
//   1  patch_resblock_bwd_ordered_kernel(PatchArgs a, float* ws, int n_chunks): chunk c = patches [8c, 8c + 8), taken in
//      ascending order by whichever CTA gets it; the partials are reset per chunk and stored to workspace slot c, which
//      ordered_colreduce then folds in a fixed order.
// It is text rather than a __device__ function because nvcc optimises a function before inlining it, without the kernel's
// __launch_bounds__ (the range of threadIdx.x), and the default kernel's code would come out different.
#if PE_BWD_ORDERED
#define PE_PUT(p, v) (*(p) = (v))
#define PE_GRAD slot_grad
#else
#define PE_PUT(p, v) atomicAdd(p, v)
#define PE_GRAD a.grad
#endif
  extern __shared__ __align__(16) uint8_t pe_raw[];
  bf16* colX = reinterpret_cast<bf16*>(pe_raw);                       // [256][40] im2col of gelu(x) (+ ones column)
  bf16* colY = colX + PE_PX * PE_KP;                                   // [256][40] flipped im2col of dY
  bf16* W1s = colY + PE_PX * PE_KP;                                    // [128][40]
  bf16* W2r = W1s + PE_C * PE_KP;                                      // [128][40]  W2r[c][co*9+tap] = w2[co][c][tap]
  bf16* h2s = W2r + PE_C * PE_KP;                                      // [256][72]  gelu(gn(h)) of the current channel half
  bf16* dhs = h2s + PE_PX * PE_HP2;                                    // [256][72]  gradient at the conv1 output
  float* gx = reinterpret_cast<float*>(dhs + PE_PX * PE_HP2);          // [3][18][18]
  float* dyp = gx + 3 * PE_PAD * PE_PAD;                               // [3][18][18]
  float* gpart = dyp + 3 * PE_PAD * PE_PAD;                            // [8 warps][64 groups][2]  s1, s2 partials
  float* gstat = gpart + 8 * 64 * 2;                                   // [64][2] mean, rstd
  float* gsum = gstat + 128;                                           // [64][2] m1, m2
  float* gws = gsum + 128;                                             // [128]
  float* gbs = gws + PE_C;                                             // [128]
  float* aff = gbs + PE_C;                                             // [8 warps][128][2] dgamma, dbeta accumulators
  float* db2s = aff + 8 * PE_C * 2;                                    // [8 warps][4]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, q = lane & 3;
  const int P = a.n_img * a.n_h * a.n_w;
  const int gs = PE_C / a.groups, gshift = 31 - __clz(gs);             // channels per group: a power of two in [2, 64]
  const STile tX{(uint32_t)__cvta_generic_to_shared(colX), PE_KP}, tY{(uint32_t)__cvta_generic_to_shared(colY), PE_KP};
  const STile tW1{(uint32_t)__cvta_generic_to_shared(W1s), PE_KP}, tW2{(uint32_t)__cvta_generic_to_shared(W2r), PE_KP};
  const STile tH2{(uint32_t)__cvta_generic_to_shared(h2s), PE_HP2}, tDH{(uint32_t)__cvta_generic_to_shared(dhs), PE_HP2};

  for (int i = tid; i < PE_C * PE_KP; i += PE_THREADS) {
    const int c = i / PE_KP, n = i - c * PE_KP;
    W1s[i] = __float2bfloat16_rn(n < 27 ? a.w1[c * 27 + n] : (n == 27 ? a.b1[c] : 0.f));
    float w2v = 0.f;
    if (n < 27) { const int co = n / 9, tap = n - co * 9; w2v = a.w2[(co * PE_C + c) * 9 + tap]; }
    W2r[i] = __float2bfloat16_rn(w2v);
  }
  for (int i = tid; i < 3 * PE_PAD * PE_PAD; i += PE_THREADS) { gx[i] = 0.f; dyp[i] = 0.f; }
  for (int i = tid; i < PE_C; i += PE_THREADS) { gws[i] = a.gw[i]; gbs[i] = a.gb[i]; }
#if PE_BWD_ORDERED
  __syncthreads();
  for (int chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
  float* slot = ws + (size_t)chunk * PS_SLOT;
  const PatchGrads slot_grad{slot + PS_DW1, slot + PS_DB1, slot + PS_DGW, slot + PS_DGB, slot + PS_DW2, slot + PS_DB2};
#endif
  for (int i = tid; i < 8 * PE_C * 2; i += PE_THREADS) aff[i] = 0.f;
  if (tid < 32) db2s[tid] = 0.f;
  __syncthreads();

  // weight-gradient accumulators, persistent over the patches between two flushes.
  // dW2r[n][c]: per channel half 2 (n m-tiles) x 8 (c n-tiles) output tiles -> warp w owns m-tile (w & 1), n-tiles 2*(w>>1), +1
  // dW1 [c][n]: per channel half 4 (c m-tiles) x 4 (n n-tiles) output tiles -> warp w owns m-tile (w >> 1), n-tiles 2*(w&1), +1
  float aw2[2][2][4], aw1[2][2][4];
#pragma unroll
  for (int hc = 0; hc < 2; ++hc)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) { aw2[hc][j][e] = 0.f; aw1[hc][j][e] = 0.f; }

#if PE_BWD_ORDERED
  for (int patch = chunk * PE_CHUNK; patch < min(P, (chunk + 1) * PE_CHUNK); ++patch) {
#else
  for (int patch = blockIdx.x; patch < P; patch += gridDim.x) {
#endif
    pe_load_patch(a, gx, nullptr, patch);
    {
      const int y = tid >> 4, x = tid & 15;
      const bf16* gy = a.dout + (size_t)patch * (3 * PE_PX);
#pragma unroll
      for (int co = 0; co < 3; ++co) {
        const float v = __bfloat162float(gy[co * PE_PX + tid]);
        dyp[(co * PE_PAD + y + 1) * PE_PAD + x + 1] = v;
        const float t = warp_sum(v);
        if (lane == 0) db2s[warp * 4 + co] += t;
      }
    }
    if (tid < a.groups) {
      gstat[2 * tid] = a.stats[((size_t)patch * a.groups + tid) * 2];
      gstat[2 * tid + 1] = a.stats[((size_t)patch * a.groups + tid) * 2 + 1];
    }
    __syncthreads();
    pe_im2col_row<false>(gx, colX, 1.0f);
    pe_im2col_row<true>(dyp, colY, 0.0f);
    __syncthreads();

    uint32_t ax[2][2][4], ay[2][2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        fa_mk(tX, warp * 32 + mt * 16, k * 16, lane, ax[mt][k]);
        fa_mk(tY, warp * 32 + mt * 16, k * 16, lane, ay[mt][k]);
      }

#pragma unroll
    for (int hc = 0; hc < 2; ++hc) {
      // ---- recompute conv1 and run the transposed conv2 for 64 channels: H, dh2 [32 px][64 c] per warp ----
      float h[2][8][4], dh[2][8][4];
#pragma unroll
      for (int n2 = 0; n2 < 4; ++n2) {
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int e = 0; e < 4; ++e) { h[mt][2 * n2][e] = h[mt][2 * n2 + 1][e] = 0.f; dh[mt][2 * n2][e] = dh[mt][2 * n2 + 1][e] = 0.f; }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          uint32_t b1f[4], b2f[4];
          fb_nk(tW1, hc * 64 + n2 * 16, k * 16, lane, b1f);
          fb_nk(tW2, hc * 64 + n2 * 16, k * 16, lane, b2f);
#pragma unroll
          for (int mt = 0; mt < 2; ++mt) {
            pe_mma(h[mt][2 * n2], ax[mt][k], b1f[0], b1f[1]);
            pe_mma(h[mt][2 * n2 + 1], ax[mt][k], b1f[2], b1f[3]);
            pe_mma(dh[mt][2 * n2], ay[mt][k], b2f[0], b2f[1]);
            pe_mma(dh[mt][2 * n2 + 1], ay[mt][k], b2f[2], b2f[3]);
          }
        }
      }
      // ---- elementwise: xhat, h2 = gelu(hn) -> h2s ; dhn = dh2 * gelu'(hn) ; group partial sums ; dgamma / dbeta ----
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int c0 = hc * 64 + nt * 8 + 2 * q;
        const int grp = c0 >> gshift;
        const float mean = gstat[2 * grp], rstd = gstat[2 * grp + 1];
        const float w0 = gws[c0], w1 = gws[c0 + 1], b0 = gbs[c0], b1 = gbs[c0 + 1];
        float s1 = 0.f, s2 = 0.f, dg0 = 0.f, dg1 = 0.f, db0 = 0.f, db1 = 0.f;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int px = warp * 32 + mt * 16 + g + hh * 8;
            const float xh0 = (h[mt][nt][2 * hh] - mean) * rstd, xh1 = (h[mt][nt][2 * hh + 1] - mean) * rstd;
            const float hn0 = xh0 * w0 + b0, hn1 = xh1 * w1 + b1;
            float y0, y1, g0, g1;
            gelu_erf_both(hn0, y0, g0);
            gelu_erf_both(hn1, y1, g1);
            *reinterpret_cast<uint32_t*>(h2s + px * PE_HP2 + nt * 8 + 2 * q) = pack_bf16x2(y0, y1);
            const float d0 = dh[mt][nt][2 * hh] * g0, d1 = dh[mt][nt][2 * hh + 1] * g1;
            h[mt][nt][2 * hh] = xh0; h[mt][nt][2 * hh + 1] = xh1;     // keep xhat
            dh[mt][nt][2 * hh] = d0; dh[mt][nt][2 * hh + 1] = d1;     // keep dhn
            dg0 += d0 * xh0; dg1 += d1 * xh1; db0 += d0; db1 += d1;
          }
        s1 = w0 * db0 + w1 * db1;
        s2 = w0 * dg0 + w1 * dg1;
        // per-channel sums over this warp's pixels (reduce over g), per-group sums additionally over the quad lanes
#pragma unroll
        for (int m = 4; m <= 16; m <<= 1) {
          dg0 += __shfl_xor_sync(0xffffffffu, dg0, m); dg1 += __shfl_xor_sync(0xffffffffu, dg1, m);
          db0 += __shfl_xor_sync(0xffffffffu, db0, m); db1 += __shfl_xor_sync(0xffffffffu, db1, m);
          s1 += __shfl_xor_sync(0xffffffffu, s1, m); s2 += __shfl_xor_sync(0xffffffffu, s2, m);
        }
        if (gs >= 4) { s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s2 += __shfl_xor_sync(0xffffffffu, s2, 1); }
        if (gs >= 8) { s1 += __shfl_xor_sync(0xffffffffu, s1, 2); s2 += __shfl_xor_sync(0xffffffffu, s2, 2); }
        if (g == 0) {
          float* af = aff + (warp * PE_C + c0) * 2;
          af[0] += dg0; af[1] += db0; af[2] += dg1; af[3] += db1;
          if (((2 * q) & (min(gs, 8) - 1)) == 0) {
            float* slot = gpart + (warp * 64 + grp) * 2;
            if ((nt * 8) & (gs - 1)) { slot[0] += s1; slot[1] += s2; } else { slot[0] = s1; slot[1] = s2; }
          }
        }
      }
      __syncthreads();
      if (tid < a.groups) {
        const int lo = (hc * 64) >> gshift, hi = (hc * 64 + 64) >> gshift;
        if (tid >= lo && tid < hi) {
          float s1 = 0.f, s2 = 0.f;
          for (int w = 0; w < 8; ++w) { s1 += gpart[(w * 64 + tid) * 2]; s2 += gpart[(w * 64 + tid) * 2 + 1]; }
          const float inv_n = 1.0f / (float)(gs * PE_PX);
          gsum[2 * tid] = s1 * inv_n; gsum[2 * tid + 1] = s2 * inv_n;
        }
      }
      __syncthreads();
      // ---- dh = rstd * (gamma * dhn - m1 - xhat * m2) -> dhs (bf16) ----
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int c0 = hc * 64 + nt * 8 + 2 * q;
        const int grp = c0 >> gshift;
        const float rstd = gstat[2 * grp + 1], m1 = gsum[2 * grp], m2 = gsum[2 * grp + 1];
        const float w0 = gws[c0], w1 = gws[c0 + 1];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            const int px = warp * 32 + mt * 16 + g + hh * 8;
            const float v0 = rstd * (w0 * dh[mt][nt][2 * hh] - m1 - h[mt][nt][2 * hh] * m2);
            const float v1 = rstd * (w1 * dh[mt][nt][2 * hh + 1] - m1 - h[mt][nt][2 * hh + 1] * m2);
            *reinterpret_cast<uint32_t*>(dhs + px * PE_HP2 + nt * 8 + 2 * q) = pack_bf16x2(v0, v1);
          }
      }
      __syncthreads();
      // ---- weight gradients over K = 256 pixels ----
      {
        const int mt2 = warp & 1, nb2 = (warp >> 1) * 16;   // dW2r tile: n rows [16*mt2, +16), channels [nb2, +16) of this half
        const int mt1 = warp >> 1, nb1 = (warp & 1) * 16;   // dW1  tile: channels [16*mt1, +16) of this half, n cols [nb1, +16)
#pragma unroll 4
        for (int k = 0; k < PE_PX / 16; ++k) {
          uint32_t af[4], bfr[4];
          fa_km(tY, k * 16, mt2 * 16, lane, af);
          fb_kn(tH2, k * 16, nb2, lane, bfr);
          pe_mma(aw2[hc][0], af, bfr[0], bfr[1]);
          pe_mma(aw2[hc][1], af, bfr[2], bfr[3]);
          fa_km(tDH, k * 16, mt1 * 16, lane, af);
          fb_kn(tX, k * 16, nb1, lane, bfr);
          pe_mma(aw1[hc][0], af, bfr[0], bfr[1]);
          pe_mma(aw1[hc][1], af, bfr[2], bfr[3]);
        }
      }
      __syncthreads();  // h2s / dhs are rewritten by the next half / patch
    }
  }

  // ---- flush the gradient partials: atomics, or stores to the chunk's slot (every element written once) ----
#pragma unroll
  for (int hc = 0; hc < 2; ++hc)
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        {  // dW2r[n][c] -> d_conv2_w[co][c][tap]
          const int n = (warp & 1) * 16 + g + (e >> 1) * 8;
          const int c = hc * 64 + (warp >> 1) * 16 + j * 8 + 2 * q + (e & 1);
          if (n < 27) { const int co = n / 9, tap = n - co * 9; PE_PUT(PE_GRAD.dw2 + ((size_t)co * PE_C + c) * 9 + tap, aw2[hc][j][e]); }
        }
        {  // dW1[c][n] -> d_conv1_w[c][ci][tap] ; column 27 (ones) is the bias gradient
          const int c = hc * 64 + (warp >> 1) * 16 + g + (e >> 1) * 8;
          const int n = (warp & 1) * 16 + j * 8 + 2 * q + (e & 1);
          if (n < 27) PE_PUT(PE_GRAD.dw1 + (size_t)c * 27 + n, aw1[hc][j][e]);
          else if (n == 27) PE_PUT(PE_GRAD.db1 + c, aw1[hc][j][e]);
        }
      }
  __syncthreads();
  for (int c = tid; c < PE_C; c += PE_THREADS) {
    float dg = 0.f, db = 0.f;
    for (int w = 0; w < 8; ++w) { dg += aff[(w * PE_C + c) * 2]; db += aff[(w * PE_C + c) * 2 + 1]; }
    PE_PUT(PE_GRAD.dgw + c, dg);
    PE_PUT(PE_GRAD.dgb + c, db);
  }
  if (tid < 3) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += db2s[w * 4 + tid];
    PE_PUT(PE_GRAD.db2 + tid, s);
  }
#if PE_BWD_ORDERED
  __syncthreads();   // the next chunk re-zeroes the shared accumulators just read
  }
#endif
#undef PE_PUT
#undef PE_GRAD
