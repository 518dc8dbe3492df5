// One row block of the column-owner LayerNorm backward kernels (layernorm.cu), included into the row-block loop of
// layernorm_bwd_kernel (LN_COLS_STAGED 0) and of layernorm_bwd_staged_kernel (1) after each has loaded its rows into xv, dv,
// rv: the row statistics, their block-wide reduction, dx_resid, the (masked) branch gradient to dx_bf16, and the column sums
// ag, ab, ac.  The staged kernel refills the ring slot it has just read once every thread is past the block reduction's barrier.
// It is text rather than a __device__ function because nvcc optimises a function before inlining it, without the kernel's
// context, and the default kernels' code would come out different.
    float sred[2 * LNB_ROWS];
    float4 gy[LNB_ROWS], xh[LNB_ROWS];
#pragma unroll
    for (int r = 0; r < LNB_ROWS; ++r) {
      const float2 d01 = unpack_bf16x2(dv[r].x), d23 = unpack_bf16x2(dv[r].y);
      xh[r] = make_float4((xv[r].x - mu[r]) * rs[r], (xv[r].y - mu[r]) * rs[r], (xv[r].z - mu[r]) * rs[r], (xv[r].w - mu[r]) * rs[r]);
      gy[r] = make_float4(d01.x * g.x, d01.y * g.y, d23.x * g.z, d23.y * g.w);
      sred[r] = (gy[r].x + gy[r].y) + (gy[r].z + gy[r].w);
      sred[LNB_ROWS + r] = (gy[r].x * xh[r].x + gy[r].y * xh[r].y) + (gy[r].z * xh[r].z + gy[r].w * xh[r].w);
      // column sums of dy and dy * xhat
      ab.x += d01.x; ab.y += d01.y; ab.z += d23.x; ab.w += d23.y;
      ag.x += d01.x * xh[r].x; ag.y += d01.y * xh[r].y; ag.z += d23.x * xh[r].z; ag.w += d23.y * xh[r].w;
    }
#pragma unroll
    for (int i = 0; i < 2 * LNB_ROWS; ++i) sred[i] = warp_sum(sred[i]);
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < 2 * LNB_ROWS; ++i) red[parity][wid][i] = sred[i];
    }
#if LN_COLS_STAGED
    __syncthreads();   // every thread has read its slice of ring slot s: the slot may be refilled
    if (threadIdx.x == 0 && it + stages < n_iter) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(it + stages);
    }
#else
    __syncthreads();
#endif
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
        if (drop.seed) {  // gradient entering the dropped-out residual branch: mask * scale * dx
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
