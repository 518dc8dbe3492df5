// One row of the warp-per-row LayerNorm backward (layernorm.cu), included into the body of the row loop of
// layernorm_bwd_rows_kernel and of layernorm_bwd_ordered_kernel: dx_resid += LN'(dy), the (masked) branch gradient to dx_bf16,
// and dy * xhat | dy | branch gradient added to this warp's accumulators wacc [3][d].  The lanes own float4 columns lane,
// lane + 32, ...; sg is gamma in shared memory.
//   LN_ROW_GUARD   any d % 4 == 0 up to 2048: lanes skip the float4 columns past nv4 = d / 4 (defined by the kernel), and
//                  dx_resid is read where it is used (held across the row reduction at up to NV = 16, it would cost registers)
//   LN_ROW_COLSUM  whether the branch gradient is summed
// It is text rather than a __device__ function because nvcc optimises a function before inlining it, without the kernel's
// context, and the default kernel's code would come out different.
{
  const size_t off = (size_t)row * d;
  const float4* x4 = reinterpret_cast<const float4*>(x + off);
  const uint2* d2 = reinterpret_cast<const uint2*>(dy + off);
  float4* r4 = reinterpret_cast<float4*>(dx_resid + off);
  float4 xv[NV];
  uint2 dv[NV];
#if LN_ROW_GUARD
#pragma unroll
  for (int k = 0; k < NV; ++k)
    if (lane + 32 * k < nv4) { xv[k] = x4[lane + 32 * k]; dv[k] = d2[lane + 32 * k]; }
#else
  float4 rv[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) { xv[k] = x4[lane + 32 * k]; dv[k] = d2[lane + 32 * k]; rv[k] = r4[lane + 32 * k]; }
#endif
  const float mu = __ldg(mean + row), rs = __ldg(rstd + row);
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int c4 = lane + 32 * k;
#if LN_ROW_GUARD
    if (c4 >= nv4) continue;
#endif
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
#if LN_ROW_GUARD
    if (c4 >= nv4) continue;
#endif
    const float4 g = *reinterpret_cast<const float4*>(sg + 4 * c4);
    const float2 d01 = unpack_bf16x2(dv[k].x), d23 = unpack_bf16x2(dv[k].y);
#if LN_ROW_GUARD
    float4 o = r4[c4];
#else
    float4 o = rv[k];
#endif
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
    if (LN_ROW_COLSUM) {
      float4* ac = reinterpret_cast<float4*>(wacc + 2 * d + 4 * c4);
      float4 t = *ac;
      t.x += o.x; t.y += o.y; t.z += o.z; t.w += o.w;
      *ac = t;
    }
  }
}
