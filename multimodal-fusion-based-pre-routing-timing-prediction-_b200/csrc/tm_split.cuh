// Operand splits that let 16- and 19-bit tensor-core formats carry fp32-class products.
//
// fp16 two-term split (GNN cell MLP, resident-weight self MLPs):
//   x s = hi + lo,  hi = fp16(x s),  lo' = fp16((x s - hi) 2^11)
// with s a per-row power of two that brings the row's largest magnitude into [1, 2) (exact, undone in the
// epilogue), so values of any size keep 22 significant bits; the 2^11 keeps lo' out of the fp16 subnormals.
//   acc_main += hi hi;  acc_corr += hi lo' + lo' hi      (both fp32)
//   result = (acc_main + 2^-11 acc_corr) / s            -- ~22-bit products, fp32 accumulation
//
// 3xTF32 residual (tcgen05 kind::tf32 GEMM and convolutions): the MMA reads the upper 19 bits of an fp32 word,
// so the fp32 word itself is the "hi" operand and only lo = x - trunc_tf32(x), exact in fp32, is formed;
// hi hi + hi lo + lo hi keeps ~21 mantissa bits.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace tmk {

constexpr float LO_SCALE = 2048.f, LO_INV = 1.f / 2048.f;

__device__ __forceinline__ void split_h(float x, __half& hi, __half& lo) {
  hi = __float2half_rn(x);
  lo = __float2half_rn((x - __half2float(hi)) * LO_SCALE);
}
__device__ __forceinline__ uint32_t pack_h2(__half a, __half b) {
  return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
}
__device__ __forceinline__ void split_h4(float4 x, uint2& hi, uint2& lo) {
  __half h0, h1, h2, h3, l0, l1, l2, l3;
  split_h(x.x, h0, l0); split_h(x.y, h1, l1); split_h(x.z, h2, l2); split_h(x.w, h3, l3);
  hi = make_uint2(pack_h2(h0, h1), pack_h2(h2, h3));
  lo = make_uint2(pack_h2(l0, l1), pack_h2(l2, l3));
}
// Two values in [0, 2) -> packed (hi, hi) and (lo', lo') words.  hi is taken by Veltkamp's splitting (x rounded to 11
// significant bits in fp32: exactly an fp16 number when x >= 2^-14) so that only TWO packed conversions are issued
// per pair instead of six scalar ones -- the conversions, not the FMAs, bounded the generator; below 2^-14 the
// conversion of hi rounds once more, by at most 2^-25 of the row's scale.
__device__ __forceinline__ void split_pair(float y0, float y1, uint32_t& hi, uint32_t& lo) {
  const float C = 8193.f;                                     // 2^13 + 1
  const float t0 = __fmul_rn(y0, C), t1 = __fmul_rn(y1, C);
  const float h0 = __fsub_rn(t0, __fsub_rn(t0, y0)), h1 = __fsub_rn(t1, __fsub_rn(t1, y1));
  const __half2 hh = __floats2half2_rn(h0, h1);
  const __half2 ll = __floats2half2_rn(__fmul_rn(__fsub_rn(y0, h0), LO_SCALE), __fmul_rn(__fsub_rn(y1, h1), LO_SCALE));
  hi = *reinterpret_cast<const uint32_t*>(&hh);
  lo = *reinterpret_cast<const uint32_t*>(&ll);
}
// power-of-two scale of a row whose largest magnitude is rowmax: s = 2^-e, inv = 2^e, e = floor(log2(rowmax))
// clamped to [emin, 100].  With an upper bound in place of rowmax, every |value| <= bound lands in [0, 2).
__device__ __forceinline__ void row_scale(float rowmax, int emin, float& s, float& inv) {
  int e = (int)((__float_as_uint(rowmax) >> 23) & 0xffu) - 127;
  e = max(emin, min(e, 100));
  s = __uint_as_float((uint32_t)(127 - e) << 23);
  inv = __uint_as_float((uint32_t)(127 + e) << 23);
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// lo = x - trunc_tf32(x) per element, exact in fp32
__device__ __forceinline__ float4 tf32_lo(float4 x) {
  constexpr uint32_t TF32_MASK = 0xFFFFE000u;
  float4 l;
  l.x = x.x - __uint_as_float(__float_as_uint(x.x) & TF32_MASK);
  l.y = x.y - __uint_as_float(__float_as_uint(x.y) & TF32_MASK);
  l.z = x.z - __uint_as_float(__float_as_uint(x.z) & TF32_MASK);
  l.w = x.w - __uint_as_float(__float_as_uint(x.w) & TF32_MASK);
  return l;
}

}  // namespace tmk
