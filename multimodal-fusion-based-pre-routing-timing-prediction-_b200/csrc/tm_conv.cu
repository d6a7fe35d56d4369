// G4 (fp32 path): U-Net / LayoutNet image branch on NHWC activations.
//
// Replaces the cuDNN / ATen calls behind src/Unet.py:16-21 (Conv2d 3x3 + BatchNorm2d + ReLU),
// :53 (ConvTranspose2d k2 s2), :75-77 (1x1 conv, pool, ReLU), :89-91 (pooling) and
// src/model.py:227-243 (LayoutNet 9x9 / 7x7 convs).  Convolutions are implicit GEMMs on the shared
// fp32 GEMM core (tm_gemm.cuh) with im2col performed by the operand loader; every activation
// carries an explicit pixel stride so torch.cat (Unet.py:67) is free: producers write straight
// into the halves of the concat buffer.  The tensor-core paths live in tm_tc.cu (cp.async-fed, every precision) and
// tm_tma.cu (TMA-fed, bf16 activations); the batch-norm / pooling / OutConv kernels below serve all of them.
#include <cuda_bf16.h>
#include <initializer_list>
#include <utility>

#include "tm_gemm.cuh"

using namespace tmk;

namespace {
// ------------------------------------------------------------------------------ layout kernels
__global__ void nchw_to_nhwc_kernel(int64_t B, int64_t C, int64_t HW, const float* __restrict__ in,
                                    float* __restrict__ out, int64_t ld) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C * HW) return;
  const int64_t c = i % C, p = (i / C) % HW, b = i / (C * HW);
  out[(b * HW + p) * ld + c] = in[(b * C + c) * HW + p];
}
__global__ void nhwc_to_nchw_kernel(int64_t B, int64_t C, int64_t HW, const float* __restrict__ in,
                                    int64_t ld, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C * HW) return;
  const int64_t p = i % HW, c = (i / HW) % C, b = i / (C * HW);
  out[i] = in[(b * HW + p) * ld + c];
}
__global__ void conv_pack_kernel(int64_t Cout, int64_t Cin, int64_t k, const float* __restrict__ w,
                                 float* __restrict__ wf, float* __restrict__ wb) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cout * Cin * k * k) return;
  const int64_t tx = i % k, ty = (i / k) % k, ci = (i / (k * k)) % Cin, co = i / (k * k * Cin);
  const float v = w[i];
  if (wf) wf[((ty * k + tx) * Cin + ci) * Cout + co] = v;
  if (wb) wb[(((k - 1 - ty) * k + (k - 1 - tx)) * Cout + co) * Cin + ci] = v;
}
__global__ void conv_unpack_kernel(int64_t Cout, int64_t Cin, int64_t k, const float* __restrict__ dwf,
                                   float* __restrict__ dw) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cout * Cin * k * k) return;
  const int64_t tx = i % k, ty = (i / k) % k, ci = (i / (k * k)) % Cin, co = i / (k * k * Cin);
  dw[i] = dwf[((ty * k + tx) * Cin + ci) * Cout + co];
}
__global__ void convt_pack_kernel(int64_t Cin, int64_t Cout, const float* __restrict__ w,
                                  float* __restrict__ wt, float* __restrict__ wtT) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cin * Cout * 4) return;
  const int64_t q = i % 4, co = (i / 4) % Cout, ci = i / (4 * Cout);  // w[ci][co][dy][dx], q = dy*2+dx
  const float v = w[i];
  if (wt) wt[ci * 4 * Cout + q * Cout + co] = v;
  if (wtT) wtT[(q * Cout + co) * Cin + ci] = v;
}
__global__ void convt_unpack_kernel(int64_t Cin, int64_t Cout, const float* __restrict__ dwt,
                                    float* __restrict__ dw) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Cin * Cout * 4) return;
  const int64_t q = i % 4, co = (i / 4) % Cout, ci = i / (4 * Cout);
  dw[i] = dwt[ci * 4 * Cout + q * Cout + co];
}
__global__ void fold4_kernel(int64_t Cout, const float* __restrict__ cs, float* __restrict__ dbias) {
  const int64_t co = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (co < Cout) dbias[co] = cs[co] + cs[Cout + co] + cs[2 * Cout + co] + cs[3 * Cout + co];
}

// ------------------------------------------------------------------------------ batch norm
// Statistics: a fixed number of blocks (BN_BLOCKS, independent of the image size) each sweep a contiguous
// pixel range; a thread owns VEC consecutive channels (128-bit loads when the layout allows) of every
// (256 / groups)-th pixel, accumulates in fp64 and the block folds its pixel lanes in shared memory:
// part[block][C][2].  The finalize kernels add the <= BN_BLOCKS partials per channel in a fixed order.
// The forward sums are shifted: every pixel contributes x - K_c and (x - K_c)^2, K_c = the image's first pixel of
// channel c, so that E[x^2] - mean^2 does not cancel catastrophically on a channel whose mean is large against its
// spread (a constant background: at mean/std = 3000 the unshifted sums lost 3e-3 of the variance).  K_c is the same
// for every block of an image, so the segmented and single-image results stay bit-identical.
// Segmented form (several images of npix pixels each, one U-Net batch with per-image statistics): blockIdx.y is the
// image; image k sweeps its own pixels with the block partition a single-image call uses, and every per-channel,
// per-image array ([nseg][C]) is offset by k, so each image's numbers are bit-identical to a call on that image.
constexpr int BN_BLOCKS = 592;           // 4 per SM
constexpr int BN_THREADS = 256;

__device__ __forceinline__ uint32_t bn_pack_bf16(float a, float b) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&h);
}

// The normalised pre-activation, with every rounding pinned (no FMA contraction): the backward pass re-evaluates it
// to rebuild the ReLU mask bit-for-bit instead of reading the stored activation.
__device__ __forceinline__ float bn_affine(float x, float mu, float is, float ga, float be) {
  return __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(x, mu), is), ga), be);
}

template <int VEC, bool BWD>
__global__ void __launch_bounds__(BN_THREADS)
bn_stats_kernel(int64_t npix, int C, const float* __restrict__ x, int64_t ldx, const float* __restrict__ y, int64_t ldy,
                const float* __restrict__ dy, int64_t lddy, const float* __restrict__ mean,
                const float* __restrict__ invstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                double* __restrict__ part) {
  extern __shared__ double sh[];                       // [lanes][C][2]
  const int64_t seg = blockIdx.y;
  x += seg * npix * ldx;
  if (y) y += seg * npix * ldy;
  if (BWD) { dy += seg * npix * lddy; mean += seg * C; invstd += seg * C; }
  part += seg * gridDim.x * C * 2;
  const int groups = (C + VEC - 1) / VEC;              // channel groups per pixel
  const int lanes = BN_THREADS / groups;               // pixel lanes (groups <= 256)
  const int g = threadIdx.x % groups, pl = threadIdx.x / groups;
  const int c0 = g * VEC;
  const int64_t per = (npix + gridDim.x - 1) / gridDim.x;
  const int64_t p0 = (int64_t)blockIdx.x * per, p1 = p0 + per < npix ? p0 + per : npix;
  double a[VEC], b[VEC];
  float mu[VEC], is[VEC], ga[VEC], be[VEC], kk[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    a[j] = 0.0; b[j] = 0.0;
    kk[j] = (!BWD && c0 + j < C) ? x[c0 + j] : 0.f;     // the forward's shift K_c
    mu[j] = (BWD && c0 + j < C) ? mean[c0 + j] : 0.f;
    is[j] = (BWD && c0 + j < C) ? invstd[c0 + j] : 0.f;
    ga[j] = (BWD && !y && c0 + j < C) ? gamma[c0 + j] : 0.f;
    be[j] = (BWD && !y && c0 + j < C) ? beta[c0 + j] : 0.f;
  }
  if (pl < lanes) {
    // short runs (<= 8 pixels) are summed in fp32 and folded into the fp64 accumulators: the conversions and
    // fp64 adds, not the loads, bound this kernel when every element went through fp64
    float sa[VEC], sb[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) { sa[j] = 0.f; sb[j] = 0.f; }
    auto fold = [&]() {
#pragma unroll
      for (int j = 0; j < VEC; ++j) { a[j] += (double)sa[j]; b[j] += (double)sb[j]; sa[j] = 0.f; sb[j] = 0.f; }
    };
    auto accumulate = [&](const float (&xv)[VEC], const float (&yv)[VEC], const float (&gv)[VEC]) {
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        if (BWD) {
          const float gg = yv[j] > 0.f ? gv[j] : 0.f;
          sa[j] += gg;
          sb[j] = fmaf(gg, (xv[j] - mu[j]) * is[j], sb[j]);
        } else {
          const float d = xv[j] - kk[j];
          sa[j] += d;
          sb[j] = fmaf(d, d, sb[j]);
        }
      }
    };
    if constexpr (VEC == 4) {
      // four pixels per iteration, every load issued before the first use: all loads of an iteration in flight together
      constexpr int U = 2;
      const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f), k4 = make_float4(kk[0], kk[1], kk[2], kk[3]);
      int it = 0;
      for (int64_t p = p0 + pl; p < p1; p += (int64_t)U * lanes) {
        float4 tx[U], tg[U], ty[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int64_t pu = p + (int64_t)u * lanes;
          const bool on = pu < p1;                       // a skipped pixel contributes exact zeros
          tx[u] = on ? ld4_stream(x + pu * ldx + c0) : k4;
          tg[u] = (BWD && on) ? ld4_stream(dy + pu * lddy + c0) : z4;
          ty[u] = (BWD && y && on) ? ld4_stream(y + pu * ldy + c0) : z4;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const float xv[VEC] = {tx[u].x, tx[u].y, tx[u].z, tx[u].w};
          const float gv[VEC] = {tg[u].x, tg[u].y, tg[u].z, tg[u].w};
          float yv[VEC] = {ty[u].x, ty[u].y, ty[u].z, ty[u].w};
          if (BWD && !y) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) yv[j] = bn_affine(xv[j], mu[j], is[j], ga[j], be[j]);
          }
          accumulate(xv, yv, gv);
        }
        if ((++it & 3) == 0) fold();
      }
      fold();
    } else {
      for (int64_t p = p0 + pl; p < p1; p += lanes) {
        float xv[VEC], yv[VEC], gv[VEC];
        xv[0] = c0 < C ? x[p * ldx + c0] : 0.f;
        gv[0] = (BWD && c0 < C) ? dy[p * lddy + c0] : 0.f;
        yv[0] = (!BWD || c0 >= C) ? 0.f : y ? y[p * ldy + c0] : bn_affine(xv[0], mu[0], is[0], ga[0], be[0]);
        accumulate(xv, yv, gv);
        fold();
      }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j)
      if (c0 + j < C) { sh[((int64_t)pl * C + c0 + j) * 2] = a[j]; sh[((int64_t)pl * C + c0 + j) * 2 + 1] = b[j]; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += BN_THREADS) {
    double s = 0.0;
    for (int l = 0; l < lanes; ++l) s += sh[(int64_t)l * C * 2 + i];
    part[(int64_t)blockIdx.x * C * 2 + i] = s;
  }
}

// one block of 256 threads per channel: thread t adds partials t, t+256, ...; warps and then the 8 warp sums are
// folded in a fixed order (deterministic).  (One warp per channel was latency-bound once the fused convolution
// statistics brought thousands of partials per channel.)
__device__ __forceinline__ void bn_block_sum2(double& a, double& b) {
  __shared__ double sa[8], sb[8];
  a = warp_sum(a);
  b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) { sa[threadIdx.x >> 5] = a; sb[threadIdx.x >> 5] = b; }
  __syncthreads();
  a = 0.0; b = 0.0;
  for (int i = 0; i < 8; ++i) { a += sa[i]; b += sb[i]; }
}

__global__ void __launch_bounds__(256)
bn_finalize_kernel(int64_t npix, int64_t C, int nblk, int nseg, const double* __restrict__ part,
                   const float* __restrict__ shift_x, int64_t ldx, float* __restrict__ running_mean,
                   float* __restrict__ running_var, float momentum, float eps, float* __restrict__ save_mean,
                   float* __restrict__ save_invstd) {   // shift_x: the images whose first pixel shifted the sums, or NULL
  const int c = blockIdx.x;
  // images in order: the running statistics see image 0's update first, as nseg single-image calls would
  for (int k = 0; k < nseg; ++k) {
    const double* pk = part + (int64_t)k * nblk * C * 2;
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < nblk; i += 256) { a += pk[((int64_t)i * C + c) * 2]; b += pk[((int64_t)i * C + c) * 2 + 1]; }
    bn_block_sum2(a, b);
    if (threadIdx.x == 0) {
      const double m1 = a / (double)npix;              // mean of x - K_c
      const double mean = (shift_x ? (double)shift_x[(int64_t)k * npix * ldx + c] : 0.0) + m1;
      double var = b / (double)npix - m1 * m1;
      if (var < 0.0) var = 0.0;
      save_mean[k * C + c] = (float)mean;
      save_invstd[k * C + c] = (float)(1.0 / sqrt(var + (double)eps));
      if (running_mean) {
        const double unbiased = npix > 1 ? var * (double)npix / (double)(npix - 1) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
      }
    }
    __syncthreads();                                   // bn_block_sum2's shared slots are reused by the next image
  }
}

// y = relu((x - mean) * invstd * gamma + beta); optionally also a compact bf16 copy yb [npix][C] (the TMA
// operand of the next convolution).  VEC == 4: one thread per 4 channels, 128-bit loads and stores.
template <int VEC>
__global__ void bn_relu_apply_kernel(int64_t npix, int C, const float* __restrict__ x, int64_t ldx,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     const float* __restrict__ mean, const float* __restrict__ invstd,
                                     float* __restrict__ y, int64_t ldy, __nv_bfloat16* __restrict__ yb) {
  const int groups = C / VEC;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * groups) return;
  const int64_t seg = blockIdx.y;                      // image (segmented call): its rows and statistics
  x += seg * npix * ldx;
  if (y) y += seg * npix * ldy;
  if (yb) yb += seg * npix * C;
  mean += seg * C;
  invstd += seg * C;
  const int64_t p = i / groups;
  const int c = (int)(i - p * groups) * VEC;
  float v[VEC];
  if (VEC == 4) {
    const float4 t = ld4_stream(x + p * ldx + c);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    v[0] = x[p * ldx + c];
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j)
    v[j] = fmaxf(bn_affine(v[j], __ldg(mean + c + j), __ldg(invstd + c + j), __ldg(gamma + c + j), __ldg(beta + c + j)), 0.f);
  if (VEC == 4) {
    if (y) st4(y + p * ldy + c, make_float4(v[0], v[1], v[2], v[3]));
    if (yb) *reinterpret_cast<uint2*>(yb + p * C + c) = make_uint2(bn_pack_bf16(v[0], v[1]), bn_pack_bf16(v[2], v[3]));
  } else {
    if (y) y[p * ldy + c] = v[0];
    if (yb) yb[p * C + c] = __float2bfloat16(v[0]);
  }
}

__global__ void __launch_bounds__(256)
bn_bwd_finalize_kernel(int64_t C, int nblk, int nseg, const double* __restrict__ part, float* dgamma_seg, float* dbeta_seg,
                       float* dgamma, float* dbeta) {   // (not restrict: nseg == 1 passes the same arrays twice)
  const int c = blockIdx.x;
  double ga = 0.0, be = 0.0;                           // fold over the images, in image order
  for (int k = 0; k < nseg; ++k) {
    const double* pk = part + (int64_t)k * nblk * C * 2;
    double a = 0.0, b = 0.0;
    for (int i = threadIdx.x; i < nblk; i += 256) { a += pk[((int64_t)i * C + c) * 2]; b += pk[((int64_t)i * C + c) * 2 + 1]; }
    bn_block_sum2(a, b);
    if (threadIdx.x == 0) {
      dbeta_seg[k * C + c] = (float)a;                 // image k's own sums: its data gradient needs them
      dgamma_seg[k * C + c] = (float)b;
      be += (double)(float)a;
      ga += (double)(float)b;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { dbeta[c] = (float)be; dgamma[c] = (float)ga; }
}

template <int VEC>
__global__ void bn_bwd_apply_kernel(int64_t npix, int C, const float* __restrict__ x, int64_t ldx,
                                    const float* __restrict__ y, int64_t ldy, const float* __restrict__ dy,
                                    int64_t lddy, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, const float* __restrict__ mean,
                                    const float* __restrict__ invstd, const float* __restrict__ dgamma,
                                    const float* __restrict__ dbeta, float* __restrict__ dx, int64_t lddx,
                                    __nv_bfloat16* __restrict__ dxb) {
  const int groups = C / VEC;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * groups) return;
  const int64_t seg = blockIdx.y;
  x += seg * npix * ldx;
  if (y) y += seg * npix * ldy;
  dy += seg * npix * lddy;
  if (dx) dx += seg * npix * lddx;
  if (dxb) dxb += seg * npix * C;
  mean += seg * C; invstd += seg * C; dgamma += seg * C; dbeta += seg * C;
  const int64_t p = i / groups;
  const int c = (int)(i - p * groups) * VEC;
  float xv[VEC], yv[VEC], gv[VEC], o[VEC];
  if (VEC == 4) {
    const float4 t = ld4_stream(x + p * ldx + c), w = ld4_stream(dy + p * lddy + c);
    xv[0] = t.x; xv[1] = t.y; xv[2] = t.z; xv[3] = t.w;
    gv[0] = w.x; gv[1] = w.y; gv[2] = w.z; gv[3] = w.w;
    if (y) {
      const float4 u = ld4_stream(y + p * ldy + c);
      yv[0] = u.x; yv[1] = u.y; yv[2] = u.z; yv[3] = u.w;
    }
  } else {
    xv[0] = x[p * ldx + c]; gv[0] = dy[p * lddy + c];
    if (y) yv[0] = y[p * ldy + c];
  }
  if (!y) {
#pragma unroll
    for (int j = 0; j < VEC; ++j)
      yv[j] = bn_affine(xv[j], __ldg(mean + c + j), __ldg(invstd + c + j), __ldg(gamma + c + j), __ldg(beta + c + j));
  }
  const float inv_n = 1.f / (float)npix;
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    const float g = (yv[j] > 0.f) ? gv[j] : 0.f;
    const float is = __ldg(invstd + c + j);
    const float xh = (xv[j] - __ldg(mean + c + j)) * is;
    o[j] = __ldg(gamma + c + j) * is * (g - __ldg(dbeta + c + j) * inv_n - xh * __ldg(dgamma + c + j) * inv_n);
  }
  if (VEC == 4) {
    if (dx) st4(dx + p * lddx + c, make_float4(o[0], o[1], o[2], o[3]));
    if (dxb) *reinterpret_cast<uint2*>(dxb + p * C + c) = make_uint2(bn_pack_bf16(o[0], o[1]), bn_pack_bf16(o[2], o[3]));
  } else {
    if (dx) dx[p * lddx + c] = o[0];
    if (dxb) dxb[p * C + c] = __float2bfloat16(o[0]);
  }
}

// ------------------------------------------------------------------------------ OutConv (1x1, one output channel)
// Unet.py:74-75: nn.Conv2d(16, 1, kernel_size=1).  Three streaming kernels (exact fp32): a 1x1 convolution with a
// single output channel is a dot product per pixel, its data gradient an outer product, its weight gradient a
// column reduction -- none of them is a GEMM worth a tensor-core launch.
template <int VEC>
__global__ void conv1x1_c1_fwd_kernel(int64_t npix, int C, const float* __restrict__ x, int64_t ldx,
                                      const float* __restrict__ w, const float* __restrict__ bias, float* __restrict__ y,
                                      int64_t ldy) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npix) return;
  float s = bias ? __ldg(bias) : 0.f;
  const float* xp = x + p * ldx;
  if (VEC == 4) {
    for (int c = 0; c < C; c += 4) {
      const float4 t = ld4_stream(xp + c);
      s += t.x * __ldg(w + c) + t.y * __ldg(w + c + 1) + t.z * __ldg(w + c + 2) + t.w * __ldg(w + c + 3);
    }
  } else {
    for (int c = 0; c < C; ++c) s += xp[c] * __ldg(w + c);
  }
  y[p * ldy] = s;
}
template <int VEC>
__global__ void conv1x1_c1_dgrad_kernel(int64_t npix, int C, const float* __restrict__ dy, int64_t lddy,
                                        const float* __restrict__ w, float* __restrict__ dx, int64_t lddx) {
  const int groups = C / VEC;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * groups) return;
  const int64_t p = i / groups;
  const int c = (int)(i - p * groups) * VEC;
  const float g = dy[p * lddy];
  if (VEC == 4) st4(dx + p * lddx + c, make_float4(g * __ldg(w + c), g * __ldg(w + c + 1), g * __ldg(w + c + 2), g * __ldg(w + c + 3)));
  else dx[p * lddx + c] = g * __ldg(w + c);
}
// part[block][C + 1]: sum_p x[p][c] * dy[p] for c < C, sum_p dy[p] at index C
__global__ void __launch_bounds__(BN_THREADS)
conv1x1_c1_wgrad_kernel(int64_t npix, int C, const float* __restrict__ x, int64_t ldx, const float* __restrict__ dy,
                        int64_t lddy, double* __restrict__ part) {
  extern __shared__ double sh[];                       // [lanes][C + 1]
  const int lanes = BN_THREADS / C;
  const int c = threadIdx.x % C, pl = threadIdx.x / C;
  const int64_t per = (npix + gridDim.x - 1) / gridDim.x;
  const int64_t p0 = (int64_t)blockIdx.x * per, p1 = p0 + per < npix ? p0 + per : npix;
  double a = 0.0, b = 0.0;
  if (pl < lanes) {
    for (int64_t p = p0 + pl; p < p1; p += lanes) {
      const float g = dy[p * lddy];
      a += (double)x[p * ldx + c] * (double)g;
      if (c == 0) b += (double)g;
    }
    sh[pl * (C + 1) + c] = a;
    if (c == 0) sh[pl * (C + 1) + C] = b;
  }
  __syncthreads();
  for (int i = threadIdx.x; i <= C; i += BN_THREADS) {
    double s2 = 0.0;
    for (int l = 0; l < lanes; ++l) s2 += sh[l * (C + 1) + i];
    part[(int64_t)blockIdx.x * (C + 1) + i] = s2;
  }
}
__global__ void conv1x1_c1_wgrad_final_kernel(int C, int nblk, const double* __restrict__ part, float* __restrict__ dw,
                                              float* __restrict__ dbias) {
  const int lane = threadIdx.x & 31;
  const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (c > C) return;
  double a = 0.0;
  for (int i = lane; i < nblk; i += 32) a += part[(int64_t)i * (C + 1) + c];
  a = warp_sum(a);
  if (lane != 0) return;
  if (c < C) dw[c] = (float)a;
  else if (dbias) dbias[0] = (float)a;
}

// ------------------------------------------------------------------------------ narrow data gradient (input image)
// dx = conv_transpose2d(dy, w) of the first convolution of each image network (U-Net inc: k = 3, 16 -> 3; LayoutNet
// encode.0: k = 9, 32 -> 2).  With 2-4 output channels an implicit GEMM padded to 16 would waste 4-8x of every MMA, so
// this is a direct correlation with the flipped taps on CUDA cores: a CTA owns a 32 x 32 tile of dx for every input
// channel; dy (tile + halo, NDG_CC channels at a time) and the weights live in shared memory; a thread owns a column of
// NDG_RPT pixels, loads the NDG_RPT + K - 1 dy values a tap column needs once and reuses them over the K taps of that
// column.  fp32 accumulate in a fixed order (deterministic); dx is written straight to NCHW.
constexpr int NDG_THREADS = 128, NDG_RPT = 8, NDG_TW = 32, NDG_TH = NDG_RPT * NDG_THREADS / 32, NDG_CC = 8;

__host__ __device__ constexpr int ndg_cinp(int cin) { return cin == 3 ? 4 : cin; }

__device__ __forceinline__ void ndg_load8(const float* p, float* v) {
  const float4 a = ld4(p), b = ld4(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ndg_load8(const __nv_bfloat16* p, float* v) {
  const uint4 a = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&a);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 f = __bfloat1622float2(h[j]);
    v[2 * j] = f.x;
    v[2 * j + 1] = f.y;
  }
}

template <int K, int CIN, typename T>
__global__ void __launch_bounds__(NDG_THREADS)
conv_dgrad_narrow_kernel(int H, int W, int Cout, const T* __restrict__ dy, int64_t lddy, const float* __restrict__ w,
                         float* __restrict__ dx) {
  constexpr int P = K / 2, SW = NDG_TW + K - 1, SH = NDG_TH + K - 1, CP = ndg_cinp(CIN);
  extern __shared__ float4 ndg_sh[];
  float* sw = reinterpret_cast<float*>(ndg_sh);       // [Cout][K][K][CP], taps flipped
  float* sd = sw + Cout * K * K * CP;                  // [NDG_CC][SH][SW]
  const int b = blockIdx.z, x0 = blockIdx.x * NDG_TW, y0 = blockIdx.y * NDG_TH;
  for (int i = threadIdx.x; i < Cout * K * K * CP; i += NDG_THREADS) {
    const int ci = i % CP, tap = (i / CP) % (K * K), co = i / (CP * K * K);
    sw[i] = ci < CIN ? __ldg(w + ((int64_t)co * CIN + ci) * K * K + (K * K - 1 - tap)) : 0.f;
  }
  const int lane = threadIdx.x & 31, r0 = (threadIdx.x >> 5) * NDG_RPT;
  float acc[NDG_RPT][CIN];
#pragma unroll
  for (int i = 0; i < NDG_RPT; ++i)
#pragma unroll
    for (int ci = 0; ci < CIN; ++ci) acc[i][ci] = 0.f;
  const T* dyb = dy + (int64_t)b * H * W * lddy;
  for (int c0 = 0; c0 < Cout; c0 += NDG_CC) {
    __syncthreads();
    for (int p = threadIdx.x; p < SH * SW; p += NDG_THREADS) {
      const int ly = p / SW, lx = p - ly * SW, gy = y0 - P + ly, gx = x0 - P + lx;
      float v[NDG_CC];
      if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
        ndg_load8(dyb + ((int64_t)gy * W + gx) * lddy + c0, v);
      } else {
#pragma unroll
        for (int c = 0; c < NDG_CC; ++c) v[c] = 0.f;
      }
#pragma unroll
      for (int c = 0; c < NDG_CC; ++c) sd[(c * SH + ly) * SW + lx] = v[c];
    }
    __syncthreads();
    for (int c = 0; c < NDG_CC; ++c) {
      const float* s = sd + (c * SH + r0) * SW + lane;
      const float* wc = sw + (c0 + c) * K * K * CP;
#pragma unroll
      for (int v = 0; v < K; ++v) {
        float col[NDG_RPT + K - 1];
#pragma unroll
        for (int i = 0; i < NDG_RPT + K - 1; ++i) col[i] = s[i * SW + v];
#pragma unroll
        for (int u = 0; u < K; ++u) {
          float wv[CP];
          const float* wp = wc + (u * K + v) * CP;
          if constexpr (CP == 4) {
            const float4 t = *reinterpret_cast<const float4*>(wp);
            wv[0] = t.x; wv[1] = t.y; wv[2] = t.z; wv[3] = t.w;
          } else if constexpr (CP == 2) {
            const float2 t = *reinterpret_cast<const float2*>(wp);
            wv[0] = t.x; wv[1] = t.y;
          } else {
            wv[0] = wp[0];
          }
#pragma unroll
          for (int i = 0; i < NDG_RPT; ++i)
#pragma unroll
            for (int ci = 0; ci < CIN; ++ci) acc[i][ci] = fmaf(col[i + u], wv[ci], acc[i][ci]);
        }
      }
    }
  }
  const int gx = x0 + lane;
  if (gx >= W) return;
#pragma unroll
  for (int i = 0; i < NDG_RPT; ++i) {
    const int gy = y0 + r0 + i;
    if (gy < H) {
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) dx[(((int64_t)b * CIN + ci) * H + gy) * W + gx] = acc[i][ci];
    }
  }
}

// ------------------------------------------------------------------------------ pooling etc.
__global__ void pool_fwd_kernel(int64_t B, int64_t H, int64_t W, int64_t C, int mode,
                                const float* __restrict__ x, int64_t ldx, float* __restrict__ y, int64_t ldy,
                                uint8_t* __restrict__ idx, int relu) {
  const int64_t Ho = H / 2, Wo = W / 2;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Ho * Wo * C) return;
  const int64_t c = i % C, xo = (i / C) % Wo, yo = (i / (C * Wo)) % Ho, b = i / (C * Wo * Ho);
  const float* base = x + ((b * H + 2 * yo) * W + 2 * xo) * ldx + c;
  const float v0 = base[0], v1 = base[ldx], v2 = base[W * ldx], v3 = base[W * ldx + ldx];
  float out;
  if (mode == 0) {
    int am = 0;
    out = v0;
    if (v1 > out || v1 != v1) { out = v1; am = 1; }   // first maximum wins, NaN propagates (ATen rule)
    if (v2 > out || v2 != v2) { out = v2; am = 2; }
    if (v3 > out || v3 != v3) { out = v3; am = 3; }
    if (idx) idx[i] = (uint8_t)am;
  } else {
    out = 0.25f * (v0 + v1 + v2 + v3);
  }
  if (relu) out = fmaxf(out, 0.f);
  y[((b * Ho + yo) * Wo + xo) * ldy + c] = out;
}

// 128-bit variant: one thread per (output pixel, 4 channels); same first-maximum / NaN rule per channel
__global__ void pool_fwd_vec_kernel(int B, int H, int W, int C, int mode, const float* __restrict__ x, int64_t ldx,
                                    float* __restrict__ y, int64_t ldy, uint8_t* __restrict__ idx, int relu) {
  const int Ho = H / 2, Wo = W / 2, cg = C / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * Ho * Wo * cg) return;
  const int c = (int)(i % cg) * 4;
  const int64_t o = i / cg;
  const int xo = (int)(o % Wo);
  const int64_t t = o / Wo;
  const int yo = (int)(t % Ho), b = (int)(t / Ho);
  const float* base = x + (((int64_t)b * H + 2 * yo) * W + 2 * xo) * ldx + c;
  const float4 q0 = ld4_stream(base), q1 = ld4_stream(base + ldx), q2 = ld4_stream(base + (int64_t)W * ldx),
               q3 = ld4_stream(base + (int64_t)W * ldx + ldx);
  const float v[4][4] = {{q0.x, q0.y, q0.z, q0.w}, {q1.x, q1.y, q1.z, q1.w}, {q2.x, q2.y, q2.z, q2.w}, {q3.x, q3.y, q3.z, q3.w}};
  float out[4];
  uint32_t am = 0;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (mode == 0) {
      int a = 0;
      float m = v[0][j];
#pragma unroll
      for (int q = 1; q < 4; ++q)
        if (v[q][j] > m || v[q][j] != v[q][j]) { m = v[q][j]; a = q; }
      out[j] = m;
      am |= (uint32_t)a << (8 * j);
    } else {
      out[j] = 0.25f * (v[0][j] + v[1][j] + v[2][j] + v[3][j]);
    }
    if (relu) out[j] = fmaxf(out[j], 0.f);
  }
  if (mode == 0 && idx) *reinterpret_cast<uint32_t*>(idx + o * C + c) = am;
  st4(y + o * ldy + c, make_float4(out[0], out[1], out[2], out[3]));
}

__global__ void pool_bwd_kernel(int64_t B, int64_t H, int64_t W, int64_t C, int mode,
                                const float* __restrict__ dy, int64_t lddy, const float* __restrict__ y,
                                int64_t ldy, const uint8_t* __restrict__ idx, float* __restrict__ dx,
                                int64_t lddx, int relu) {
  const int64_t Ho = H / 2, Wo = W / 2;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H * W * C) return;
  const int64_t c = i % C, xi = (i / C) % W, yi = (i / (C * W)) % H, b = i / (C * W * H);
  const int64_t yo = yi / 2, xo = xi / 2;
  float g = 0.f;
  if (yo < Ho && xo < Wo) {
    const int64_t o = ((b * Ho + yo) * Wo + xo);
    g = dy[o * lddy + c];
    if (relu && !(y[o * ldy + c] > 0.f)) g = 0.f;
    if (mode == 0) {
      const int am = idx[o * C + c];
      if (am != (int)((yi & 1) * 2 + (xi & 1))) g = 0.f;
    } else {
      g *= 0.25f;
    }
  }
  dx[((b * H + yi) * W + xi) * lddx + c] = g;
}

// 128-bit variant: one thread per (output pixel, 4 channels) writes the 2x2 input window (H, W even, C % 4 == 0)
__global__ void pool_bwd_vec_kernel(int B, int H, int W, int C, int mode, const float* __restrict__ dy, int64_t lddy,
                                    const float* __restrict__ y, int64_t ldy, const uint8_t* __restrict__ idx,
                                    float* __restrict__ dx, int64_t lddx, int relu, const float* __restrict__ add,
                                    int64_t ldadd) {
  const int Ho = H / 2, Wo = W / 2, cg = C / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * Ho * Wo * cg) return;
  const int c = (int)(i % cg) * 4;
  const int64_t o = i / cg;                              // output pixel (b, yo, xo)
  const int xo = (int)(o % Wo);
  const int64_t t = o / Wo;
  const int yo = (int)(t % Ho), b = (int)(t / Ho);
  float4 g = ld4_stream(dy + o * lddy + c);
  if (relu) {
    const float4 yy = ld4(y + o * ldy + c);
    if (!(yy.x > 0.f)) g.x = 0.f;
    if (!(yy.y > 0.f)) g.y = 0.f;
    if (!(yy.z > 0.f)) g.z = 0.f;
    if (!(yy.w > 0.f)) g.w = 0.f;
  }
  uint32_t am = 0;
  if (mode == 0) am = *reinterpret_cast<const uint32_t*>(idx + o * C + c);
  else { g.x *= 0.25f; g.y *= 0.25f; g.z *= 0.25f; g.w *= 0.25f; }
  float* base = dx + (((int64_t)b * H + 2 * yo) * W + 2 * xo) * lddx + c;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float4 v = g;
    if (mode == 0) {
      if ((am & 0xFF) != (uint32_t)q) v.x = 0.f;
      if (((am >> 8) & 0xFF) != (uint32_t)q) v.y = 0.f;
      if (((am >> 16) & 0xFF) != (uint32_t)q) v.z = 0.f;
      if (((am >> 24) & 0xFF) != (uint32_t)q) v.w = 0.f;
    }
    const int64_t off = (int64_t)(q >> 1) * W + (q & 1);
    if (add) {                                           // + gradient arriving through the skip connection
      const float4 s4 = ld4_stream(add + ((((int64_t)b * H + 2 * yo) * W + 2 * xo) + off) * ldadd + c);
      v.x += s4.x; v.y += s4.y; v.z += s4.z; v.w += s4.w;
    }
    st4(base + off * lddx, v);
  }
}

__global__ void lrelu_fwd_kernel(int64_t n, const float* __restrict__ x, float slope, float* __restrict__ y) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { const float v = x[i]; y[i] = v > 0.f ? v : v * slope; }
}
__global__ void lrelu_bwd_kernel(int64_t n, const float* __restrict__ y, const float* __restrict__ dy,
                                 float slope, float* __restrict__ dx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dx[i] = y[i] > 0.f ? dy[i] : dy[i] * slope;
}
__global__ void add_strided_kernel(int64_t npix, int64_t C, const float* __restrict__ src, int64_t lds,
                                   float* __restrict__ dst, int64_t ldd) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * C) return;
  const int64_t p = i / C, c = i - p * C;
  dst[p * ldd + c] += src[p * lds + c];
}

inline unsigned blocks_for(int64_t n) { return (unsigned)cdiv(n, 256); }
}  // namespace

#define ST ((cudaStream_t)stream)

extern "C" int tm_nchw_to_nhwc(int64_t B, int64_t C, int64_t H, int64_t W, const float* in, float* out,
                               int64_t ld, void* stream) {
  if (B * C * H * W <= 0) return 0;
  nchw_to_nhwc_kernel<<<blocks_for(B * C * H * W), 256, 0, ST>>>(B, C, H * W, in, out, ld);
  return check_launch("nchw_to_nhwc");
}
extern "C" int tm_nhwc_to_nchw(int64_t B, int64_t C, int64_t H, int64_t W, const float* in, int64_t ld,
                               float* out, void* stream) {
  if (B * C * H * W <= 0) return 0;
  nhwc_to_nchw_kernel<<<blocks_for(B * C * H * W), 256, 0, ST>>>(B, C, H * W, in, ld, out);
  return check_launch("nhwc_to_nchw");
}
extern "C" int tm_conv_pack_weight(int64_t Cout, int64_t Cin, int64_t k, const float* w, float* wf,
                                   float* wb, void* stream) {
  conv_pack_kernel<<<blocks_for(Cout * Cin * k * k), 256, 0, ST>>>(Cout, Cin, k, w, wf, wb);
  return check_launch("conv_pack");
}
extern "C" int tm_conv_unpack_wgrad(int64_t Cout, int64_t Cin, int64_t k, const float* dwf, float* dw,
                                    void* stream) {
  conv_unpack_kernel<<<blocks_for(Cout * Cin * k * k), 256, 0, ST>>>(Cout, Cin, k, dwf, dw);
  return check_launch("conv_unpack");
}

extern "C" int tm_conv2d_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                              const float* x, int64_t ldx, const float* wf, const float* bias, float* y,
                              int64_t ldy, int flags, void* stream) {
  TM_REQUIRE(k >= 1 && (k & 1), "tm_conv2d_nhwc: odd kernel sizes only");
  Im2colLoader al{x, ldx, (int)H, (int)W, (int)Cin, (int)k, (int)(k / 2)};
  PlainEpilogue ep{y, ldy, nullptr, bias, nullptr, 0, (flags & TM_EPI_RELU) | (bias ? TM_EPI_BIAS : 0)};
  const bool veca = (Cin % 4 == 0) && (ldx % 4 == 0) && aligned16(x);
  return launch_gemm_nn(al, veca, wf, Cout, ep, B * H * W, Cout, k * k * Cin, ST);
}

extern "C" size_t tm_conv2d_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k) {
  return tn_ws_bytes(k * k * Cin, Cout, B * H * W);
}
extern "C" int tm_conv2d_wgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                                    const float* x, int64_t ldx, const float* dy, int64_t lddy, float* dwf,
                                    float* dbias, void* ws, size_t ws_bytes, void* stream) {
  Im2colLoader al{x, ldx, (int)H, (int)W, (int)Cin, (int)k, (int)(k / 2)};
  PlainLoader bl{dy, lddy, nullptr};
  const bool veca = (Cin % 4 == 0) && (ldx % 4 == 0) && aligned16(x);
  const bool vecb = (Cout % 4 == 0) && (lddy % 4 == 0) && aligned16(dy);
  return launch_gemm_tn(al, veca, bl, vecb, k * k * Cin, Cout, B * H * W, dwf, Cout, nullptr, dbias, 0, ws, ws_bytes, ST);
}

extern "C" int tm_convt_pack_weight(int64_t Cin, int64_t Cout, const float* w, float* wt, float* wtT,
                                    void* stream) {
  convt_pack_kernel<<<blocks_for(Cin * Cout * 4), 256, 0, ST>>>(Cin, Cout, w, wt, wtT);
  return check_launch("convt_pack");
}
extern "C" int tm_convt_unpack_wgrad(int64_t Cin, int64_t Cout, const float* dwt, float* dw, void* stream) {
  convt_unpack_kernel<<<blocks_for(Cin * Cout * 4), 256, 0, ST>>>(Cin, Cout, dwt, dw);
  return check_launch("convt_unpack");
}
extern "C" int tm_convt2x2_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* x,
                                int64_t ldx, const float* wt, const float* bias, float* y, int64_t ldy,
                                int64_t Hy, int64_t Wy, int64_t oy, int64_t ox, void* stream) {
  TM_REQUIRE(2 * H + oy <= Hy && 2 * W + ox <= Wy && oy >= 0 && ox >= 0, "tm_convt2x2: window outside y");
  PlainLoader al{x, ldx, nullptr};
  ConvtEpilogue ep{y, ldy, bias, (int)H, (int)W, (int)Cout, (int)Hy, (int)Wy, (int)oy, (int)ox};
  const bool veca = (Cin % 4 == 0) && (ldx % 4 == 0) && aligned16(x);
  return launch_gemm_nn(al, veca, wt, 4 * Cout, ep, B * H * W, 4 * Cout, Cin, ST);
}
extern "C" int tm_convt2x2_dgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout,
                                      const float* dyo, int64_t lddy, int64_t Hy, int64_t Wy, int64_t oy,
                                      int64_t ox, const float* wtT, float* dx, int64_t lddx, void* stream) {
  ConvtLoader al{dyo, lddy, (int)H, (int)W, (int)Cout, (int)Hy, (int)Wy, (int)oy, (int)ox};
  PlainEpilogue ep{dx, lddx, nullptr, nullptr, nullptr, 0, 0};
  const bool veca = (Cout % 4 == 0) && (lddy % 4 == 0) && aligned16(dyo);
  return launch_gemm_nn(al, veca, wtT, Cin, ep, B * H * W, Cin, 4 * Cout, ST);
}
extern "C" size_t tm_convt2x2_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  return tn_ws_bytes(Cin, 4 * Cout, B * H * W) + (size_t)4 * Cout * sizeof(float) + 256;
}
extern "C" int tm_convt2x2_wgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout,
                                      const float* x, int64_t ldx, const float* dyo, int64_t lddy,
                                      int64_t Hy, int64_t Wy, int64_t oy, int64_t ox, float* dwt,
                                      float* dbias, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(ws_bytes >= tm_convt2x2_wgrad_ws(B, H, W, Cin, Cout), "tm_convt2x2_wgrad: workspace too small");
  PlainLoader al{x, ldx, nullptr};
  ConvtLoader bl{dyo, lddy, (int)H, (int)W, (int)Cout, (int)Hy, (int)Wy, (int)oy, (int)ox};
  const bool veca = (Cin % 4 == 0) && (ldx % 4 == 0) && aligned16(x);
  const bool vecb = (Cout % 4 == 0) && (lddy % 4 == 0) && aligned16(dyo);
  float* cs = (float*)ws;                                   // [4*Cout] column sums
  char* rest = (char*)ws + align_up((size_t)4 * Cout * sizeof(float), 256);
  TM_TRY(launch_gemm_tn(al, veca, bl, vecb, Cin, 4 * Cout, B * H * W, dwt, 4 * Cout, nullptr, dbias ? cs : nullptr, 0,
                        rest, ws_bytes - (size_t)(rest - (char*)ws), ST));
  if (dbias) {
    fold4_kernel<<<blocks_for(Cout), 256, 0, ST>>>(Cout, cs, dbias);
    TM_TRY(check_launch("fold4"));
  }
  return 0;
}

namespace {
// Blocks of the statistics sweep: at most BN_BLOCKS, and at least two pixels per pixel lane of a block (a block of
// 256 threads has 256 / (C / VEC) lanes).  The small deep maps (32 x 32 x 128: 1 024 pixels) ran 592 blocks of one
// or two pixels each, whose fixed fp64 fold cost more than the sweep (14 - 16 us against 6 - 9 us for 256 x 256 x 16).
inline int bn_blocks(int64_t npix, int64_t C = 0, bool v4 = false) {
  int64_t n = npix < BN_BLOCKS ? npix : BN_BLOCKS;
  if (C > 0) {
    const int64_t groups = v4 ? C / 4 : C;
    const int64_t lanes = groups < BN_THREADS ? BN_THREADS / groups : 1;
    const int64_t cap = npix / (2 * lanes);
    if (n > cap) n = cap;
  }
  return (int)(n < 1 ? 1 : n);
}
inline bool bn_vec4(int64_t C, std::initializer_list<std::pair<const void*, int64_t>> ts) {
  if (C % 4 != 0 || C > 1024) return false;
  for (auto& t : ts)
    if (t.first && ((reinterpret_cast<uintptr_t>(t.first) % 16 != 0) || (t.second % 4 != 0))) return false;
  return true;
}
}  // namespace

extern "C" size_t tm_bn_ws(int64_t npix, int64_t C) {
  return (size_t)BN_BLOCKS * C * 2 * sizeof(double) + 256;
}

extern "C" size_t tm_bn_seg_ws(int64_t nseg, int64_t npix, int64_t C) {
  return (size_t)nseg * (BN_BLOCKS * C * 2 * sizeof(double) + 2 * C * sizeof(float)) + 256;
}

namespace {
// nseg images of npix pixels each: image k's rows start at x + k * npix * ldx (likewise y, dy, dx; the bf16 copies
// are compact), its statistics at save_mean + k * C.  nseg == 1 is the plain batch-norm call.
int bn_relu_forward_impl(int64_t nseg, int64_t npix, int64_t C, const float* x, int64_t ldx, const float* gamma,
                         const float* beta, float* running_mean, float* running_var, float momentum, float eps, float* y,
                         int64_t ldy, float* save_mean, float* save_invstd, void* y_bf16, const void* stats_part,
                         int64_t nparts, void* ws, size_t ws_bytes, cudaStream_t stream) {
  double* part = (double*)ws;
  const bool v4 = bn_vec4(C, {{x, ldx}, {y, ldy}});
  const int nblk = bn_blocks(npix, C, v4);
  const int groups = v4 ? (int)C / 4 : (int)C;
  const size_t sh = (size_t)(BN_THREADS / groups) * C * 2 * sizeof(double);
  const dim3 sgrid((unsigned)nblk, (unsigned)nseg);
  int nfin = nblk;
  if (stats_part) {                      // statistics already taken by the producing convolution's epilogue
    part = (double*)stats_part;
    nfin = (int)nparts;
  } else {
    if (v4) bn_stats_kernel<4, false><<<sgrid, BN_THREADS, sh, ST>>>(npix, (int)C, x, ldx, nullptr, 0, nullptr, 0, nullptr, nullptr, nullptr, nullptr, part);
    else bn_stats_kernel<1, false><<<sgrid, BN_THREADS, sh, ST>>>(npix, (int)C, x, ldx, nullptr, 0, nullptr, 0, nullptr, nullptr, nullptr, nullptr, part);
    TM_TRY(check_launch("bn_stats"));
  }
  bn_finalize_kernel<<<(unsigned)C, 256, 0, ST>>>(npix, C, nfin, (int)nseg, part, stats_part ? nullptr : x, ldx,
                                                  running_mean, running_var, momentum, eps, save_mean, save_invstd);
  TM_TRY(check_launch("bn_finalize"));
  if (v4) bn_relu_apply_kernel<4><<<dim3(blocks_for(npix * (C / 4)), (unsigned)nseg), 256, 0, ST>>>(npix, (int)C, x, ldx, gamma, beta, save_mean, save_invstd, y, ldy, (__nv_bfloat16*)y_bf16);
  else bn_relu_apply_kernel<1><<<dim3(blocks_for(npix * C), (unsigned)nseg), 256, 0, ST>>>(npix, (int)C, x, ldx, gamma, beta, save_mean, save_invstd, y, ldy, (__nv_bfloat16*)y_bf16);
  return check_launch("bn_relu_apply");
}

int bn_relu_backward_impl(int64_t nseg, int64_t npix, int64_t C, const float* x, int64_t ldx, const float* y,
                          int64_t ldy, const float* dy, int64_t lddy, const float* gamma, const float* beta,
                          const float* save_mean, const float* save_invstd, float* dx, int64_t lddx, float* dgamma,
                          float* dbeta, void* dx_bf16, void* ws, cudaStream_t stream) {
  const bool v4 = bn_vec4(C, {{x, ldx}, {y, ldy}, {dy, lddy}, {dx, lddx}});
  const int nblk = bn_blocks(npix, C, v4);
  double* part = (double*)ws;
  // per-image dgamma / dbeta (what image k's data gradient uses); a single image uses the outputs themselves
  float* dg_seg = nseg > 1 ? reinterpret_cast<float*>(part + nseg * nblk * C * 2) : dgamma;
  float* db_seg = nseg > 1 ? dg_seg + nseg * C : dbeta;
  const int groups = v4 ? (int)C / 4 : (int)C;
  const size_t sh = (size_t)(BN_THREADS / groups) * C * 2 * sizeof(double);
  const dim3 sgrid((unsigned)nblk, (unsigned)nseg);
  if (v4) bn_stats_kernel<4, true><<<sgrid, BN_THREADS, sh, ST>>>(npix, (int)C, x, ldx, y, ldy, dy, lddy, save_mean, save_invstd, gamma, beta, part);
  else bn_stats_kernel<1, true><<<sgrid, BN_THREADS, sh, ST>>>(npix, (int)C, x, ldx, y, ldy, dy, lddy, save_mean, save_invstd, gamma, beta, part);
  TM_TRY(check_launch("bn_bwd_stats"));
  bn_bwd_finalize_kernel<<<(unsigned)C, 256, 0, ST>>>(C, nblk, (int)nseg, part, dg_seg, db_seg, dgamma, dbeta);
  TM_TRY(check_launch("bn_bwd_finalize"));
  if (v4) bn_bwd_apply_kernel<4><<<dim3(blocks_for(npix * (C / 4)), (unsigned)nseg), 256, 0, ST>>>(npix, (int)C, x, ldx, y, ldy, dy, lddy, gamma, beta, save_mean, save_invstd, dg_seg, db_seg, dx, lddx, (__nv_bfloat16*)dx_bf16);
  else bn_bwd_apply_kernel<1><<<dim3(blocks_for(npix * C), (unsigned)nseg), 256, 0, ST>>>(npix, (int)C, x, ldx, y, ldy, dy, lddy, gamma, beta, save_mean, save_invstd, dg_seg, db_seg, dx, lddx, (__nv_bfloat16*)dx_bf16);
  return check_launch("bn_bwd_apply");
}
}  // namespace

/* y_bf16 (optional): compact bf16 copy [npix][C] of y, written by the same pass */
extern "C" int tm_bn_relu_forward(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* gamma,
                                  const float* beta, float* running_mean, float* running_var,
                                  float momentum, float eps, float* y, int64_t ldy, float* save_mean,
                                  float* save_invstd, void* y_bf16, const void* stats_part, int64_t nparts, void* ws,
                                  size_t ws_bytes, void* stream) {
  TM_REQUIRE(npix > 0 && C > 0 && C <= 256, "tm_bn_relu_forward: bad sizes (C <= 256)");
  TM_REQUIRE(ws_bytes >= tm_bn_ws(npix, C), "tm_bn_relu_forward: workspace too small");
  TM_REQUIRE(y || y_bf16, "tm_bn_relu_forward: neither y nor y_bf16 given");
  return bn_relu_forward_impl(1, npix, C, x, ldx, gamma, beta, running_mean, running_var, momentum, eps, y, ldy,
                              save_mean, save_invstd, y_bf16, stats_part, nparts, ws, ws_bytes, ST);
}

extern "C" int tm_bn_relu_forward_seg(int64_t nseg, int64_t npix, int64_t C, const float* x, int64_t ldx,
                                      const float* gamma, const float* beta, float* running_mean, float* running_var,
                                      float momentum, float eps, float* y, int64_t ldy, float* save_mean,
                                      float* save_invstd, void* y_bf16, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(nseg > 0 && nseg <= 65535 && npix > 0 && C > 0 && C <= 256, "tm_bn_relu_forward_seg: bad sizes (C <= 256)");
  TM_REQUIRE(ws_bytes >= tm_bn_seg_ws(nseg, npix, C), "tm_bn_relu_forward_seg: workspace too small");
  TM_REQUIRE(y || y_bf16, "tm_bn_relu_forward_seg: neither y nor y_bf16 given");
  return bn_relu_forward_impl(nseg, npix, C, x, ldx, gamma, beta, running_mean, running_var, momentum, eps, y, ldy,
                              save_mean, save_invstd, y_bf16, nullptr, 0, ws, ws_bytes, ST);
}

namespace {
__global__ void bn_eval_stats_kernel(int C, const float* __restrict__ rm, const float* __restrict__ rv, float eps,
                                     float* __restrict__ mean, float* __restrict__ invstd) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) { mean[c] = rm[c]; invstd[c] = rsqrtf(rv[c] + eps); }
}
}  // namespace

/* nn.BatchNorm2d in EVAL mode + ReLU: y = relu(gamma * (x - running_mean) * rsqrt(running_var + eps) + beta) */
extern "C" int tm_bn_relu_eval(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* gamma, const float* beta,
                               const float* running_mean, const float* running_var, float eps, float* y, int64_t ldy,
                               float* save_mean, float* save_invstd, void* y_bf16, void* stream) {
  TM_REQUIRE(npix > 0 && C > 0 && C <= 256, "tm_bn_relu_eval: bad sizes (C <= 256)");
  TM_REQUIRE(y || y_bf16, "tm_bn_relu_eval: neither y nor y_bf16 given");
  TM_REQUIRE(running_mean && running_var && save_mean && save_invstd, "tm_bn_relu_eval: statistics missing");
  bn_eval_stats_kernel<<<(unsigned)cdiv(C, 128), 128, 0, ST>>>((int)C, running_mean, running_var, eps, save_mean, save_invstd);
  TM_TRY(check_launch("bn_eval_stats"));
  const bool v4 = bn_vec4(C, {{x, ldx}, {y, ldy}});
  if (v4) bn_relu_apply_kernel<4><<<blocks_for(npix * (C / 4)), 256, 0, ST>>>(npix, (int)C, x, ldx, gamma, beta, save_mean, save_invstd, y, ldy, (__nv_bfloat16*)y_bf16);
  else bn_relu_apply_kernel<1><<<blocks_for(npix * C), 256, 0, ST>>>(npix, (int)C, x, ldx, gamma, beta, save_mean, save_invstd, y, ldy, (__nv_bfloat16*)y_bf16);
  return check_launch("bn_relu_apply(eval)");
}

/* dx_bf16 (optional): compact bf16 copy [npix][C] of dx, written by the same pass */
extern "C" int tm_bn_relu_backward(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* y,
                                   int64_t ldy, const float* dy, int64_t lddy, const float* gamma, const float* beta,
                                   const float* save_mean, const float* save_invstd, float* dx,
                                   int64_t lddx, float* dgamma, float* dbeta, void* dx_bf16, void* ws, size_t ws_bytes,
                                   void* stream) {
  TM_REQUIRE(npix > 0 && C > 0 && C <= 256, "tm_bn_relu_backward: bad sizes (C <= 256)");
  TM_REQUIRE(dx || dx_bf16, "tm_bn_relu_backward: neither dx nor dx_bf16 given");
  TM_REQUIRE(y || beta, "tm_bn_relu_backward: without the stored activation y the mask is rebuilt from beta");
  TM_REQUIRE(ws_bytes >= tm_bn_ws(npix, C), "tm_bn_relu_backward: workspace too small");
  return bn_relu_backward_impl(1, npix, C, x, ldx, y, ldy, dy, lddy, gamma, beta, save_mean, save_invstd, dx, lddx,
                               dgamma, dbeta, dx_bf16, ws, ST);
}

extern "C" int tm_bn_relu_backward_seg(int64_t nseg, int64_t npix, int64_t C, const float* x, int64_t ldx,
                                       const float* y, int64_t ldy, const float* dy, int64_t lddy, const float* gamma,
                                       const float* beta, const float* save_mean, const float* save_invstd, float* dx,
                                       int64_t lddx, float* dgamma, float* dbeta, void* dx_bf16, void* ws,
                                       size_t ws_bytes, void* stream) {
  TM_REQUIRE(nseg > 0 && nseg <= 65535 && npix > 0 && C > 0 && C <= 256, "tm_bn_relu_backward_seg: bad sizes (C <= 256)");
  TM_REQUIRE(dx || dx_bf16, "tm_bn_relu_backward_seg: neither dx nor dx_bf16 given");
  TM_REQUIRE(y || beta, "tm_bn_relu_backward_seg: without the stored activation y the mask is rebuilt from beta");
  TM_REQUIRE(ws_bytes >= tm_bn_seg_ws(nseg, npix, C), "tm_bn_relu_backward_seg: workspace too small");
  return bn_relu_backward_impl(nseg, npix, C, x, ldx, y, ldy, dy, lddy, gamma, beta, save_mean, save_invstd, dx, lddx,
                               dgamma, dbeta, dx_bf16, ws, ST);
}

extern "C" int tm_conv1x1_c1_forward(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* w,
                                     const float* bias, float* y, int64_t ldy, void* stream) {
  if (npix <= 0) return 0;
  const bool v4 = (C % 4 == 0) && (ldx % 4 == 0) && aligned16(x);
  if (v4) conv1x1_c1_fwd_kernel<4><<<blocks_for(npix), 256, 0, ST>>>(npix, (int)C, x, ldx, w, bias, y, ldy);
  else conv1x1_c1_fwd_kernel<1><<<blocks_for(npix), 256, 0, ST>>>(npix, (int)C, x, ldx, w, bias, y, ldy);
  return check_launch("conv1x1_c1_fwd");
}
extern "C" int tm_conv1x1_c1_dgrad(int64_t npix, int64_t C, const float* dy, int64_t lddy, const float* w, float* dx,
                                   int64_t lddx, void* stream) {
  if (npix <= 0) return 0;
  if ((C % 4 == 0) && (lddx % 4 == 0) && aligned16(dx))
    conv1x1_c1_dgrad_kernel<4><<<blocks_for(npix * (C / 4)), 256, 0, ST>>>(npix, (int)C, dy, lddy, w, dx, lddx);
  else
    conv1x1_c1_dgrad_kernel<1><<<blocks_for(npix * C), 256, 0, ST>>>(npix, (int)C, dy, lddy, w, dx, lddx);
  return check_launch("conv1x1_c1_dgrad");
}
extern "C" size_t tm_conv1x1_c1_wgrad_ws(int64_t C) { return (size_t)BN_BLOCKS * (C + 1) * sizeof(double) + 256; }
extern "C" int tm_conv1x1_c1_wgrad(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* dy, int64_t lddy,
                                   float* dw, float* dbias, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(npix > 0 && C > 0 && C <= BN_THREADS, "tm_conv1x1_c1_wgrad: bad sizes");
  TM_REQUIRE(ws_bytes >= tm_conv1x1_c1_wgrad_ws(C), "tm_conv1x1_c1_wgrad: workspace too small");
  const int nblk = bn_blocks(npix);
  const size_t sh = (size_t)(BN_THREADS / C) * (C + 1) * sizeof(double);
  conv1x1_c1_wgrad_kernel<<<nblk, BN_THREADS, sh, ST>>>(npix, (int)C, x, ldx, dy, lddy, (double*)ws);
  TM_TRY(check_launch("conv1x1_c1_wgrad"));
  conv1x1_c1_wgrad_final_kernel<<<(unsigned)cdiv((C + 1) * 32, 128), 128, 0, ST>>>((int)C, nblk, (const double*)ws, dw, dbias);
  return check_launch("conv1x1_c1_wgrad_final");
}

namespace {
template <int K, int CIN, typename T>
int conv_dgrad_narrow_launch(int64_t B, int64_t H, int64_t W, int64_t Cout, const void* dy, int64_t lddy, const float* w,
                             float* dx, cudaStream_t st) {
  auto kern = conv_dgrad_narrow_kernel<K, CIN, T>;
  const size_t sh = sizeof(float) * ((size_t)Cout * K * K * ndg_cinp(CIN) + (size_t)NDG_CC * (NDG_TH + K - 1) *
                                     (NDG_TW + K - 1));
  TM_REQUIRE(sh <= 227 * 1024, "tm_conv_dgrad_narrow: Cout = %lld needs %zu bytes of shared memory", (long long)Cout, sh);
  TM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sh));
  const dim3 grid((unsigned)cdiv(W, NDG_TW), (unsigned)cdiv(H, NDG_TH), (unsigned)B);
  kern<<<grid, NDG_THREADS, sh, st>>>((int)H, (int)W, (int)Cout, (const T*)dy, lddy, w, dx);
  return check_launch("conv_dgrad_narrow");
}
template <int K, typename T>
int conv_dgrad_narrow_cin(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const void* dy, int64_t lddy,
                          const float* w, float* dx, cudaStream_t st) {
  switch (Cin) {
    case 1: return conv_dgrad_narrow_launch<K, 1, T>(B, H, W, Cout, dy, lddy, w, dx, st);
    case 2: return conv_dgrad_narrow_launch<K, 2, T>(B, H, W, Cout, dy, lddy, w, dx, st);
    case 3: return conv_dgrad_narrow_launch<K, 3, T>(B, H, W, Cout, dy, lddy, w, dx, st);
    default: return conv_dgrad_narrow_launch<K, 4, T>(B, H, W, Cout, dy, lddy, w, dx, st);
  }
}
template <typename T>
int conv_dgrad_narrow_k(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k, const void* dy,
                        int64_t lddy, const float* w, float* dx, cudaStream_t st) {
  switch (k) {
    case 3: return conv_dgrad_narrow_cin<3, T>(B, H, W, Cin, Cout, dy, lddy, w, dx, st);
    default: return conv_dgrad_narrow_cin<9, T>(B, H, W, Cin, Cout, dy, lddy, w, dx, st);
  }
}
}  // namespace

extern "C" int tm_conv_dgrad_narrow(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                                    const void* dy, int64_t lddy, int dy_bf16, const float* w, float* dx,
                                    void* stream) {
  TM_REQUIRE(B > 0 && H > 0 && W > 0 && B <= 65535 && H * W <= INT32_MAX, "tm_conv_dgrad_narrow: bad sizes");
  TM_REQUIRE(Cin >= 1 && Cin <= 4, "tm_conv_dgrad_narrow: Cin must be 1..4 (got %lld)", (long long)Cin);
  TM_REQUIRE(k == 3 || k == 9, "tm_conv_dgrad_narrow: k must be 3 or 9 (got %lld)", (long long)k);
  TM_REQUIRE(Cout > 0 && Cout % NDG_CC == 0 && lddy >= Cout && lddy % 8 == 0 && ((uintptr_t)dy & 15) == 0,
             "tm_conv_dgrad_narrow: dy needs Cout %% 8 == 0, a pixel stride lddy >= Cout with lddy %% 8 == 0 and 16-byte "
             "alignment (Cout %lld, lddy %lld)", (long long)Cout, (long long)lddy);
  if (dy_bf16)
    return conv_dgrad_narrow_k<__nv_bfloat16>(B, H, W, Cin, Cout, k, dy, lddy, w, dx, ST);
  return conv_dgrad_narrow_k<float>(B, H, W, Cin, Cout, k, dy, lddy, w, dx, ST);
}

extern "C" int tm_pool2x2_forward(int64_t B, int64_t H, int64_t W, int64_t C, int mode, const float* x,
                                  int64_t ldx, float* y, int64_t ldy, uint8_t* idx, int flags, void* stream) {
  TM_REQUIRE(mode == 0 || mode == 1, "tm_pool2x2: mode must be 0 (max) or 1 (avg)");
  const int64_t n = B * (H / 2) * (W / 2) * C;
  if (n <= 0) return 0;
  if (C % 4 == 0 && H % 2 == 0 && W % 2 == 0 && ldx % 4 == 0 && ldy % 4 == 0 && aligned16(x) && aligned16(y) &&
      (!idx || reinterpret_cast<uintptr_t>(idx) % 4 == 0) && B * H * W < (1ll << 31)) {
    pool_fwd_vec_kernel<<<blocks_for(n / 4), 256, 0, ST>>>((int)B, (int)H, (int)W, (int)C, mode, x, ldx, y, ldy, idx,
                                                         (flags & TM_EPI_RELU) != 0);
    return check_launch("pool_fwd_vec");
  }
  pool_fwd_kernel<<<blocks_for(n), 256, 0, ST>>>(B, H, W, C, mode, x, ldx, y, ldy, idx, (flags & TM_EPI_RELU) != 0);
  return check_launch("pool_fwd");
}
extern "C" int tm_pool2x2_backward(int64_t B, int64_t H, int64_t W, int64_t C, int mode, const float* dy,
                                   int64_t lddy, const float* y, int64_t ldy, const uint8_t* idx, float* dx,
                                   int64_t lddx, int flags, const float* add, int64_t ldadd, void* stream) {
  TM_REQUIRE(mode == 0 || mode == 1, "tm_pool2x2: mode must be 0 (max) or 1 (avg)");
  TM_REQUIRE(mode == 1 || idx, "tm_pool2x2_backward: max pooling needs idx");
  const int64_t n = B * H * W * C;
  if (n <= 0) return 0;
  const bool relu = (flags & TM_EPI_RELU) != 0;
  if (C % 4 == 0 && H % 2 == 0 && W % 2 == 0 && lddy % 4 == 0 && lddx % 4 == 0 && aligned16(dy) && aligned16(dx) &&
      (!relu || (ldy % 4 == 0 && aligned16(y))) && (mode != 0 || reinterpret_cast<uintptr_t>(idx) % 4 == 0) &&
      (!add || (ldadd % 4 == 0 && aligned16(add))) && B * H * W < (1ll << 31)) {
    pool_bwd_vec_kernel<<<blocks_for(n / 16), 256, 0, ST>>>((int)B, (int)H, (int)W, (int)C, mode, dy, lddy, y, ldy, idx,
                                                          dx, lddx, relu, add, ldadd);
    return check_launch("pool_bwd_vec");
  }
  pool_bwd_kernel<<<blocks_for(n), 256, 0, ST>>>(B, H, W, C, mode, dy, lddy, y, ldy, idx, dx, lddx, relu);
  if (add) {
    TM_TRY(check_launch("pool_bwd"));
    add_strided_kernel<<<blocks_for(B * H * W * C), 256, 0, ST>>>(B * H * W, C, add, ldadd, dx, lddx);
  }
  return check_launch("pool_bwd");
}
extern "C" int tm_leaky_relu_forward(int64_t n, const float* x, float slope, float* y, void* stream) {
  if (n <= 0) return 0;
  lrelu_fwd_kernel<<<blocks_for(n), 256, 0, ST>>>(n, x, slope, y);
  return check_launch("lrelu_fwd");
}
extern "C" int tm_leaky_relu_backward(int64_t n, const float* y, const float* dy, float slope, float* dx,
                                      void* stream) {
  if (n <= 0) return 0;
  lrelu_bwd_kernel<<<blocks_for(n), 256, 0, ST>>>(n, y, dy, slope, dx);
  return check_launch("lrelu_bwd");
}
extern "C" int tm_add_strided(int64_t npix, int64_t C, const float* src, int64_t lds, float* dst, int64_t ldd,
                              void* stream) {
  if (npix * C <= 0) return 0;
  add_strided_kernel<<<blocks_for(npix * C), 256, 0, ST>>>(npix, C, src, lds, dst, ldd);
  return check_launch("add_strided");
}
