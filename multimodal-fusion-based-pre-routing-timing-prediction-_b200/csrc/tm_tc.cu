// Tensor-core (tcgen05 / TMEM) entry points: dense layers, weight gradients and NHWC convolutions.
//
// Same contracts as the fp32 CUDA-core entry points in tm_gemm.cu / tm_conv.cu (which they replace on
// the hot path); `precision` selects 0 = bf16 operands (U-Net bf16 mode, rtol 2e-2) or 1 = split-bf16
// x3 (fp32-class accuracy, rtol 1e-3).  `err` is an optional device int set to 1 if a tensor-core
// barrier ever times out (never expected; it turns a would-be hang into a detectable failure).
#include "tm_tc.cuh"

using namespace tmk;

namespace {
// widest vector load the operand rows allow: 2 = 256-bit, 1 = 128-bit, 0 = scalar
inline int vec_mode(const void* p, int64_t ld) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  if ((ld % 8 == 0) && (a % 32 == 0)) return 2;
  if ((ld % 4 == 0) && (a % 16 == 0)) return 1;
  return 0;
}
// splits of the reduction dimension so that (tiles x splits) fills the persistent grid once
inline void tn_split(int64_t M, int64_t N, int64_t R, int bn, int* splits, int64_t* k_per_split) {
  const int64_t tiles = cdiv(M, tc::BM) * cdiv(N, bn);
  int64_t want = (int64_t)sm_count() / tiles;
  const int64_t cap = cdiv(R, 4 * tc::BK);
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  int64_t kps = cdiv(cdiv(R, want), tc::BK) * tc::BK;
  *splits = (int)cdiv(R, kps);
  *k_per_split = kps;
}
}  // namespace

extern "C" int tm_tc_gemm_nn(int64_t M, int64_t N, int64_t K, const float* A, int64_t lda,
                             const int32_t* a_rows, const float* B, int64_t ldb, int b_is_nk, float* C,
                             int64_t ldc, const int32_t* c_rows, const float* bias, const float* mask,
                             int64_t ldmask, int flags, int precision, int* err, void* stream) {
  TM_REQUIRE(M >= 0 && N >= 0 && K >= 0, "tm_tc_gemm_nn: negative size");
  TM_REQUIRE(!(flags & TM_EPI_BIAS) || bias, "tm_tc_gemm_nn: TM_EPI_BIAS without bias");
  TM_REQUIRE(!(flags & TM_EPI_MASK) || mask, "tm_tc_gemm_nn: TM_EPI_MASK without mask");
  cudaStream_t st = (cudaStream_t)stream;
  tc::RowLoader al{A, lda, a_rows, M, K, vec_mode(A, lda)};
  PlainEpilogue ep{C, ldc, c_rows, bias, mask, ldmask, flags};
  if (b_is_nk) {
    tc::RowLoader bl{B, ldb, nullptr, N, K, vec_mode(B, ldb)};
    return tc::launch(al, bl, ep, M, N, K, 1, K > 0 ? cdiv(K, tc::BK) * tc::BK : tc::BK, precision, err, st);
  }
  tc::ColLoader bl{B, ldb, nullptr, N, K, vec_mode(B, ldb)};
  return tc::launch(al, bl, ep, M, N, K, 1, K > 0 ? cdiv(K, tc::BK) * tc::BK : tc::BK, precision, err, st);
}

namespace {
// part [slots = G * EPI_WARPS][3][N] -> db1[n], dW1[n][kx].  Block = 32 columns x 8 slot groups (group w adds slots
// w, w+8, ...; coalesced 128-byte loads), folded in a fixed order: deterministic.  (One thread per column walking all
// ~600 slots took 53 us for 2 MB on the backward chain.)
__global__ void __launch_bounds__(256)
mlp1_reduce_kernel(const float* __restrict__ part, int slots, int64_t N, int kx, float* __restrict__ dW1,
                   float* __restrict__ db1) {
  __shared__ float sm[8][3][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t n = (int64_t)blockIdx.x * 32 + lane;
  float s[3] = {0.f, 0.f, 0.f};
  if (n < N) {
#pragma unroll 4
    for (int g = w; g < slots; g += 8)
#pragma unroll
      for (int k = 0; k < 3; ++k) s[k] += part[((int64_t)g * 3 + k) * N + n];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) sm[w][k][lane] = s[k];
  __syncthreads();
  if (w == 0 && n < N) {
#pragma unroll
    for (int k = 0; k < 3; ++k)
      for (int i = 1; i < 8; ++i) s[k] += sm[i][k][lane];
    db1[n] = s[0];
    dW1[n * kx] = s[1];
    if (kx > 1) dW1[n * kx + 1] = s[2];
  }
}
}  // namespace

extern "C" size_t tm_tc_mlp1_bwd_ws(int64_t N) {
  return (size_t)sm_count() * tc::EPI_WARPS * 3 * N * sizeof(float) + 256;
}

extern "C" int tm_tc_mlp1_bwd_fused(int64_t M, int64_t N, int64_t K, const float* G, int64_t ldg, const int32_t* g_rows,
                                    const float* W2t, const float* H, int64_t ldh, const float* X, int64_t ldx,
                                    const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, float* dW1,
                                    float* db1, void* ws, size_t ws_bytes, int* err, void* stream) {
  TM_REQUIRE(M > 0 && N > 0 && N <= 256 && N % 4 == 0 && K > 0, "tm_tc_mlp1_bwd_fused: needs 0 < N <= 256, N % 4 == 0");
  TM_REQUIRE(kx == 1 || kx == 2, "tm_tc_mlp1_bwd_fused: the first layer must have 1 or 2 inputs");
  TM_REQUIRE(H ? ((ldh % 4 == 0) && aligned16(H)) : (W1 && b1),
             "tm_tc_mlp1_bwd_fused: H rows must be 16-byte aligned (or pass W1, b1 to regenerate the mask)");
  TM_REQUIRE(ws && ws_bytes >= tm_tc_mlp1_bwd_ws(N), "tm_tc_mlp1_bwd_fused: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  const int64_t tiles = cdiv(M, tc::BM) * cdiv(N, 128);
  const int grid = (int)(tiles < sm_count() ? tiles : sm_count());
  tc::RowLoader al{G, ldg, g_rows, M, K, vec_mode(G, ldg)};
  tc::RowLoader bl{W2t, K, nullptr, N, K, vec_mode(W2t, K)};
  tc::ReduceEpilogue ep{H, ldh, X, ldx, x_rows, (int)kx, part, W1, b1};
  TM_TRY((tc::launch_tf<tc::RowLoader, tc::RowLoader, tc::ReduceEpilogue, 128, 2>(al, bl, ep, M, N, K, 1, cdiv(K, tc::BK) * tc::BK, err, st)));
  mlp1_reduce_kernel<<<(unsigned)cdiv(N, 32), 256, 0, st>>>(part, grid * tc::EPI_WARPS, N, (int)kx, dW1, db1);
  return check_launch("mlp1_reduce");
}

// out[out_rows[m], :] = relu(X[x_rows[m], 0:kx] @ W1^T + b1) @ W2^T + b2 with the hidden layer generated in
// the A-operand loader (never stored).  W2: [N,K] row-major as nn.Linear stores it (K = hidden width).
extern "C" int tm_tc_mlp2_smallk_forward(int64_t M, int64_t K, int64_t N, const float* X, int64_t ldx,
                                         const int32_t* x_rows, int64_t kx, const float* W1, const float* b1,
                                         const float* W2, const float* b2, float* out, int64_t ldo,
                                         const int32_t* out_rows, int precision, int* err, void* stream) {
  TM_REQUIRE(kx == 1 || kx == 2, "tm_tc_mlp2_smallk_forward: the first layer must have 1 or 2 inputs");
  if (M <= 0 || N <= 0) return 0;
  tc::Hidden2 h{X, ldx, x_rows, W1, b1, (int)kx};
  tc::GenRowLoader al{h, M, K};
  tc::RowLoader bl{W2, K, nullptr, N, K, vec_mode(W2, K)};
  PlainEpilogue ep{out, ldo, out_rows, b2, nullptr, 0, b2 ? TM_EPI_BIAS : 0};
  return tc::launch(al, bl, ep, M, N, K, 1, cdiv(K, tc::BK) * tc::BK, precision, err, (cudaStream_t)stream);
}

// dW2[M_out, hid] = G[g_rows]^T @ hidden, hidden generated in the B-operand loader (R = samples)
extern "C" int tm_tc_mlp2_smallk_wgrad2(int64_t Mo, int64_t hid, int64_t R, const float* G, int64_t ldg,
                                        const int32_t* g_rows, const float* X, int64_t ldx, const int32_t* x_rows,
                                        int64_t kx, const float* W1, const float* b1, float* dW2, int precision,
                                        void* ws, size_t ws_bytes, int* err, void* stream) {
  TM_REQUIRE(kx == 1 || kx == 2, "tm_tc_mlp2_smallk_wgrad2: the first layer must have 1 or 2 inputs");
  if (Mo <= 0 || hid <= 0) return 0;
  TM_REQUIRE(ws_bytes >= tm_tc_gemm_tn_ws(Mo, hid, R), "tm_tc_mlp2_smallk_wgrad2: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  int splits;
  int64_t kps;
  tn_split(Mo, hid, R, tc::pick_bn(hid, precision), &splits, &kps);
  tc::Hidden2 h{X, ldx, x_rows, W1, b1, (int)kx};
  tc::ColLoader al{G, ldg, g_rows, Mo, R, vec_mode(G, ldg)};
  tc::GenColLoader bl{h, hid, R};
  tc::PartialEpilogue ep{(float*)ws, Mo, hid};
  TM_TRY(tc::launch(al, bl, ep, Mo, hid, R, splits, kps, precision, err, st));
  split_reduce_kernel<<<(unsigned)cdiv(Mo * hid, 64), 256, 0, st>>>((const float*)ws, Mo * hid, splits, dW2, hid, hid, 0);
  return check_launch("split_reduce(smallk wgrad2)");
}

extern "C" size_t tm_tc_gemm_tn_ws(int64_t M, int64_t N, int64_t R) {
  size_t worst = 0;                       // the N tile depends on the precision chosen at launch
  for (int prec = 0; prec < 5; ++prec) {
    int splits;
    int64_t kps;
    tn_split(M, N, R, tc::pick_bn(N, prec), &splits, &kps);
    if ((size_t)splits > worst) worst = (size_t)splits;
  }
  return worst * M * N * sizeof(float) + 256;
}

extern "C" int tm_tc_gemm_tn(int64_t M, int64_t N, int64_t R, const float* A, int64_t lda,
                             const int32_t* a_rows, const float* B, int64_t ldb, const int32_t* b_rows,
                             float* C, int64_t ldc, int accumulate, int precision, void* ws, size_t ws_bytes,
                             int* err, void* stream) {
  TM_REQUIRE(M >= 0 && N >= 0 && R >= 0, "tm_tc_gemm_tn: negative size");
  if (M == 0 || N == 0) return 0;
  TM_REQUIRE(ws_bytes >= tm_tc_gemm_tn_ws(M, N, R), "tm_tc_gemm_tn: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  int splits;
  int64_t kps;
  tn_split(M, N, R, tc::pick_bn(N, precision), &splits, &kps);
  tc::ColLoader al{A, lda, a_rows, M, R, vec_mode(A, lda)};
  tc::ColLoader bl{B, ldb, b_rows, N, R, vec_mode(B, ldb)};
  tc::PartialEpilogue ep{(float*)ws, M, N};
  TM_TRY(tc::launch(al, bl, ep, M, N, R, splits, kps, precision, err, st));
  split_reduce_kernel<<<(unsigned)cdiv(M * N, 64), 256, 0, st>>>((const float*)ws, M * N, splits, C, N, ldc, accumulate);
  return check_launch("split_reduce(tc)");
}

extern "C" int tm_tc_conv2d_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                                 const float* x, int64_t ldx, const float* wf, const float* bias, float* y,
                                 int64_t ldy, int flags, int precision, int* err, void* stream) {
  TM_REQUIRE(k >= 1 && (k & 1), "tm_tc_conv2d_nhwc: odd kernel sizes only");
  const int64_t M = B * H * W, K = k * k * Cin;
  tc::Im2colLoader8 al{x, ldx, (int)H, (int)W, (int)Cin, (int)k, (int)(k / 2), M, K,
                       (Cin % 4 == 0) ? vec_mode(x, ldx) : 0};
  tc::ColLoader bl{wf, Cout, nullptr, Cout, K, vec_mode(wf, Cout)};
  PlainEpilogue ep{y, ldy, nullptr, bias, nullptr, 0, (flags & TM_EPI_RELU) | (bias ? TM_EPI_BIAS : 0)};
  return tc::launch(al, bl, ep, M, Cout, K, 1, cdiv(K, tc::BK) * tc::BK, precision, err, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------------
// Split-K form of the convolution for the deep, small-map layers.  One U-Net step at 256 x 256 has layers of
// 64 x 64 and 32 x 32 pixels: 32 and 8 output tiles of 128 pixels -- 22 % and 5 % of the SMs -- each walking
// K = 9 Cin = 576 .. 1152 (measured 34 - 74 us per layer on 8 - 32 CTAs).  Here the K range is cut so that
// tiles x splits fills the GPU; every CTA writes an fp32 partial tile, and one pass adds them in a fixed order
// (deterministic) with the bias / ReLU of the plain epilogue.
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256)
conv_split_reduce_kernel(const float* __restrict__ P, int64_t M, int64_t N, int splits, const float* __restrict__ bias,
                         int relu, float* __restrict__ Y, int64_t ldy) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // one float4 of the M x N result
  const int64_t n4 = N >> 2;
  if (i >= M * n4) return;
  const int64_t m = i / n4, n = (i - m * n4) << 2;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  const float4* p = reinterpret_cast<const float4*>(P + m * N + n);
  const int64_t stride4 = (M * N) >> 2;
#pragma unroll 4
  for (int k = 0; k < splits; ++k) {
    const float4 v = p[(int64_t)k * stride4];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  if (bias) { s.x += bias[n]; s.y += bias[n + 1]; s.z += bias[n + 2]; s.w += bias[n + 3]; }
  if (relu) { s.x = fmaxf(s.x, 0.f); s.y = fmaxf(s.y, 0.f); s.z = fmaxf(s.z, 0.f); s.w = fmaxf(s.w, 0.f); }
  float* y = Y + m * ldy + n;
  if ((ldy & 3) == 0 && (reinterpret_cast<uintptr_t>(Y) & 15) == 0) *reinterpret_cast<float4*>(y) = s;
  else { y[0] = s.x; y[1] = s.y; y[2] = s.z; y[3] = s.w; }
}

// number of K splits of a convolution GEMM (1 = the plain kernel) and the K range of one split
inline int conv_splits(int64_t M, int64_t N, int64_t K, int precision, int64_t* kps) {
  *kps = cdiv(K, tc::BK) * tc::BK;
  static const bool off = getenv("TM_CONV_SPLITK") && atoi(getenv("TM_CONV_SPLITK")) == 0;
  if (off || precision < 3 || (N & 3) || M <= 0) return 1;
  const int64_t tiles = cdiv(M, tc::BM) * cdiv(N, tc::pick_bn(N, precision));
  const int64_t nkb = cdiv(K, tc::BK);
  int64_t want = (int64_t)sm_count() / tiles;
  if (want > nkb / 2) want = nkb / 2;                   // at least two k-blocks per split
  if (want < 2) return 1;
  *kps = cdiv(nkb, want) * tc::BK;
  return (int)cdiv(K, *kps);
}
}  // namespace

namespace tmk {
namespace tc {
int conv_split_fold(const float* part, int64_t M, int64_t N, int splits, const float* bias, int relu, float* y, int64_t ldy,
                    cudaStream_t st) {
  conv_split_reduce_kernel<<<(unsigned)cdiv(M * (N >> 2), 256), 256, 0, st>>>(part, M, N, splits, bias, relu, y, ldy);
  return check_launch("conv_split_reduce");
}
}  // namespace tc
}  // namespace tmk

extern "C" size_t tm_tc_conv2d_splitk_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k, int precision) {
  int64_t kps;
  const int splits = conv_splits(B * H * W, Cout, k * k * Cin, precision, &kps);
  return splits > 1 ? (size_t)splits * (size_t)(B * H * W) * (size_t)Cout * sizeof(float) + 256 : 0;
}

extern "C" int tm_tc_conv2d_nhwc_splitk(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                                        const float* x, int64_t ldx, const float* wf, const float* bias, float* y,
                                        int64_t ldy, int flags, int precision, void* ws, size_t ws_bytes, int* err,
                                        void* stream) {
  TM_REQUIRE(k >= 1 && (k & 1), "tm_tc_conv2d_nhwc_splitk: odd kernel sizes only");
  const int64_t M = B * H * W, K = k * k * Cin;
  int64_t kps;
  const int splits = conv_splits(M, Cout, K, precision, &kps);
  if (splits <= 1) return tm_tc_conv2d_nhwc(B, H, W, Cin, Cout, k, x, ldx, wf, bias, y, ldy, flags, precision, err, stream);
  TM_REQUIRE(ws && ws_bytes >= tm_tc_conv2d_splitk_ws(B, H, W, Cin, Cout, k, precision),
             "tm_tc_conv2d_nhwc_splitk: workspace too small (tm_tc_conv2d_splitk_ws)");
  cudaStream_t st = (cudaStream_t)stream;
  float* part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  tc::Im2colLoader8 al{x, ldx, (int)H, (int)W, (int)Cin, (int)k, (int)(k / 2), M, K,
                       (Cin % 4 == 0) ? vec_mode(x, ldx) : 0};
  tc::ColLoader bl{wf, Cout, nullptr, Cout, K, vec_mode(wf, Cout)};
  tc::PartialEpilogue ep{part, M, Cout};
  const int bn = tc::pick_bn(Cout, precision);
#define TM_CONV_SPLIT_CASE(BN_)                                                                                              \
  TM_TRY((precision == 3 ? tc::launch_tf<tc::Im2colLoader8, tc::ColLoader, tc::PartialEpilogue, BN_, 2>(al, bl, ep, M, Cout, K, splits, kps, err, st) \
                         : tc::launch_tf<tc::Im2colLoader8, tc::ColLoader, tc::PartialEpilogue, BN_, 1>(al, bl, ep, M, Cout, K, splits, kps, err, st)))
  switch (bn) {
    case 128: TM_CONV_SPLIT_CASE(128); break;
    case 64: TM_CONV_SPLIT_CASE(64); break;
    default: TM_CONV_SPLIT_CASE(32); break;
  }
#undef TM_CONV_SPLIT_CASE
  return tc::conv_split_fold(part, M, Cout, splits, bias, (flags & TM_EPI_RELU) ? 1 : 0, y, ldy, st);
}

extern "C" size_t tm_tc_conv2d_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k) {
  return tm_tc_gemm_tn_ws(k * k * Cin, Cout, B * H * W);
}

extern "C" int tm_tc_conv2d_wgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                                       const float* x, int64_t ldx, const float* dy, int64_t lddy, float* dwf,
                                       int precision, void* ws, size_t ws_bytes, int* err, void* stream) {
  const int64_t M = k * k * Cin, N = Cout, R = B * H * W;
  TM_REQUIRE(ws_bytes >= tm_tc_gemm_tn_ws(M, N, R), "tm_tc_conv2d_wgrad: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  int splits;
  int64_t kps;
  tn_split(M, N, R, tc::pick_bn(N, precision), &splits, &kps);
  tc::Im2colColLoader al{x, ldx, (int)H, (int)W, (int)Cin, (int)k, (int)(k / 2), M, R, (Cin % 4 == 0) ? vec_mode(x, ldx) : 0};
  tc::ColLoader bl{dy, lddy, nullptr, N, R, vec_mode(dy, lddy)};
  tc::PartialEpilogue ep{(float*)ws, M, N};
  TM_TRY(tc::launch(al, bl, ep, M, N, R, splits, kps, precision, err, st));
  split_reduce_kernel<<<(unsigned)cdiv(M * N, 64), 256, 0, st>>>((const float*)ws, M * N, splits, dwf, N, N, 0);
  return check_launch("split_reduce(tc conv)");
}

/* At most `cap` persistent CTAs for the tcgen05 GEMM / convolution launches made by the calling thread from now on
 * (0 = one per SM, the default).  Returns the previous value. */
extern "C" int tm_tc_set_grid_cap(int cap) {
  const int prev = tc::tc_grid_cap();
  tc::tc_grid_cap() = cap < 0 ? 0 : cap;
  return prev;
}
