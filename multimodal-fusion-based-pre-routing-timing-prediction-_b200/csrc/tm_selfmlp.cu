// Hoisted self-term MLP of the net pins, fused (round 2):  out[out_rows[m]] = W2 relu(W1 x[x_rows[m]] + b1) + b2
// with x of width 1 or 2 (fc_net_self, model.py:46,151: Linear(2, 256) -> ReLU -> Linear(256, 128) over every odd-level
// pin -- 229 819 rows in config 2).  The hidden layer costs two FMAs per element, so it is never stored: generator
// warps write it straight into the tensor-core operand planes, chunk by chunk, and the second layer runs on
// tcgen05.mma with the accumulator in TMEM.
//
// Why a kernel of its own: the generic streaming GEMM (tm_tc.cuh) is bound by the shared-memory traffic of fp32-sized
// operands -- 2 100 cycles per 32-wide k-block, 266 us for this product.  Here
//   * operands are the fp16 two-term split (tm_split.cuh) with a per-row scale: ~22-bit products at the fp16 MMA rate
//     and half the operand bytes;
//   * W2 is split ONCE (tm_selfmlp_pack) and stays resident in shared memory (2 x 64 KB planes), so a k-step reads
//     8 KB instead of 24 KB and nothing is re-staged per tile;
//   * the per-row scale comes from a bound (|x0| max|w0| + |x1| max|w1| + max|b1| >= every hidden unit of the row), so
//     the row is generated once, with no maximum pass.
// Roles of the 416 threads of a persistent CTA (one per SM): warps 0-3 epilogue (TMEM lane quarter = warp, a lane
// owns one output row and writes it as 128-bit stores), warp 4 issues the MMAs, warps 5-12 generate.  The hidden
// tile moves through two 64-wide chunk buffers (full / empty mbarriers), the accumulators (main + corr, 128 columns
// each) are double-buffered in TMEM so the epilogue of tile t overlaps the products of tile t+1.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "tm_common.cuh"
#include "tm_sm100.cuh"
#include "tm_split.cuh"

using namespace tmk;
using namespace tmk::sm100;

namespace tmk {   // tm_gemm.cu: C[m][n] (+)= sum_k P[k][m*N + n], fixed order
__global__ void split_reduce_kernel(const float* __restrict__ P, int64_t count, int splits, float* __restrict__ C, int64_t N,
                                    int64_t ldc, int accumulate);
}

namespace {
constexpr int TM = 128;            // rows per tile (MMA M)
constexpr int HIDF = 256;          // hidden width (MMA K)
constexpr int NOUT = 128;          // outputs (MMA N)
constexpr int KC = 64;             // hidden units per chunk buffer
constexpr int NCH = HIDF / KC;     // chunks per tile
constexpr int EPI_W = 4, GEN_W = 8;
constexpr int MMA_WARP = EPI_W, GEN_WARP0 = EPI_W + 1;
constexpr int THREADS = (EPI_W + 1 + GEN_W) * 32;    // 416
static_assert(GEN_W == KC / 8, "one generator warp per k-group of a chunk");

// K-major SWIZZLE_NONE operand planes (core matrix = 8 rows x 16 bytes):
//   off(row, k) = (row / 8) * SBO + (k / 8) * LBO + (row % 8) * 16 + (k % 8) * 2          [bytes, fp16]
constexpr uint32_t W_LBO = 128, W_SBO = (HIDF / 8) * W_LBO, W_PLANE = (NOUT / 8) * W_SBO;   // 64 KB
// (hidden chunk planes: the k-group stride is padded by 16 bytes so that the 8-byte stores of the loaders -- a lane
//  holds four consecutive k of one row -- spread over the banks)
constexpr uint32_t H_LBO = 144, H_SBO = (KC / 8) * H_LBO, H_PLANE = (TM / 8) * H_SBO;      // 18 KB
constexpr uint32_t OFF_W = 0;                              // Whi, Wlo
constexpr uint32_t OFF_H = OFF_W + 2 * W_PLANE;            // [buffer 2][hi, lo]
constexpr uint32_t OFF_P = OFF_H + 4 * H_PLANE;            // w0[256], w1[256], b1[256], b2[128], maxima[4]
constexpr uint32_t OFF_BAR = OFF_P + (3 * HIDF + NOUT + 4) * 4;
constexpr uint32_t SMEM_BYTES = OFF_BAR + 16 * 8 + 16;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");
constexpr uint32_t TM_COLS = 512;                          // [acc buffer 2][main 128 | corr 128]
constexpr uint32_t MBAR_SPINS = 1u << 22;                  // mbarrier waits trap after this many probes

// W2 [NOUT][HIDF] fp32 (nn.Linear layout: K-major as it is) -> the shared-memory image of the (hi, lo') planes
__global__ void selfmlp_pack_kernel(const float* __restrict__ W2, uint8_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NOUT * HIDF) return;
  const int n = i / HIDF, k = i - n * HIDF;
  __half h, l;
  split_h(W2[i], h, l);
  const uint32_t off = (uint32_t)(n >> 3) * W_SBO + (uint32_t)(k >> 3) * W_LBO + (uint32_t)(n & 7) * 16 + (uint32_t)(k & 7) * 2;
  *reinterpret_cast<__half*>(out + off) = h;
  *reinterpret_cast<__half*>(out + W_PLANE + off) = l;
}

struct Args {
  int64_t M;
  const float* X;
  int64_t ldx;
  const int* x_rows;
  int kx;
  const float* W1;      // [HIDF][kx]
  const float* b1;
  const float* b2;
  const uint8_t* wplanes;
  float* out;
  int64_t ldo;
  const int* out_rows;
  // LOADED form (tm_selfmlp_rows_forward): the hidden layer is read, not generated
  const float* H;         // [.][ldh] stored hidden activations
  int64_t ldh;
  const int* h_rows;      // row of H (and of rowmax) for row m (NULL: m)
  const float* rowmax;    // max |H[r]| per row (tm_selfmlp_lin1_relu writes it): the per-row operand scale
};

// LOADED == false: the hidden layer is generated from 1-2 inputs (fc_net_self).  LOADED == true: second layer of an MLP
// whose hidden activations are stored (fc_cell_self): the same pipeline with loaders in place of the generators.
template <bool LOADED>
__global__ void __launch_bounds__(THREADS, 1) selfmlp_gen_fwd_kernel(Args a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  float* w0_s = reinterpret_cast<float*>(smem + OFF_P);
  float* w1_s = w0_s + HIDF;
  float* b1_s = w1_s + HIDF;
  float* b2_s = b1_s + HIDF;
  float* max_s = b2_s + NOUT;                                  // max|w0|, max|w1|, max|b1|
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t *h_full = bars, *h_empty = bars + 2, *acc_full = bars + 4, *acc_empty = bars + 6, *wbar = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t ntiles = (a.M + TM - 1) / TM;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&h_full[i], GEN_W); mbar_init(&h_empty[i], 1);
      mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], EPI_W);
    }
    mbar_init(wbar, 1);
    fence_mbarrier_init();
    fence_async_smem();
    // resident weight planes: 128 KB in four bulk copies
    mbar_expect_tx(wbar, 2 * W_PLANE);
    for (int i = 0; i < 4; ++i)
      bulk_copy_g2s(smem_u32(smem + OFF_W + i * (W_PLANE / 2)), a.wplanes + (size_t)i * (W_PLANE / 2), W_PLANE / 2, wbar);
  }
  for (int j = tid; j < HIDF; j += THREADS) {
    w0_s[j] = LOADED ? 0.f : a.W1[(size_t)j * a.kx];
    w1_s[j] = (!LOADED && a.kx > 1) ? a.W1[(size_t)j * a.kx + 1] : 0.f;
    b1_s[j] = LOADED ? 0.f : a.b1[j];
  }
  for (int j = tid; j < NOUT; j += THREADS) b2_s[j] = a.b2 ? a.b2[j] : 0.f;
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) {                                            // bounds of the first layer (for the per-row scale)
    float m0 = 0.f, m1 = 0.f, mb = 0.f;
    for (int j = lane; j < HIDF; j += 32) { m0 = fmaxf(m0, fabsf(w0_s[j])); m1 = fmaxf(m1, fabsf(w1_s[j])); mb = fmaxf(mb, fabsf(b1_s[j])); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o));
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
      mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, o));
    }
    if (lane == 0) { max_s[0] = m0; max_s[1] = m1; max_s[2] = mb; }
  }
  __syncthreads();
  const uint32_t tmem_base = *tmem_slot;
  const float wm0 = max_s[0], wm1 = max_s[1], bm = max_s[2];
  auto row_x = [&](int64_t m, float& x0, float& x1) {
    x0 = 0.f; x1 = 0.f;
    if (m < a.M) {
      const float* xp = a.X + (a.x_rows ? (int64_t)a.x_rows[m] : m) * a.ldx;
      x0 = xp[0];
      if (a.kx > 1) x1 = xp[1];
    }
  };

  if (LOADED && warp >= GEN_WARP0) {
    // ======================= loaders: stored hidden rows -> operand planes =======================
    // Warp gw owns rows 16 gw .. 16 gw + 15 of the tile.  Per chunk (64 hidden units = 256 bytes of a row) a load
    // instruction reads TWO whole 256-byte row pieces (half a warp each, 16 bytes per lane), so a lane holds four
    // consecutive k of one row: one 8-byte store per plane.  The next chunk's eight loads are issued before the
    // current chunk is split and stored.
    const int gw = warp - GEN_WARP0;
    const int sub = lane >> 4, kq = lane & 15;                 // which of the two rows of a load; 4-wide k piece
    uint32_t g = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
      const float* hp[8];
      float sc[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int64_t m = t * TM + gw * 16 + 2 * i + sub;
        hp[i] = nullptr; sc[i] = 1.f;
        if (m < a.M) {
          const int64_t r = a.h_rows ? (int64_t)a.h_rows[m] : m;
          hp[i] = a.H + r * a.ldh + kq * 4;
          float inv;
          row_scale(a.rowmax[r], -100, sc[i], inv);
        }
      }
      float4 cur[8], nxt[8];
      auto fetch = [&](int c, float4 (&v)[8]) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (hp[i]) v[i] = __ldg(reinterpret_cast<const float4*>(hp[i] + c * KC));
        }
      };
      fetch(0, cur);
#pragma unroll
      for (int c = 0; c < NCH; ++c, ++g) {
        if (c + 1 < NCH) fetch(c + 1, nxt);
        const uint32_t buf = g & 1u;
        mbar_wait_trap<MBAR_SPINS>(&h_empty[buf], ((g >> 1) & 1u) ^ 1u);
        uint8_t* hi_p = smem + OFF_H + buf * 2 * H_PLANE + (uint32_t)(kq >> 1) * H_LBO + (uint32_t)(kq & 1) * 8;
        uint8_t* lo_p = hi_p + H_PLANE;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int row = gw * 16 + 2 * i + sub;
          uint32_t h0, l0, h1, l1;
          split_pair(cur[i].x * sc[i], cur[i].y * sc[i], h0, l0);
          split_pair(cur[i].z * sc[i], cur[i].w * sc[i], h1, l1);
          const uint32_t off = (uint32_t)(row >> 3) * H_SBO + (uint32_t)(row & 7) * 16;
          *reinterpret_cast<uint2*>(hi_p + off) = make_uint2(h0, h1);
          *reinterpret_cast<uint2*>(lo_p + off) = make_uint2(l0, l1);
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_full[buf]);
        if (c + 1 < NCH) {
#pragma unroll
          for (int i = 0; i < 8; ++i) cur[i] = nxt[i];
        }
      }
    }
  } else if (warp >= GEN_WARP0) {
    // ======================= generators: hidden chunks -> operand planes =======================
    // Warp gw owns k-group gw of EVERY chunk (hidden units c*64 + 8 gw .. + 7): their first-layer parameters live in
    // registers for the whole kernel (96 values, identical in every lane), a lane owns four rows of the tile.  No
    // shared-memory reads in the loop: it shares the shared-memory pipe with the MMA operand fetch.
    const int gw = warp - GEN_WARP0;
    float pw0[NCH][8], pw1[NCH][8], pb[NCH][8];
#pragma unroll
    for (int c = 0; c < NCH; ++c)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int j = c * KC + gw * 8 + e;
        pw0[c][e] = w0_s[j]; pw1[c][e] = w1_s[j]; pb[c][e] = b1_s[j];
      }
    uint32_t g = 0;                                           // chunk counter (buffer = g & 1)
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
      float x0[4], x1[4], sc[4];
#pragma unroll
      for (int rb = 0; rb < 4; ++rb) {
        row_x(t * TM + rb * 32 + lane, x0[rb], x1[rb]);
        float inv;
        row_scale(fmaf(fabsf(x0[rb]), wm0, fmaf(fabsf(x1[rb]), wm1, bm)), -100, sc[rb], inv);
      }
#pragma unroll
      for (int c = 0; c < NCH; ++c, ++g) {
        const uint32_t buf = g & 1u;
        mbar_wait_trap<MBAR_SPINS>(&h_empty[buf], ((g >> 1) & 1u) ^ 1u);       // the MMAs that read this buffer two chunks ago are done
        uint8_t* hi_p = smem + OFF_H + buf * 2 * H_PLANE + (uint32_t)gw * H_LBO;
        uint8_t* lo_p = hi_p + H_PLANE;
#pragma unroll
        for (int rb = 0; rb < 4; ++rb) {
          const int row = rb * 32 + lane;
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int e = 0; e < 8; e += 2) {
            const float y0 = fmaxf(fmaf(pw0[c][e], x0[rb], fmaf(pw1[c][e], x1[rb], pb[c][e])), 0.f) * sc[rb];
            const float y1 = fmaxf(fmaf(pw0[c][e + 1], x0[rb], fmaf(pw1[c][e + 1], x1[rb], pb[c][e + 1])), 0.f) * sc[rb];
            split_pair(y0, y1, hw[e >> 1], lw[e >> 1]);
          }
          const uint32_t off = (uint32_t)(row >> 3) * H_SBO + (uint32_t)(row & 7) * 16;
          *reinterpret_cast<uint4*>(hi_p + off) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(lo_p + off) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
        fence_async_smem();                                   // generic stores -> async proxy (UMMA reads)
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_full[buf]);
      }
    }
  } else if (warp == MMA_WARP) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      mbar_wait_trap<MBAR_SPINS>(wbar, 0);
      const uint32_t idesc = make_idesc(Fmt::F16, NOUT);
      const uint32_t w_hi = smem_u32(smem + OFF_W), w_lo = w_hi + W_PLANE;
      uint32_t g = 0;
      int li = 0;
      for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
        const uint32_t ab = (uint32_t)li & 1u;
        mbar_wait_trap<MBAR_SPINS>(&acc_empty[ab], (((uint32_t)li >> 1) & 1u) ^ 1u);   // the epilogue drained this accumulator pair
        tc_fence_after();
        const uint32_t t_main = tmem_base + ab * 256u, t_corr = t_main + 128u;
        for (int c = 0; c < NCH; ++c, ++g) {
          const uint32_t buf = g & 1u;
          mbar_wait_trap<MBAR_SPINS>(&h_full[buf], (g >> 1) & 1u);
          tc_fence_after();
          const uint32_t h_hi = smem_u32(smem + OFF_H + buf * 2 * H_PLANE), h_lo = h_hi + H_PLANE;
#pragma unroll
          for (int ks = 0; ks < KC / 16; ++ks) {
            const uint32_t wk = (uint32_t)(c * (KC / 8) + ks * 2) * W_LBO;
            const uint64_t ah = smem_desc(h_hi + ks * 2 * H_LBO, H_LBO, H_SBO), al = smem_desc(h_lo + ks * 2 * H_LBO, H_LBO, H_SBO);
            const uint64_t bh = smem_desc(w_hi + wk, W_LBO, W_SBO), bl = smem_desc(w_lo + wk, W_LBO, W_SBO);
            const uint32_t acc = (c > 0 || ks > 0) ? 1u : 0u;
            umma_f16(t_main, ah, bh, idesc, acc);
            umma_f16(t_corr, ah, bl, idesc, acc);
            umma_f16(t_corr, al, bh, idesc, 1u);
          }
          umma_commit(&h_empty[buf]);                          // buffer reusable once these MMAs retire
        }
        umma_commit(&acc_full[ab]);                            // covers every MMA of the tile
      }
    }
    __syncwarp();
  } else {
    // ======================= epilogue: a lane owns one output row =======================
    int li = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
      const uint32_t ab = (uint32_t)li & 1u;
      const int64_t m = t * TM + warp * 32 + lane;
      float s, inv;
      if constexpr (LOADED) {
        s = 1.f; inv = 1.f;
        if (m < a.M) row_scale(a.rowmax[a.h_rows ? (int64_t)a.h_rows[m] : m], -100, s, inv);
      } else {
        float x0, x1;
        row_x(m, x0, x1);
        row_scale(fmaf(fabsf(x0), wm0, fmaf(fabsf(x1), wm1, bm)), -100, s, inv);
      }
      float* op = nullptr;
      if (m < a.M) op = a.out + (a.out_rows ? (int64_t)a.out_rows[m] : m) * a.ldo;
      mbar_wait_trap<MBAR_SPINS>(&acc_full[ab], ((uint32_t)li >> 1) & 1u);
      tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + ab * 256u;
#pragma unroll 1
      for (int c = 0; c < NOUT; c += 32) {
        float vm[32], vc[32];
        tmem_ld32(trow + (uint32_t)c, vm);
        tmem_ld32(trow + 128u + (uint32_t)c, vc);
        if (op) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float4 o;
            o.x = fmaf(fmaf(vc[4 * j], LO_INV, vm[4 * j]), inv, b2_s[c + 4 * j]);
            o.y = fmaf(fmaf(vc[4 * j + 1], LO_INV, vm[4 * j + 1]), inv, b2_s[c + 4 * j + 1]);
            o.z = fmaf(fmaf(vc[4 * j + 2], LO_INV, vm[4 * j + 2]), inv, b2_s[c + 4 * j + 2]);
            o.w = fmaf(fmaf(vc[4 * j + 3], LO_INV, vm[4 * j + 3]), inv, b2_s[c + 4 * j + 3]);
            st4(op + c + 4 * j, o);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[ab]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(tmem_base, TM_COLS);
}

// =============================================================================================
// Second-layer weight gradient:  dW2[o][j] = sum_r G[g_rows[r]][o] * relu(w0_j x0[r] + w1_j x1[r] + b_j)
//   D[M = 128 o][N = 256 j] += A[o][k = row] . B[j][k = row]^T, 64 rows per step, both operands K-major with k = row:
//   A = G transposed on the way in (a lane owns one o and eight consecutive rows: eight coalesced 128-byte loads per
//       warp, one 16-byte store per plane), B = the hidden layer generated by the thread that owns hidden unit j
//       (its three first-layer parameters in registers, the step's 64 inputs broadcast from shared memory).
// The contraction runs over the rows, so the operand scales must not depend on the row: G is scaled by a power of two
// from max|G| (gmax, device scalar), the hidden layer by one from the largest row bound (a small pass over X).  Values
// 2^-14 below the maximum keep fewer than 22 bits (absolute error <= 2^-36 of the maximum per product).
// One accumulator pair (main / corr, 256 columns each) stays in TMEM for the whole kernel; every CTA owns a contiguous
// range of steps and writes one partial dW2 at the end (folded by split_reduce in a fixed order: deterministic).
// =============================================================================================
constexpr int WG_KS = 64;                                   // rows per step (MMA K = 4 x 16)
constexpr int WG_TR_W = 4;                                  // transposer warps
constexpr int WG_THREADS = (1 + GEN_W + WG_TR_W) * 32;      // warp 0 MMA, 1..8 generators, 9..12 transposers = 416
constexpr uint32_t WG_LBO = 128, WG_SBO = (WG_KS / 8) * WG_LBO;             // 1024
// A planes: the 8-row-group stride is padded by 16 bytes so that the transposers' stores (lane = 4 outputs) hit 8
// different 16-byte columns per quarter warp
constexpr uint32_t WG_A_SBO = WG_SBO + 16;
constexpr uint32_t WG_A_PLANE = (NOUT / 8) * WG_A_SBO, WG_B_PLANE = (HIDF / 8) * WG_SBO;   // 16.25 KB, 32 KB
constexpr uint32_t WG_BUF = 2 * WG_A_PLANE + 2 * WG_B_PLANE;                // 96 KB: Ahi, Alo, Bhi, Blo
constexpr uint32_t WG_OFF_X = 2 * WG_BUF;                                   // [buffer 2][x0 64 | x1 64] fp32
constexpr uint32_t WG_OFF_BAR = WG_OFF_X + 2 * 2 * WG_KS * 4;
constexpr uint32_t WG_SMEM = WG_OFF_BAR + 8 * 8 + 16;
static_assert(WG_SMEM <= 232448, "shared memory budget");

// max |x0|, max |x1| over the rows (non-negative floats order like their bit patterns)
__global__ void selfmlp_xmax_kernel(int64_t M, const float* __restrict__ X, int64_t ldx, const int* __restrict__ x_rows, int kx,
                                    unsigned int* __restrict__ out2) {
  float m0 = 0.f, m1 = 0.f;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < M; r += (int64_t)gridDim.x * blockDim.x) {
    const float* xp = X + (x_rows ? (int64_t)x_rows[r] : r) * ldx;
    m0 = fmaxf(m0, fabsf(xp[0]));
    if (kx > 1) m1 = fmaxf(m1, fabsf(xp[1]));
  }
  for (int o = 16; o > 0; o >>= 1) {
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
  }
  if ((threadIdx.x & 31) == 0) {
    if (m0 > 0.f) atomicMax(out2, __float_as_uint(m0));
    if (m1 > 0.f) atomicMax(out2 + 1, __float_as_uint(m1));
  }
}

struct WgArgs {
  int64_t M;
  const float* G;
  int64_t ldg;
  const int* g_rows;
  const float* X;
  int64_t ldx;
  const int* x_rows;
  int kx;
  const float* W1;
  const float* b1;
  const float* gmax;      // device: max |G|
  const float* xmax;      // device: max |x0|, max |x1|
  float* part;            // [grid][128][256]
};

__global__ void __launch_bounds__(WG_THREADS, 1) selfmlp_gen_wgrad2_kernel(WgArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + WG_OFF_BAR);
  uint64_t *full = bars, *empty = bars + 2, *done = bars + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  __shared__ float wmax_s[3];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t nsteps = (a.M + WG_KS - 1) / WG_KS;
  const int64_t per = (nsteps + gridDim.x - 1) / gridDim.x;
  const int64_t s0 = (int64_t)blockIdx.x * per, s1 = (s0 + per < nsteps) ? s0 + per : nsteps;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) { mbar_init(&full[i], GEN_W + WG_TR_W); mbar_init(&empty[i], 1); }
    mbar_init(done, 1);
    fence_mbarrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, TM_COLS);
  if (warp == 1) {                                            // bounds of the first layer
    float m0 = 0.f, m1 = 0.f, mb = 0.f;
    for (int j = lane; j < HIDF; j += 32) {
      m0 = fmaxf(m0, fabsf(a.W1[(size_t)j * a.kx]));
      if (a.kx > 1) m1 = fmaxf(m1, fabsf(a.W1[(size_t)j * a.kx + 1]));
      mb = fmaxf(mb, fabsf(a.b1[j]));
    }
    for (int o = 16; o > 0; o >>= 1) {
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o));
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o));
      mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, o));
    }
    if (lane == 0) { wmax_s[0] = m0; wmax_s[1] = m1; wmax_s[2] = mb; }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // global operand scales (powers of two)
  float sg, ig, sh, ih;
  row_scale(fmaxf(a.gmax[0], 1e-37f), -100, sg, ig);
  row_scale(fmaf(a.xmax[0], wmax_s[0], fmaf(a.xmax[1], wmax_s[1], wmax_s[2])), -100, sh, ih);

  if (warp == 0) {
    // ======================= MMA issuer =======================
    if (lane == 0 && s1 > s0) {
      const uint32_t idesc = make_idesc(Fmt::F16, HIDF);
      const uint32_t t_main = tmem_base, t_corr = tmem_base + 256u;
      uint32_t g = 0;
      for (int64_t st = s0; st < s1; ++st, ++g) {
        const uint32_t buf = g & 1u;
        mbar_wait_trap<MBAR_SPINS>(&full[buf], (g >> 1) & 1u);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(smem + buf * WG_BUF), a_lo = a_hi + WG_A_PLANE;
        const uint32_t b_hi = a_hi + 2 * WG_A_PLANE, b_lo = b_hi + WG_B_PLANE;
#pragma unroll
        for (int ks = 0; ks < WG_KS / 16; ++ks) {
          const uint64_t ah = smem_desc(a_hi + ks * 2 * WG_LBO, WG_LBO, WG_A_SBO), al = smem_desc(a_lo + ks * 2 * WG_LBO, WG_LBO, WG_A_SBO);
          const uint64_t bh = smem_desc(b_hi + ks * 2 * WG_LBO, WG_LBO, WG_SBO), bl = smem_desc(b_lo + ks * 2 * WG_LBO, WG_LBO, WG_SBO);
          const uint32_t acc = (g > 0 || ks > 0) ? 1u : 0u;
          umma_f16(t_main, ah, bh, idesc, acc);
          umma_f16(t_corr, ah, bl, idesc, acc);
          umma_f16(t_corr, al, bh, idesc, 1u);
        }
        umma_commit(&empty[buf]);
      }
      umma_commit(done);
    }
    __syncwarp();
  } else if (warp <= GEN_W) {
    // ======================= generators: thread = hidden unit j, B[j][k = row] =======================
    const int j = tid - 32;
    const float w0 = a.W1[(size_t)j * a.kx], w1 = a.kx > 1 ? a.W1[(size_t)j * a.kx + 1] : 0.f, bj = a.b1[j];
    const uint32_t jbase = (uint32_t)(j >> 3) * WG_SBO + (uint32_t)(j & 7) * 16;
    uint32_t g = 0;
    for (int64_t st = s0; st < s1; ++st, ++g) {
      const uint32_t buf = g & 1u;
      mbar_wait_trap<MBAR_SPINS>(&empty[buf], ((g >> 1) & 1u) ^ 1u);
      float* xs = reinterpret_cast<float*>(smem + WG_OFF_X) + buf * 2 * WG_KS;
      if (j < WG_KS) {                                        // the step's inputs (rows past M: 0, and G is 0 there too)
        const int64_t r = st * WG_KS + j;
        float x0 = 0.f, x1 = 0.f;
        if (r < a.M) {
          const float* xp = a.X + (a.x_rows ? (int64_t)a.x_rows[r] : r) * a.ldx;
          x0 = xp[0];
          if (a.kx > 1) x1 = xp[1];
        }
        xs[j] = x0; xs[WG_KS + j] = x1;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(GEN_W * 32) : "memory");
      uint8_t* hi_p = smem + buf * WG_BUF + 2 * WG_A_PLANE + jbase;
      uint8_t* lo_p = hi_p + WG_B_PLANE;
#pragma unroll 2
      for (int rg = 0; rg < WG_KS / 8; ++rg) {
        const float4 xa = *reinterpret_cast<const float4*>(xs + rg * 8), xb = *reinterpret_cast<const float4*>(xs + rg * 8 + 4);
        const float4 ya = *reinterpret_cast<const float4*>(xs + WG_KS + rg * 8), yb = *reinterpret_cast<const float4*>(xs + WG_KS + rg * 8 + 4);
        const float x0v[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
        const float x1v[8] = {ya.x, ya.y, ya.z, ya.w, yb.x, yb.y, yb.z, yb.w};
        uint32_t hw[4], lw[4];
#pragma unroll
        for (int e = 0; e < 8; e += 2) {
          const float y0 = fmaxf(fmaf(w0, x0v[e], fmaf(w1, x1v[e], bj)), 0.f) * sh;
          const float y1 = fmaxf(fmaf(w0, x0v[e + 1], fmaf(w1, x1v[e + 1], bj)), 0.f) * sh;
          split_pair(y0, y1, hw[e >> 1], lw[e >> 1]);
        }
        *reinterpret_cast<uint4*>(hi_p + rg * WG_LBO) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4*>(lo_p + rg * WG_LBO) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[buf]);
    }
  } else {
    // ======================= transposers: A[o][k = row] from G rows =======================
    // Warp tw owns row groups tw and tw + 4 of the step (8 consecutive rows each).  A lane reads 16 bytes (4 outputs
    // o = 4 lane ..) of each row -- a warp-wide load is one whole 512-byte row -- and then holds, for each of its four
    // outputs, eight consecutive rows: one 16-byte store per output and plane.  The rows of the NEXT step are loaded
    // into registers right after this step's stores, so they are in flight while the generators and the MMAs work.
    const int tw = warp - (1 + GEN_W);
    float4 v[2][8];
    auto fetch = [&](int64_t st) {
      const int64_t r0 = st * WG_KS;
      int id0 = -1, id1 = -1;                               // row ids: two coalesced index loads, handed round by shuffles
      if (r0 + lane < a.M) id0 = a.g_rows ? a.g_rows[r0 + lane] : (int)(r0 + lane);
      if (r0 + 32 + lane < a.M) id1 = a.g_rows ? a.g_rows[r0 + 32 + lane] : (int)(r0 + 32 + lane);
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int row = (tw + 4 * h) * 8 + e;               // 0 .. 63; h == 1 rows are >= 32
          const int src = __shfl_sync(0xffffffffu, h ? id1 : id0, row & 31);
          v[h][e] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (src >= 0) v[h][e] = __ldg(reinterpret_cast<const float4*>(a.G + (int64_t)src * a.ldg) + lane);
        }
    };
    if (s0 < s1) fetch(s0);
    uint32_t g = 0;
    for (int64_t st = s0; st < s1; ++st, ++g) {
      const uint32_t buf = g & 1u;
      mbar_wait_trap<MBAR_SPINS>(&empty[buf], ((g >> 1) & 1u) ^ 1u);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int rg = tw + 4 * h;
#pragma unroll
        for (int c = 0; c < 4; ++c) {                         // output o = 4 lane + c, rows rg*8 .. rg*8 + 7
          const int o = lane * 4 + c;
          float x[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) x[e] = (c == 0 ? v[h][e].x : c == 1 ? v[h][e].y : c == 2 ? v[h][e].z : v[h][e].w) * sg;
          uint32_t hw[4], lw[4];
#pragma unroll
          for (int e = 0; e < 8; e += 2) split_pair(x[e], x[e + 1], hw[e >> 1], lw[e >> 1]);
          uint8_t* hi_p = smem + buf * WG_BUF + (uint32_t)(o >> 3) * WG_A_SBO + (uint32_t)(o & 7) * 16 + (uint32_t)rg * WG_LBO;
          *reinterpret_cast<uint4*>(hi_p) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
          *reinterpret_cast<uint4*>(hi_p + WG_A_PLANE) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
        }
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&full[buf]);
      if (st + 1 < s1) fetch(st + 1);
    }
  }
  // ======================= epilogue: warps 1..4 (TMEM lane quarter = warp % 4), once =======================
  if (warp >= 1 && warp <= 4) {
    const int q = warp & 3;
    float* prow = a.part + ((size_t)blockIdx.x * NOUT + (q * 32 + lane)) * HIDF;
    if (s1 > s0) {
      mbar_wait_trap<MBAR_SPINS>(done, 0);
      tc_fence_after();
      const float unscale = ig * ih;
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int c = 0; c < HIDF; c += 32) {
        float vm[32], vc[32];
        tmem_ld32(trow + (uint32_t)c, vm);
        tmem_ld32(trow + 256u + (uint32_t)c, vc);
#pragma unroll
        for (int e = 0; e < 8; ++e)
          st4(prow + c + 4 * e, make_float4(fmaf(vc[4 * e], LO_INV, vm[4 * e]) * unscale, fmaf(vc[4 * e + 1], LO_INV, vm[4 * e + 1]) * unscale,
                                            fmaf(vc[4 * e + 2], LO_INV, vm[4 * e + 2]) * unscale, fmaf(vc[4 * e + 3], LO_INV, vm[4 * e + 3]) * unscale));
      }
    } else {
      for (int c = 0; c < HIDF; c += 4) st4(prow + c, make_float4(0.f, 0.f, 0.f, 0.f));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, TM_COLS);
}

// =============================================================================================
// First-layer gradients:  dh = (G W2) * (pre > 0),  db1[j] = sum_r dh[r][j],  dW1[j][c] = sum_r dh[r][j] x_c[r]
//   D[M = 128 rows][N = 256 j] = A[row][k = o] . B[j][k = o]^T:  A = the G rows (per-row power-of-two scale: the
//   contraction runs over o), B = W2 transposed, split once and resident (2 x 64 KB).  The 256 columns are two
//   halves with their own accumulator pair, so the epilogue of one half overlaps the MMAs of the other and of the
//   next tile.  dh is never written: an epilogue warp masks its 32 x 32 block with the regenerated pre-activation
//   sign (the forward's own expression), transposes it through shared memory and adds it into per-lane column
//   accumulators that live in registers for the whole kernel (8 columns x 3 sums per lane); one partial per warp at
//   the end, folded in a fixed order.
// =============================================================================================
constexpr uint32_t B1_W_SBO = (NOUT / 8) * 128, B1_W_PLANE = (HIDF / 8) * B1_W_SBO;        // B[j][o]: 2048, 64 KB
constexpr uint32_t B1_A_LBO = 144, B1_A_SBO = (NOUT / 8) * B1_A_LBO, B1_A_PLANE = (TM / 8) * B1_A_SBO;   // 2304, 36 KB
constexpr uint32_t B1_OFF_W = 0;
constexpr uint32_t B1_OFF_A = 2 * B1_W_PLANE;
constexpr uint32_t B1_OFF_P = B1_OFF_A + 2 * B1_A_PLANE;                 // w0, w1, b1 [256]
constexpr uint32_t B1_OFF_INV = B1_OFF_P + 3 * HIDF * 4;                 // [tile parity 2][128]
constexpr uint32_t B1_OFF_SCR = B1_OFF_INV + 2 * TM * 4;                 // per epilogue warp: 32 x 33 block + x0[32] + x1[32]
constexpr uint32_t B1_SCR_W = (32 * 33 + 64) * 4;
constexpr uint32_t B1_OFF_BAR = B1_OFF_SCR + EPI_W * B1_SCR_W;
constexpr uint32_t B1_SMEM = B1_OFF_BAR + 8 * 8 + 16;
static_assert(B1_SMEM <= 232448, "shared memory budget");

// W2 [NOUT o][HIDF j] fp32 -> planes of B[j][k = o]
__global__ void selfmlp_pack_t_kernel(const float* __restrict__ W2, uint8_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= NOUT * HIDF) return;
  const int o = i / HIDF, j = i - o * HIDF;
  __half h, l;
  split_h(W2[i], h, l);
  const uint32_t off = (uint32_t)(j >> 3) * B1_W_SBO + (uint32_t)(o >> 3) * 128 + (uint32_t)(j & 7) * 16 + (uint32_t)(o & 7) * 2;
  *reinterpret_cast<__half*>(out + off) = h;
  *reinterpret_cast<__half*>(out + B1_W_PLANE + off) = l;
}

// part [slots][3][HIDF] -> db1[j], dW1[j][kx]: 32 columns x 8 slot groups per block, fixed order
__global__ void __launch_bounds__(256)
selfmlp_bwd1_reduce_kernel(const float* __restrict__ part, int slots, int kx, float* __restrict__ dW1, float* __restrict__ db1) {
  __shared__ float sm[8][3][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + lane;
  float s[3] = {0.f, 0.f, 0.f};
#pragma unroll 4
  for (int g = w; g < slots; g += 8)
#pragma unroll
    for (int k = 0; k < 3; ++k) s[k] += part[((size_t)g * 3 + k) * HIDF + n];
#pragma unroll
  for (int k = 0; k < 3; ++k) sm[w][k][lane] = s[k];
  __syncthreads();
  if (w == 0) {
#pragma unroll
    for (int k = 0; k < 3; ++k)
      for (int i = 1; i < 8; ++i) s[k] += sm[i][k][lane];
    db1[n] = s[0];
    dW1[n * kx] = s[1];
    if (kx > 1) dW1[n * kx + 1] = s[2];
  }
}

struct B1Args {
  int64_t M;
  const float* G;
  int64_t ldg;
  const int* g_rows;
  const float* X;
  int64_t ldx;
  const int* x_rows;
  int kx;
  const float* W1;
  const float* b1;
  const uint8_t* wplanes;
  float* part;            // [grid * EPI_W][3][256]
  // STORE form (tm_selfmlp_rows_dh): dh rows are written, masked by a STORED hidden activation
  const float* H;         // [.][ldh] hidden activations of the forward
  int64_t ldh;
  const int* h_rows;      // row of H (and of DH) that belongs to row m (NULL: m)
  float* DH;
  int64_t lddh;
  // DX form (tm_selfmlp_gen_bwd1_dx, tm_selfmlp_rows_dx): the input's data gradient dh W1, written to the row of X the
  // forward read (x_rows)
  float* dX;
  int64_t lddx;
  const int* m_dev;       // DEVM: device row count; M is then the capacity the grid was sized for
};

// STORE == false: first-layer gradients of the generated MLP (above); DX adds the data gradient dX = dh W1, two FMAs per
// hidden unit in the lane that owns the row, in hidden-unit order; WG == false (with DX) drops the first-layer weight
// gradients and leaves dX the same bits.  STORE == true: the same product with the epilogue of the general MLP
// backward -- dh = (G W2) * (H > 0) written to DH (fc_cell_self: 36 inputs, the hidden layer is stored); with DX, dh is
// not written but multiplied into dX = dh W1 (kx <= 48 inputs) in the lane that owns the row, in hidden-unit order.
// DEVM: the row count is *m_dev (at most M), read on the device; CTAs past it have no tile.
template <bool STORE, bool DX, bool WG = true, bool DEVM = false>
__global__ void __launch_bounds__(THREADS, 1) selfmlp_gen_bwd1_kernel(B1Args a) {
  if constexpr (DEVM) a.M = max((int64_t)0, min(a.M, (int64_t)*a.m_dev));
  extern __shared__ __align__(1024) uint8_t smem[];
  float* w0_s = reinterpret_cast<float*>(smem + B1_OFF_P);
  float* w1_s = w0_s + HIDF;
  float* b1_s = w1_s + HIDF;
  float* inv_s = reinterpret_cast<float*>(smem + B1_OFF_INV);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + B1_OFF_BAR);
  uint64_t *a_full = bars, *a_empty = bars + 1, *acc_full = bars + 2, *acc_empty = bars + 4, *wbar = bars + 6;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t ntiles = (a.M + TM - 1) / TM;

  if (tid == 0) {
    mbar_init(a_full, GEN_W); mbar_init(a_empty, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], EPI_W); }
    mbar_init(wbar, 1);
    fence_mbarrier_init();
    fence_async_smem();
    mbar_expect_tx(wbar, 2 * B1_W_PLANE);
    for (int i = 0; i < 4; ++i)
      bulk_copy_g2s(smem_u32(smem + B1_OFF_W + i * (B1_W_PLANE / 2)), a.wplanes + (size_t)i * (B1_W_PLANE / 2), B1_W_PLANE / 2, wbar);
  }
  if constexpr (!STORE) {
    for (int j = tid; j < HIDF; j += THREADS) {
      w0_s[j] = a.W1[(size_t)j * a.kx];
      w1_s[j] = a.kx > 1 ? a.W1[(size_t)j * a.kx + 1] : 0.f;
      b1_s[j] = a.b1[j];
    }
  }
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= GEN_WARP0) {
    // ======================= loaders: G rows -> A planes (warp lw: rows 16 lw .. 16 lw + 15 of the tile) ==========
    const int lw = warp - GEN_WARP0;
    float4 v[16];
    auto fetch = [&](int64_t t) {
      const int64_t r = t * TM + lw * 16 + (lane & 15);
      int id = -1;
      if (r < a.M) id = a.g_rows ? a.g_rows[r] : (int)r;
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const int src = __shfl_sync(0xffffffffu, id, e);
        v[e] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (src >= 0) v[e] = __ldg(reinterpret_cast<const float4*>(a.G + (int64_t)src * a.ldg) + lane);
      }
    };
    if ((int64_t)blockIdx.x < ntiles) fetch(blockIdx.x);
    uint32_t li = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
      mbar_wait_trap<MBAR_SPINS>(a_empty, (li & 1u) ^ 1u);                      // the MMAs of the previous tile are done with the planes
      uint8_t* hi_p = smem + B1_OFF_A + (uint32_t)(lane >> 1) * B1_A_LBO + (uint32_t)(lane & 1) * 8;
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const int row = lw * 16 + e;
        const float4 x = v[e];
        float rm = fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) rm = fmaxf(rm, __shfl_xor_sync(0xffffffffu, rm, o));
        float sc, inv;
        row_scale(rm, -100, sc, inv);
        uint32_t h0, l0, h1, l1;
        split_pair(x.x * sc, x.y * sc, h0, l0);
        split_pair(x.z * sc, x.w * sc, h1, l1);
        const uint32_t off = (uint32_t)(row >> 3) * B1_A_SBO + (uint32_t)(row & 7) * 16;
        *reinterpret_cast<uint2*>(hi_p + off) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(hi_p + B1_A_PLANE + off) = make_uint2(l0, l1);
        if (lane == 0) inv_s[(li & 1u) * TM + row] = inv;
      }
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full);
      if (t + gridDim.x < ntiles) fetch(t + gridDim.x);
    }
  } else if (warp == MMA_WARP) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      mbar_wait_trap<MBAR_SPINS>(wbar, 0);
      const uint32_t idesc = make_idesc(Fmt::F16, NOUT);             // N = 128 columns per half
      const uint32_t a_hi = smem_u32(smem + B1_OFF_A), a_lo = a_hi + B1_A_PLANE;
      const uint32_t w_hi = smem_u32(smem + B1_OFF_W), w_lo = w_hi + B1_W_PLANE;
      uint32_t li = 0;
      for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
        mbar_wait_trap<MBAR_SPINS>(a_full, li & 1u);
        tc_fence_after();
        for (uint32_t half = 0; half < 2; ++half) {
          mbar_wait_trap<MBAR_SPINS>(&acc_empty[half], (li & 1u) ^ 1u);         // the epilogue drained this half's accumulators
          tc_fence_after();
          const uint32_t t_main = tmem_base + half * 256u, t_corr = t_main + 128u;
          const uint32_t wh = w_hi + half * 16u * B1_W_SBO, wl = w_lo + half * 16u * B1_W_SBO;
#pragma unroll
          for (int ks = 0; ks < NOUT / 16; ++ks) {
            const uint64_t ah = smem_desc(a_hi + ks * 2 * B1_A_LBO, B1_A_LBO, B1_A_SBO), al = smem_desc(a_lo + ks * 2 * B1_A_LBO, B1_A_LBO, B1_A_SBO);
            const uint64_t bh = smem_desc(wh + ks * 2 * 128u, 128u, B1_W_SBO), bl = smem_desc(wl + ks * 2 * 128u, 128u, B1_W_SBO);
            const uint32_t acc = ks > 0 ? 1u : 0u;
            umma_f16(t_main, ah, bh, idesc, acc);
            umma_f16(t_corr, ah, bl, idesc, acc);
            umma_f16(t_corr, al, bh, idesc, 1u);
          }
          umma_commit(&acc_full[half]);
        }
        umma_commit(a_empty);                                  // planes reusable once both halves' MMAs retire
      }
    }
    __syncwarp();
  } else if constexpr (STORE && DX) {
    // ======================= epilogue (rows_dx): a lane owns one row: mask from H, dX = dh W1 in registers ==========
    // W1 [256][kx] rows are read as warp-uniform 16-byte loads (one transaction per warp, L1-resident)
    const int nk4 = a.kx >> 2;
    float* dsc = reinterpret_cast<float*>(smem + B1_OFF_SCR + warp * B1_SCR_W) + lane * 9;   // this row's 8 gated dh values
    uint32_t li = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
      const int64_t m = t * TM + warp * 32 + lane;
      const float* hp = nullptr;
      if (m < a.M) hp = a.H + (a.h_rows ? (int64_t)a.h_rows[m] : m) * a.ldh;
      float dx[48];
#pragma unroll
      for (int k = 0; k < 48; ++k) dx[k] = 0.f;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        mbar_wait_trap<MBAR_SPINS>(&acc_full[half], li & 1u);
        tc_fence_after();
        const float inv = inv_s[(li & 1u) * TM + warp * 32 + lane];
        const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)half * 256u;
#pragma unroll 1
        for (int c = 0; c < 16; ++c) {
          const int j0 = half * 128 + c * 8;
          float4 mk[2];
#pragma unroll
          for (int e = 0; e < 2; ++e) mk[e] = hp ? ld4(hp + j0 + 4 * e) : make_float4(0.f, 0.f, 0.f, 0.f);
          float vm[8], vc[8];
          tmem_ld8(trow + (uint32_t)(c * 8), vm);
          tmem_ld8(trow + 128u + (uint32_t)(c * 8), vc);
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            dsc[4 * e] = mk[e].x > 0.f ? fmaf(vc[4 * e], LO_INV, vm[4 * e]) * inv : 0.f;
            dsc[4 * e + 1] = mk[e].y > 0.f ? fmaf(vc[4 * e + 1], LO_INV, vm[4 * e + 1]) * inv : 0.f;
            dsc[4 * e + 2] = mk[e].z > 0.f ? fmaf(vc[4 * e + 2], LO_INV, vm[4 * e + 2]) * inv : 0.f;
            dsc[4 * e + 3] = mk[e].w > 0.f ? fmaf(vc[4 * e + 3], LO_INV, vm[4 * e + 3]) * inv : 0.f;
          }
#pragma unroll 1
          for (int i = 0; i < 8; ++i) {                      // (the loop stays rolled: 48 accumulators fill the budget)
            const float d = dsc[i];
            const float4* wr = reinterpret_cast<const float4*>(a.W1 + (size_t)(j0 + i) * a.kx);
#pragma unroll
            for (int k4 = 0; k4 < 12; ++k4) {
              if (k4 < nk4) {
                const float4 w = __ldg(wr + k4);
                dx[4 * k4] = fmaf(d, w.x, dx[4 * k4]);
                dx[4 * k4 + 1] = fmaf(d, w.y, dx[4 * k4 + 1]);
                dx[4 * k4 + 2] = fmaf(d, w.z, dx[4 * k4 + 2]);
                dx[4 * k4 + 3] = fmaf(d, w.w, dx[4 * k4 + 3]);
              }
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[half]);
      }
      if (m < a.M) {
        float* dp = a.dX + (a.x_rows ? (int64_t)a.x_rows[m] : m) * a.lddx;
#pragma unroll
        for (int k4 = 0; k4 < 12; ++k4)
          if (k4 < nk4) st4(dp + 4 * k4, make_float4(dx[4 * k4], dx[4 * k4 + 1], dx[4 * k4 + 2], dx[4 * k4 + 3]));
      }
    }
  } else if constexpr (STORE) {
    // ======================= epilogue (STORE): a lane owns one row: mask from H, 128-bit stores to DH ===============
    uint32_t li = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
      const int64_t m = t * TM + warp * 32 + lane;
      const float* hp = nullptr;
      float* dp = nullptr;
      if (m < a.M) {
        const int64_t r = a.h_rows ? (int64_t)a.h_rows[m] : m;
        hp = a.H + r * a.ldh;
        dp = a.DH + r * a.lddh;
      }
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        mbar_wait_trap<MBAR_SPINS>(&acc_full[half], li & 1u);
        tc_fence_after();
        const float inv = inv_s[(li & 1u) * TM + warp * 32 + lane];
        const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)half * 256u;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int j0 = half * 128 + c * 32;
          float4 mk[8];
          if (hp) {
#pragma unroll
            for (int e = 0; e < 8; ++e) mk[e] = ld4(hp + j0 + 4 * e);        // (in flight under the TMEM loads)
          }
          float vm[32], vc[32];
          tmem_ld32(trow + (uint32_t)(c * 32), vm);
          tmem_ld32(trow + 128u + (uint32_t)(c * 32), vc);
          if (dp) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              float4 o;
              o.x = mk[e].x > 0.f ? fmaf(vc[4 * e], LO_INV, vm[4 * e]) * inv : 0.f;
              o.y = mk[e].y > 0.f ? fmaf(vc[4 * e + 1], LO_INV, vm[4 * e + 1]) * inv : 0.f;
              o.z = mk[e].z > 0.f ? fmaf(vc[4 * e + 2], LO_INV, vm[4 * e + 2]) * inv : 0.f;
              o.w = mk[e].w > 0.f ? fmaf(vc[4 * e + 3], LO_INV, vm[4 * e + 3]) * inv : 0.f;
              st4(dp + j0 + 4 * e, o);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[half]);
      }
    }
  } else {
    // ======================= epilogue: mask, transpose, column sums in registers =======================
    float* scr = reinterpret_cast<float*>(smem + B1_OFF_SCR + warp * B1_SCR_W);
    float* xs0 = scr + 32 * 33;
    float* xs1 = xs0 + 32;
    float acc[8][3];
#pragma unroll
    for (int i = 0; i < 8; ++i) { acc[i][0] = 0.f; acc[i][1] = 0.f; acc[i][2] = 0.f; }
    uint32_t li = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
      const int64_t m = t * TM + warp * 32 + lane;
      float x0 = 0.f, x1 = 0.f;
      if (m < a.M) {
        const float* xp = a.X + (a.x_rows ? (int64_t)a.x_rows[m] : m) * a.ldx;
        x0 = xp[0];
        if (a.kx > 1) x1 = xp[1];
      }
      __syncwarp();
      xs0[lane] = x0; xs1[lane] = x1;
      __syncwarp();
      float dx0 = 0.f, dx1 = 0.f;                                      // (DX) this row's data gradient
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        mbar_wait_trap<MBAR_SPINS>(&acc_full[half], li & 1u);
        tc_fence_after();
        const float inv = inv_s[(li & 1u) * TM + warp * 32 + lane];   // (written before a_full of this tile was signalled)
        const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)half * 256u;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float vm[32], vc[32];
          tmem_ld32(trow + (uint32_t)(c * 32), vm);
          tmem_ld32(trow + 128u + (uint32_t)(c * 32), vc);
          const int j0 = half * 128 + c * 32;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float pre = fmaf(w0_s[j0 + i], x0, fmaf(w1_s[j0 + i], x1, b1_s[j0 + i]));
            const float dh = fmaf(vc[i], LO_INV, vm[i]) * inv;
            const float d = pre > 0.f ? dh : 0.f;
            if constexpr (WG) scr[lane * 33 + i] = d;
            if constexpr (DX) {
              dx0 = fmaf(d, w0_s[j0 + i], dx0);
              dx1 = fmaf(d, w1_s[j0 + i], dx1);
            }
          }
          if constexpr (WG) {
            __syncwarp();
            float s = 0.f, s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int r = 0; r < 32; r += 4) {                    // (the rows' inputs: broadcast 16-byte reads)
              const float4 p = *reinterpret_cast<const float4*>(xs0 + r), q = *reinterpret_cast<const float4*>(xs1 + r);
              const float d0 = scr[r * 33 + lane], d1 = scr[(r + 1) * 33 + lane], d2 = scr[(r + 2) * 33 + lane], d3 = scr[(r + 3) * 33 + lane];
              s += (d0 + d1) + (d2 + d3);
              s0 = fmaf(d0, p.x, fmaf(d1, p.y, fmaf(d2, p.z, fmaf(d3, p.w, s0))));
              s1 = fmaf(d0, q.x, fmaf(d1, q.y, fmaf(d2, q.z, fmaf(d3, q.w, s1))));
            }
            acc[half * 4 + c][0] += s; acc[half * 4 + c][1] += s0; acc[half * 4 + c][2] += s1;
            __syncwarp();
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[half]);
      }
      if constexpr (DX) {
        if (m < a.M) {
          float* dp = a.dX + (a.x_rows ? (int64_t)a.x_rows[m] : m) * a.lddx;
          dp[0] = dx0;
          if (a.kx > 1) dp[1] = dx1;
        }
      }
    }
    if constexpr (WG) {
      float* pp = a.part + ((size_t)blockIdx.x * EPI_W + warp) * 3 * HIDF;
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int k = 0; k < 3; ++k) pp[(size_t)k * HIDF + i * 32 + lane] = acc[i][k];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(tmem_base, TM_COLS);
}

// =============================================================================================
// First layer of a stored-hidden MLP:  HID[m][0:256] = relu(X[x_rows[m]][0:kin] W1^T + b1), kin <= 48 (fc_cell_self: 36).
// Output-bound (1 KB written per 144 bytes read): A = the x rows (a loader thread owns one row: per-row scale without
// shuffles, K padded to 48 = three k-steps), B = W1 split once and resident (2 x 24 KB), two column halves with their
// own accumulator pair, row-direct storing epilogue with bias + ReLU.
// =============================================================================================
constexpr int L1_K = 48;
constexpr uint32_t L1_SBO = (L1_K / 8) * 128;                                   // 768
constexpr uint32_t L1_A_PLANE = (TM / 8) * L1_SBO, L1_W_PLANE = (HIDF / 8) * L1_SBO;   // 12 KB, 24 KB
constexpr uint32_t L1_OFF_W = 0, L1_OFF_A = 2 * L1_W_PLANE, L1_OFF_B = L1_OFF_A + 2 * L1_A_PLANE;
constexpr uint32_t L1_OFF_INV = L1_OFF_B + HIDF * 4, L1_OFF_BAR = L1_OFF_INV + 2 * TM * 4;
// (requested size: more than half an SM's shared memory, so that two of these CTAs -- each allocates all 512 TMEM
//  columns -- can never be resident on one SM)
constexpr uint32_t L1_SMEM = (L1_OFF_BAR + 8 * 8 + 16) > 120 * 1024 ? (L1_OFF_BAR + 8 * 8 + 16) : 120 * 1024;
constexpr int L1_LOAD_W = TM / 32;                                              // loader warps that own rows

__global__ void selfmlp_pack_w1_kernel(const float* __restrict__ W1, int kin, uint8_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= HIDF * L1_K) return;
  const int j = i / L1_K, k = i - j * L1_K;
  __half h, l;
  split_h(k < kin ? W1[(size_t)j * kin + k] : 0.f, h, l);
  const uint32_t off = (uint32_t)(j >> 3) * L1_SBO + (uint32_t)(k >> 3) * 128 + (uint32_t)(j & 7) * 16 + (uint32_t)(k & 7) * 2;
  *reinterpret_cast<__half*>(out + off) = h;
  *reinterpret_cast<__half*>(out + L1_W_PLANE + off) = l;
}

struct L1Args {
  int64_t M;
  const float* X;
  int64_t ldx;
  const int* x_rows;
  int kin;                // multiple of 4, <= 48
  const float* b1;
  const uint8_t* wplanes;
  float* out;
  int64_t ldo;
  float* rowmax;          // optional: max over the row's 256 outputs (the scale of tm_selfmlp_rows_forward)
  const int* m_dev;       // DEVM: device row count; M is then the capacity the grid was sized for
};

// DEVM: the row count is *m_dev (at most M), read on the device; CTAs past it have no tile.
template <bool DEVM = false>
__global__ void __launch_bounds__(THREADS, 1) selfmlp_lin1_kernel(L1Args a) {
  if constexpr (DEVM) a.M = max((int64_t)0, min(a.M, (int64_t)*a.m_dev));
  extern __shared__ __align__(1024) uint8_t smem[];
  float* b1_s = reinterpret_cast<float*>(smem + L1_OFF_B);
  float* inv_s = reinterpret_cast<float*>(smem + L1_OFF_INV);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L1_OFF_BAR);
  uint64_t *a_full = bars, *a_empty = bars + 1, *acc_full = bars + 2, *acc_empty = bars + 4, *wbar = bars + 6;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 7);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t ntiles = (a.M + TM - 1) / TM;

  if (tid == 0) {
    mbar_init(a_full, L1_LOAD_W); mbar_init(a_empty, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], EPI_W); }
    mbar_init(wbar, 1);
    fence_mbarrier_init();
    fence_async_smem();
    mbar_expect_tx(wbar, 2 * L1_W_PLANE);
    for (int i = 0; i < 2; ++i)
      bulk_copy_g2s(smem_u32(smem + L1_OFF_W + i * L1_W_PLANE), a.wplanes + (size_t)i * L1_W_PLANE, L1_W_PLANE, wbar);
  }
  for (int j = tid; j < HIDF; j += THREADS) b1_s[j] = a.b1[j];
  if (warp == MMA_WARP) tmem_alloc(tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= GEN_WARP0 && warp < GEN_WARP0 + L1_LOAD_W) {
    // ======================= loaders: thread = one row of the tile =======================
    const int row = tid - GEN_WARP0 * 32;
    const int nq = a.kin >> 2;
    float4 v[L1_K / 4];
    auto fetch = [&](int64_t t) {
      const int64_t m = t * TM + row;
#pragma unroll
      for (int q = 0; q < L1_K / 4; ++q) v[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m < a.M) {
        const float4* xp = reinterpret_cast<const float4*>(a.X + (a.x_rows ? (int64_t)a.x_rows[m] : m) * a.ldx);
#pragma unroll
        for (int q = 0; q < L1_K / 4; ++q)
          if (q < nq) v[q] = __ldg(xp + q);
      }
    };
    if ((int64_t)blockIdx.x < ntiles) fetch(blockIdx.x);
    uint32_t li = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
      mbar_wait_trap<MBAR_SPINS>(a_empty, (li & 1u) ^ 1u);
      float rm = 0.f;
#pragma unroll
      for (int q = 0; q < L1_K / 4; ++q) rm = fmaxf(rm, fmaxf(fmaxf(fabsf(v[q].x), fabsf(v[q].y)), fmaxf(fabsf(v[q].z), fabsf(v[q].w))));
      float sc, inv;
      row_scale(rm, -100, sc, inv);
      uint8_t* hi_p = smem + L1_OFF_A + (uint32_t)(row >> 3) * L1_SBO + (uint32_t)(row & 7) * 16;
#pragma unroll
      for (int kg = 0; kg < L1_K / 8; ++kg) {
        uint32_t hw[4], lw[4];
        split_pair(v[2 * kg].x * sc, v[2 * kg].y * sc, hw[0], lw[0]);
        split_pair(v[2 * kg].z * sc, v[2 * kg].w * sc, hw[1], lw[1]);
        split_pair(v[2 * kg + 1].x * sc, v[2 * kg + 1].y * sc, hw[2], lw[2]);
        split_pair(v[2 * kg + 1].z * sc, v[2 * kg + 1].w * sc, hw[3], lw[3]);
        *reinterpret_cast<uint4*>(hi_p + kg * 128) = make_uint4(hw[0], hw[1], hw[2], hw[3]);
        *reinterpret_cast<uint4*>(hi_p + L1_A_PLANE + kg * 128) = make_uint4(lw[0], lw[1], lw[2], lw[3]);
      }
      inv_s[(li & 1u) * TM + row] = inv;
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full);
      if (t + gridDim.x < ntiles) fetch(t + gridDim.x);
    }
  } else if (warp == MMA_WARP) {
    if (lane == 0) {
      mbar_wait_trap<MBAR_SPINS>(wbar, 0);
      const uint32_t idesc = make_idesc(Fmt::F16, NOUT);
      const uint32_t a_hi = smem_u32(smem + L1_OFF_A), a_lo = a_hi + L1_A_PLANE;
      const uint32_t w_hi = smem_u32(smem + L1_OFF_W), w_lo = w_hi + L1_W_PLANE;
      uint32_t li = 0;
      for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
        mbar_wait_trap<MBAR_SPINS>(a_full, li & 1u);
        tc_fence_after();
        for (uint32_t half = 0; half < 2; ++half) {
          mbar_wait_trap<MBAR_SPINS>(&acc_empty[half], (li & 1u) ^ 1u);
          tc_fence_after();
          const uint32_t t_main = tmem_base + half * 256u, t_corr = t_main + 128u;
          const uint32_t wh = w_hi + half * 16u * L1_SBO, wl = w_lo + half * 16u * L1_SBO;
#pragma unroll
          for (int ks = 0; ks < L1_K / 16; ++ks) {
            const uint64_t ah = smem_desc(a_hi + ks * 256u, 128u, L1_SBO), al = smem_desc(a_lo + ks * 256u, 128u, L1_SBO);
            const uint64_t bh = smem_desc(wh + ks * 256u, 128u, L1_SBO), bl = smem_desc(wl + ks * 256u, 128u, L1_SBO);
            const uint32_t acc = ks > 0 ? 1u : 0u;
            umma_f16(t_main, ah, bh, idesc, acc);
            umma_f16(t_corr, ah, bl, idesc, acc);
            umma_f16(t_corr, al, bh, idesc, 1u);
          }
          umma_commit(&acc_full[half]);
        }
        umma_commit(a_empty);
      }
    }
    __syncwarp();
  } else if (warp < EPI_W) {
    // ======================= epilogue: a lane owns one row: bias, ReLU, 128-bit stores =======================
    uint32_t li = 0;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++li) {
      const int64_t m = t * TM + warp * 32 + lane;
      float* op = m < a.M ? a.out + m * a.ldo : nullptr;
      float rmax = 0.f;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        mbar_wait_trap<MBAR_SPINS>(&acc_full[half], li & 1u);
        tc_fence_after();
        const float inv = inv_s[(li & 1u) * TM + warp * 32 + lane];
        const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)half * 256u;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          const int j0 = half * 128 + c * 32;
          float vm[32], vc[32];
          tmem_ld32(trow + (uint32_t)(c * 32), vm);
          tmem_ld32(trow + 128u + (uint32_t)(c * 32), vc);
          if (op) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const float4 b = *reinterpret_cast<const float4*>(b1_s + j0 + 4 * e);
              float4 o;
              o.x = fmaxf(fmaf(fmaf(vc[4 * e], LO_INV, vm[4 * e]), inv, b.x), 0.f);
              o.y = fmaxf(fmaf(fmaf(vc[4 * e + 1], LO_INV, vm[4 * e + 1]), inv, b.y), 0.f);
              o.z = fmaxf(fmaf(fmaf(vc[4 * e + 2], LO_INV, vm[4 * e + 2]), inv, b.z), 0.f);
              o.w = fmaxf(fmaf(fmaf(vc[4 * e + 3], LO_INV, vm[4 * e + 3]), inv, b.w), 0.f);
              rmax = fmaxf(fmaxf(rmax, fmaxf(o.x, o.y)), fmaxf(o.z, o.w));
              st4(op + j0 + 4 * e, o);
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[half]);
      }
      if (a.rowmax && op) a.rowmax[m] = rmax;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(tmem_base, TM_COLS);
}
}  // namespace

extern "C" size_t tm_selfmlp_ws_bytes() { return 2 * (size_t)W_PLANE + 256; }

/* out[out_rows[m], 0:128] = W2 relu(W1 X[x_rows[m], 0:kx] + b1) + b2 for m < M, with W1 [256][kx] (kx = 1 or 2),
 * W2 [128][256] as nn.Linear stores them.  `ws`: tm_selfmlp_ws_bytes() bytes (the split planes of W2). */
extern "C" int tm_selfmlp_gen_forward(int64_t M, const float* X, int64_t ldx, const int32_t* x_rows, int64_t kx,
                                      const float* W1, const float* b1, const float* W2, const float* b2, float* out,
                                      int64_t ldo, const int32_t* out_rows, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(kx == 1 || kx == 2, "tm_selfmlp_gen_forward: the first layer must have 1 or 2 inputs");
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_ws_bytes(), "tm_selfmlp_gen_forward: workspace too small (tm_selfmlp_ws_bytes)");
  TM_REQUIRE((ldo & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "tm_selfmlp_gen_forward: out rows must be 16-byte aligned");
  if (M <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_kernel<<<(NOUT * HIDF + 255) / 256, 256, 0, st>>>(W2, planes);
  TM_TRY(check_launch("selfmlp_pack"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES + 1024));
  Args a{M, X, ldx, x_rows, (int)kx, W1, b1, b2, planes, out, ldo, out_rows, nullptr, 0, nullptr, nullptr};
  const int64_t ntiles = (M + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  selfmlp_gen_fwd_kernel<false><<<grid, THREADS, SMEM_BYTES + 1024, st>>>(a);
  return check_launch("selfmlp_gen_fwd");
}

extern "C" size_t tm_selfmlp_wgrad2_ws_bytes() { return (size_t)sm_count() * NOUT * HIDF * sizeof(float) + 1024; }

extern "C" int tm_selfmlp_gen_wgrad2(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* X, int64_t ldx,
                                     const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, const float* gmax,
                                     float* dW2, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(kx == 1 || kx == 2, "tm_selfmlp_gen_wgrad2: the first layer must have 1 or 2 inputs");
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_wgrad2_ws_bytes(), "tm_selfmlp_gen_wgrad2: workspace too small (tm_selfmlp_wgrad2_ws_bytes)");
  TM_REQUIRE(gmax, "tm_selfmlp_gen_wgrad2: gmax (device scalar, max |G|: tm_colsum_absmax) missing");
  TM_REQUIRE((ldg & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0, "tm_selfmlp_gen_wgrad2: G rows must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (M <= 0) {
    TM_CUDA(cudaMemsetAsync(dW2, 0, (size_t)NOUT * HIDF * sizeof(float), st));
    return 0;
  }
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  unsigned int* xmax = reinterpret_cast<unsigned int*>(base);
  float* part = reinterpret_cast<float*>(base + 256);
  TM_CUDA(cudaMemsetAsync(xmax, 0, 2 * sizeof(float), st));
  selfmlp_xmax_kernel<<<(unsigned)(sm_count() * 2), 256, 0, st>>>(M, X, ldx, x_rows, (int)kx, xmax);
  TM_TRY(check_launch("selfmlp_xmax"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_wgrad2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG_SMEM + 1024));
  const int64_t nsteps = (M + WG_KS - 1) / WG_KS;
  const int grid = (int)(nsteps < sm_count() ? nsteps : sm_count());
  WgArgs a{M, G, ldg, g_rows, X, ldx, x_rows, (int)kx, W1, b1, gmax, reinterpret_cast<const float*>(xmax), part};
  selfmlp_gen_wgrad2_kernel<<<grid, WG_THREADS, WG_SMEM + 1024, st>>>(a);
  TM_TRY(check_launch("selfmlp_gen_wgrad2"));
  split_reduce_kernel<<<(unsigned)cdiv((int64_t)NOUT * HIDF, 64), 256, 0, st>>>(part, (int64_t)NOUT * HIDF, grid, dW2, HIDF, HIDF, 0);
  return check_launch("split_reduce(selfmlp wgrad2)");
}

extern "C" size_t tm_selfmlp_bwd1_ws_bytes() { return 2 * (size_t)B1_W_PLANE + (size_t)sm_count() * EPI_W * 3 * HIDF * sizeof(float) + 1024; }

namespace {
// tm_selfmlp_gen_bwd1 (dX == nullptr) and tm_selfmlp_gen_bwd1_dx
int gen_bwd1(const char* name, int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* X, int64_t ldx,
             const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, const float* W2, float* dW1, float* db1,
             float* dX, int64_t lddx, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(kx == 1 || kx == 2, "%s: the first layer must have 1 or 2 inputs", name);
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_bwd1_ws_bytes(), "%s: workspace too small (tm_selfmlp_bwd1_ws_bytes)", name);
  TM_REQUIRE((ldg & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0, "%s: G rows must be 16-byte aligned", name);
  TM_REQUIRE((dW1 == nullptr) == (db1 == nullptr), "%s: dW1 and db1 must be both set or both NULL", name);
  TM_REQUIRE(dW1 || dX, "%s: dW1 / db1 NULL is served with dX only (tm_selfmlp_gen_bwd1_dx)", name);
  cudaStream_t st = (cudaStream_t)stream;
  if (M <= 0 && !dW1) return 0;
  if (M <= 0) {
    TM_CUDA(cudaMemsetAsync(dW1, 0, (size_t)HIDF * kx * sizeof(float), st));
    TM_CUDA(cudaMemsetAsync(db1, 0, (size_t)HIDF * sizeof(float), st));
    return 0;
  }
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  float* part = reinterpret_cast<float*>(planes + 2 * B1_W_PLANE);
  selfmlp_pack_t_kernel<<<(NOUT * HIDF + 255) / 256, 256, 0, st>>>(W2, planes);
  TM_TRY(check_launch("selfmlp_pack_t"));
  const int64_t ntiles = (M + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  B1Args a{M, G, ldg, g_rows, X, ldx, x_rows, (int)kx, W1, b1, planes, part, nullptr, 0, nullptr, nullptr, 0, dX, lddx};
  if (!dW1) {                 // data gradient only: no column accumulators, no partials, no reduction
    TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_bwd1_kernel<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B1_SMEM + 1024));
    selfmlp_gen_bwd1_kernel<false, true, false><<<grid, THREADS, B1_SMEM + 1024, st>>>(a);
    return check_launch("selfmlp_gen_bwd1_dx(no wgrad)");
  }
  if (dX) {
    TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_bwd1_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B1_SMEM + 1024));
    selfmlp_gen_bwd1_kernel<false, true><<<grid, THREADS, B1_SMEM + 1024, st>>>(a);
    TM_TRY(check_launch("selfmlp_gen_bwd1_dx"));
  } else {
    TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_bwd1_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B1_SMEM + 1024));
    selfmlp_gen_bwd1_kernel<false, false><<<grid, THREADS, B1_SMEM + 1024, st>>>(a);
    TM_TRY(check_launch("selfmlp_gen_bwd1"));
  }
  selfmlp_bwd1_reduce_kernel<<<HIDF / 32, 256, 0, st>>>(part, grid * EPI_W, (int)kx, dW1, db1);
  return check_launch("selfmlp_bwd1_reduce");
}
}  // namespace

extern "C" int tm_selfmlp_gen_bwd1(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* X, int64_t ldx,
                                   const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, const float* W2,
                                   float* dW1, float* db1, void* ws, size_t ws_bytes, void* stream) {
  return gen_bwd1("tm_selfmlp_gen_bwd1", M, G, ldg, g_rows, X, ldx, x_rows, kx, W1, b1, W2, dW1, db1, nullptr, 0, ws,
                  ws_bytes, stream);
}

/* ... and the input's data gradient dX[x_rows ? x_rows[m] : m, 0:kx] = dh W1 (declared in tm_b200.h). */
extern "C" int tm_selfmlp_gen_bwd1_dx(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* X,
                                      int64_t ldx, const int32_t* x_rows, int64_t kx, const float* W1, const float* b1,
                                      const float* W2, float* dW1, float* db1, float* dX, int64_t lddx, void* ws,
                                      size_t ws_bytes, void* stream) {
  TM_REQUIRE(dX && lddx >= kx, "tm_selfmlp_gen_bwd1_dx: dX missing or its row stride lddx < kx");
  return gen_bwd1("tm_selfmlp_gen_bwd1_dx", M, G, ldg, g_rows, X, ldx, x_rows, kx, W1, b1, W2, dW1, db1, dX, lddx, ws,
                  ws_bytes, stream);
}

extern "C" size_t tm_selfmlp_rows_dh_ws_bytes() { return 2 * (size_t)B1_W_PLANE + 256; }

/* DH[r, 0:256] = (G[g_rows[m], 0:128] @ W2) * (H[r, 0:256] > 0), r = h_rows ? h_rows[m] : m, for m < M: the hidden-layer
 * gradient of Linear(., 256) -> ReLU -> Linear(256, 128) whose hidden activations H were stored (fc_cell_self). */
extern "C" int tm_selfmlp_rows_dh(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* W2, const float* H,
                                  int64_t ldh, const int32_t* h_rows, float* DH, int64_t lddh, void* ws, size_t ws_bytes,
                                  void* stream) {
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_rows_dh_ws_bytes(), "tm_selfmlp_rows_dh: workspace too small (tm_selfmlp_rows_dh_ws_bytes)");
  TM_REQUIRE((ldg & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0 && (ldh & 3) == 0 && (reinterpret_cast<uintptr_t>(H) & 15) == 0 &&
                 (lddh & 3) == 0 && (reinterpret_cast<uintptr_t>(DH) & 15) == 0,
             "tm_selfmlp_rows_dh: G, H and DH rows must be 16-byte aligned");
  if (M <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_t_kernel<<<(NOUT * HIDF + 255) / 256, 256, 0, st>>>(W2, planes);
  TM_TRY(check_launch("selfmlp_pack_t"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_bwd1_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B1_SMEM + 1024));
  const int64_t ntiles = (M + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  B1Args a{M, G, ldg, g_rows, nullptr, 0, nullptr, 0, nullptr, nullptr, planes, nullptr, H, ldh, h_rows, DH, lddh};
  selfmlp_gen_bwd1_kernel<true, false><<<grid, THREADS, B1_SMEM + 1024, st>>>(a);
  return check_launch("selfmlp_rows_dh");
}

/* dX[x_rows[m], 0:kin] = ((G[g_rows[m]] @ W2) * (H[h_rows[m]] > 0)) @ W1 for m < M: the data gradient of
 * Linear(kin, 256) -> ReLU -> Linear(256, 128) whose hidden activations H were stored (fc_cell_self), in one pass; the
 * hidden gradient never leaves the SM.  W1 [256][kin] as stored, kin % 4 == 0, kin <= 48.  ws: tm_selfmlp_rows_dh_ws_bytes(). */
extern "C" int tm_selfmlp_rows_dx(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* W2, const float* H,
                                  int64_t ldh, const int32_t* h_rows, const float* W1, int64_t kin, float* dX, int64_t lddx,
                                  const int32_t* x_rows, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(kin > 0 && kin <= 48 && (kin & 3) == 0, "tm_selfmlp_rows_dx: kin must be a multiple of 4, <= 48");
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_rows_dh_ws_bytes(), "tm_selfmlp_rows_dx: workspace too small (tm_selfmlp_rows_dh_ws_bytes)");
  TM_REQUIRE(G && W2 && H && W1 && dX, "tm_selfmlp_rows_dx: G, W2, H, W1 and dX are required");
  TM_REQUIRE((ldg & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0 && (ldh & 3) == 0 && (reinterpret_cast<uintptr_t>(H) & 15) == 0 &&
                 (lddx & 3) == 0 && lddx >= kin && (reinterpret_cast<uintptr_t>(dX) & 15) == 0 && (reinterpret_cast<uintptr_t>(W1) & 15) == 0,
             "tm_selfmlp_rows_dx: G, H, W1 and dX rows must be 16-byte aligned (lddx >= kin)");
  if (M <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_t_kernel<<<(NOUT * HIDF + 255) / 256, 256, 0, st>>>(W2, planes);
  TM_TRY(check_launch("selfmlp_pack_t"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_bwd1_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B1_SMEM + 1024));
  const int64_t ntiles = (M + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  B1Args a{M, G, ldg, g_rows, nullptr, 0, x_rows, (int)kin, W1, nullptr, planes, nullptr, H, ldh, h_rows, nullptr, 0, dX, lddx};
  selfmlp_gen_bwd1_kernel<true, true, false><<<grid, THREADS, B1_SMEM + 1024, st>>>(a);
  return check_launch("selfmlp_rows_dx");
}

extern "C" size_t tm_selfmlp_lin1_ws_bytes() { return 2 * (size_t)L1_W_PLANE + 256; }

/* HID[m, 0:256] = relu(X[x_rows[m], 0:kin] @ W1^T + b1) for m < M (W1 [256][kin] as stored; kin % 4 == 0, kin <= 48). */
extern "C" int tm_selfmlp_lin1_relu(int64_t M, const float* X, int64_t ldx, const int32_t* x_rows, int64_t kin, const float* W1,
                                    const float* b1, float* HID, int64_t ldh, float* rowmax, void* ws, size_t ws_bytes,
                                    void* stream) {
  TM_REQUIRE(kin > 0 && kin <= L1_K && (kin & 3) == 0, "tm_selfmlp_lin1_relu: kin must be a multiple of 4, <= 48");
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_lin1_ws_bytes(), "tm_selfmlp_lin1_relu: workspace too small (tm_selfmlp_lin1_ws_bytes)");
  TM_REQUIRE((ldx & 3) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && (ldh & 3) == 0 && (reinterpret_cast<uintptr_t>(HID) & 15) == 0,
             "tm_selfmlp_lin1_relu: X and HID rows must be 16-byte aligned");
  if (M <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_w1_kernel<<<(HIDF * L1_K + 255) / 256, 256, 0, st>>>(W1, (int)kin, planes);
  TM_TRY(check_launch("selfmlp_pack_w1"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_lin1_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L1_SMEM + 1024));
  const int64_t ntiles = (M + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  L1Args a{M, X, ldx, x_rows, (int)kin, b1, planes, HID, ldh, rowmax};
  selfmlp_lin1_kernel<false><<<grid, THREADS, L1_SMEM + 1024, st>>>(a);
  return check_launch("selfmlp_lin1");
}

/* out[out_rows[m], 0:128] = H[h_rows[m], 0:256] @ W2^T + b2: second layer of an MLP whose hidden activations are stored;
 * rowmax[r] >= max |H[r, :]| (tm_selfmlp_lin1_relu writes it).  ws: tm_selfmlp_ws_bytes(). */
extern "C" int tm_selfmlp_rows_forward(int64_t M, const float* H, int64_t ldh, const int32_t* h_rows, const float* rowmax,
                                       const float* W2, const float* b2, float* out, int64_t ldo, const int32_t* out_rows,
                                       void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_ws_bytes(), "tm_selfmlp_rows_forward: workspace too small (tm_selfmlp_ws_bytes)");
  TM_REQUIRE(rowmax, "tm_selfmlp_rows_forward: rowmax missing");
  TM_REQUIRE((ldo & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (ldh & 3) == 0 && (reinterpret_cast<uintptr_t>(H) & 15) == 0,
             "tm_selfmlp_rows_forward: H and out rows must be 16-byte aligned");
  if (M <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_kernel<<<(NOUT * HIDF + 255) / 256, 256, 0, st>>>(W2, planes);
  TM_TRY(check_launch("selfmlp_pack"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES + 1024));
  Args a{M, nullptr, 0, nullptr, 1, nullptr, nullptr, b2, planes, out, ldo, out_rows, H, ldh, h_rows, rowmax};
  const int64_t ntiles = (M + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  selfmlp_gen_fwd_kernel<true><<<grid, THREADS, SMEM_BYTES + 1024, st>>>(a);
  return check_launch("selfmlp_rows_fwd");
}

// ------------------------------------------------------------------------------------------
// The same data-gradient products over a row count that exists only on the device (*m_dev, at most `cap`): the grid is
// sized by the capacity and the kernels read the count (a fan-in cone's class lists, tm_fanin_cone).  Each is its own
// template instance, so the entry points above compile as before.
// ------------------------------------------------------------------------------------------
extern "C" int tm_selfmlp_lin1_relu_dcount(int64_t cap, const int32_t* m_dev, const float* X, int64_t ldx,
                                           const int32_t* x_rows, int64_t kin, const float* W1, const float* b1, float* HID,
                                           int64_t ldh, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(m_dev && X && x_rows && W1 && b1 && HID, "tm_selfmlp_lin1_relu_dcount: NULL operand");
  TM_REQUIRE(kin > 0 && kin <= L1_K && (kin & 3) == 0, "tm_selfmlp_lin1_relu_dcount: kin must be a multiple of 4, <= 48");
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_lin1_ws_bytes(), "tm_selfmlp_lin1_relu_dcount: workspace too small (tm_selfmlp_lin1_ws_bytes)");
  TM_REQUIRE((ldx & 3) == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && (ldh & 3) == 0 && (reinterpret_cast<uintptr_t>(HID) & 15) == 0,
             "tm_selfmlp_lin1_relu_dcount: X and HID rows must be 16-byte aligned");
  if (cap <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_w1_kernel<<<(HIDF * L1_K + 255) / 256, 256, 0, st>>>(W1, (int)kin, planes);
  TM_TRY(check_launch("selfmlp_pack_w1"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_lin1_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L1_SMEM + 1024));
  const int64_t ntiles = (cap + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  L1Args a{cap, X, ldx, x_rows, (int)kin, b1, planes, HID, ldh, nullptr, m_dev};
  selfmlp_lin1_kernel<true><<<grid, THREADS, L1_SMEM + 1024, st>>>(a);
  return check_launch("selfmlp_lin1(device count)");
}

extern "C" int tm_selfmlp_rows_dx_dcount(int64_t cap, const int32_t* m_dev, const float* G, int64_t ldg,
                                         const int32_t* g_rows, const float* W2, const float* H, int64_t ldh,
                                         const int32_t* h_rows, const float* W1, int64_t kin, float* dX, int64_t lddx,
                                         const int32_t* x_rows, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(m_dev && G && W2 && H && W1 && dX, "tm_selfmlp_rows_dx_dcount: NULL operand");
  TM_REQUIRE(kin > 0 && kin <= 48 && (kin & 3) == 0, "tm_selfmlp_rows_dx_dcount: kin must be a multiple of 4, <= 48");
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_rows_dh_ws_bytes(), "tm_selfmlp_rows_dx_dcount: workspace too small (tm_selfmlp_rows_dh_ws_bytes)");
  TM_REQUIRE((ldg & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0 && (ldh & 3) == 0 && (reinterpret_cast<uintptr_t>(H) & 15) == 0 &&
                 (lddx & 3) == 0 && lddx >= kin && (reinterpret_cast<uintptr_t>(dX) & 15) == 0 && (reinterpret_cast<uintptr_t>(W1) & 15) == 0,
             "tm_selfmlp_rows_dx_dcount: G, H, W1 and dX rows must be 16-byte aligned (lddx >= kin)");
  if (cap <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_t_kernel<<<(NOUT * HIDF + 255) / 256, 256, 0, st>>>(W2, planes);
  TM_TRY(check_launch("selfmlp_pack_t"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_bwd1_kernel<true, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B1_SMEM + 1024));
  const int64_t ntiles = (cap + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  B1Args a{cap, G, ldg, g_rows, nullptr, 0, x_rows, (int)kin, W1, nullptr, planes, nullptr, H, ldh, h_rows, nullptr, 0, dX, lddx,
           m_dev};
  selfmlp_gen_bwd1_kernel<true, true, false, true><<<grid, THREADS, B1_SMEM + 1024, st>>>(a);
  return check_launch("selfmlp_rows_dx(device count)");
}

extern "C" int tm_selfmlp_gen_bwd1_dx_dcount(int64_t cap, const int32_t* m_dev, const float* G, int64_t ldg,
                                             const int32_t* g_rows, const float* X, int64_t ldx, const int32_t* x_rows,
                                             int64_t kx, const float* W1, const float* b1, const float* W2, float* dX,
                                             int64_t lddx, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(m_dev && G && X && W1 && b1 && W2 && dX, "tm_selfmlp_gen_bwd1_dx_dcount: NULL operand");
  TM_REQUIRE(kx == 1 || kx == 2, "tm_selfmlp_gen_bwd1_dx_dcount: the first layer must have 1 or 2 inputs");
  TM_REQUIRE(lddx >= kx, "tm_selfmlp_gen_bwd1_dx_dcount: dX row stride lddx < kx");
  TM_REQUIRE(ws && ws_bytes >= tm_selfmlp_bwd1_ws_bytes(), "tm_selfmlp_gen_bwd1_dx_dcount: workspace too small (tm_selfmlp_bwd1_ws_bytes)");
  TM_REQUIRE((ldg & 3) == 0 && (reinterpret_cast<uintptr_t>(G) & 15) == 0, "tm_selfmlp_gen_bwd1_dx_dcount: G rows must be 16-byte aligned");
  if (cap <= 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* planes = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  selfmlp_pack_t_kernel<<<(NOUT * HIDF + 255) / 256, 256, 0, st>>>(W2, planes);
  TM_TRY(check_launch("selfmlp_pack_t"));
  TM_CUDA(cudaFuncSetAttribute(selfmlp_gen_bwd1_kernel<false, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)B1_SMEM + 1024));
  const int64_t ntiles = (cap + TM - 1) / TM;
  const int grid = (int)(ntiles < sm_count() ? ntiles : sm_count());
  B1Args a{cap, G, ldg, g_rows, X, ldx, x_rows, (int)kx, W1, b1, planes, nullptr, nullptr, 0, nullptr, nullptr, 0, dX, lddx,
           m_dev};
  selfmlp_gen_bwd1_kernel<false, true, false, true><<<grid, THREADS, B1_SMEM + 1024, st>>>(a);
  return check_launch("selfmlp_gen_bwd1_dx(device count)");
}
