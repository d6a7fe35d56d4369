// TMA-fed tcgen05 3x3 convolutions on bf16 NHWC activations (U-Net bf16 mode, Unet.py:8-22), and the same kernels
// with k x k taps for LayoutNet's 7x7 / 9x9 layers (model.py:227-243; end of the file).
//
// The activation is a compact bf16 tensor [B][H][W][C] (C a multiple of 16).  A 4-D tensor map
// (C, W, H, B) lets ONE cp.async.bulk.tensor per (tile, tap) fetch the 128 input pixels a tile of
// 128 output pixels needs for that tap -- the box is simply shifted by (tap_x-1, tap_y-1) and TMA's
// out-of-bounds zero fill IS the convolution's zero padding (and the tail of the batch).  The box
// lands in shared memory in exactly the swizzled K-major layout tcgen05.mma reads (32/64/128-byte
// swizzle for 16/32/64 channels per step), so no thread ever touches an operand:
//
//   warp 0   one thread: TMA producer (activation box + weight box per k-step, mbarrier expect_tx)
//   warp 1   one thread: tcgen05.mma issuer, fp32 accumulator double-buffered in tensor memory
//   warps 2-9 epilogue (two per TMEM lane quarter): tcgen05.ld -> (+bias, ReLU, BN statistics) -> transposed 128-bit stores
//
//   fprop / dgrad (conv3x3_tma_kernel):  Y[pix, n] = sum_{tap, c} X[pix + tap, c] * Wq[tap][n][c]
//       (the data gradient is the same kernel on dY with the tap-reversed, transposed weights)
//   wgrad (conv3x3_wgrad_tma_kernel):    dW[tap][co][ci] = sum_pix dY[pix, co] * X[pix + tap, ci]
//       both operands are MN-major (channels contiguous, pixels = K): the same activation boxes,
//       no transposition anywhere; split over pixel blocks x kernel rows, fp32 partials reduced in
//       a fixed order (deterministic).
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>

#include "tm_tc.cuh"

using namespace tmk;
using namespace tmk::tc;

namespace {

// ------------------------------------------------------------------------------------------------
// tensor maps (the encoder lives in libcuda; resolved at run time so the library links without it)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encoder() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

inline CUtensorMapSwizzle swizzle_for(int inner_bytes) {
  return inner_bytes >= 128 ? CU_TENSOR_MAP_SWIZZLE_128B : inner_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                                            : CU_TENSOR_MAP_SWIZZLE_32B;
}

// [B][H][W][C] with a box of (boxC channels, TW, TH, TB); bf16 (esz 2) or fp32 (esz 4) elements, pixel stride ld
// elements (0: C).  mn32: fp32 boxes of 32 channels read as MN-major operands -- 128-byte swizzle with 32-byte atoms,
// the layout tcgen05 calls SWIZZLE_128B_BASE32B (descriptor layout type 1)
int encode_act(CUtensorMap* m, const void* ptr, int64_t C, int64_t W, int64_t H, int64_t B, int boxC, int TW,
               int TH, int TB, int step = 1, int esz = 2, int64_t ld = 0, bool mn32 = false) {   // step 2: every other pixel in W and H (transposed-conv gradients)
  EncodeTiledFn enc = encoder();
  if (!enc) return fail(TM_EINVAL, "cuTensorMapEncodeTiled is not available from the driver");
  if (ld <= 0) ld = C;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)(ld * esz), (cuuint64_t)(W * ld * esz), (cuuint64_t)(H * W * ld * esz)};
  cuuint32_t box[4] = {(cuuint32_t)boxC, (cuuint32_t)(TW * step), (cuuint32_t)(TH * step), (cuuint32_t)TB};
  cuuint32_t es[4] = {1, (cuuint32_t)step, (cuuint32_t)step, 1};
  CUresult r = enc(m, esz == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                   const_cast<void*>(ptr), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   mn32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : swizzle_for(boxC * esz), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(TM_EINVAL, "cuTensorMapEncodeTiled(activation) failed: %d", (int)r);
  return 0;
}

// [rows][C] with a box of (boxC, boxRows); bf16 (esz 2) or fp32 (esz 4)
int encode_2d(CUtensorMap* m, const void* ptr, int64_t C, int64_t rows, int boxC, int boxRows, int esz = 2) {
  EncodeTiledFn enc = encoder();
  if (!enc) return fail(TM_EINVAL, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(C * esz)};
  cuuint32_t box[2] = {(cuuint32_t)boxC, (cuuint32_t)boxRows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, esz == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                   const_cast<void*>(ptr), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(boxC * esz), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(TM_EINVAL, "cuTensorMapEncodeTiled(weights) failed: %d", (int)r);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void prefetch_map(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// shared-memory descriptor layout of a swizzled row of inner_bytes: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B
__host__ __device__ constexpr uint32_t sw_type(int inner_bytes) { return inner_bytes >= 128 ? 2u : inner_bytes == 64 ? 4u : 6u; }

// Store one 16-column chunk of a 32-row accumulator slab.  After tcgen05.ld lane = row; writing from that layout
// would touch 32 different lines with 16 bytes each per instruction.  The chunk is transposed through a padded
// per-warp scratch instead, so that four neighbouring lanes write the 64 contiguous bytes of one row (8 rows per
// instruction, only full 32-byte sectors).  rowp[pass]: output row pass * 8 + lane / 4 (nullptr = outside the batch).
__device__ __forceinline__ void store_chunk16(float* scr, int lane, const float (&v)[16], float* const (&rowp)[4], int64_t coff,
                                              double* stat = nullptr) {
#pragma unroll
  for (int i = 0; i < 16; ++i) scr[lane * 17 + i] = v[i];
  __syncwarp();
  const int c4 = (lane & 3) * 4;
  float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int pass = 0; pass < 4; ++pass) {
    const float* sp = scr + (pass * 8 + (lane >> 2)) * 17 + c4;
    const float4 o = make_float4(sp[0], sp[1], sp[2], sp[3]);
    if (rowp[pass]) st4(rowp[pass] + coff + c4, o);
    if (stat) {          // rows outside the batch are exact zeros (zero-filled input, no bias): they add nothing
      s1[0] += o.x; s1[1] += o.y; s1[2] += o.z; s1[3] += o.w;
      s2[0] = fmaf(o.x, o.x, s2[0]); s2[1] = fmaf(o.y, o.y, s2[1]); s2[2] = fmaf(o.z, o.z, s2[2]); s2[3] = fmaf(o.w, o.w, s2[3]);
    }
  }
  if (stat) {
    // batch-norm statistics of the convolution's output, from the fp32 accumulators: fold the 8 lanes that own
    // the same 4 columns (fixed shuffle tree), then lanes 0..3 add the chunk's 32-row sums into the warp's fp64 slots
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], o);
        s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], o);
      }
    }
    if (lane < 4) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { stat[(c4 + j) * 2] += (double)s1[j]; stat[(c4 + j) * 2 + 1] += (double)s2[j]; }
    }
  }
  __syncwarp();
}

struct Geom {
  int B, H, W, TW, TH, TB, tiles_x, tiles_y;
  int64_t ntiles;
  __host__ __device__ void origin(int64_t t, int& x0, int& y0, int& b0) const {
    x0 = (int)(t % tiles_x) * TW;
    y0 = (int)((t / tiles_x) % tiles_y) * TH;
    b0 = (int)(t / ((int64_t)tiles_x * tiles_y)) * TB;
  }
};

inline bool pow2(int64_t v) { return v > 0 && (v & (v - 1)) == 0; }

// tiles of `tile` pixels (128: one MMA row block; the tf32x3 weight gradient also takes 64 / 32 per pipeline stage)
inline Geom make_geom(int64_t B, int64_t H, int64_t W, int tile = 128) {
  Geom g;
  g.B = (int)B; g.H = (int)H; g.W = (int)W;
  g.TW = (int)(W < tile ? W : tile);
  g.TH = (int)(H < tile / g.TW ? H : tile / g.TW);
  g.TB = tile / (g.TW * g.TH);
  g.tiles_x = (int)(W / g.TW);
  g.tiles_y = (int)(H / g.TH);
  g.ntiles = (int64_t)g.tiles_x * g.tiles_y * cdiv(B, g.TB);
  return g;
}

constexpr int CONV_THREADS = 192;
constexpr int STAT_MAX_N = 128;          // widest accumulator row the fused batch-norm statistics support
constexpr int CONV_MAX_STAGES = 8;
constexpr uint32_t CONV_SMEM_BUDGET = 200 * 1024;
// forward / data-gradient kernels: 8 epilogue warps (two per TMEM lane quarter, splitting the columns / rows of a
// tile) -- the epilogue, not TMA, is what the MMA stream waits for
constexpr int FWD_EPI_WARPS = 8;
constexpr int FWD_THREADS = (2 + FWD_EPI_WARPS) * 32;
constexpr uint32_t FWD_SMEM_BUDGET = 184 * 1024;

// Operand formats.  FMT_BF16: one bf16 plane per operand, kind::f16.  FMT_TF32X3: fp32 operands read in place by TMA
// (tcgen05.mma.kind::tf32 uses the upper 19 bits of each word, so the fp32 word is the "hi" operand); the residual
// lo = x - trunc_tf32(x) (tm_split.cuh) is formed in shared memory next to it, and every 32-byte K chunk issues
// hi*hi + hi*lo + lo*hi into one fp32 accumulator -- the 3xTF32 product of tf_gemm_kernel (tm_tc.cuh).
constexpr int FMT_BF16 = 0, FMT_TF32X3 = 1;
// tf32x3 forward / data gradient: warps that form the lo planes of a stage once TMA has landed its hi planes
constexpr int SPLIT_WARPS = 4;

// lo = x - trunc_tf32(x) for the `bytes` of hi operand at st, written at st + lo_off.  Elementwise at the same
// offset, so the lo plane has the hi plane's swizzled layout whatever the swizzle.
__device__ __forceinline__ void split_lo(uint8_t* st, uint32_t bytes, uint32_t lo_off, int t, int nthr) {
  const float4* hi = reinterpret_cast<const float4*>(st);
  float4* lo = reinterpret_cast<float4*>(st + lo_off);
#pragma unroll 4
  for (int i = t; i < (int)(bytes >> 4); i += nthr) lo[i] = tf32_lo(hi[i]);
}

struct ConvArgs {
  Geom g;                            // geometry in PACKED pixels (rows of P pixels)
  int Cin, N, stages;                // channels per packed row: Cin = P * cin, N = P * cout
  int P, cpx;                        // pixels per row, output channels per pixel
  int ntaps, cscale, convt;          // taps (k*k / 4 / 1), coordinate scale of the input map, transposed-conv scatter epilogue
  signed char tdx[81], tdy[81];      // input offset of every tap (up to 9x9)
  uint32_t a_bytes, b_bytes, stage_bytes;
  uint32_t hi_bytes;                 // FMT_TF32X3: offset of the lo planes inside a stage
  int ksplit, kper;                  // FMT_TF32X3: K splits (k-steps kper each); split z writes y + z * zstride
  int64_t zstride;
  float* y;
  int64_t ldy;
  const float* bias;
  int flags;
  int* err;
  double* stats;                     // optional [gridDim.x * 4][N][2]: per epilogue warp sum / sum of squares per column
};

// ------------------------------------------------------------------------------------------------
// fprop / dgrad
// ------------------------------------------------------------------------------------------------
// FMT_TF32X3: CK fp32 channels per k-step (128- or 64-byte rows); a stage holds the hi planes of A and B (TMA) and,
// hi_bytes further, their lo planes (SPLIT_WARPS warps).  ksplit > 1: work unit = (tile, K split), fp32 partials.
template <int CK, int FMT>
__global__ void __launch_bounds__(FWD_THREADS + (FMT == FMT_TF32X3 ? SPLIT_WARPS * 32 : 0), 1)
conv3x3_tma_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmw, ConvArgs a) {
  constexpr bool TF = FMT == FMT_TF32X3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ __align__(8) uint64_t full_bar[CONV_MAX_STAGES], empty_bar[CONV_MAX_STAGES], acc_full[2], acc_empty[2];
  __shared__ __align__(8) uint64_t lo_bar[TF ? CONV_MAX_STAGES : 1];   // TF: lo planes of the stage written
  __shared__ float epi_scr[FWD_EPI_WARPS][32 * 17];
  __shared__ double epi_stat[FWD_EPI_WARPS][STAT_MAX_N * 2];       // per epilogue warp: column sums / sums of squares (a.stats)
  __shared__ uint32_t tmem_base_s;
  __shared__ int abort_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NS = a.stages, N = a.N;
  const uint32_t tmem_cols = 2 * N < 32 ? 32u : (uint32_t)(2 * N);

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) {
      mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1);
      if (TF) mbar_init(&lo_bar[i], SPLIT_WARPS);
    }
    mbar_init(&acc_full[0], 1); mbar_init(&acc_full[1], 1);
    mbar_init(&acc_empty[0], FWD_EPI_WARPS); mbar_init(&acc_empty[1], FWD_EPI_WARPS);
    abort_s = 0;
    fence_mbarrier_init();
    prefetch_map(&tmx);
    prefetch_map(&tmw);
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  volatile int* abortp = &abort_s;
  bool ok = true;
  const int64_t G = gridDim.x;
  const int csteps = a.Cin / CK;
  const int ksteps = a.ntaps * csteps;
  const int64_t nunits = TF ? a.g.ntiles * a.ksplit : a.g.ntiles;
  // work unit u -> tile t, K split z, k-steps [k0, k1)
  auto unit = [&](int64_t u, int64_t& t, int& z, int& k0, int& k1) {
    if (TF) {
      t = u / a.ksplit; z = (int)(u - t * a.ksplit);
      k0 = z * a.kper; k1 = k0 + a.kper < ksteps ? k0 + a.kper : ksteps;
    } else {
      t = u; z = 0; k0 = 0; k1 = ksteps;
    }
  };

  if (warp == 0) {
    // ======================= TMA producer =======================
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      for (int64_t u = blockIdx.x; u < nunits && ok; u += G) {
        int64_t t; int z, k0, k1;
        unit(u, t, z, k0, k1);
        int x0, y0, b0;
        a.g.origin(t, x0, y0, b0);
        for (int tap = 0; tap < a.ntaps && ok; ++tap) {
          const int dx = a.tdx[tap], dy = a.tdy[tap];
          for (int cs = 0; cs < csteps; ++cs) {
            if (TF && (tap * csteps + cs < k0 || tap * csteps + cs >= k1)) continue;
            ok = mbar_wait_abort(&empty_bar[s], ph ^ 1u, abortp);
            if (!ok) break;
            const uint32_t base = smem_u32(ring + (size_t)s * a.stage_bytes);
            mbar_expect_tx(&full_bar[s], a.a_bytes + a.b_bytes);
            tma_load_4d(base, &tmx, cs * CK, x0 * a.cscale + dx, y0 * a.cscale + dy, b0, &full_bar[s]);
            tma_load_2d(base + a.a_bytes, &tmw, cs * CK, tap * N, &full_bar[s]);
            if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      const uint32_t idesc = TF ? make_idesc(Fmt::TF32, N) : make_idesc(Fmt::BF16, N);
      constexpr int RB = CK * (TF ? 4 : 2);                 // bytes per operand row; one MMA takes 32 of them
      constexpr uint32_t TY = sw_type(RB), SBO = 8u * RB;
      uint32_t s = 0, ph = 0;
      int li = 0;
      for (int64_t u = blockIdx.x; u < nunits && ok; u += G, ++li) {
        int64_t t; int z, k0, k1;
        unit(u, t, z, k0, k1);
        const int buf = li & 1;
        ok = mbar_wait_abort(&acc_empty[buf], (((uint32_t)(li >> 1)) & 1u) ^ 1u, abortp);
        if (!ok) break;
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(buf * N);
        for (int ks = k0; ks < k1; ++ks) {
          ok = mbar_wait_abort(TF ? &lo_bar[s] : &full_bar[s], ph, abortp);
          if (!ok) break;
          tc_fence_after();
          const uint32_t base = smem_u32(ring + (size_t)s * a.stage_bytes);
#pragma unroll
          for (int j = 0; j < RB / 32; ++j) {
            const uint64_t da = smem_desc(base + j * 32, 16, SBO, TY);
            const uint64_t db = smem_desc(base + a.a_bytes + j * 32, 16, SBO, TY);
            if (TF) {
              const uint64_t dal = smem_desc(base + a.hi_bytes + j * 32, 16, SBO, TY);
              const uint64_t dbl = smem_desc(base + a.hi_bytes + a.a_bytes + j * 32, 16, SBO, TY);
              umma_tf32(tmem_d, da, db, idesc, (ks > k0 || j > 0) ? 1u : 0u);
              umma_tf32(tmem_d, da, dbl, idesc, 1u);
              umma_tf32(tmem_d, dal, db, idesc, 1u);
            } else {
              umma_f16(tmem_d, da, db, idesc, (ks > k0 || j > 0) ? 1u : 0u);
            }
          }
          umma_commit(&empty_bar[s]);
          if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
        }
        if (!ok) break;
        umma_commit(&acc_full[buf]);
      }
    }
    __syncwarp();
  } else if (TF && warp >= 2 + FWD_EPI_WARPS) {
    // ======================= lo planes (tf32x3) =======================
    const int rt = tid - (2 + FWD_EPI_WARPS) * 32;
    uint32_t s = 0, ph = 0;
    for (int64_t u = blockIdx.x; u < nunits && ok; u += G) {
      int64_t t; int z, k0, k1;
      unit(u, t, z, k0, k1);
      for (int ks = k0; ks < k1; ++ks) {
        ok = mbar_wait_abort(&full_bar[s], ph, abortp);
        if (!ok) break;
        split_lo(ring + (size_t)s * a.stage_bytes, a.a_bytes + a.b_bytes, a.hi_bytes, rt, SPLIT_WARPS * 32);
        fence_async_smem();                                // generic stores -> async proxy (the MMAs)
        __syncwarp();
        if (lane == 0) mbar_arrive(&lo_bar[s]);
        if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
      }
    }
  } else {
    // ======================= epilogue =======================
    const int q = warp & 3;                               // TMEM lane quarter this warp may read
    const int e = warp - 2, half = e >> 2;                // two warps per quarter: even / odd 16-column chunks
    float* scr = epi_scr[e];
    double* wstat = epi_stat[e];
    if (a.stats) {
      for (int i = lane; i < 2 * N; i += 32) wstat[i] = 0.0;
      __syncwarp();
    }
    int li = 0;
    for (int64_t u = blockIdx.x; u < nunits && ok; u += G, ++li) {
      int64_t t; int z, k0, k1;
      unit(u, t, z, k0, k1);
      float* const yz = TF ? a.y + z * a.zstride : a.y;
      const int buf = li & 1;
      ok = mbar_wait_abort(&acc_full[buf], ((uint32_t)(li >> 1)) & 1u, abortp);
      if (!ok) break;
      tc_fence_after();
      int x0, y0, b0;
      a.g.origin(t, x0, y0, b0);
      float* rowp[4];
#pragma unroll
      for (int pass = 0; pass < 4; ++pass) {                // the rows this lane stores after the transposition
        const int m = q * 32 + pass * 8 + (lane >> 2);
        const int tw = m % a.g.TW, th = (m / a.g.TW) % a.g.TH, tb = m / (a.g.TW * a.g.TH);
        if (a.convt)       // transposed conv k2 s2: the row is the 2x2 output window of input pixel (y0+th, x0+tw)
          rowp[pass] = b0 + tb < a.g.B
                           ? yz + (((int64_t)(b0 + tb) * 2 * a.g.H + 2 * (y0 + th)) * 2 * a.g.W + 2 * (x0 + tw)) * a.ldy
                           : nullptr;
        else
          rowp[pass] = b0 + tb < a.g.B
                           ? yz + (((int64_t)(b0 + tb) * a.g.H + (y0 + th)) * a.g.W + (x0 + tw)) * a.P * a.ldy
                           : nullptr;
      }
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * N);
      for (int c = half * 16; c < N; c += 32) {
        float v[16];
        tmem_ld16(trow + (uint32_t)c, v);
        const int po = c / a.cpx, co = c - po * a.cpx;     // pixel inside the packed row, its first channel
        if (a.flags & TM_EPI_BIAS) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] += __ldg(a.bias + co + i);
        }
        if (a.flags & TM_EPI_RELU) {
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
        }
        // po: pixel inside the packed row -- or, for the transposed conv, the quadrant (dy, dx) of the 2x2 window
        const int64_t coff = a.convt ? ((int64_t)(po >> 1) * 2 * a.g.W + (po & 1)) * a.ldy + co : (int64_t)po * a.ldy + co;
        store_chunk16(scr, lane, v, rowp, coff, a.stats ? wstat + c * 2 : nullptr);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
    }
    if (a.stats && ok) {
      __syncwarp();
      for (int i = lane; i < 2 * N; i += 32) a.stats[((int64_t)blockIdx.x * FWD_EPI_WARPS + e) * 2 * N + i] = wstat[i];
    }
  }
  if (!ok) {
    abort_s = 1;
    if (a.err) atomicExch(a.err, 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------
// fprop / dgrad, row-reuse variant for layers whose whole packed weight (9 taps x N x 64 channels, N <= 64)
// stays resident in shared memory and whose rows are >= 128 packed pixels wide.
// A tile is 128 packed pixels x ROWS image rows.  Every input row y0-1 .. y0+ROWS is fetched ONCE per horizontal
// shift (3 boxes) and feeds the three output rows it touches (kernel rows r = 0..2 -> accumulators j = iy+1-r):
// shared-memory fill per output row drops from 9 activation boxes + 9 weight boxes to 3 (ROWS+2)/ROWS boxes.
// ------------------------------------------------------------------------------------------------
constexpr int V2_ROWS = 4;

template <int ROWS>
__global__ void __launch_bounds__(FWD_THREADS, 1)
conv3x3_tma_rows_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmw, ConvArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* wsm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int N = a.N;
  const uint32_t w_tap = (uint32_t)N * 128u;                       // one tap: N rows x 64 channels bf16
  uint8_t* ring = wsm + 9 * (size_t)w_tap;                          // 9 * N * 128 is a multiple of 1024 (N % 16 == 0 -> check on host)
  __shared__ __align__(8) uint64_t full_bar[CONV_MAX_STAGES], empty_bar[CONV_MAX_STAGES], acc_full[2], acc_empty[2], w_full;
  __shared__ float epi_scr[FWD_EPI_WARPS][32 * 17];
  __shared__ double epi_stat[FWD_EPI_WARPS][STAT_MAX_N * 2];       // per epilogue warp: column sums / sums of squares (a.stats)
  __shared__ uint32_t tmem_base_s;
  __shared__ int abort_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NS = a.stages;
  uint32_t tmem_cols = 32;
  while (tmem_cols < (uint32_t)(2 * ROWS * N)) tmem_cols <<= 1;

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    mbar_init(&acc_full[0], 1); mbar_init(&acc_full[1], 1);
    mbar_init(&acc_empty[0], FWD_EPI_WARPS); mbar_init(&acc_empty[1], FWD_EPI_WARPS);
    mbar_init(&w_full, 1);
    abort_s = 0;
    fence_mbarrier_init();
    prefetch_map(&tmx);
    prefetch_map(&tmw);
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  volatile int* abortp = &abort_s;
  bool ok = true;
  const int64_t G = gridDim.x;
  // tiles: (x block of 128 packed pixels, group of ROWS image rows, image)
  const int tiles_x = a.g.W / 128, tiles_y = a.g.H / ROWS;
  const int64_t ntiles = (int64_t)tiles_x * tiles_y * a.g.B;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(&w_full, 9u * w_tap);
      // resident order: for every horizontal shift S the kernel rows r = 2, 1, 0 are stacked, so that the taps that
      // read the same input row write NEIGHBOURING accumulators and fuse into one MMA of up to 3N columns
      for (int t = 0; t < 9; ++t)
        tma_load_2d(smem_u32(wsm + (size_t)((t % 3) * 3 + (2 - t / 3)) * w_tap), &tmw, 0, t * N, &w_full);
      uint32_t s = 0, ph = 0;
      for (int64_t t = blockIdx.x; t < ntiles && ok; t += G) {
        const int x0 = (int)(t % tiles_x) * 128, y0 = (int)((t / tiles_x) % tiles_y) * ROWS;
        const int b = (int)(t / ((int64_t)tiles_x * tiles_y));
        for (int iy = -1; iy <= ROWS && ok; ++iy) {
          for (int S = 0; S < 3; ++S) {
            ok = mbar_wait_abort(&empty_bar[s], ph ^ 1u, abortp);
            if (!ok) break;
            if (a.flags & 0x400) { mbar_arrive(&full_bar[s]); }
            else {
            mbar_expect_tx(&full_bar[s], a.a_bytes);
            tma_load_4d(smem_u32(ring + (size_t)s * a.a_bytes), &tmx, 0, x0 + S - 1, y0 + iy, b, &full_bar[s]);
            }
            if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc(Fmt::BF16, N);
      ok = mbar_wait_abort(&w_full, 0, abortp);
      uint32_t s = 0, ph = 0;
      int li = 0;
      for (int64_t t = blockIdx.x; t < ntiles && ok; t += G, ++li) {
        const int buf = li & 1;
        ok = mbar_wait_abort(&acc_empty[buf], (((uint32_t)(li >> 1)) & 1u) ^ 1u, abortp);
        if (!ok) break;
        tc_fence_after();
        const uint32_t acc0 = tmem_base + (uint32_t)(buf * ROWS * N);
        for (int iy = -1; iy <= ROWS && ok; ++iy) {
          for (int S = 0; S < 3; ++S) {
            ok = mbar_wait_abort(&full_bar[s], ph, abortp);
            if (!ok) break;
            tc_fence_after();
            const uint32_t abase = smem_u32(ring + (size_t)s * a.a_bytes);
            // input row iy feeds output rows j = iy + 1 - r through kernel row r; valid r: 0 <= j < ROWS
            const int r_lo = iy + 1 - (ROWS - 1) > 0 ? iy + 1 - (ROWS - 1) : 0;
            const int r_hi = iy + 1 < 2 ? iy + 1 : 2;
            if (!(a.flags & 0x200)) {
              const uint32_t wS = smem_u32(wsm + (size_t)(S * 3) * w_tap);       // stacked [r=2; r=1; r=0] for this shift
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint64_t da = smem_desc(abase + k * 32, 16, 1024, 2);
                int hi = r_hi;
                if (S == 0 && k == 0 && r_lo == 0) {
                  // first touch of accumulator j = iy + 1 (kernel row 0): overwrite instead of accumulate
                  umma_f16(acc0 + (uint32_t)((iy + 1) * N), da, smem_desc(wS + 2 * w_tap + k * 32, 16, 1024, 2), idesc, 0u);
                  if (r_hi == 0) continue;
                  // the remaining rows r = 1 .. r_hi accumulate: handled below with r_lo' = 1
                  const int nr = r_hi;                                             // rows 1 .. r_hi
                  umma_f16(acc0 + (uint32_t)((iy + 1 - r_hi) * N), da, smem_desc(wS + (uint32_t)(2 - r_hi) * w_tap + k * 32, 16, 1024, 2),
                       make_idesc(Fmt::BF16, nr * N), 1u);
                  continue;
                }
                const int nr = hi - r_lo + 1;
                umma_f16(acc0 + (uint32_t)((iy + 1 - hi) * N), da, smem_desc(wS + (uint32_t)(2 - hi) * w_tap + k * 32, 16, 1024, 2),
                     make_idesc(Fmt::BF16, nr * N), 1u);
              }
            }
            umma_commit(&empty_bar[s]);
            if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
          }
        }
        if (!ok) break;
        umma_commit(&acc_full[buf]);
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3;
    const int e = warp - 2, half = e >> 2;                // two warps per quarter: even / odd image rows of the tile
    float* scr = epi_scr[e];
    double* wstat = epi_stat[e];
    if (a.stats) {
      for (int i = lane; i < 2 * N; i += 32) wstat[i] = 0.0;
      __syncwarp();
    }
    int li = 0;
    for (int64_t t = blockIdx.x; t < ntiles && ok; t += G, ++li) {
      const int buf = li & 1;
      ok = mbar_wait_abort(&acc_full[buf], ((uint32_t)(li >> 1)) & 1u, abortp);
      if (!ok) break;
      tc_fence_after();
      const int x0 = (int)(t % tiles_x) * 128, y0 = (int)((t / tiles_x) % tiles_y) * ROWS;
      const int b = (int)(t / ((int64_t)tiles_x * tiles_y));
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * ROWS * N);
      for (int j = half; j < ROWS; j += 2) {
        float* rowp[4];
#pragma unroll
        for (int pass = 0; pass < 4; ++pass)
          rowp[pass] = a.y + (((int64_t)b * a.g.H + (y0 + j)) * a.g.W + (x0 + q * 32 + pass * 8 + (lane >> 2))) * a.P * a.ldy;
        for (int c = 0; c < N; c += 16) {
          float v[16];
          tmem_ld16(trow + (uint32_t)(j * N + c), v);
          const int po = c / a.cpx, co = c - po * a.cpx;
          if (a.flags & TM_EPI_BIAS) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] += __ldg(a.bias + co + i);
          }
          if (a.flags & TM_EPI_RELU) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
          }
          if (!(a.flags & 0x100))
            store_chunk16(scr, lane, v, rowp, (int64_t)po * a.ldy + co, a.stats ? wstat + (c) * 2 : nullptr);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
    }
    if (a.stats && ok) {
      __syncwarp();
      for (int i = lane; i < 2 * N; i += 32) a.stats[((int64_t)blockIdx.x * FWD_EPI_WARPS + e) * 2 * N + i] = wstat[i];
    }
  }
  if (!ok) {
    abort_s = 1;
    if (a.err) atomicExch(a.err, 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------
// wgrad: grid (pixel splits, k kernel rows x tap groups); CTA (z, r, grp) accumulates taps (r, grp*tg ..) over its
// pixel blocks
// ------------------------------------------------------------------------------------------------
struct WgradArgs {
  Geom g;
  int Cin, Cout, stages;
  int cbx, nbx, cby, nby;            // channels per TMA box / boxes per tile, x and dy
  uint32_t x_bytes, dy_bytes, stage_bytes;
  float* part;                       // [splits][taps][Cout][Cin]
  int* err;
  int cscale;                        // coordinate scale of the tapped map (2: transposed-conv gradient, every other pixel)
  signed char tdx[4], tdy[4];        // NT == 4: offsets of the four taps (transposed conv); NT == 3 / 1 / 0 use (s - k/2, r - k/2)
  int k, tg, groups;                 // NT == 0 (k x k): kernel size, taps per group, groups per kernel row
  uint32_t hi_bytes;                 // FMT_TF32X3: offset of the lo planes inside a stage
  int tp;                            // FMT_TF32X3: pixels per stage (128 / 64 / 32: the tile of a.g)
};

// NT: tapped tiles per stage -- 4: transposed conv; 3: a 3x3 kernel row fused; 1: one tap per stage; 0: k x k, a group
// of a kernel row's taps fused (runtime k / tg / groups; NT == 3 is this with k = tg = 3 as compile-time constants)
// FMT_TF32X3: fp32 boxes of 32 channels, MN-major SWIZZLE_128B_BASE32B; a.tp pixels per stage; the epilogue warps,
// idle until the last MMA, form each stage's lo planes first.
template <int NT, int FMT>
__global__ void __launch_bounds__(CONV_THREADS, 1)
conv3x3_wgrad_tma_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmdy, WgradArgs a) {
  constexpr bool TF = FMT == FMT_TF32X3;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  __shared__ __align__(8) uint64_t full_bar[CONV_MAX_STAGES], empty_bar[CONV_MAX_STAGES], acc_full;
  __shared__ __align__(8) uint64_t lo_bar[TF ? CONV_MAX_STAGES : 1];
  __shared__ uint32_t tmem_base_s;
  __shared__ int abort_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NS = a.stages, Cin = a.Cin, Cout = a.Cout;
  // NT == 0: a kernel row's taps are split into groups of tg, so that a group's accumulators (tg * Cin columns) fit
  // one MMA (N <= 256); the CTA (z, r, grp) accumulates taps s0 .. s0 + nt - 1 of kernel row r
  constexpr bool KXK = NT == 0;
  constexpr int NTOT = NT == 4 ? 4 : 3;                   // taps accumulated by one CTA (NT != 0)
  const int r = KXK ? (int)blockIdx.y / a.groups : (int)blockIdx.y;
  const int s0 = KXK ? ((int)blockIdx.y % a.groups) * a.tg : 0;
  const int nt = KXK ? (a.k - s0 < a.tg ? a.k - s0 : a.tg) : NTOT;
  const int kw = KXK ? a.k : NTOT;                        // taps per kernel row
  const int TT = KXK ? a.k * a.k : NT == 4 ? 4 : 9;       // taps in the whole gradient
  const int half_k = KXK ? a.k / 2 : 1;
  const int nload = KXK ? nt : NT;                        // tapped tiles per stage
  uint32_t tmem_cols = 32;
  while (tmem_cols < (uint32_t)((KXK ? a.tg : NTOT) * Cin)) tmem_cols <<= 1;

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) {
      mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1);
      if (TF) mbar_init(&lo_bar[i], 4);
    }
    mbar_init(&acc_full, 1);
    abort_s = 0;
    fence_mbarrier_init();
    prefetch_map(&tmx);
    prefetch_map(&tmdy);
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  volatile int* abortp = &abort_s;
  bool ok = true;
  const int64_t G = gridDim.x;
  constexpr int STEPS = NT == 1 ? 3 : 1;                  // stages per pixel block

  if (warp == 0) {
    if (lane == 0) {
      uint32_t s = 0, ph = 0;
      for (int64_t t = blockIdx.x; t < a.g.ntiles && ok; t += G) {
        int x0, y0, b0;
        a.g.origin(t, x0, y0, b0);
        for (int st = 0; st < STEPS && ok; ++st) {
          ok = mbar_wait_abort(&empty_bar[s], ph ^ 1u, abortp);
          if (!ok) break;
          const uint32_t base = smem_u32(ring + (size_t)s * a.stage_bytes);
          mbar_expect_tx(&full_bar[s], a.dy_bytes + nload * a.x_bytes);
          for (int j = 0; j < a.nby; ++j)
            tma_load_4d(base + j * (a.dy_bytes / a.nby), &tmdy, j * a.cby, x0, y0, b0, &full_bar[s]);
#pragma unroll
          for (int u = 0; u < nload; ++u) {
            const int cx = NT == 4 ? x0 * a.cscale + a.tdx[u] : x0 + s0 + (NT == 1 ? st : u) - half_k;
            const int cy = NT == 4 ? y0 * a.cscale + a.tdy[u] : y0 + r - half_k;
            for (int j = 0; j < a.nbx; ++j)
              tma_load_4d(base + a.dy_bytes + u * a.x_bytes + j * (a.x_bytes / a.nbx), &tmx, j * a.cbx, cx, cy, b0,
                          &full_bar[s]);
          }
          if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = TF ? make_idesc(Fmt::TF32, Cin, true, true) : make_idesc(Fmt::BF16, Cin, true, true);
      // MN-major operand tiles: pixel row k at k * (cb*2) bytes; 8-pixel groups at SBO; the next 64-channel box at LBO
      const uint32_t a_ty = sw_type(a.cby * 2), b_ty = sw_type(a.cbx * 2);
      const uint32_t a_sbo = 8u * a.cby * 2u, b_sbo = 8u * a.cbx * 2u;
      const uint32_t a_lbo = a.nby > 1 ? a.dy_bytes / a.nby : 0u, b_lbo = a.nbx > 1 ? a.x_bytes / a.nbx : 0u;
      const uint32_t a_kstep = 16u * a.cby * 2u, b_kstep = 16u * a.cbx * 2u;   // 16 pixels per MMA
      uint32_t s = 0, ph = 0;
      bool first = true;
      for (int64_t t = blockIdx.x; t < a.g.ntiles && ok; t += G) {
        for (int st = 0; st < STEPS && ok; ++st) {
          ok = mbar_wait_abort(TF ? &lo_bar[s] : &full_bar[s], ph, abortp);
          if (!ok) break;
          tc_fence_after();
          const uint32_t base = smem_u32(ring + (size_t)s * a.stage_bytes);
          if (TF) {
            // 32-channel boxes of tp pixels x 128 bytes: 4-pixel groups at SBO = 512, 8 pixels (one MMA) = 1024 bytes,
            // the next 32 channels (box) at LBO; the tapped tiles' boxes are uniformly spaced, so NT != 1 is again ONE
            // MMA of nload * Cin columns.  LBO 0: a single box, re-read for M rows beyond Cout (never stored).
            const uint32_t box_y = a.dy_bytes / a.nby, box_x = a.x_bytes / a.nbx;
            const uint32_t lbo_y = a.nby > 1 ? box_y : 0u;
            const uint32_t idn = NT != 1 ? make_idesc(Fmt::TF32, nload * Cin, true, true) : idesc;
            const uint32_t tmem_d = tmem_base + (uint32_t)(NT != 1 ? 0 : st * Cin);
            const uint32_t xb = base + a.dy_bytes;
            for (int j = 0; j < a.tp / 8; ++j) {
              const uint64_t da = smem_desc(base + j * 1024, lbo_y, 512, 1);
              const uint64_t db = smem_desc(xb + j * 1024, box_x, 512, 1);
              const uint64_t dal = smem_desc(base + a.hi_bytes + j * 1024, lbo_y, 512, 1);
              const uint64_t dbl = smem_desc(xb + a.hi_bytes + j * 1024, box_x, 512, 1);
              umma_tf32(tmem_d, da, db, idn, (!first || j > 0) ? 1u : 0u);
              umma_tf32(tmem_d, da, dbl, idn, 1u);
              umma_tf32(tmem_d, dal, db, idn, 1u);
            }
          } else if (NT != 1) {
            // the tapped tiles are one MN-major operand of nload * Cin columns (tile stride = leading byte
            // offset), their accumulators neighbours in TMEM: ONE MMA per 16 pixels instead of nload
            const uint32_t idesc3 = make_idesc(Fmt::BF16, nload * Cin, true, true);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint64_t da = smem_desc(base + j * a_kstep, a_lbo, a_sbo, a_ty);
              const uint64_t db = smem_desc(base + a.dy_bytes + j * b_kstep, a.x_bytes, b_sbo, b_ty);
              umma_f16(tmem_base, da, db, idesc3, (!first || j > 0) ? 1u : 0u);
            }
          } else {
            const uint32_t tmem_d = tmem_base + (uint32_t)(st * Cin);       // tap inside the kernel row
            const uint32_t xb = base + a.dy_bytes;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const uint64_t da = smem_desc(base + j * a_kstep, a_lbo, a_sbo, a_ty);
              const uint64_t db = smem_desc(xb + j * b_kstep, b_lbo, b_sbo, b_ty);
              umma_f16(tmem_d, da, db, idesc, (!first || j > 0) ? 1u : 0u);
            }
          }
          umma_commit(&empty_bar[s]);
          if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
          if (NT != 1 || st == STEPS - 1) first = false;
        }
      }
      if (ok) umma_commit(&acc_full);
    }
    __syncwarp();
  } else {
    const int q = warp & 3;
    const int co = q * 32 + lane;
    if (TF) {
      // lo planes of every stage of this CTA, in the producer's order
      uint32_t s = 0, ph = 0;
      for (int64_t t = blockIdx.x; t < a.g.ntiles && ok; t += G) {
        for (int st = 0; st < STEPS && ok; ++st) {
          ok = mbar_wait_abort(&full_bar[s], ph, abortp);
          if (!ok) break;
          split_lo(ring + (size_t)s * a.stage_bytes, a.dy_bytes + nload * a.x_bytes, a.hi_bytes, tid - 64, 128);
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(&lo_bar[s]);
          if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
        }
      }
    }
    if (ok) ok = mbar_wait_abort(&acc_full, 0, abortp);
    if (ok) {
      tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
      for (int tl = 0; tl < nt; ++tl) {
        float* pp = a.part + (((int64_t)blockIdx.x * TT + r * kw + s0 + tl) * Cout + co) * Cin;
        for (int c = 0; c < Cin; c += 16) {
          float v[16];
          tmem_ld16(trow + (uint32_t)(tl * Cin + c), v);
          if (co < Cout) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) st4(pp + c + i, make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
          }
        }
      }
    }
  }
  if (!ok) {
    abort_s = 1;
    if (a.err) atomicExch(a.err, 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

// part [splits][(r,S)][po*Cout+co][pi*CinP+ci] (packed rows of P pixels) -> dw [Cout][Cin][k][k] (torch layout):
// tap (r, s) collects every (S, po, pi) with S*P + pi - po + k/2 == s.  One warp per output element: lane z owns the
// splits z, z+32, ..., the lanes are folded by a fixed shuffle tree (deterministic).
// KC: the kernel size as a compile-time constant (3), or 0: k_rt
template <int KC>
__global__ void wgrad_reduce_kernel(const float* __restrict__ part, int splits, int P, int Cout, int CinP, int Cin, int k_rt,
                                    float* __restrict__ dw) {
  const int lane = threadIdx.x & 31;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int k = KC ? KC : k_rt, kk = k * k, h = k / 2;
  if (i >= (int64_t)kk * Cout * Cin) return;
  // ci fastest: neighbouring warps read neighbouring partials
  const int ci = (int)(i % Cin), co = (int)((i / Cin) % Cout), tap = (int)(i / ((int64_t)Cin * Cout));
  const int r = tap / k, sx = tap % k;
  const int64_t ldn = (int64_t)P * CinP, per_tap = (int64_t)P * Cout * ldn;
  float s = 0.f;
  for (int z = lane; z < splits; z += 32)
    for (int S = -h; S <= h; ++S)
      for (int po = 0; po < P; ++po) {
        const int pi = sx - h + po - S * P;
        if (pi < 0 || pi >= P) continue;
        s += part[((int64_t)z * kk + r * k + S + h) * per_tap + ((int64_t)po * Cout + co) * ldn + (int64_t)pi * CinP + ci];
      }
  s = warp_sum(s);
  if (lane == 0) dw[((int64_t)co * Cin + ci) * kk + tap] = s;
}

// fp32 rows (stride ld) -> compact bf16 rows of Cp >= C channels (zero padded); 8 channels per thread
__global__ void to_bf16_kernel(int64_t npix, int C, const float* __restrict__ x, int64_t ld, __nv_bfloat16* __restrict__ out,
                               int Cp, int vec) {
  const int groups = Cp / 8;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix * groups) return;
  const int64_t p = i / groups;
  const int c0 = (int)(i % groups) * 8;
  float v[8];
  const float* xp = x + p * ld + c0;
  if (vec && c0 + 8 <= C) {
    const float4 a = ld4_stream(xp), b = ld4_stream(xp + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = c0 + j < C ? xp[j] : 0.f;
  }
  uint4 o;
  o.x = pack_bf16(v[0], v[1]); o.y = pack_bf16(v[2], v[3]); o.z = pack_bf16(v[4], v[5]); o.w = pack_bf16(v[6], v[7]);
  *reinterpret_cast<uint4*>(out + p * Cp + c0) = o;
}

// w [Cout][Cin][ks][ks] fp32 -> operand of the convolution over rows of P packed pixels:
//   q[(r,S)][n = po*Nc + nc][k = pi*KcP + kc],  S in {-ks/2..ks/2} = neighbouring packed row, po / pi = pixel inside
//   the output / input row; the entry is the tap s = S*P + pi - po + ks/2 of kernel row r when 0 <= s < ks, else 0.
//   dgrad == 0: n = output channel co, k = input channel ci                    (forward operand)
//   dgrad == 1: n = ci, k = co, taps reversed (r, s) -> (ks-1-r, ks-1-s)       (data-gradient operand)
__device__ __forceinline__ void put(__nv_bfloat16* q, int64_t i, float v) { q[i] = __float2bfloat16(v); }
__device__ __forceinline__ void put(float* q, int64_t i, float v) { q[i] = v; }
template <typename T>
__global__ void pack_w_kernel(int Cout, int Cin, int ks, const float* __restrict__ w, T* __restrict__ q, int P, int KcP,
                              int dgrad) {
  const int Nc = dgrad ? Cin : Cout, Kc = dgrad ? Cout : Cin;
  const int64_t ldk = (int64_t)P * KcP, rows = (int64_t)P * Nc;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)ks * ks * rows * ldk) return;
  const int k = (int)(i % ldk), n = (int)((i / ldk) % rows), t = (int)(i / (ldk * rows));
  const int h = ks / 2, r = t / ks, S = t % ks - h;
  const int pi = k / KcP, kc = k % KcP, po = n / Nc, nc = n % Nc;
  const int sx = S * P + pi - po + h;
  float v = 0.f;
  if (sx >= 0 && sx < ks && kc < Kc) {
    const int co = dgrad ? kc : nc, ci = dgrad ? nc : kc;
    const int tap = dgrad ? (ks - 1 - r) * ks + (ks - 1 - sx) : r * ks + sx;
    v = w[((int64_t)co * Cin + ci) * ks * ks + tap];
  }
  put(q, i, v);
}

inline bool conv_shape_ok(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N) {
  return B > 0 && pow2(H) && pow2(W) && H * W >= 1 && Cin % 16 == 0 && Cin >= 16 && Cin <= 256 &&
         (Cin <= 64 ? pow2(Cin) : Cin % 64 == 0) && N % 16 == 0 && N >= 16 && N <= 256 && W <= 65536 && H <= 65536;
}

// pixels packed into one operand row: narrow layers (16 / 32 channels) are run as 64-channel layers over rows of
// 4 / 2 horizontally adjacent pixels (block-sparse packed weights), so that every TMA row is a full 128-byte line
inline int conv_pack(int64_t W, int64_t cin, int64_t cout) {
  int P = 1;
  while (P * cin < 64 && 2 * P <= W && 2 * P * cout <= 256) P *= 2;
  return P;
}
inline int wgrad_pack(int64_t W, int64_t cin, int64_t cout) {
  const int64_t lo = cin < cout ? cin : cout, hi = cin < cout ? cout : cin;
  int P = 1;
  while (P * lo < 64 && 2 * P <= W && 2 * P * hi <= 128) P *= 2;
  return P;
}
}  // namespace

extern "C" int tm_conv3x3_bf16_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  if (W <= 0 || Cin <= 0 || Cout <= 0 || Cin % 16 || Cout % 16) return 0;
  const int P = conv_pack(W, Cin, Cout), Pw = wgrad_pack(W, Cin, Cout);
  return conv_shape_ok(B, H, W / P, P * Cin, P * Cout) && conv_shape_ok(B, H, W / Pw, Pw * Cin, Pw * Cout) &&
         Pw * Cin <= 128 && Pw * Cout <= 128 && pow2(Cin) && pow2(Cout) ? 1 : 0;
}

extern "C" int tm_conv3x3_bf16_pack(int64_t W, int64_t Cin, int64_t Cout) { return conv_pack(W, Cin, Cout); }

namespace {
int launch_taps(const ConvArgs& a, const CUtensorMap& tmx, const CUtensorMap& tmw, int CK, cudaStream_t st);
}

extern "C" int tm_to_bf16_rows(int64_t npix, int64_t C, const float* x, int64_t ldx, void* out, int64_t Cp, void* stream) {
  TM_REQUIRE(Cp % 8 == 0 && Cp >= C, "tm_to_bf16_rows: padded width must be a multiple of 8 and >= C");
  if (npix <= 0) return 0;
  const int vec = (ldx % 4 == 0) && (reinterpret_cast<uintptr_t>(x) % 16 == 0);
  const int64_t n = npix * (Cp / 8);
  to_bf16_kernel<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(npix, (int)C, x, ldx, (__nv_bfloat16*)out, (int)Cp, vec);
  return check_launch("to_bf16");
}

// q: bf16 [9][P*Nc][P*KcP]; dgrad = 0: Nc = Cout, Kc = Cin (padded to KcP); dgrad = 1: Nc = Cin, Kc = Cout
extern "C" int tm_conv3x3_pack_bf16(int64_t Cout, int64_t Cin, const float* w, void* q, int64_t P, int64_t KcP, int dgrad,
                                    void* stream) {
  TM_REQUIRE(P >= 1 && KcP >= (dgrad ? Cout : Cin), "tm_conv3x3_pack_bf16: bad packing");
  const int64_t n = 9 * P * (dgrad ? Cin : Cout) * P * KcP;
  pack_w_kernel<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((int)Cout, (int)Cin, 3, w, (__nv_bfloat16*)q,
                                                                             (int)P, (int)KcP, dgrad);
  return check_launch("pack_w_bf16");
}

// Y[pix, 0:N] = sum_{tap,c} X[pix+tap, c] * W[tap][n][c]  (3x3, stride 1, zero padding 1)
// xb: bf16 [B][H][W][Cin] compact; wq: tm_conv3x3_pack_bf16 operand for P = tm_conv3x3_bf16_pack(W, Cin, N);
// y: fp32 rows of stride ldy.
extern "C" size_t tm_conv3x3_bf16_stats_bytes(int64_t N, int64_t P) {
  return (size_t)sm_count() * FWD_EPI_WARPS * 2 * (size_t)(N * P) * sizeof(double);
}

// stats (optional, tm_conv3x3_bf16_stats_bytes(N, P) bytes, no bias): per-column sum / sum of squares of the output,
// [sm_count * 4 slots][P * N][2] fp64 -- the batch-norm statistics pass fused into the epilogue (slot s, pixel po,
// channel c at ((s * P + po) * N + c) * 2: tm_bn_relu_forward reads it as sm_count * 4 * P partials of N channels).
extern "C" int tm_conv3x3_bf16(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t P, const void* xb,
                               const void* wq, const float* bias, float* y, int64_t ldy, int flags, void* stats, int* err,
                               void* stream) {
  TM_REQUIRE(P >= 1 && W % P == 0 && conv_shape_ok(B, H, W / P, P * Cin, P * N) && N % 16 == 0,
             "tm_conv3x3_bf16: unsupported shape (H, W powers of two; channels multiples of 16)");
  TM_REQUIRE(ldy % 4 == 0 && reinterpret_cast<uintptr_t>(y) % 16 == 0, "tm_conv3x3_bf16: output rows must be 16-byte aligned");
  TM_REQUIRE(reinterpret_cast<uintptr_t>(xb) % 16 == 0 && reinterpret_cast<uintptr_t>(wq) % 16 == 0, "tm_conv3x3_bf16: operands must be 16-byte aligned");
  const int64_t Wp = W / P, Cp = P * Cin, Np = P * N;
  const int CK = Cp >= 64 ? 64 : (int)Cp;
  ConvArgs a;
  a.g = make_geom(B, H, Wp);
  a.Cin = (int)Cp; a.N = (int)Np; a.P = (int)P; a.cpx = (int)N;
  a.a_bytes = 128u * CK * 2u;
  a.b_bytes = (uint32_t)Np * CK * 2u;
  a.stage_bytes = a.a_bytes + (uint32_t)align_up(a.b_bytes, 1024);
  int ns = (int)(FWD_SMEM_BUDGET / a.stage_bytes);
  a.stages = ns > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns;
  a.y = y; a.ldy = ldy; a.bias = bias;
  a.stats = (double*)stats;
  if (stats) {
    TM_REQUIRE(!bias && Np <= STAT_MAX_N, "tm_conv3x3_bf16: fused statistics need no bias and P * N <= 128");
    TM_CUDA(cudaMemsetAsync(stats, 0, tm_conv3x3_bf16_stats_bytes(N, P), (cudaStream_t)stream));   // slots of idle CTAs
  }
  a.ntaps = 9; a.cscale = 1; a.convt = 0;
  for (int t = 0; t < 9; ++t) { a.tdx[t] = (signed char)(t % 3 - 1); a.tdy[t] = (signed char)(t / 3 - 1); }
  a.flags = (flags & TM_EPI_RELU) | (bias ? TM_EPI_BIAS : 0);
  if (getenv("TM_CONV_DEBUG")) a.flags |= atoi(getenv("TM_CONV_DEBUG")) & 0x700;   // bottleneck bisection (rows kernel)
  a.err = err;
  CUtensorMap tmx, tmw;
  cudaStream_t st = (cudaStream_t)stream;
  static const bool rows_on = !(getenv("TM_CONV_ROWS") && atoi(getenv("TM_CONV_ROWS")) == 0);
  if (rows_on && Cp == 64 && Np <= 64 && Wp >= 128 && H % V2_ROWS == 0) {
    // whole packed weight resident in shared memory, every input row fetched once per horizontal shift
    const size_t wbytes = (size_t)9 * Np * 128;
    int ns2 = (int)((FWD_SMEM_BUDGET - wbytes) / a.a_bytes);
    a.stages = ns2 > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns2;
    TM_TRY(encode_act(&tmx, xb, Cp, Wp, H, B, 64, 128, 1, 1));
    TM_TRY(encode_2d(&tmw, wq, Cp, 9 * Np, 64, (int)Np));
    const int64_t nt = (Wp / 128) * (H / V2_ROWS) * B;
    const int grid2 = (int)(nt < sm_count() ? nt : sm_count());
    const size_t smem2 = wbytes + (size_t)a.stages * a.a_bytes + 1024;
    static bool optin2 = false;
    if (!optin2) {
      TM_CUDA(cudaFuncSetAttribute(conv3x3_tma_rows_kernel<V2_ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int)FWD_SMEM_BUDGET + 1024));
      optin2 = true;
    }
    conv3x3_tma_rows_kernel<V2_ROWS><<<grid2, FWD_THREADS, smem2, st>>>(tmx, tmw, a);
    return check_launch("conv3x3_tma_rows");
  }
  TM_TRY(encode_act(&tmx, xb, Cp, Wp, H, B, CK, a.g.TW, a.g.TH, a.g.TB));
  TM_TRY(encode_2d(&tmw, wq, Cp, 9 * Np, CK, (int)Np));
  return launch_taps(a, tmx, tmw, CK, st);
}

namespace {
int launch_taps(const ConvArgs& a, const CUtensorMap& tmx, const CUtensorMap& tmw, int CK, cudaStream_t st) {
  const size_t smem = (size_t)a.stages * a.stage_bytes + 1024;
  const int grid = (int)(a.g.ntiles < sm_count() ? a.g.ntiles : sm_count());
#define TM_LAUNCH_CONV(CK_)                                                                                   \
  do {                                                                                                        \
    static bool optin = false;                                                                                \
    if (!optin) {                                                                                             \
      TM_CUDA(cudaFuncSetAttribute(conv3x3_tma_kernel<CK_, FMT_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize,       \
                                   (int)FWD_SMEM_BUDGET + 1024));                                             \
      optin = true;                                                                                           \
    }                                                                                                         \
    conv3x3_tma_kernel<CK_, FMT_BF16><<<grid, FWD_THREADS, smem, st>>>(tmx, tmw, a);                                    \
  } while (0)
  if (CK == 64) TM_LAUNCH_CONV(64);
  else if (CK == 32) TM_LAUNCH_CONV(32);
  else TM_LAUNCH_CONV(16);
#undef TM_LAUNCH_CONV
  return check_launch("conv_tma");
}

template <typename T>
__global__ void pack_convt_kernel(int Cin, int Cout, const float* __restrict__ w, T* __restrict__ wf, T* __restrict__ wd) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)Cin * Cout * 4) return;
  const int q = (int)(i % 4), co = (int)((i / 4) % Cout), ci = (int)(i / (4 * Cout));   // w[ci][co][dy][dx], q = dy*2+dx
  const float v = w[i];
  if (wf) put(wf, ((int64_t)q * Cout + co) * Cin + ci, v);     // forward operand  [(q,co)][ci]
  if (wd) put(wd, ((int64_t)q * Cin + ci) * Cout + co, v);     // data-gradient operand, tap q: [ci][co]
}
}  // namespace

// nn.ConvTranspose2d(k=2, s=2) weight w [Cin][Cout][2][2] fp32 -> wf bf16 [4*Cout][Cin], wd bf16 [4][Cin][Cout]
extern "C" int tm_convt2x2_pack_bf16(int64_t Cin, int64_t Cout, const float* w, void* wf, void* wd, void* stream) {
  pack_convt_kernel<<<(unsigned)cdiv(Cin * Cout * 4, 256), 256, 0, (cudaStream_t)stream>>>((int)Cin, (int)Cout, w,
                                                                                              (__nv_bfloat16*)wf, (__nv_bfloat16*)wd);
  return check_launch("pack_convt_bf16");
}

namespace {
inline bool convt_shape_ok(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  return conv_shape_ok(B, H, W, Cin, 4 * Cout) && conv_shape_ok(B, H, W, Cout, Cin);
}
void fill_common(ConvArgs& a, int64_t B, int64_t H, int64_t W, int64_t K, int64_t N, int CK, float* y, int64_t ldy,
                 const float* bias, int* err) {
  a.g = make_geom(B, H, W);
  a.Cin = (int)K; a.N = (int)N; a.P = 1;
  a.a_bytes = 128u * CK * 2u;
  a.b_bytes = (uint32_t)N * CK * 2u;
  a.stage_bytes = a.a_bytes + (uint32_t)align_up(a.b_bytes, 1024);
  const int ns = (int)(FWD_SMEM_BUDGET / a.stage_bytes);
  a.stages = ns > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns;
  a.y = y; a.ldy = ldy; a.bias = bias;
  a.flags = bias ? TM_EPI_BIAS : 0;
  a.err = err;
  a.stats = nullptr;
}
}  // namespace

extern "C" int tm_convt2x2_bf16_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  return convt_shape_ok(B, H, W, Cin, Cout) ? 1 : 0;
}

// y[b, 2y+dy, 2x+dx, co] (fp32, pixel stride ldy, (B,2H,2W,*)) = bias[co] + sum_ci xb[b,y,x,ci] * w[ci][co][dy][dx]
// One tap; the accumulator row of an input pixel is its 2x2 output window (4*Cout columns), scattered by the epilogue.
extern "C" int tm_convt2x2_bf16(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const void* xb, const void* wf,
                                const float* bias, float* y, int64_t ldy, int* err, void* stream) {
  TM_REQUIRE(convt_shape_ok(B, H, W, Cin, Cout), "tm_convt2x2_bf16: unsupported shape");
  TM_REQUIRE(ldy % 4 == 0 && reinterpret_cast<uintptr_t>(y) % 16 == 0, "tm_convt2x2_bf16: output rows must be 16-byte aligned");
  const int CK = Cin >= 64 ? 64 : (int)Cin;
  ConvArgs a;
  fill_common(a, B, H, W, Cin, 4 * Cout, CK, y, ldy, bias, err);
  a.cpx = (int)Cout; a.ntaps = 1; a.cscale = 1; a.convt = 1;
  a.tdx[0] = 0; a.tdy[0] = 0;
  CUtensorMap tmx, tmw;
  TM_TRY(encode_act(&tmx, xb, Cin, W, H, B, CK, a.g.TW, a.g.TH, a.g.TB));
  TM_TRY(encode_2d(&tmw, wf, Cin, 4 * Cout, CK, (int)(4 * Cout)));
  return launch_taps(a, tmx, tmw, CK, (cudaStream_t)stream);
}

// dx[b,y,x,ci] (fp32, stride lddx) = sum_{dy,dx,co} dyb[b, 2y+dy, 2x+dx, co] * w[ci][co][dy][dx]
// Four taps; tap (dy,dx) reads every other pixel of the compact bf16 gradient [B][2H][2W][Cout] through a tensor
// map with element strides (1, 2, 2, 1).
extern "C" int tm_convt2x2_bf16_dgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const void* dyb,
                                      const void* wd, float* dx, int64_t lddx, int* err, void* stream) {
  TM_REQUIRE(convt_shape_ok(B, H, W, Cin, Cout), "tm_convt2x2_bf16_dgrad: unsupported shape");
  TM_REQUIRE(lddx % 4 == 0 && reinterpret_cast<uintptr_t>(dx) % 16 == 0, "tm_convt2x2_bf16_dgrad: output rows must be 16-byte aligned");
  const int CK = Cout >= 64 ? 64 : (int)Cout;
  ConvArgs a;
  fill_common(a, B, H, W, Cout, Cin, CK, dx, lddx, nullptr, err);
  a.cpx = (int)Cin; a.ntaps = 4; a.cscale = 2; a.convt = 0;
  for (int q = 0; q < 4; ++q) { a.tdx[q] = (signed char)(q & 1); a.tdy[q] = (signed char)(q >> 1); }
  CUtensorMap tmx, tmw;
  TM_TRY(encode_act(&tmx, dyb, Cout, 2 * W, 2 * H, B, CK, a.g.TW, a.g.TH, a.g.TB, 2));
  TM_TRY(encode_2d(&tmw, wd, Cout, 4 * Cin, CK, (int)Cin));
  return launch_taps(a, tmx, tmw, CK, (cudaStream_t)stream);
}

namespace {
// gy: CTAs per pixel split (kernel rows x tap groups)
inline int wgrad_splits(const Geom& g, int gy = 3) {
  const int want = sm_count() / gy > 0 ? sm_count() / gy : 1;
  return (int)(g.ntiles < want ? g.ntiles : want);
}
}  // namespace

extern "C" size_t tm_conv3x3_bf16_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  const int P = wgrad_pack(W, Cin, Cout);
  const Geom g = make_geom(B, H, W / P);
  return (size_t)wgrad_splits(g) * 9 * (P * Cout) * (P * Cin) * sizeof(float) + 256;
}

namespace {
// part [splits][q][ci][co] -> dw [Cin][Cout][2][2] (torch ConvTranspose2d layout), fixed order
__global__ void convt_wgrad_reduce_kernel(const float* __restrict__ part, int splits, int Cin, int Cout, float* __restrict__ dw) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)4 * Cin * Cout) return;
  const int co = (int)(i % Cout), ci = (int)((i / Cout) % Cin), q = (int)(i / ((int64_t)Cout * Cin));
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += part[(int64_t)z * 4 * Cin * Cout + i];
  dw[((int64_t)ci * Cout + co) * 4 + q] = s;
}
inline int convt_wgrad_splits(const Geom& g) { return (int)(g.ntiles < sm_count() ? g.ntiles : sm_count()); }
}  // namespace

extern "C" size_t tm_convt2x2_bf16_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  const Geom g = make_geom(B, H, W);
  return (size_t)convt_wgrad_splits(g) * 4 * Cin * Cout * sizeof(float) + 256;
}

// dw[ci][co][dy][dx] = sum_{b,y,x} xb[b,y,x,ci] * dyb[b, 2y+dy, 2x+dx, co]   (the bias gradient is a column sum of dy)
// xb: bf16 [B][H][W][Cin]; dyb: bf16 compact [B][2H][2W][Cout].  A = x (M = Cin), B = the four strided taps of dy
// fused into one MN-major operand of 4*Cout columns.
extern "C" int tm_convt2x2_bf16_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const void* xb,
                                      const void* dyb, float* dw, void* ws, size_t ws_bytes, int* err, void* stream) {
  TM_REQUIRE(convt_shape_ok(B, H, W, Cin, Cout) && Cin <= 128 && Cout <= 64 && pow2(Cin) && pow2(Cout),
             "tm_convt2x2_bf16_wgrad: unsupported shape");
  TM_REQUIRE(ws && ws_bytes >= tm_convt2x2_bf16_wgrad_ws(B, H, W, Cin, Cout), "tm_convt2x2_bf16_wgrad: workspace too small");
  WgradArgs a;
  a.g = make_geom(B, H, W);
  // kernel roles: "dy" slot = the untapped M-side operand (here x), "x" slot = the tapped N-side operand (here dy)
  a.Cin = (int)Cout; a.Cout = (int)Cin;
  a.cbx = (int)Cout; a.nbx = 1;
  a.cby = Cin > 64 ? 64 : (int)Cin; a.nby = (int)Cin / a.cby;
  a.x_bytes = 128u * (uint32_t)Cout * 2u;
  a.dy_bytes = 128u * (uint32_t)Cin * 2u;
  a.stage_bytes = (uint32_t)align_up(a.dy_bytes + 4 * a.x_bytes, 1024);
  const int ns = (int)(CONV_SMEM_BUDGET / a.stage_bytes);
  a.stages = ns > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns;
  TM_REQUIRE(a.stages >= 2, "tm_convt2x2_bf16_wgrad: tile does not fit shared memory");
  a.part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  a.err = err;
  a.cscale = 2;
  for (int q = 0; q < 4; ++q) { a.tdx[q] = (signed char)(q & 1); a.tdy[q] = (signed char)(q >> 1); }
  CUtensorMap tm_tap, tm_m;
  TM_TRY(encode_act(&tm_tap, dyb, Cout, 2 * W, 2 * H, B, a.cbx, a.g.TW, a.g.TH, a.g.TB, 2));
  TM_TRY(encode_act(&tm_m, xb, Cin, W, H, B, a.cby, a.g.TW, a.g.TH, a.g.TB));
  const int splits = convt_wgrad_splits(a.g);
  const size_t smem = (size_t)a.stages * a.stage_bytes + 1024;
  cudaStream_t st = (cudaStream_t)stream;
  static bool optin = false;
  if (!optin) {
    TM_CUDA(cudaFuncSetAttribute(conv3x3_wgrad_tma_kernel<4, FMT_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CONV_SMEM_BUDGET + 1024));
    optin = true;
  }
  conv3x3_wgrad_tma_kernel<4, FMT_BF16><<<dim3((unsigned)splits, 1), CONV_THREADS, smem, st>>>(tm_tap, tm_m, a);
  TM_TRY(check_launch("convt_wgrad_tma"));
  convt_wgrad_reduce_kernel<<<(unsigned)cdiv(4 * Cin * Cout, 256), 256, 0, st>>>(a.part, splits, (int)Cin, (int)Cout, dw);
  return check_launch("convt_wgrad_reduce");
}

// dw[co][ci][ky][kx] (ci < Cin_real) = sum_pix dY[pix, co] * X[pix + (ky-1, kx-1), ci]
// xb: bf16 [B][H][W][Cin]; dyb: bf16 [B][H][W][Cout]; both compact, channels multiples of 16.
extern "C" int tm_conv3x3_bf16_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cin_real, int64_t Cout,
                                     const void* xb, const void* dyb, float* dw, void* ws, size_t ws_bytes, int* err,
                                     void* stream) {
  TM_REQUIRE(W > 0 && Cin > 0 && Cout > 0, "tm_conv3x3_bf16_wgrad: bad sizes");
  const int P = wgrad_pack(W, Cin, Cout);
  const int64_t Wp = W / P, Cp = P * Cin, Np = P * Cout;
  TM_REQUIRE(conv_shape_ok(B, H, Wp, Cp, Np) && Cp <= 128 && Np <= 128 && pow2(Cp) && pow2(Np),
             "tm_conv3x3_bf16_wgrad: unsupported shape");
  TM_REQUIRE(ws && ws_bytes >= tm_conv3x3_bf16_wgrad_ws(B, H, W, Cin, Cout), "tm_conv3x3_bf16_wgrad: workspace too small");
  WgradArgs a;
  a.g = make_geom(B, H, Wp);
  a.Cin = (int)Cp; a.Cout = (int)Np;
  a.cbx = Cp > 64 ? 64 : (int)Cp; a.nbx = (int)Cp / a.cbx;
  a.cby = Np > 64 ? 64 : (int)Np; a.nby = (int)Np / a.cby;
  a.x_bytes = 128u * (uint32_t)Cp * 2u;
  a.dy_bytes = 128u * (uint32_t)Np * 2u;
  const int NT = Cp <= 64 ? 3 : 1;
  a.stage_bytes = (uint32_t)align_up(a.dy_bytes + NT * a.x_bytes, 1024);
  int ns = (int)(CONV_SMEM_BUDGET / a.stage_bytes);
  a.stages = ns > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns;
  TM_REQUIRE(a.stages >= 2, "tm_conv3x3_bf16_wgrad: tile does not fit shared memory");
  a.part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  a.err = err;
  CUtensorMap tmx, tmdy;
  TM_TRY(encode_act(&tmx, xb, Cp, Wp, H, B, a.cbx, a.g.TW, a.g.TH, a.g.TB));
  TM_TRY(encode_act(&tmdy, dyb, Np, Wp, H, B, a.cby, a.g.TW, a.g.TH, a.g.TB));
  const int splits = wgrad_splits(a.g);
  const size_t smem = (size_t)a.stages * a.stage_bytes + 1024;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid((unsigned)splits, 3);
  static bool optin = false;
  if (!optin) {
    TM_CUDA(cudaFuncSetAttribute(conv3x3_wgrad_tma_kernel<3, FMT_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CONV_SMEM_BUDGET + 1024));
    TM_CUDA(cudaFuncSetAttribute(conv3x3_wgrad_tma_kernel<1, FMT_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CONV_SMEM_BUDGET + 1024));
    optin = true;
  }
  if (NT == 3) conv3x3_wgrad_tma_kernel<3, FMT_BF16><<<grid, CONV_THREADS, smem, st>>>(tmx, tmdy, a);
  else conv3x3_wgrad_tma_kernel<1, FMT_BF16><<<grid, CONV_THREADS, smem, st>>>(tmx, tmdy, a);
  TM_TRY(check_launch("conv3x3_wgrad_tma"));
  const int64_t n = 9 * Cout * Cin_real;
  wgrad_reduce_kernel<3><<<(unsigned)cdiv(n * 32, 256), 256, 0, st>>>(a.part, splits, P, (int)Cout, (int)Cin, (int)Cin_real, 3, dw);
  return check_launch("wgrad_reduce");
}

// ------------------------------------------------------------------------------------------------
// tf32x3 (fp32-class) forms of the 3x3 and transposed convolutions: the kernels above with FMT_TF32X3.  The operands
// are the fp32 activations themselves, read in place through their pixel stride; the weights are packed in fp32.
// Rows of 32 fp32 channels are 128 bytes, so narrow layers pack P = 2 pixels per row (16 channels), not 4.
// ------------------------------------------------------------------------------------------------
namespace {
inline int conv_pack_f32(int64_t W, int64_t cin, int64_t cout) {
  int P = 1;
  while (P * cin < 32 && 2 * P <= W && 2 * P * cout <= 256) P *= 2;
  return P;
}
inline int wgrad_pack_f32(int64_t W, int64_t cin, int64_t cout) {
  const int64_t lo = cin < cout ? cin : cout, hi = cin < cout ? cout : cin;
  int P = 1;
  while (P * lo < 32 && 2 * P <= W && 2 * P * hi <= 128) P *= 2;
  return P;
}
// MN-major fp32 operands come in boxes of 32 channels (128 bytes; the only MN-major 32-bit layout tcgen05 takes)
inline bool wgrad_f32_ok(int64_t Cp, int64_t Np) {
  return Cp % 32 == 0 && Np % 32 == 0 && Cp <= 128 && Np <= 128 && pow2(Cp) && pow2(Np);
}

// Stage geometry of a forward / data-gradient launch (a.Cin = K, a.N set): CK fp32 channels per k-step, 32 (128-byte
// rows) unless that leaves fewer than 3 stages -- then 16.  A stage is twice a bf16 stage of the same CK (hi and lo
// planes), so the 184 KB ring holds 2-4 stages of CK = 32 (N = 128 / 64 / 32); N = 128 and the transposed
// convolution's N = 256 run at CK = 16 with 5 / 3 stages.  K splits when the tiles leave SMs idle, as
// tm_tc_conv2d_splitk_ws does: tiles x splits fills the GPU, at least two k-steps per split.  Returns the splits.
int tf_plan(ConvArgs& a, int& CK) {
  auto hi = [&](int ck) { return (uint32_t)(128 * ck * 4 + align_up((size_t)a.N * ck * 4, 1024)); };
  CK = a.Cin >= 32 ? 32 : 16;
  if (CK == 32 && FWD_SMEM_BUDGET / (2 * hi(32)) < 3) CK = 16;
  a.a_bytes = 128u * CK * 4u;
  a.b_bytes = (uint32_t)a.N * CK * 4u;
  a.hi_bytes = hi(CK);
  a.stage_bytes = 2 * a.hi_bytes;
  const int ns = (int)(FWD_SMEM_BUDGET / a.stage_bytes);
  a.stages = ns > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns;
  const int ksteps = a.ntaps * (a.Cin / CK);
  a.ksplit = 1; a.kper = ksteps; a.zstride = 0;
  int64_t want = (int64_t)sm_count() / a.g.ntiles;
  if (want > ksteps / 2) want = ksteps / 2;
  if (want >= 2) {
    a.kper = (int)cdiv(ksteps, want);
    a.ksplit = (int)cdiv(ksteps, a.kper);
  }
  return a.ksplit;
}
inline size_t tf_ws(ConvArgs a, int64_t mout) {
  int CK;
  const int splits = tf_plan(a, CK);
  return splits > 1 ? (size_t)splits * mout * a.cpx * sizeof(float) + 256 : 0;
}

// a: geometry, channels, taps and stats set.  x: fp32 map (xC channels, xW x xH, pixel stride ldx elements; step 2:
// every other pixel), wq: fp32 operand of wrows rows.  mout rows of a.cpx outputs; split launches write fp32 partials
// into ws and fold them (fixed order) into y with the bias and ReLU.
int run_tf32(ConvArgs a, const float* x, int64_t xC, int64_t xW, int64_t xH, int64_t ldx, int step, const float* wq,
             int64_t wrows, int64_t mout, const float* bias, int relu, float* y, int64_t ldy, void* ws, size_t ws_bytes,
             int* err, cudaStream_t st) {
  TM_REQUIRE(ldx % 4 == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(wq) % 16 == 0,
             "tf32x3 convolution: operand rows must be 16-byte aligned");
  TM_REQUIRE(ldy % 4 == 0 && reinterpret_cast<uintptr_t>(y) % 16 == 0, "tf32x3 convolution: output rows must be 16-byte aligned");
  int CK;
  const int splits = tf_plan(a, CK);
  a.err = err;
  float* part = nullptr;
  if (splits > 1) {
    TM_REQUIRE(!a.stats, "tf32x3 convolution: fused statistics need an unsplit launch");
    TM_REQUIRE(ws && ws_bytes >= (size_t)splits * mout * a.cpx * sizeof(float) + 256, "tf32x3 convolution: workspace too small");
    part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    a.y = part; a.ldy = a.cpx; a.zstride = mout * a.cpx;
    a.bias = nullptr; a.flags = 0;
  } else {
    a.y = y; a.ldy = ldy; a.bias = bias;
    a.flags = (relu ? TM_EPI_RELU : 0) | (bias ? TM_EPI_BIAS : 0);
  }
  if (a.stats) TM_CUDA(cudaMemsetAsync(a.stats, 0, tm_conv3x3_bf16_stats_bytes(a.cpx, a.P), st));   // slots of idle CTAs
  CUtensorMap tmx, tmw;
  TM_TRY(encode_act(&tmx, x, xC, xW, xH, a.g.B, CK, a.g.TW, a.g.TH, a.g.TB, step, 4, ldx));
  TM_TRY(encode_2d(&tmw, wq, a.Cin, wrows, CK, a.N, 4));
  const int64_t units = a.g.ntiles * a.ksplit;
  const int grid = (int)(units < sm_count() ? units : sm_count());
  const size_t smem = (size_t)a.stages * a.stage_bytes + 1024;
  constexpr int threads = FWD_THREADS + SPLIT_WARPS * 32;
#define TM_LAUNCH_TF(CK_)                                                                                     \
  do {                                                                                                        \
    static bool optin = false;                                                                                \
    if (!optin) {                                                                                             \
      TM_CUDA(cudaFuncSetAttribute(conv3x3_tma_kernel<CK_, FMT_TF32X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                   (int)FWD_SMEM_BUDGET + 1024));                                             \
      optin = true;                                                                                           \
    }                                                                                                         \
    conv3x3_tma_kernel<CK_, FMT_TF32X3><<<grid, threads, smem, st>>>(tmx, tmw, a);                            \
  } while (0)
  if (CK == 32) TM_LAUNCH_TF(32);
  else TM_LAUNCH_TF(16);
#undef TM_LAUNCH_TF
  TM_TRY(check_launch("conv_tma_tf32"));
  if (splits > 1) return tc::conv_split_fold(part, mout, a.cpx, splits, bias, relu, y, ldy, st);
  return 0;
}

ConvArgs conv3x3_args(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t P) {
  ConvArgs a;
  a.g = make_geom(B, H, W / P);
  a.Cin = (int)(P * Cin); a.N = (int)(P * N); a.P = (int)P; a.cpx = (int)N;
  a.ntaps = 9; a.cscale = 1; a.convt = 0;
  for (int t = 0; t < 9; ++t) { a.tdx[t] = (signed char)(t % 3 - 1); a.tdy[t] = (signed char)(t / 3 - 1); }
  a.stats = nullptr;
  return a;
}
ConvArgs convt_args(int64_t B, int64_t H, int64_t W, int64_t K, int64_t N, int64_t cpx, int ntaps) {
  ConvArgs a;
  a.g = make_geom(B, H, W);
  a.Cin = (int)K; a.N = (int)N; a.P = 1; a.cpx = (int)cpx;
  a.ntaps = ntaps; a.cscale = ntaps == 4 ? 2 : 1; a.convt = ntaps == 1;
  for (int q = 0; q < 4; ++q) { a.tdx[q] = (signed char)(ntaps == 4 ? q & 1 : 0); a.tdy[q] = (signed char)(ntaps == 4 ? q >> 1 : 0); }
  a.stats = nullptr;
  return a;
}

// weight-gradient stage geometry: tapped tiles per stage (3: a kernel row fused, when 3 * Cin <= 192; else 1) and
// pixels per stage (128 / 64 / 32), the first that leaves at least 3 stages -- a tf32x3 stage is twice a bf16 stage
// of the same pixels, and 128 pixels of a 128-channel layer would not fit twice
void tf_wgrad_plan(WgradArgs& a, int64_t B, int64_t H, int64_t Wp, int nt_max, int& NT) {
  const int nts[2] = {nt_max, nt_max == 3 ? 1 : nt_max};    // the transposed conv (4) has no one-tap form
  for (int min_st = 3; min_st >= 2; --min_st)
    for (int i = 0; i < 2; ++i) {
      if (i == 1 && nts[1] == nts[0]) break;
      for (int tp = 128; tp >= 32; tp >>= 1) {
        const uint32_t hi = (uint32_t)align_up((size_t)tp * a.Cout * 4 + (size_t)nts[i] * tp * a.Cin * 4, 1024);
        if (CONV_SMEM_BUDGET / (2 * hi) >= (uint32_t)min_st) {
          NT = nts[i];
          a.tp = tp;
          a.g = make_geom(B, H, Wp, tp);
          a.cbx = 32; a.nbx = a.Cin / 32;
          a.cby = 32; a.nby = a.Cout / 32;
          a.x_bytes = (uint32_t)tp * a.Cin * 4;
          a.dy_bytes = (uint32_t)tp * a.Cout * 4;
          a.hi_bytes = hi;
          a.stage_bytes = 2 * hi;
          const int ns = (int)(CONV_SMEM_BUDGET / a.stage_bytes);
          a.stages = ns > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns;
          return;
        }
      }
    }
  NT = 0;   // no fit (not reached for Cin, Cout <= 128)
}

template <int NT>
int launch_wgrad_tf32(const WgradArgs& a, const CUtensorMap& tmx, const CUtensorMap& tmdy, dim3 grid, cudaStream_t st) {
  static bool optin = false;
  if (!optin) {
    TM_CUDA(cudaFuncSetAttribute(conv3x3_wgrad_tma_kernel<NT, FMT_TF32X3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)CONV_SMEM_BUDGET + 1024));
    optin = true;
  }
  conv3x3_wgrad_tma_kernel<NT, FMT_TF32X3><<<grid, CONV_THREADS, (size_t)a.stages * a.stage_bytes + 1024, st>>>(tmx, tmdy, a);
  return check_launch("wgrad_tma_tf32");
}
}  // namespace

extern "C" int tm_conv3x3_tf32_pack(int64_t W, int64_t Cin, int64_t Cout) { return conv_pack_f32(W, Cin, Cout); }

extern "C" int tm_conv3x3_tf32_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  if (W <= 0 || Cin <= 0 || Cout <= 0 || Cin % 16 || Cout % 16) return 0;
  const int P = conv_pack_f32(W, Cin, Cout), Pw = wgrad_pack_f32(W, Cin, Cout);
  return conv_shape_ok(B, H, W / P, P * Cin, P * Cout) && conv_shape_ok(B, H, W / Pw, Pw * Cin, Pw * Cout) &&
                 wgrad_f32_ok(Pw * Cin, Pw * Cout)
             ? 1
             : 0;
}

extern "C" int tm_conv3x3_pack_f32(int64_t Cout, int64_t Cin, const float* w, float* q, int64_t P, int64_t KcP, int dgrad,
                                   void* stream) {
  TM_REQUIRE(P >= 1 && KcP >= (dgrad ? Cout : Cin), "tm_conv3x3_pack_f32: bad packing");
  const int64_t n = 9 * P * (dgrad ? Cin : Cout) * P * KcP;
  pack_w_kernel<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((int)Cout, (int)Cin, 3, w, q, (int)P, (int)KcP, dgrad);
  return check_launch("pack_w_f32");
}

extern "C" size_t tm_conv3x3_tf32_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t P) {
  if (P < 1 || W % P || !conv_shape_ok(B, H, W / P, P * Cin, P * N)) return 0;
  return tf_ws(conv3x3_args(B, H, W, Cin, N, P), B * H * W);
}

extern "C" int tm_conv3x3_tf32(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t P, const float* x, int64_t ldx,
                               const float* wq, const float* bias, float* y, int64_t ldy, int flags, void* stats, void* ws,
                               size_t ws_bytes, int* err, void* stream) {
  TM_REQUIRE(P >= 1 && W % P == 0 && conv_shape_ok(B, H, W / P, P * Cin, P * N),
             "tm_conv3x3_tf32: unsupported shape (H, W powers of two; channels multiples of 16)");
  TM_REQUIRE(P == 1 || ldx == Cin, "tm_conv3x3_tf32: packed rows (P > 1) need compact input rows (ldx == Cin)");
  ConvArgs a = conv3x3_args(B, H, W, Cin, N, P);
  if (stats) {
    TM_REQUIRE(!bias && a.N <= STAT_MAX_N, "tm_conv3x3_tf32: fused statistics need no bias and P * N <= 128");
    a.stats = (double*)stats;
  }
  return run_tf32(a, x, P * Cin, W / P, H, P * ldx, 1, wq, 9 * P * N, B * H * W, bias, flags & TM_EPI_RELU, y, ldy, ws,
                  ws_bytes, err, (cudaStream_t)stream);
}

extern "C" size_t tm_conv3x3_tf32_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  const int P = wgrad_pack_f32(W, Cin, Cout);
  if (!wgrad_f32_ok(P * Cin, P * Cout)) return 0;
  WgradArgs a;
  a.Cin = (int)(P * Cin); a.Cout = (int)(P * Cout);
  int NT;
  tf_wgrad_plan(a, B, H, W / P, a.Cin <= 64 ? 3 : 1, NT);
  return (size_t)wgrad_splits(a.g) * 9 * a.Cout * a.Cin * sizeof(float) + 256;
}

// dw[co][ci][ky][kx] (ci < Cin_real) = sum_pix dy[pix, co] * x[pix + (ky-1, kx-1), ci]; x, dy fp32 rows of stride ldx / lddy
extern "C" int tm_conv3x3_tf32_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cin_real, int64_t Cout,
                                     const float* x, int64_t ldx, const float* dy, int64_t lddy, float* dw, void* ws,
                                     size_t ws_bytes, int* err, void* stream) {
  TM_REQUIRE(tm_conv3x3_tf32_supported(B, H, W, Cin, Cout), "tm_conv3x3_tf32_wgrad: unsupported shape");
  const int P = wgrad_pack_f32(W, Cin, Cout);
  TM_REQUIRE(P == 1 || (ldx == Cin && lddy == Cout), "tm_conv3x3_tf32_wgrad: packed rows (P > 1) need compact rows");
  TM_REQUIRE(ldx % 4 == 0 && lddy % 4 == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(dy) % 16 == 0,
             "tm_conv3x3_tf32_wgrad: operand rows must be 16-byte aligned");
  TM_REQUIRE(ws && ws_bytes >= tm_conv3x3_tf32_wgrad_ws(B, H, W, Cin, Cout), "tm_conv3x3_tf32_wgrad: workspace too small");
  const int64_t Wp = W / P;
  WgradArgs a;
  a.Cin = (int)(P * Cin); a.Cout = (int)(P * Cout);
  int NT;
  tf_wgrad_plan(a, B, H, Wp, a.Cin <= 64 ? 3 : 1, NT);
  TM_REQUIRE(NT > 0, "tm_conv3x3_tf32_wgrad: tile does not fit shared memory");
  a.part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  a.err = err;
  CUtensorMap tmx, tmdy;
  TM_TRY(encode_act(&tmx, x, a.Cin, Wp, H, B, 32, a.g.TW, a.g.TH, a.g.TB, 1, 4, P * ldx, true));
  TM_TRY(encode_act(&tmdy, dy, a.Cout, Wp, H, B, 32, a.g.TW, a.g.TH, a.g.TB, 1, 4, P * lddy, true));
  const int splits = wgrad_splits(a.g);
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid((unsigned)splits, 3);
  TM_TRY(NT == 3 ? launch_wgrad_tf32<3>(a, tmx, tmdy, grid, st) : launch_wgrad_tf32<1>(a, tmx, tmdy, grid, st));
  const int64_t n = 9 * Cout * Cin_real;
  wgrad_reduce_kernel<3><<<(unsigned)cdiv(n * 32, 256), 256, 0, st>>>(a.part, splits, P, (int)Cout, (int)Cin, (int)Cin_real, 3, dw);
  return check_launch("wgrad_reduce");
}

extern "C" int tm_convt2x2_tf32_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  return convt_shape_ok(B, H, W, Cin, Cout) ? 1 : 0;
}
extern "C" int tm_convt2x2_tf32_wgrad_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  return convt_shape_ok(B, H, W, Cin, Cout) && Cin % 32 == 0 && Cout % 32 == 0 && Cin <= 128 && Cout <= 64 && pow2(Cin) &&
                 pow2(Cout)
             ? 1
             : 0;
}

// w [Cin][Cout][2][2] fp32 -> wf fp32 [4*Cout][Cin], wd fp32 [4][Cin][Cout] (either may be NULL)
extern "C" int tm_convt2x2_pack_f32(int64_t Cin, int64_t Cout, const float* w, float* wf, float* wd, void* stream) {
  pack_convt_kernel<<<(unsigned)cdiv(Cin * Cout * 4, 256), 256, 0, (cudaStream_t)stream>>>((int)Cin, (int)Cout, w, wf, wd);
  return check_launch("pack_convt_f32");
}

namespace {
void convt_tf_wgrad_plan(WgradArgs& a, int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  // kernel roles: "dy" slot = the untapped M-side operand (x), "x" slot = the four tapped N-side tiles (dy)
  a.Cin = (int)Cout; a.Cout = (int)Cin;
  int NT;
  tf_wgrad_plan(a, B, H, W, 4, NT);
}
}  // namespace

// workspace of tm_convt2x2_tf32, _dgrad and _wgrad (the largest of the three)
extern "C" size_t tm_convt2x2_tf32_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout) {
  if (!convt_shape_ok(B, H, W, Cin, Cout)) return 0;
  size_t n = tf_ws(convt_args(B, H, W, Cin, 4 * Cout, Cout, 1), 4 * B * H * W);
  const size_t d = tf_ws(convt_args(B, H, W, Cout, Cin, Cin, 4), B * H * W);
  if (d > n) n = d;
  if (tm_convt2x2_tf32_wgrad_supported(B, H, W, Cin, Cout)) {
    WgradArgs a;
    convt_tf_wgrad_plan(a, B, H, W, Cin, Cout);
    const size_t w = (size_t)convt_wgrad_splits(a.g) * 4 * Cin * Cout * sizeof(float) + 256;
    if (w > n) n = w;
  }
  return n;
}

// y[b, 2y+dy, 2x+dx, co] (row stride ldy) = bias[co] + sum_ci x[b,y,x,ci] * w[ci][co][dy][dx]; x fp32 rows of stride ldx
extern "C" int tm_convt2x2_tf32(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* x, int64_t ldx,
                                const float* wf, const float* bias, float* y, int64_t ldy, void* ws, size_t ws_bytes, int* err,
                                void* stream) {
  TM_REQUIRE(convt_shape_ok(B, H, W, Cin, Cout), "tm_convt2x2_tf32: unsupported shape");
  return run_tf32(convt_args(B, H, W, Cin, 4 * Cout, Cout, 1), x, Cin, W, H, ldx, 1, wf, 4 * Cout, 4 * B * H * W, bias, 0,
                  y, ldy, ws, ws_bytes, err, (cudaStream_t)stream);
}

// dx[b,y,x,ci] (row stride lddx) = sum_{dy,dx,co} dy[b, 2y+dy, 2x+dx, co] * w[ci][co][dy][dx]; dy fp32 rows of stride lddy
extern "C" int tm_convt2x2_tf32_dgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* dy, int64_t lddy,
                                      const float* wd, float* dx, int64_t lddx, void* ws, size_t ws_bytes, int* err, void* stream) {
  TM_REQUIRE(convt_shape_ok(B, H, W, Cin, Cout), "tm_convt2x2_tf32_dgrad: unsupported shape");
  return run_tf32(convt_args(B, H, W, Cout, Cin, Cin, 4), dy, Cout, 2 * W, 2 * H, lddy, 2, wd, 4 * Cin, B * H * W, nullptr, 0,
                  dx, lddx, ws, ws_bytes, err, (cudaStream_t)stream);
}

// dw[ci][co][dy][dx] = sum_{b,y,x} x[b,y,x,ci] * dy[b, 2y+dy, 2x+dx, co]; x, dy fp32 rows of stride ldx / lddy
extern "C" int tm_convt2x2_tf32_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* x, int64_t ldx,
                                      const float* dy, int64_t lddy, float* dw, void* ws, size_t ws_bytes, int* err,
                                      void* stream) {
  TM_REQUIRE(tm_convt2x2_tf32_wgrad_supported(B, H, W, Cin, Cout), "tm_convt2x2_tf32_wgrad: unsupported shape");
  TM_REQUIRE(ldx % 4 == 0 && lddy % 4 == 0 && reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(dy) % 16 == 0,
             "tm_convt2x2_tf32_wgrad: operand rows must be 16-byte aligned");
  TM_REQUIRE(ws && ws_bytes >= tm_convt2x2_tf32_ws(B, H, W, Cin, Cout), "tm_convt2x2_tf32_wgrad: workspace too small");
  WgradArgs a;
  convt_tf_wgrad_plan(a, B, H, W, Cin, Cout);
  a.part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  a.err = err;
  a.cscale = 2;
  for (int q = 0; q < 4; ++q) { a.tdx[q] = (signed char)(q & 1); a.tdy[q] = (signed char)(q >> 1); }
  CUtensorMap tm_tap, tm_m;
  TM_TRY(encode_act(&tm_tap, dy, Cout, 2 * W, 2 * H, B, 32, a.g.TW, a.g.TH, a.g.TB, 2, 4, lddy, true));
  TM_TRY(encode_act(&tm_m, x, Cin, W, H, B, 32, a.g.TW, a.g.TH, a.g.TB, 1, 4, ldx, true));
  const int splits = convt_wgrad_splits(a.g);
  cudaStream_t st = (cudaStream_t)stream;
  TM_TRY(launch_wgrad_tf32<4>(a, tm_tap, tm_m, dim3((unsigned)splits, 1), st));
  convt_wgrad_reduce_kernel<<<(unsigned)cdiv(4 * Cin * Cout, 256), 256, 0, st>>>(a.part, splits, (int)Cin, (int)Cout, dw);
  return check_launch("convt_wgrad_reduce");
}

// ------------------------------------------------------------------------------------------------
// k x k convolutions (odd k <= 9, stride 1, zero padding k/2) on the same kernels: LayoutNet's 7x7 / 9x9 layers
// (src/model.py:227-243).  Operand rows are single pixels (P = 1); the weights stream through the ring with the
// activation boxes (a whole 7x7 / 9x9 weight does not fit shared memory next to the ring).
// ------------------------------------------------------------------------------------------------
namespace {
inline bool kxk_ok(int64_t k) { return k >= 3 && k <= 9 && (k & 1); }
// weight gradient: a kernel row's k taps in groups of tg, so that a group's accumulators fit one MMA (tg * Cin <= 256)
inline void kxk_groups(int64_t Cin, int64_t k, int& tg, int& groups) {
  tg = (int)(256 / Cin < k ? 256 / Cin : k);
  groups = (int)cdiv(k, tg);
  tg = (int)cdiv(k, groups);
}
}  // namespace

extern "C" int tm_convkxk_bf16_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k) {
  return kxk_ok(k) && conv_shape_ok(B, H, W, Cin, Cout) && conv_shape_ok(B, H, W, Cout, Cin) && pow2(Cin) && Cin <= 64 &&
                 pow2(Cout) && Cout <= 128
             ? 1
             : 0;
}

// q: bf16 [k*k][Nc][KcP]; dgrad = 0: Nc = Cout, Kc = Cin (padded to KcP); dgrad = 1: Nc = Cin, Kc = Cout, taps reversed
extern "C" int tm_convkxk_pack_bf16(int64_t Cout, int64_t Cin, int64_t k, const float* w, void* q, int64_t KcP, int dgrad,
                                    void* stream) {
  TM_REQUIRE(kxk_ok(k) && KcP >= (dgrad ? Cout : Cin), "tm_convkxk_pack_bf16: bad kernel size or packing");
  const int64_t n = k * k * (dgrad ? Cin : Cout) * KcP;
  pack_w_kernel<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>((int)Cout, (int)Cin, (int)k, w,
                                                                             (__nv_bfloat16*)q, 1, (int)KcP, dgrad);
  return check_launch("pack_w_bf16");
}

// y[pix, 0:N] (fp32, row stride ldy) = act(bias + sum_{tap,c} xb[pix + tap, c] * wq[tap][n][c]); flags: TM_EPI_RELU.
// The data gradient is the same call on bf16(dy) with the dgrad operand (no bias).
extern "C" int tm_convkxk_bf16(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t k, const void* xb,
                               const void* wq, const float* bias, float* y, int64_t ldy, int flags, int* err, void* stream) {
  TM_REQUIRE(kxk_ok(k) && conv_shape_ok(B, H, W, Cin, N),
             "tm_convkxk_bf16: unsupported shape (odd k <= 9; H, W powers of two; channels multiples of 16)");
  TM_REQUIRE(ldy % 4 == 0 && reinterpret_cast<uintptr_t>(y) % 16 == 0, "tm_convkxk_bf16: output rows must be 16-byte aligned");
  TM_REQUIRE(reinterpret_cast<uintptr_t>(xb) % 16 == 0 && reinterpret_cast<uintptr_t>(wq) % 16 == 0,
             "tm_convkxk_bf16: operands must be 16-byte aligned");
  const int CK = Cin >= 64 ? 64 : (int)Cin;
  ConvArgs a;
  fill_common(a, B, H, W, Cin, N, CK, y, ldy, bias, err);
  a.flags = (flags & TM_EPI_RELU) | (bias ? TM_EPI_BIAS : 0);
  a.cpx = (int)N; a.ntaps = (int)(k * k); a.cscale = 1; a.convt = 0;
  for (int t = 0; t < a.ntaps; ++t) { a.tdx[t] = (signed char)(t % k - k / 2); a.tdy[t] = (signed char)(t / k - k / 2); }
  CUtensorMap tmx, tmw;
  TM_TRY(encode_act(&tmx, xb, Cin, W, H, B, CK, a.g.TW, a.g.TH, a.g.TB));
  TM_TRY(encode_2d(&tmw, wq, Cin, k * k * N, CK, (int)N));
  return launch_taps(a, tmx, tmw, CK, (cudaStream_t)stream);
}

extern "C" size_t tm_convkxk_bf16_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k) {
  if (!kxk_ok(k) || Cin <= 0 || Cin > 256) return 0;
  int tg, groups;
  kxk_groups(Cin, k, tg, groups);
  return (size_t)wgrad_splits(make_geom(B, H, W), (int)k * groups) * k * k * Cout * Cin * sizeof(float) + 256;
}

// dw[co][ci][ky][kx] (torch layout) = sum_pix dyb[pix, co] * xb[pix + (ky - k/2, kx - k/2), ci]
// Grid (pixel splits, k kernel rows x tap groups); the partials are folded in a fixed order (deterministic).
extern "C" int tm_convkxk_bf16_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k, const void* xb,
                                     const void* dyb, float* dw, void* ws, size_t ws_bytes, int* err, void* stream) {
  TM_REQUIRE(tm_convkxk_bf16_supported(B, H, W, Cin, Cout, k), "tm_convkxk_bf16_wgrad: unsupported shape");
  TM_REQUIRE(ws && ws_bytes >= tm_convkxk_bf16_wgrad_ws(B, H, W, Cin, Cout, k), "tm_convkxk_bf16_wgrad: workspace too small");
  WgradArgs a;
  a.g = make_geom(B, H, W);
  a.Cin = (int)Cin; a.Cout = (int)Cout;
  a.cbx = (int)Cin; a.nbx = 1;
  a.cby = Cout > 64 ? 64 : (int)Cout; a.nby = (int)Cout / a.cby;
  a.x_bytes = 128u * (uint32_t)Cin * 2u;
  a.dy_bytes = 128u * (uint32_t)Cout * 2u;
  a.k = (int)k;
  kxk_groups(Cin, k, a.tg, a.groups);
  a.stage_bytes = (uint32_t)align_up(a.dy_bytes + a.tg * a.x_bytes, 1024);
  const int ns = (int)(CONV_SMEM_BUDGET / a.stage_bytes);
  a.stages = ns > CONV_MAX_STAGES ? CONV_MAX_STAGES : ns;
  TM_REQUIRE(a.stages >= 2, "tm_convkxk_bf16_wgrad: tile does not fit shared memory");
  a.part = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  a.err = err;
  a.cscale = 1;
  CUtensorMap tmx, tmdy;
  TM_TRY(encode_act(&tmx, xb, Cin, W, H, B, a.cbx, a.g.TW, a.g.TH, a.g.TB));
  TM_TRY(encode_act(&tmdy, dyb, Cout, W, H, B, a.cby, a.g.TW, a.g.TH, a.g.TB));
  const int gy = (int)k * a.groups;
  const int splits = wgrad_splits(a.g, gy);
  const size_t smem = (size_t)a.stages * a.stage_bytes + 1024;
  cudaStream_t st = (cudaStream_t)stream;
  static bool optin = false;
  if (!optin) {
    TM_CUDA(cudaFuncSetAttribute(conv3x3_wgrad_tma_kernel<0, FMT_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CONV_SMEM_BUDGET + 1024));
    optin = true;
  }
  conv3x3_wgrad_tma_kernel<0, FMT_BF16><<<dim3((unsigned)splits, (unsigned)gy), CONV_THREADS, smem, st>>>(tmx, tmdy, a);
  TM_TRY(check_launch("convkxk_wgrad_tma"));
  const int64_t n = k * k * Cout * Cin;
  wgrad_reduce_kernel<0><<<(unsigned)cdiv(n * 32, 256), 256, 0, st>>>(a.part, splits, 1, (int)Cout, (int)Cin, (int)Cin, (int)k, dw);
  return check_launch("wgrad_reduce");
}
