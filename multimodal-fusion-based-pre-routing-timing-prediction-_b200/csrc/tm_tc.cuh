// tcgen05 / TMEM GEMM core (sm_100a): C[M,N] = epi( A[M,K] . B[N,K]^T ), fp32 in / fp32 out.
//
// Operands are fp32 in HBM.  They are staged into shared memory by the CTA's threads, converted
// on the fly to bf16 in the canonical K-major no-swizzle UMMA layout (8-row x 16-byte core
// matrices), and multiplied by tcgen05.mma.kind::f16 with the fp32 accumulator in tensor memory:
//   SPLIT == 1 : plain bf16 operands                          (rtol 2e-2 class, conv bf16 path)
//   SPLIT == 3 : x = hi + mid (two bf16 terms); hi*hi + hi*mid + mid*hi -- ~16-17 bit products
//   SPLIT == 6 : x = hi + mid + lo (three bf16 terms = 24 bits); the six products down to 2^-16
//                relative size are accumulated in fp32: fp32-class accuracy for the rtol 1e-3 path
// Staging through threads (instead of TMA) keeps row gathers, transposed operands (weight
// gradients) and im2col (convolutions) one template parameter away.
//
// Persistent, warp-specialised CTA (one per SM), tiles of BM = 128 rows x BN in {32,64,128,256}
// columns, k-blocks of BK = 32:
//   warps 5..12  producers: cp.async of raw fp32 k-blocks ND ahead (across tile boundaries) into a
//                raw ring; once landed: raw -> registers -> bf16 split -> ring of NS stages in the
//                UMMA layout; arrive on full[stage].  K-contiguous operands are copied and
//                converted by the SAME thread (no barrier, warps drift apart and overlap their
//                copy / convert phases); transposed operands are copied cooperatively.
//   warp  4      one elected thread issues the tcgen05.mma's of a stage, tcgen05.commit releases
//                the stage (empty[stage]) and, after a tile's last k-block, publishes the
//                accumulator (acc_full[buf]); the accumulator is double-buffered in TMEM
//   warps 0..3   epilogue: tcgen05.ld of the finished accumulator (lane = tile row), transpose
//                through shared memory, fused bias / ReLU / mask / accumulate, 128-bit stores,
//                then acc_empty[buf] -- overlapping the next tile's main loop.
#pragma once
#include <cuda_bf16.h>
#include <stdlib.h>

#include "tm_gemm.cuh"
#include "tm_sm100.cuh"
#include "tm_split.cuh"

// Bottleneck-bisection switches (TM_TC_DEBUG bits) and the clock64 timeline (TM_TC_TRACE) are compiled
// in only with -DTM_TC_INSTRUMENT=1 (make INSTRUMENT=1); production kernels carry none of it.
#ifndef TM_TC_INSTRUMENT
#define TM_TC_INSTRUMENT 0
#endif
#define TM_DBGBITS (TM_TC_INSTRUMENT ? tm.dbg : 0)
#define TM_TRACEPTR (TM_TC_INSTRUMENT ? tm.trace : (long long*)nullptr)

namespace tmk {
namespace tc {

using namespace sm100;

constexpr int BM = 128;
constexpr int BK = 32;
constexpr int EPI_WARPS = 4;        // warps 0..3: TMEM lane group = warp index
constexpr int MMA_WARP = 4;
constexpr int PROD_WARP0 = 5;
constexpr int PROD_WARPS = 8;
constexpr int PROD_THREADS = PROD_WARPS * 32;
constexpr int THREADS = (EPI_WARPS + 1 + PROD_WARPS) * 32;   // 416

// cp.async (LDGSTS): global -> shared without a register round trip; bytes past `nbytes` are
// zero-filled, so out-of-matrix elements need no branch in the consumer
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int nbytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src, int nbytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(nbytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---------------------------------------------------------------------------------------------
// operand loaders.  Operands are fp32 in HBM; a k-block of a tile is first copied RAW into shared
// memory by cp.async in 16-byte chunks (4 floats), several k-blocks ahead of its use.
//   kTransposed == false: k is contiguous in HBM.  chunk = 4 consecutive k of one row.
//        St begin(row)            resolves what depends on the row once per tile
//        copy4(dst, st, k)        operand(row, k..k+3) -> 16 bytes at dst (zero outside the matrix)
//   kTransposed == true: the row index is contiguous in HBM.  chunk = 4 consecutive rows, one k.
//        St begin(row4)           (row4 % 4 == 0)
//        copy4(dst, st, k)        operand(row4..row4+3, k) -> 16 bytes at dst
// ---------------------------------------------------------------------------------------------
struct RowLoader {      // element(row, k) = A[rows ? rows[row] : row][k]   (k contiguous)
  static constexpr bool kTransposed = false;
  const float* A;
  int64_t ld;
  const int32_t* rows;
  int64_t nrows, K;
  int vec;              // != 0: ld % 4 == 0 and 16-byte aligned base
  struct St { const float* p; };
  __device__ __forceinline__ St begin(int64_t row) const {
    St s;
    s.p = nullptr;
    if (row < nrows) s.p = A + (rows ? (int64_t)rows[row] : row) * ld;
    return s;
  }
  __device__ __forceinline__ void copy4(uint32_t dst, const St& s, int64_t k) const {
    const int64_t rem = s.p ? K - k : 0;             // valid elements from k on
    const float* src = (rem > 0) ? s.p + k : A;
    if (vec) {
      cp_async16(dst, src, rem >= 4 ? 16 : (rem > 0 ? (int)rem * 4 : 0));
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) cp_async4(dst + 4 * i, rem > i ? src + i : A, rem > i ? 4 : 0);
    }
  }
};

struct ColLoader {      // element(row, k) = A[krows ? krows[k] : k][row]   (row contiguous)
  static constexpr bool kTransposed = true;
  const float* A;
  int64_t ld;
  const int32_t* krows;
  int64_t nrows, K;
  int vec;              // != 0: ld % 4 == 0 and 16-byte aligned base
  struct St { int64_t row4; int nr; };
  __device__ __forceinline__ St begin(int64_t row4) const {
    St s;
    s.row4 = row4;
    const int64_t nr = nrows - row4;
    s.nr = nr >= 4 ? 4 : (nr > 0 ? (int)nr : 0);
    return s;
  }
  __device__ __forceinline__ void copy4(uint32_t dst, const St& s, int64_t k) const {
    const int nr = (k < K) ? s.nr : 0;
    const float* src = nr ? A + (krows ? (int64_t)krows[k] : k) * ld + s.row4 : A;
    if (vec) {
      cp_async16(dst, src, nr * 4);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) cp_async4(dst + 4 * i, nr > i ? src + i : A, nr > i ? 4 : 0);
    }
  }
};

// ---------------------------------------------------------------------------------------------
// GENERATED operands: the hidden layer of an MLP whose input has 1 or 2 columns
// (fc_net_self: Linear(2,256) -> ReLU -> Linear(256,128), model.py:50) costs 2 FMAs per element to
// recompute, so it is never stored: the loaders below synthesise  hid(r, j) = relu(w1[j,:] . x[r,:] + b1[j])
// straight into the shared-memory stage (plain st.shared instead of cp.async), in the forward GEMM
// (K-major A operand) and in the weight-gradient GEMM (MN-major B operand); the fused first-layer
// backward regenerates the ReLU mask the same way.  One expression everywhere: bit-identical values.
// ---------------------------------------------------------------------------------------------
struct Hidden2 {
  const float* X;           // layer inputs [*, ldx]
  int64_t ldx;
  const int32_t* x_rows;    // optional gather
  const float* W1;          // [hid][kx] row-major (nn.Linear weight)
  const float* b1;          // [hid]
  int kx;                   // 1 or 2
  __device__ __forceinline__ float2 x_of(int64_t r) const {
    const float* p = X + (x_rows ? (int64_t)x_rows[r] : r) * ldx;
    return make_float2(p[0], kx > 1 ? p[1] : 0.f);
  }
  __device__ __forceinline__ float pre(float2 x, int64_t j) const {     // pre-activation of hidden unit j
    const float w0 = __ldg(W1 + j * kx), w1 = kx > 1 ? __ldg(W1 + j * kx + 1) : 0.f;
    return fmaf(w0, x.x, fmaf(w1, x.y, __ldg(b1 + j)));
  }
  __device__ __forceinline__ float act(float2 x, int64_t j) const { return fmaxf(pre(x, j), 0.f); }
};
__device__ __forceinline__ void st_shared4(uint32_t dst, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(dst), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

struct GenRowLoader {   // element(row, k) = hid(row, k)          (k = hidden unit, contiguous in the stage)
  static constexpr bool kTransposed = false;
  Hidden2 h;
  int64_t nrows, K;
  struct St { float2 x; bool ok; };
  __device__ __forceinline__ St begin(int64_t row) const {
    St s;
    s.ok = row < nrows;
    s.x = s.ok ? h.x_of(row) : make_float2(0.f, 0.f);
    return s;
  }
  __device__ __forceinline__ void copy4(uint32_t dst, const St& s, int64_t k) const {
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = (s.ok && k + i < K) ? h.act(s.x, k + i) : 0.f;
    st_shared4(dst, v[0], v[1], v[2], v[3]);
  }
};

struct GenColLoader {   // element(row, k) = hid(k, row)          (row = hidden unit: 4 consecutive units per chunk)
  static constexpr bool kTransposed = true;
  Hidden2 h;
  int64_t nrows, K;     // nrows = hidden width, K = number of samples
  struct St { int64_t row4; int nr; };
  __device__ __forceinline__ St begin(int64_t row4) const {
    St s;
    s.row4 = row4;
    const int64_t nr = nrows - row4;
    s.nr = nr >= 4 ? 4 : (nr > 0 ? (int)nr : 0);
    return s;
  }
  __device__ __forceinline__ void copy4(uint32_t dst, const St& s, int64_t k) const {
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (k < K && s.nr > 0) {
      const float2 x = h.x_of(k);
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < s.nr) v[i] = h.act(x, s.row4 + i);
    }
    st_shared4(dst, v[0], v[1], v[2], v[3]);
  }
};

// im2col view of an NHWC tensor: row = output pixel, k = tap * Cin + ci (stride 1, pad ks/2)
struct Im2colLoader8 {
  static constexpr bool kTransposed = false;
  const float* X;
  int64_t ldx;
  int H, W, Cin, ks, pad;
  int64_t nrows, K;
  int vec;              // != 0: Cin % 4 == 0, ldx % 4 == 0, 16-byte aligned base
  struct St { const float* p; int y, x; };
  __device__ __forceinline__ St begin(int64_t row) const {
    St s;
    s.p = nullptr; s.y = 0; s.x = 0;
    if (row < nrows) {
      const uint32_t r = (uint32_t)row, hw = (uint32_t)(H * W);
      const uint32_t rem = r % hw;
      s.y = (int)(rem / (uint32_t)W);
      s.x = (int)(rem - (uint32_t)s.y * (uint32_t)W);
      s.p = X + row * ldx;                       // pixel (b, y, x)
    }
    return s;
  }
  __device__ __forceinline__ const float* tap_ptr(const St& s, int tap) const {   // nullptr: padding
    const int ty = tap / ks, tx = tap - ty * ks;
    const int yy = s.y + ty - pad, xx = s.x + tx - pad;
    if (yy < 0 || yy >= H || xx < 0 || xx >= W) return nullptr;
    return s.p + ((int64_t)(ty - pad) * W + (tx - pad)) * ldx;
  }
  __device__ __forceinline__ void copy4(uint32_t dst, const St& s, int64_t k) const {
    const bool on = s.p && k < K;
    int tap = on ? (int)((uint32_t)k / (uint32_t)Cin) : 0, ci = on ? (int)k - tap * Cin : 0;
    if (vec) {                                   // the 4 elements share a tap
      const float* p = on ? tap_ptr(s, tap) : nullptr;
      cp_async16(dst, p ? p + ci : X, p ? 16 : 0);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float* p = (on && k + i < K) ? tap_ptr(s, tap) : nullptr;
        cp_async4(dst + 4 * i, p ? p + ci : X, p ? 4 : 0);
        if (++ci == Cin) { ci = 0; ++tap; }
      }
    }
  }
};

// transposed im2col (weight gradients): row = k index (tap, ci), reduction index = pixel
struct Im2colColLoader {
  static constexpr bool kTransposed = true;
  const float* X;
  int64_t ldx;
  int H, W, Cin, ks, pad;
  int64_t nrows, K;     // nrows = ks*ks*Cin, K = number of pixels
  int vec;              // != 0: Cin % 4 == 0, ldx % 4 == 0, 16-byte aligned base
  struct St { int row4, nr; };
  __device__ __forceinline__ St begin(int64_t row4) const {
    St s;
    s.row4 = (int)row4;
    const int64_t nr = nrows - row4;
    s.nr = nr >= 4 ? 4 : (nr > 0 ? (int)nr : 0);
    return s;
  }
  __device__ __forceinline__ void copy4(uint32_t dst, const St& s, int64_t k) const {
    const bool on = s.nr > 0 && k < K;
    int y = 0, x = 0;
    if (on) {
      const uint32_t rem = (uint32_t)k % (uint32_t)(H * W);
      y = (int)(rem / (uint32_t)W);
      x = (int)(rem - (uint32_t)y * (uint32_t)W);
    }
    int tap = on ? s.row4 / Cin : 0, ci = on ? s.row4 - tap * Cin : 0;
    const float* px = X + k * ldx;               // pixel k itself
    if (vec) {                                   // the 4 rows share a tap
      const int ty = tap / ks, tx = tap - ty * ks;
      const int yy = y + ty - pad, xx = x + tx - pad;
      const bool inb = on && yy >= 0 && yy < H && xx >= 0 && xx < W;
      cp_async16(dst, inb ? px + ((int64_t)(ty - pad) * W + (tx - pad)) * ldx + ci : X, inb ? 16 : 0);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ty = tap / ks, tx = tap - ty * ks;
        const int yy = y + ty - pad, xx = x + tx - pad;
        const bool inb = on && i < s.nr && yy >= 0 && yy < H && xx >= 0 && xx < W;
        cp_async4(dst + 4 * i, inb ? px + ((int64_t)(ty - pad) * W + (tx - pad)) * ldx + ci : X, inb ? 4 : 0);
        if (++ci == Cin) { ci = 0; ++tap; }
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------
// staging: fp32 -> bf16 parts into the UMMA K-major no-swizzle layout (BK = 32: 4 k-groups of 8)
//   byte offset of (row, kgroup) = (row / 8) * 512 + kgroup * 128 + (row % 8) * 16
// A warp-level work unit covers 32 (row, kgroup) items.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

template <bool TRANSPOSED>
__device__ __forceinline__ void unit_coords(int u, int lane, int& row, int& kg) {
  if (TRANSPOSED) { row = (u >> 2) * 32 + lane; kg = u & 3; }
  else { row = u * 8 + (lane & 7); kg = lane >> 3; }
}

// PARTS bf16 terms of v[0..7] -> 16-byte stores at `off` of each part buffer (part stride PSTRIDE)
template <int PARTS>
__device__ __forceinline__ void split_store(float (&v)[8], uint8_t* base, uint32_t off, uint32_t pstride) {
#pragma unroll
  for (int part = 0; part < PARTS; ++part) {
    uint4 h;
    h.x = pack_bf16(v[0], v[1]); h.y = pack_bf16(v[2], v[3]); h.z = pack_bf16(v[4], v[5]); h.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(base + (size_t)part * pstride + off) = h;
    if (part + 1 < PARTS) {
      const uint32_t hh[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {            // exact: the residual is representable in fp32
        v[2 * i] -= __uint_as_float(hh[i] << 16);
        v[2 * i + 1] -= __uint_as_float(hh[i] & 0xFFFF0000u);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// epilogues write 4 consecutive columns of one row (vector path when the layout allows)
// ---------------------------------------------------------------------------------------------
struct PartialEpilogue {
  float* P;
  int64_t M, N;
  struct Row { float* p; };
};

// Data-gradient GEMM of a first layer with <= 2 inputs (fc_net_self.layers.0: Linear(2,256)), fused
// with everything its output is needed for: dh = (g @ W2) * (h > 0) is never written; the epilogue
// reduces it straight into  db1[n] = sum_m dh[m,n]  and  dW1[n,c] = sum_m dh[m,n] * x[m,c].
// Partial sums are owned per (CTA, epilogue warp) and added up in a fixed order: deterministic.
struct ReduceEpilogue {
  const float* mask;        // hidden activations h (ReLU mask), rows indexed like the GEMM rows;
  int64_t ldmask;           //   NULL: the mask is regenerated from (X, W1, b1) below
  const float* X;           // layer inputs
  int64_t ldx;
  const int32_t* x_rows;    // optional gather of the input rows
  int kx;                   // 1 or 2 input columns
  float* part;              // [grid][EPI_WARPS][3][N]
  const float* W1;          // [N][kx], b1 [N]: only read when mask == NULL
  const float* b1;
  struct Row { int64_t r; };
  __device__ __forceinline__ Row row(int64_t m) const { return Row{m}; }
  __device__ __forceinline__ void store(const Row&, int64_t, float) const {}
};
template <class EP> struct IsReduce { static constexpr bool value = false; };
template <> struct IsReduce<ReduceEpilogue> { static constexpr bool value = true; };
constexpr uint32_t REDUCE_ACC_BYTES = EPI_WARPS * 2 * 3 * 128 * 4;   // per warp [n tiles <= 2][3][BN <= 128] fp32

template <class EP>
__device__ __forceinline__ typename EP::Row epi_row(const EP& ep, int64_t m, int z) { return ep.row(m); }
template <>
__device__ __forceinline__ PartialEpilogue::Row epi_row<PartialEpilogue>(const PartialEpilogue& ep, int64_t m, int z) {
  return PartialEpilogue::Row{ep.P + ((int64_t)z * ep.M + m) * ep.N};
}

// Column-only epilogue terms (bias) are fetched once per 32-column chunk, row handles once per tile:
// a load issued after a store to memory that may alias it cannot be hoisted by the compiler and
// would otherwise serialise one L2 round trip per store.
template <class EP>
__device__ __forceinline__ float4 epi_bias4(const EP& ep, int64_t n, int64_t N) { return make_float4(0.f, 0.f, 0.f, 0.f); }
template <>
__device__ __forceinline__ float4 epi_bias4<PlainEpilogue>(const PlainEpilogue& ep, int64_t n, int64_t N) {
  float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ep.flags & TM_EPI_BIAS) {
    if (n < N) b.x = ep.bias[n];
    if (n + 1 < N) b.y = ep.bias[n + 1];
    if (n + 2 < N) b.z = ep.bias[n + 2];
    if (n + 3 < N) b.w = ep.bias[n + 3];
  }
  return b;
}

// Row operands of the epilogue (ReLU-backward mask, old C for accumulation) are fetched for all 8
// store passes of a chunk BEFORE the first store, for the same reason.
struct EpiAux { float4 mask, old; };
template <class EP>
__device__ __forceinline__ EpiAux epi_aux(const EP& ep, const typename EP::Row& rw, int64_t n, int64_t N) { return EpiAux{}; }
template <>
__device__ __forceinline__ EpiAux epi_aux<PlainEpilogue>(const PlainEpilogue& ep, const PlainEpilogue::Row& rw, int64_t n, int64_t N) {
  EpiAux a;
  a.mask = make_float4(1.f, 1.f, 1.f, 1.f);
  a.old = make_float4(0.f, 0.f, 0.f, 0.f);
  if (ep.flags & TM_EPI_MASK) {
    const float* mp = ep.mask + rw.r * ep.ldmask + n;
    if ((n + 4 <= N) && ((ep.ldmask & 3) == 0) && ((reinterpret_cast<uintptr_t>(ep.mask) & 15) == 0)) a.mask = ld4(mp);
    else {
      if (n < N) a.mask.x = mp[0];
      if (n + 1 < N) a.mask.y = mp[1];
      if (n + 2 < N) a.mask.z = mp[2];
      if (n + 3 < N) a.mask.w = mp[3];
    }
  }
  if (ep.flags & TM_EPI_ACCUM) {
    const float* cp = ep.C + rw.r * ep.ldc + n;
    if ((n + 4 <= N) && ((ep.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(ep.C) & 15) == 0)) a.old = ld4(cp);
    else {
      if (n < N) a.old.x = cp[0];
      if (n + 1 < N) a.old.y = cp[1];
      if (n + 2 < N) a.old.z = cp[2];
      if (n + 3 < N) a.old.w = cp[3];
    }
  }
  return a;
}

template <class EP>
__device__ __forceinline__ void store4(const EP& ep, const typename EP::Row& rw, int64_t n, int64_t N, const float (&v)[4],
                                       const float4& b4, const EpiAux& ax) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
    if (n + i < N) ep.store(rw, n + i, v[i]);
}
template <>
__device__ __forceinline__ void store4<PartialEpilogue>(const PartialEpilogue& ep, const PartialEpilogue::Row& rw, int64_t n,
                                                        int64_t N, const float (&v)[4], const float4& b4, const EpiAux& ax) {
  if (n + 4 <= N && (N & 3) == 0) {
    st4(rw.p + n, make_float4(v[0], v[1], v[2], v[3]));
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (n + i < N) rw.p[n + i] = v[i];
  }
}
// PlainEpilogue: one 128-bit store per lane when rows are 16-byte aligned
template <>
__device__ __forceinline__ void store4<PlainEpilogue>(const PlainEpilogue& ep, const PlainEpilogue::Row& rw, int64_t n,
                                                      int64_t N, const float (&v)[4], const float4& b4, const EpiAux& ax) {
  float4 o = make_float4(v[0] + b4.x + ax.old.x, v[1] + b4.y + ax.old.y, v[2] + b4.z + ax.old.z, v[3] + b4.w + ax.old.w);
  if (ep.flags & TM_EPI_RELU) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
  if (ep.flags & TM_EPI_MASK) {
    o.x = ax.mask.x > 0.f ? o.x : 0.f; o.y = ax.mask.y > 0.f ? o.y : 0.f; o.z = ax.mask.z > 0.f ? o.z : 0.f; o.w = ax.mask.w > 0.f ? o.w : 0.f;
  }
  float* p = ep.C + rw.r * ep.ldc + n;
  if ((n + 4 <= N) && ((ep.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(ep.C) & 15) == 0)) {
    st4(p, o);
  } else {
    if (n < N) p[0] = o.x;
    if (n + 1 < N) p[1] = o.y;
    if (n + 2 < N) p[2] = o.z;
    if (n + 3 < N) p[3] = o.w;
  }
}

// ---------------------------------------------------------------------------------------------
// Row-direct epilogue (tf_gemm_kernel): a lane owns ONE row of the tile (TMEM lane = tile row) and writes the 32
// columns of a chunk straight from the tcgen05.ld registers as eight 128-bit stores -- no shared-memory transpose, the
// row handle and the vector-path predicates resolved once per tile.  Measured on the 229 819 x 128 x 256 product the
// transposing epilogue was the critical path of the whole kernel: 23 000 cycles per 128 x 128 tile (a single warp per
// scheduler walking ~1 500 dependent 64-bit index / predicate instructions) against 17 000 for the main loop.  The
// eight stores of a lane fill one 128-byte line, so L2 sees whole lines.
// ---------------------------------------------------------------------------------------------
template <class EP>
struct RowStore {                 // generic: element-wise through EP::store
  typename EP::Row rw;
  __device__ __forceinline__ void open(const EP& ep, int64_t m, int z, int64_t N) { rw = epi_row<EP>(ep, m, z); }
  __device__ __forceinline__ void chunk(const EP& ep, int64_t n, int64_t N, const float (&v)[32]) const {
#pragma unroll
    for (int i = 0; i < 32; ++i)
      if (n + i < N) ep.store(rw, n + i, v[i]);
  }
};
template <>
struct RowStore<PartialEpilogue> {
  float* p;
  bool vec;
  __device__ __forceinline__ void open(const PartialEpilogue& ep, int64_t m, int z, int64_t N) {
    p = ep.P + ((int64_t)z * ep.M + m) * ep.N;
    vec = (N & 3) == 0 && (reinterpret_cast<uintptr_t>(ep.P) & 15) == 0;
  }
  __device__ __forceinline__ void chunk(const PartialEpilogue& ep, int64_t n, int64_t N, const float (&v)[32]) const {
    float* q = p + n;
    if (vec && n + 32 <= N) {
#pragma unroll
      for (int j = 0; j < 8; ++j) st4(q + 4 * j, make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (n + i < N) q[i] = v[i];
    }
  }
};
template <>
struct RowStore<PlainEpilogue> {
  float* p;
  const float* mp;
  bool vec;
  __device__ __forceinline__ void open(const PlainEpilogue& ep, int64_t m, int z, int64_t N) {
    const int64_t r = ep.c_rows ? (int64_t)ep.c_rows[m] : m;
    p = ep.C + r * ep.ldc;
    mp = (ep.flags & TM_EPI_MASK) ? ep.mask + r * ep.ldmask : nullptr;
    vec = (ep.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(ep.C) & 15) == 0 &&
          (!(ep.flags & TM_EPI_BIAS) || (reinterpret_cast<uintptr_t>(ep.bias) & 15) == 0) &&
          (!mp || ((ep.ldmask & 3) == 0 && (reinterpret_cast<uintptr_t>(ep.mask) & 15) == 0));
  }
  __device__ __forceinline__ void chunk(const PlainEpilogue& ep, int64_t n, int64_t N, const float (&v)[32]) const {
    const int flags = ep.flags;
    if (vec && n + 32 <= N) {
      float4 mk[8], old[8];
      if (flags & TM_EPI_MASK) {                   // row operands first: all loads in flight before the first store
#pragma unroll
        for (int j = 0; j < 8; ++j) mk[j] = ld4(mp + n + 4 * j);
      }
      if (flags & TM_EPI_ACCUM) {
#pragma unroll
        for (int j = 0; j < 8; ++j) old[j] = ld4(p + n + 4 * j);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        if (flags & TM_EPI_BIAS) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(ep.bias + n + 4 * j));
          o.x += b.x; o.y += b.y; o.z += b.z; o.w += b.w;
        }
        if (flags & TM_EPI_ACCUM) { o.x += old[j].x; o.y += old[j].y; o.z += old[j].z; o.w += old[j].w; }
        if (flags & TM_EPI_RELU) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
        if (flags & TM_EPI_MASK) {
          o.x = mk[j].x > 0.f ? o.x : 0.f; o.y = mk[j].y > 0.f ? o.y : 0.f;
          o.z = mk[j].z > 0.f ? o.z : 0.f; o.w = mk[j].w > 0.f ? o.w : 0.f;
        }
        st4(p + n + 4 * j, o);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        if (n + i < N) {
          float o = v[i];
          if (flags & TM_EPI_BIAS) o += ep.bias[n + i];
          if (flags & TM_EPI_ACCUM) o += p[n + i];
          if (flags & TM_EPI_RELU) o = fmaxf(o, 0.f);
          if (flags & TM_EPI_MASK) o = (mp[n + i] > 0.f) ? o : 0.f;
          p[n + i] = o;
        }
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------
// kernel configuration
// ---------------------------------------------------------------------------------------------
__host__ __device__ constexpr int parts_of(int split) { return split == 1 ? 1 : (split == 3 ? 2 : 3); }
constexpr uint32_t EPI_SCRATCH = EPI_WARPS * 32 * 33 * 4;   // one 32 x 33 fp32 transpose tile per epilogue warp
constexpr uint32_t SMEM_BUDGET = 218 * 1024;
constexpr int MAX_STAGES = 8;

template <int BN, int SPLIT>
struct Cfg {
  static constexpr int PARTS = parts_of(SPLIT);
  static constexpr uint32_t A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2;
  static constexpr uint32_t STAGE = (A_BYTES + B_BYTES) * PARTS;      // one k-block of bf16 parts (UMMA layout)
  static constexpr int A_UNITS = BM / 8, B_UNITS = BN / 8;          // 32-item conversion units per stage
  static constexpr int A_PER = A_UNITS / PROD_WARPS;                // 2
  static constexpr int B_PER = (B_UNITS + PROD_WARPS - 1) / PROD_WARPS;   // 1..4
  // raw fp32 k-block (cp.async target): thread-private items of 32 bytes, 256 threads (transposed
  // operands use the same area as a [k][row] tile image, which is never larger)
  static constexpr uint32_t RAW_A = A_PER * 32 * PROD_THREADS, RAW_B = B_PER * 32 * PROD_THREADS;
  static constexpr uint32_t RAW = RAW_A + RAW_B;
  static constexpr uint32_t RING = SMEM_BUDGET - EPI_SCRATCH - 1024;
  static constexpr int NS = (PARTS == 3 || 3 * STAGE + 2 * RAW > RING) ? 2 : 3;          // bf16 stages
  static constexpr int ND_RAW = (int)((RING - NS * STAGE) / RAW);
  static constexpr int ND = ND_RAW > 6 ? 6 : ND_RAW;                  // raw k-blocks in flight
  static_assert(ND >= 2, "shared-memory budget too small for this tile");
  static constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;   // two accumulators, power of two
  static constexpr size_t SMEM = (size_t)NS * STAGE + (size_t)ND * RAW + EPI_SCRATCH + 1024 /*alignment slack*/;
  static constexpr int A_CH = BM * BK / 4 / PROD_THREADS;           // 16-byte copy chunks per thread (4)
  static constexpr int B_CH = (BN * BK / 4 + PROD_THREADS - 1) / PROD_THREADS;   // 1..8
};

// tile index -> (m tile, n tile, k split): splits fastest, then n, so that concurrently running
// CTAs share A rows through L2
struct TileMap {
  int64_t total, K, k_per_split;
  int nt, z;
  long long* trace;   // TM_TC_TRACE: clock64 stamps of CTA 0 (producer warp 0 / MMA thread / epilogue warp 0)
  int dbg;    // TM_TC_DEBUG bits (bottleneck bisection): 1 no epilogue stores, 2 no global loads, 4 no staging, 8 no MMA
  // nq = n tile INDEX (the kernel scales it by its BN)
  __device__ __forceinline__ void decode(int64_t t, int64_t& m0, int64_t& nq, int& zi, int64_t& kbeg, int& nkb) const {
    zi = (int)(t % z);
    const int64_t q = t / z;
    nq = q % nt;
    m0 = (q / nt) * BM;
    kbeg = (int64_t)zi * k_per_split;
    const int64_t kend = (kbeg + k_per_split < K) ? kbeg + k_per_split : K;
    const int64_t nb = (kend > kbeg) ? (kend - kbeg + BK - 1) / BK : 0;
    nkb = nb > 0 ? (int)nb : 1;                  // K == 0 still produces a (zero) accumulator
  }
};

// ---------------------------------------------------------------------------------------------
// the kernel.  grid = min(#tiles, #SMs) persistent CTAs
// ---------------------------------------------------------------------------------------------
template <class AL, class BL, class EP, int BN, int SPLIT>
__global__ void __launch_bounds__(THREADS, 1)
tc_gemm_kernel(AL al, BL bl, EP ep, int64_t M, int64_t N, TileMap tm, int* __restrict__ err) {
  using C = Cfg<BN, SPLIT>;
  constexpr int PARTS = C::PARTS, NS = C::NS, A_PER = C::A_PER, B_PER = C::B_PER;
  constexpr uint32_t A_BYTES = C::A_BYTES, B_BYTES = C::B_BYTES, STAGE = C::STAGE;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* rawring = ring + (size_t)NS * STAGE;
  float* scratch = reinterpret_cast<float*>(rawring + (size_t)C::ND * C::RAW);
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ int abort_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(&full_bar[i], PROD_WARPS); mbar_init(&empty_bar[i], 1); }
    mbar_init(&acc_full[0], 1); mbar_init(&acc_full[1], 1);
    mbar_init(&acc_empty[0], EPI_WARPS); mbar_init(&acc_empty[1], EPI_WARPS);
    abort_s = 0;
    fence_mbarrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(&tmem_base_s, C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  volatile int* abortp = &abort_s;
  bool ok = true;
  const int64_t G = gridDim.x;

  if (warp >= PROD_WARP0) {
    // ======================= producers =======================
    constexpr int ND = C::ND, A_CH = C::A_CH, B_CH = C::B_CH;
    constexpr uint32_t RAW = C::RAW, RAW_A = C::RAW_A;
    constexpr bool COOP = AL::kTransposed || BL::kTransposed;       // any cooperative copy -> producer-wide barriers
    const int pw = warp - PROD_WARP0;
    const int ptid = tid - PROD_WARP0 * 32;
    // ---- conversion items (fixed per thread): (row, k group) of the tile, 8 consecutive k each
    int a_row[A_PER], a_kg[A_PER], b_row[B_PER], b_kg[B_PER];
    uint32_t a_off[A_PER], b_off[B_PER];
    bool b_on[B_PER];
#pragma unroll
    for (int i = 0; i < A_PER; ++i) {
      unit_coords<AL::kTransposed>(pw * A_PER + i, lane, a_row[i], a_kg[i]);
      a_off[i] = (uint32_t)(a_row[i] >> 3) * 512u + (uint32_t)a_kg[i] * 128u + (uint32_t)(a_row[i] & 7) * 16u;
    }
#pragma unroll
    for (int i = 0; i < B_PER; ++i) {
      const int u = pw * B_PER + i;
      b_on[i] = u < C::B_UNITS;
      unit_coords<BL::kTransposed>(b_on[i] ? u : 0, lane, b_row[i], b_kg[i]);
      b_off[i] = (uint32_t)(b_row[i] >> 3) * 512u + (uint32_t)b_kg[i] * 128u + (uint32_t)(b_row[i] & 7) * 16u;
    }
    // raw layouts.  K-contiguous operand: thread-private, item i half h at ((2i + h) * 256 + ptid) * 16
    // (conflict-free for the warp's 128-bit accesses).  Transposed operand: tile image [k][row].
    auto priv = [&](int i, int h) { return (uint32_t)((2 * i + h) * PROD_THREADS + ptid) * 16u; };
    // ---- load cursor (ND k-blocks ahead of the conversion, across tile boundaries)
    constexpr int A_NST = AL::kTransposed ? 1 : A_PER;
    constexpr int B_NST = BL::kTransposed ? 1 : B_PER;
    typename AL::St ast[A_NST];
    typename BL::St bst[B_NST];
    int64_t lt = blockIdx.x, lk = 0;
    int lkb = 0, lnkb = 0;
    bool lvalid = false;
    uint32_t total = 0;
    for (int64_t t = blockIdx.x; t < tm.total; t += G) {
      int64_t m0, nq, kb0; int zi, nkb;
      tm.decode(t, m0, nq, zi, kb0, nkb);
      total += (uint32_t)nkb;
    }
    auto open_tile = [&]() {
      lvalid = lt < tm.total;
      if (!lvalid) return;
      int64_t m0, nq; int zi;
      tm.decode(lt, m0, nq, zi, lk, lnkb);
      lkb = 0;
      if (AL::kTransposed) { ast[0] = al.begin(m0 + (ptid & (BM / 4 - 1)) * 4); }
      else {
#pragma unroll
        for (int i = 0; i < A_NST; ++i) ast[i] = al.begin(m0 + a_row[i]);
      }
      if (BL::kTransposed) { bst[0] = bl.begin(nq * BN + (ptid & (BN / 4 - 1)) * 4); }
      else {
#pragma unroll
        for (int i = 0; i < B_NST; ++i) bst[i] = bl.begin(nq * BN + b_row[i]);
      }
    };
    uint32_t ls = 0;                                               // raw slot of the next k-block to load
    auto issue = [&]() {                                           // always commits exactly one group
      if (lvalid && !(TM_DBGBITS & 2)) {
        const uint32_t ra = smem_u32(rawring + (size_t)ls * RAW), rb = ra + RAW_A;
        if (AL::kTransposed) {
#pragma unroll
          for (int j = 0; j < A_CH; ++j) {
            const int q = j * PROD_THREADS + ptid, kk = q / (BM / 4), rc = q % (BM / 4);
            al.copy4(ra + (uint32_t)(kk * BM + rc * 4) * 4u, ast[0], lk + kk);
          }
        } else {
#pragma unroll
          for (int i = 0; i < A_PER; ++i) {
            al.copy4(ra + priv(i, 0), ast[i], lk + a_kg[i] * 8);
            al.copy4(ra + priv(i, 1), ast[i], lk + a_kg[i] * 8 + 4);
          }
        }
        if (BL::kTransposed) {
#pragma unroll
          for (int j = 0; j < B_CH; ++j) {
            const int q = j * PROD_THREADS + ptid, kk = q / (BN / 4), rc = q % (BN / 4);
            if (kk < BK) bl.copy4(rb + (uint32_t)(kk * BN + rc * 4) * 4u, bst[0], lk + kk);
          }
        } else {
#pragma unroll
          for (int i = 0; i < B_PER; ++i) {
            if (b_on[i]) {
              bl.copy4(rb + priv(i, 0), bst[i < B_NST ? i : 0], lk + b_kg[i] * 8);
              bl.copy4(rb + priv(i, 1), bst[i < B_NST ? i : 0], lk + b_kg[i] * 8 + 4);
            }
          }
        }
      }
      if (lvalid) {
        lk += BK;
        if (++lkb == lnkb) { lt += G; open_tile(); }
      }
      cp_async_commit();
      if (++ls == (uint32_t)ND) ls = 0;
    };
    auto read_item = [&](bool transposed, const uint8_t* raw, int i, int row, int kg, int rows, float (&v)[8]) {
      if (transposed) {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = *reinterpret_cast<const float*>(raw + (uint32_t)((kg * 8 + e) * rows + row) * 4u);
      } else {
        const float4 x = *reinterpret_cast<const float4*>(raw + priv(i, 0));
        const float4 y = *reinterpret_cast<const float4*>(raw + priv(i, 1));
        v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
      }
    };
    open_tile();
#pragma unroll 1
    for (int d = 0; d < ND; ++d) issue();

    uint32_t s = 0, ph = 0, rs = 0;
    uint32_t tr_n = 0;
    const bool tr_on = TM_TRACEPTR && blockIdx.x == 0 && pw == 0 && lane == 0;
#pragma unroll 1
    for (uint32_t g = 0; g < total; ++g) {
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 0] = clock64();
      cp_async_wait<ND - 1>();                                         // my copies of k-block g have landed
      if (!mbar_wait_abort(&empty_bar[s], ph ^ 1u, abortp)) abort_s = 1;    // MMAs that read this stage are done
      if (COOP) asm volatile("bar.sync 1, %0;" ::"n"(PROD_THREADS) : "memory");   // everybody's copies landed
      else __syncwarp();
      if (*abortp) { ok = false; break; }                              // (uniform across the barrier)
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 1] = clock64();
      const uint8_t* raw_a = rawring + (size_t)rs * RAW;
      const uint8_t* raw_b = raw_a + RAW_A;
      uint8_t* a_base = ring + (size_t)s * STAGE;
      uint8_t* b_base = a_base + A_BYTES * PARTS;
      if (!(TM_DBGBITS & 4)) {
#pragma unroll
        for (int i = 0; i < A_PER; ++i) {
          float v[8];
          read_item(AL::kTransposed, raw_a, i, a_row[i], a_kg[i], BM, v);
          split_store<PARTS>(v, a_base, a_off[i], A_BYTES);
        }
#pragma unroll
        for (int i = 0; i < B_PER; ++i) {
          if (b_on[i]) {
            float v[8];
            read_item(BL::kTransposed, raw_b, i, b_row[i], b_kg[i], BN, v);
            split_store<PARTS>(v, b_base, b_off[i], B_BYTES);
          }
        }
      }
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 2] = clock64();
      fence_async_smem();                                              // generic-proxy stores -> async proxy (UMMA)
      if (COOP) asm volatile("bar.sync 2, %0;" ::"n"(PROD_THREADS) : "memory");   // everyone is done reading raw slot rs
      else __syncwarp();
      if (lane == 0) mbar_arrive(&full_bar[s]);                        // one arrival per producer warp
      if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
      if (++rs == (uint32_t)ND) rs = 0;
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 3] = clock64();
      ++tr_n;
      issue();                                                         // refill the slot just freed (k-block g + ND)
    }
    cp_async_wait<0>();
  } else if (warp == MMA_WARP) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(Fmt::BF16, BN);
      uint32_t s = 0, ph = 0;
      int li = 0;
      for (int64_t t = blockIdx.x; t < tm.total && ok; t += G, ++li) {
        const int buf = li & 1;
        const uint32_t aph = (uint32_t)(li >> 1) & 1u;
        ok = mbar_wait_abort(&acc_empty[buf], aph ^ 1u, abortp);               // epilogue drained this accumulator
        if (!ok) break;
        tc_fence_after();
        int64_t m0, nq, kb0; int zi, nkb;
        tm.decode(t, m0, nq, zi, kb0, nkb);
        const uint32_t tmem_d = tmem_base + (uint32_t)(buf * BN);
        for (int kb = 0; kb < nkb; ++kb) {
          const bool tr_on = TM_TRACEPTR && blockIdx.x == 0 && li == 0 + (kb >> 6) && kb < 64;
          if (tr_on) TM_TRACEPTR[256 + kb * 4 + 0] = clock64();
          ok = mbar_wait_abort(&full_bar[s], ph, abortp);
          if (!ok) break;
          tc_fence_after();
          if (tr_on) TM_TRACEPTR[256 + kb * 4 + 1] = clock64();
          const uint32_t sa = smem_u32(ring + (size_t)s * STAGE), sb = sa + A_BYTES * PARTS;
          if (!(TM_DBGBITS & 8))
#pragma unroll
          for (int ks = 0; ks < BK / 16; ++ks) {
            const uint32_t koff = (uint32_t)ks * 256u;                   // two 128-byte core matrices per K = 16
            uint64_t da[PARTS], db[PARTS];
#pragma unroll
            for (int p = 0; p < PARTS; ++p) {
              da[p] = smem_desc(sa + p * A_BYTES + koff, 128, 512);
              db[p] = smem_desc(sb + p * B_BYTES + koff, 128, 512);
            }
            // products in decreasing magnitude; parts: 0 = hi, 1 = mid, 2 = lo
            umma_f16(tmem_d, da[0], db[0], idesc, (kb > 0 || ks > 0) ? 1u : 0u);
            if (PARTS >= 2) { umma_f16(tmem_d, da[0], db[1], idesc, 1u); umma_f16(tmem_d, da[1], db[0], idesc, 1u); }
            if (PARTS >= 3) {
              umma_f16(tmem_d, da[1], db[1], idesc, 1u);
              umma_f16(tmem_d, da[0], db[2], idesc, 1u);
              umma_f16(tmem_d, da[2], db[0], idesc, 1u);
            }
          }
          umma_commit(&empty_bar[s]);                                    // stage reusable once these MMAs retire
          if (tr_on) TM_TRACEPTR[256 + kb * 4 + 2] = clock64();
          if (++s == (uint32_t)NS) { s = 0; ph ^= 1u; }
        }
        if (!ok) break;
        umma_commit(&acc_full[buf]);                                     // covers every MMA of the tile
      }
    }
    __syncwarp();
  } else {
    // ======================= epilogue =======================
    float* scr = scratch + warp * (32 * 33);
    int li = 0;
    for (int64_t t = blockIdx.x; t < tm.total && ok; t += G, ++li) {
      const int buf = li & 1;
      const uint32_t aph = (uint32_t)(li >> 1) & 1u;
      const bool tr_on = TM_TRACEPTR && blockIdx.x == 0 && warp == 0 && lane == 0 && li < 16;
      if (tr_on) TM_TRACEPTR[512 + li * 4 + 0] = clock64();
      ok = mbar_wait_abort(&acc_full[buf], aph, abortp);
      if (!ok) break;
      tc_fence_after();
      if (tr_on) TM_TRACEPTR[512 + li * 4 + 1] = clock64();
      int64_t m0, nq, kb0; int zi, nkb;
      tm.decode(t, m0, nq, zi, kb0, nkb);
      const int64_t n0 = nq * BN;
      typename EP::Row rws[8];                                            // this lane's rows of the 8 store passes
#pragma unroll
      for (int pass = 0; pass < 8; ++pass) {
        const int64_t m = m0 + warp * 32 + pass * 4 + (lane >> 3);
        rws[pass] = epi_row<EP>(ep, m < M ? m : M - 1, zi);
      }
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * BN);
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        if (n0 + c >= N) break;
        const float4 b4 = epi_bias4<EP>(ep, n0 + c + (lane & 7) * 4, N);
        float v[32];
        tmem_ld32(trow + (uint32_t)c, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) scr[lane * 33 + i] = v[i];
        __syncwarp();
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          EpiAux aux[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {                                   // row operands first (loads in flight together)
            const int pass = half * 4 + q;
            const int64_t m = m0 + warp * 32 + pass * 4 + (lane >> 3);
            const int64_t n = n0 + c + (lane & 7) * 4;
            aux[q] = (m < M && n < N) ? epi_aux<EP>(ep, rws[pass], n, N) : EpiAux{};
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {                                   // 8 lanes x 4 columns per row, 4 rows per pass
            const int pass = half * 4 + q;
            const int r = pass * 4 + (lane >> 3), cq = (lane & 7) * 4;
            const int64_t m = m0 + warp * 32 + r;
            const int64_t n = n0 + c + cq;
            if (m < M && n < N && !(TM_DBGBITS & 1)) {
              const float o[4] = {scr[r * 33 + cq], scr[r * 33 + cq + 1], scr[r * 33 + cq + 2], scr[r * 33 + cq + 3]};
              store4<EP>(ep, rws[pass], n, N, o, b4, aux[q]);
            }
          }
        }
        __syncwarp();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
      if (tr_on) TM_TRACEPTR[512 + li * 4 + 2] = clock64();
    }
  }
  if (!ok) {
    abort_s = 1;
    if (err) atomicExch(err, 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// =============================================================================================
// 3xTF32 kernel (precision 3, the default fp32-class mode; precision 4 = single-pass TF32).
//
// tcgen05.mma.kind::tf32 reads fp32 words from shared memory and uses their upper 19 bits, so the
// RAW fp32 k-block that cp.async drops into the stage *is* the "hi" operand -- no conversion and
// no second staging buffer.  Only the residual  lo = x - trunc_tf32(x)  (exact in fp32) is
// computed, elementwise and layout-preserving, by the thread that copied the chunk (no barrier
// between producer warps).  Products hi*hi + hi*lo + lo*hi keep ~21 mantissa bits.
//
// Shared-memory layouts (per operand plane, ROWS x 32 fp32 = ROWS*128 bytes, 1024-byte aligned):
//   K-contiguous operand  -> K-major SWIZZLE_128B:  off(row, c) = row*128 + ((c ^ (row&7)) << 4),
//                            c = 16-byte chunk (4 consecutive k)
//   transposed operand    -> MN-major SWIZZLE_128B_BASE32B (the only MN-major layout of 32-bit
//                            operands): atoms of 4 k x 128 bytes (32 rows), the 32-byte chunk index
//                            XOR-ed with k & 3.  chunk = 4 consecutive rows (16-byte index rc) of one k:
//                            off(k, rc) = (rc>>3)*4096 + (k>>2)*512 + (k&3)*128 + (((((rc&7)>>1) ^ (k&3)) << 1 | (rc&1)) << 4)
// Both are written directly by 16-byte cp.async's (whole 128-byte lines per quarter warp in HBM
// and in shared memory), so weight gradients (both operands transposed) need no transposition.
// =============================================================================================
// 16 producer warps: the copy phase is bound by cp.async issue and the lo pass by ALU latency, both of
// which scale with the number of warps in flight (the kernel needs < 64 registers per thread)
constexpr int TF_PROD_WARPS = 16;
constexpr int TF_PROD_THREADS = TF_PROD_WARPS * 32;
constexpr int TF_THREADS = (EPI_WARPS + 1 + TF_PROD_WARPS) * 32;   // 672

// byte offset of the 16-byte chunk (k, rc) of an MN-major plane
__device__ __forceinline__ uint32_t mn_chunk_off(int k, int rc) {
  const uint32_t j = (uint32_t)(rc & 7), k4 = (uint32_t)(k & 3);
  return (uint32_t)(rc >> 3) * 4096u + (uint32_t)(k >> 2) * 512u + k4 * 128u + (((((j >> 1) ^ k4) << 1) | (j & 1u)) << 4);
}
template <int BN, int PLANES>
struct TfCfg {
  static constexpr uint32_t PLANE_A = BM * BK * 4, PLANE_B = BN * BK * 4;
  static constexpr uint32_t SLOT = (PLANE_A + PLANE_B) * PLANES;
  static constexpr uint32_t RING = SMEM_BUDGET - EPI_SCRATCH - 1024;
  static constexpr int ND_RAW = (int)(RING / SLOT);
  static constexpr int ND = ND_RAW > MAX_STAGES ? MAX_STAGES : ND_RAW;
  static_assert(ND >= 2, "shared-memory budget too small for this tile");
  static constexpr uint32_t TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr size_t SMEM = (size_t)ND * SLOT + EPI_SCRATCH + 1024;
  static constexpr int A_CH = BM * 8 / TF_PROD_THREADS;                          // 16-byte chunks per thread (4)
  static constexpr int B_CH = (BN * 8 + TF_PROD_THREADS - 1) / TF_PROD_THREADS;     // 1..8
};

template <class AL, class BL, class EP, int BN, int PLANES>
__global__ void __launch_bounds__(TF_THREADS, 1)
tf_gemm_kernel(AL al, BL bl, EP ep, int64_t M, int64_t N, TileMap tm, int* __restrict__ err) {
  using C = TfCfg<BN, PLANES>;
  constexpr int ND = C::ND, A_CH = C::A_CH, B_CH = C::B_CH;
  constexpr uint32_t PLANE_A = C::PLANE_A, PLANE_B = C::PLANE_B, SLOT = C::SLOT;
  constexpr uint32_t OFF_AHI = 0, OFF_ALO = PLANE_A, OFF_BHI = PLANE_A * PLANES, OFF_BLO = PLANE_A * PLANES + PLANE_B;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* scratch = reinterpret_cast<float*>(ring + (size_t)ND * SLOT);
  float* reduce_acc = scratch + EPI_SCRATCH / 4;                 // only allocated for ReduceEpilogue launches
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES], empty_bar[MAX_STAGES], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ int abort_s;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < ND; ++i) { mbar_init(&full_bar[i], TF_PROD_WARPS); mbar_init(&empty_bar[i], 1); }
    mbar_init(&acc_full[0], 1); mbar_init(&acc_full[1], 1);
    mbar_init(&acc_empty[0], EPI_WARPS); mbar_init(&acc_empty[1], EPI_WARPS);
    abort_s = 0;
    fence_mbarrier_init();
  }
  if (warp == MMA_WARP) tmem_alloc(&tmem_base_s, C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  volatile int* abortp = &abort_s;
  bool ok = true;
  const int64_t G = gridDim.x;

  if (warp >= PROD_WARP0) {
    // ======================= producers =======================
    const int ptid = tid - PROD_WARP0 * 32;
    // chunk j of this thread -> byte offset inside the operand plane (same for hi and lo)
    uint32_t a_o[A_CH], b_o[B_CH];
    bool b_on[B_CH];
#pragma unroll
    for (int j = 0; j < A_CH; ++j) {
      const int q = j * TF_PROD_THREADS + ptid;
      if (AL::kTransposed) {
        const int rc = q % (BM / 4), k = q / (BM / 4);
        a_o[j] = mn_chunk_off(k, rc);
      } else {
        const int row = q >> 3, c = q & 7;
        a_o[j] = (uint32_t)row * 128u + (uint32_t)((c ^ (row & 7)) << 4);
      }
    }
#pragma unroll
    for (int j = 0; j < B_CH; ++j) {
      const int q = j * TF_PROD_THREADS + ptid;
      b_on[j] = q < BN * 8;
      if (BL::kTransposed) {
        const int rc = q % (BN / 4), k = q / (BN / 4);
        b_o[j] = mn_chunk_off(k, rc);
      } else {
        const int row = q >> 3, c = q & 7;
        b_o[j] = (uint32_t)row * 128u + (uint32_t)((c ^ (row & 7)) << 4);
      }
    }
    constexpr int A_NST = AL::kTransposed ? 1 : A_CH;
    constexpr int B_NST = BL::kTransposed ? 1 : B_CH;
    typename AL::St ast[A_NST];
    typename BL::St bst[B_NST];
    int64_t lt = blockIdx.x, lk = 0;
    int lkb = 0, lnkb = 0;
    bool lvalid = false;
    uint32_t total = 0;
    for (int64_t t = blockIdx.x; t < tm.total; t += G) {
      int64_t m0, nq, kb0; int zi, nkb;
      tm.decode(t, m0, nq, zi, kb0, nkb);
      total += (uint32_t)nkb;
    }
    auto open_tile = [&]() {
      lvalid = lt < tm.total;
      if (!lvalid) return;
      int64_t m0, nq; int zi;
      tm.decode(lt, m0, nq, zi, lk, lnkb);
      lkb = 0;
      if (AL::kTransposed) { ast[0] = al.begin(m0 + (ptid % (BM / 4)) * 4); }
      else {
#pragma unroll
        for (int j = 0; j < A_NST; ++j) ast[j] = al.begin(m0 + j * (TF_PROD_THREADS / 8) + (ptid >> 3));
      }
      if (BL::kTransposed) { bst[0] = bl.begin(nq * BN + (ptid % (BN / 4)) * 4); }
      else {
#pragma unroll
        for (int j = 0; j < B_NST; ++j) bst[j] = bl.begin(nq * BN + j * (TF_PROD_THREADS / 8) + (ptid >> 3));
      }
    };
    uint32_t ls = 0, lph = 0;                                        // slot / phase of the next k-block to load
    auto issue = [&]() -> bool {                                     // always commits exactly one group
      if (lvalid) {
        if (!mbar_wait_abort(&empty_bar[ls], lph ^ 1u, abortp)) return false;   // MMAs that read this slot are done
        if (!(TM_DBGBITS & 2)) {
          const uint32_t base = smem_u32(ring + (size_t)ls * SLOT);
#pragma unroll
          for (int j = 0; j < A_CH; ++j) {
            if (AL::kTransposed) al.copy4(base + OFF_AHI + a_o[j], ast[0], lk + (j * TF_PROD_THREADS + ptid) / (BM / 4));
            else al.copy4(base + OFF_AHI + a_o[j], ast[j], lk + (ptid & 7) * 4);
          }
#pragma unroll
          for (int j = 0; j < B_CH; ++j) {
            if (b_on[j]) {
              if (BL::kTransposed) bl.copy4(base + OFF_BHI + b_o[j], bst[0], lk + (j * TF_PROD_THREADS + ptid) / (BN / 4));
              else bl.copy4(base + OFF_BHI + b_o[j], bst[j < B_NST ? j : 0], lk + (ptid & 7) * 4);
            }
          }
        }
        lk += BK;
        if (++lkb == lnkb) { lt += G; open_tile(); }
        if (++ls == (uint32_t)ND) { ls = 0; lph ^= 1u; }
      }
      cp_async_commit();
      return true;
    };
    constexpr int D = ND - 1;                                        // k-blocks in flight
    open_tile();
#pragma unroll 1
    for (int d = 0; d < D && ok; ++d) ok = issue();

    uint32_t s = 0;
    uint32_t tr_n = 0;
    const bool tr_on = TM_TRACEPTR && blockIdx.x == 0 && warp == PROD_WARP0 && lane == 0;
#pragma unroll 1
    for (uint32_t g = 0; g < total && ok; ++g) {
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 0] = clock64();
      cp_async_wait<D - 1>();                                          // my chunks of k-block g have landed
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 1] = clock64();
      if (PLANES == 2 && !(TM_DBGBITS & 4)) {
        uint8_t* base = ring + (size_t)s * SLOT;
        auto residual = [&](uint32_t hi_off, uint32_t lo_off) {
          *reinterpret_cast<float4*>(base + lo_off) = tf32_lo(*reinterpret_cast<const float4*>(base + hi_off));
        };
#pragma unroll
        for (int j = 0; j < A_CH; ++j) residual(OFF_AHI + a_o[j], OFF_ALO + a_o[j]);
#pragma unroll
        for (int j = 0; j < B_CH; ++j)
          if (b_on[j]) residual(OFF_BHI + b_o[j], OFF_BLO + b_o[j]);
      }
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 2] = clock64();
      fence_async_smem();                                              // cp.async + generic stores -> async proxy (UMMA)
      __syncwarp();
      if (lane == 0) mbar_arrive(&full_bar[s]);                        // one arrival per producer warp
      if (++s == (uint32_t)ND) s = 0;
      if (tr_on && tr_n < 64) TM_TRACEPTR[tr_n * 4 + 3] = clock64();
      ++tr_n;
      ok = issue();                                                    // k-block g + D
    }
    cp_async_wait<0>();
  } else if (warp == MMA_WARP) {
    // ======================= MMA issuer =======================
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(Fmt::TF32, BN, AL::kTransposed, BL::kTransposed);
      // per MMA (K = 8): K-major advances 32 bytes inside the swizzle atom, MN-major two 512-byte k groups
      constexpr uint32_t A_KSTEP = AL::kTransposed ? 1024u : 32u, B_KSTEP = BL::kTransposed ? 1024u : 32u;
      constexpr uint32_t A_LBO = AL::kTransposed ? 4096u : 16u, B_LBO = BL::kTransposed ? 4096u : 16u;
      constexpr uint32_t A_SBO = AL::kTransposed ? 512u : 1024u, B_SBO = BL::kTransposed ? 512u : 1024u;
      constexpr uint32_t A_TY = AL::kTransposed ? 1u : 2u, B_TY = BL::kTransposed ? 1u : 2u;
      uint32_t s = 0, ph = 0;
      int li = 0;
      for (int64_t t = blockIdx.x; t < tm.total && ok; t += G, ++li) {
        const int buf = li & 1;
        const uint32_t aph = (uint32_t)(li >> 1) & 1u;
        ok = mbar_wait_abort(&acc_empty[buf], aph ^ 1u, abortp);               // epilogue drained this accumulator
        if (!ok) break;
        tc_fence_after();
        int64_t m0, nq, kb0; int zi, nkb;
        tm.decode(t, m0, nq, zi, kb0, nkb);
        const uint32_t tmem_d = tmem_base + (uint32_t)(buf * BN);
        for (int kb = 0; kb < nkb; ++kb) {
          const bool tr_on = TM_TRACEPTR && blockIdx.x == 0 && li == 0 && kb < 64;
          if (tr_on) TM_TRACEPTR[256 + kb * 4 + 0] = clock64();
          ok = mbar_wait_abort(&full_bar[s], ph, abortp);
          if (!ok) break;
          tc_fence_after();
          if (tr_on) TM_TRACEPTR[256 + kb * 4 + 1] = clock64();
          const uint32_t base = smem_u32(ring + (size_t)s * SLOT);
          if (!(TM_DBGBITS & 8))
#pragma unroll
          for (int ks = 0; ks < BK / 8; ++ks) {
            const uint64_t ah = smem_desc(base + OFF_AHI + ks * A_KSTEP, A_LBO, A_SBO, A_TY);
            const uint64_t bh = smem_desc(base + OFF_BHI + ks * B_KSTEP, B_LBO, B_SBO, B_TY);
            umma_tf32(tmem_d, ah, bh, idesc, (kb > 0 || ks > 0) ? 1u : 0u);
            if (PLANES == 2) {
              const uint64_t alo = smem_desc(base + OFF_ALO + ks * A_KSTEP, A_LBO, A_SBO, A_TY);
              const uint64_t blo = smem_desc(base + OFF_BLO + ks * B_KSTEP, B_LBO, B_SBO, B_TY);
              umma_tf32(tmem_d, ah, blo, idesc, 1u);
              umma_tf32(tmem_d, alo, bh, idesc, 1u);
            }
          }
          umma_commit(&empty_bar[s]);                                    // slot reusable once these MMAs retire
          if (tr_on) TM_TRACEPTR[256 + kb * 4 + 2] = clock64();
          if (++s == (uint32_t)ND) { s = 0; ph ^= 1u; }
        }
        if (!ok) break;
        umma_commit(&acc_full[buf]);                                     // covers every MMA of the tile
      }
    }
    __syncwarp();
  } else {
    // ======================= epilogue =======================
    float* scr = scratch + warp * (32 * 33);
    int li = 0;
    if constexpr (IsReduce<EP>::value) {
      float* racc = reduce_acc + warp * (2 * 3 * BN);              // [n tile][3][BN]
      for (int i = lane; i < 2 * 3 * BN; i += 32) racc[i] = 0.f;
      __syncwarp();
      for (int64_t t = blockIdx.x; t < tm.total && ok; t += G, ++li) {
        const int buf = li & 1;
        const uint32_t aph = (uint32_t)(li >> 1) & 1u;
        ok = mbar_wait_abort(&acc_full[buf], aph, abortp);
        if (!ok) break;
        tc_fence_after();
        int64_t m0, nq, kb0; int zi, nkb;
        tm.decode(t, m0, nq, zi, kb0, nkb);
        const int64_t n0 = nq * BN;
        const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * BN);
        // this lane's rows of the 8 passes: input values x0, x1 (0 for rows past M)
        float x0[8], x1[8];
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
          const int64_t m = m0 + warp * 32 + pass * 4 + (lane >> 3);
          x0[pass] = 0.f; x1[pass] = 0.f;
          if (m < M) {
            const float* xp = ep.X + (ep.x_rows ? (int64_t)ep.x_rows[m] : m) * ep.ldx;
            x0[pass] = xp[0];
            if (ep.kx > 1) x1[pass] = xp[1];
          }
        }
#pragma unroll 1
        for (int c = 0; c < BN; c += 32) {
          if (n0 + c >= N) break;
          float v[32];
          tmem_ld32(trow + (uint32_t)c, v);
#pragma unroll
          for (int i = 0; i < 32; ++i) scr[lane * 33 + i] = v[i];
          __syncwarp();
          const int cq = (lane & 7) * 4;
          const int64_t n = n0 + c + cq;
          float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            float4 mk[4];
            if (ep.mask) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {                               // mask rows first (loads in flight together)
                const int64_t m = m0 + warp * 32 + (half * 4 + q) * 4 + (lane >> 3);
                mk[q] = (m < M && n + 4 <= N) ? ld4(ep.mask + m * ep.ldmask + n) : make_float4(0.f, 0.f, 0.f, 0.f);
              }
            } else {                                                      // regenerate the pre-activations (Hidden2::pre)
              float w0[4], w1[4], bb[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const bool on = n + j < N;
                w0[j] = on ? __ldg(ep.W1 + (n + j) * ep.kx) : 0.f;
                w1[j] = (on && ep.kx > 1) ? __ldg(ep.W1 + (n + j) * ep.kx + 1) : 0.f;
                bb[j] = on ? __ldg(ep.b1 + n + j) : -1.f;
              }
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int pass = half * 4 + q;
                const int64_t m = m0 + warp * 32 + pass * 4 + (lane >> 3);
                const bool on = m < M;
                mk[q].x = on ? fmaf(w0[0], x0[pass], fmaf(w1[0], x1[pass], bb[0])) : 0.f;
                mk[q].y = on ? fmaf(w0[1], x0[pass], fmaf(w1[1], x1[pass], bb[1])) : 0.f;
                mk[q].z = on ? fmaf(w0[2], x0[pass], fmaf(w1[2], x1[pass], bb[2])) : 0.f;
                mk[q].w = on ? fmaf(w0[3], x0[pass], fmaf(w1[3], x1[pass], bb[3])) : 0.f;
              }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int pass = half * 4 + q, r = pass * 4 + (lane >> 3);
              const float mq[4] = {mk[q].x, mk[q].y, mk[q].z, mk[q].w};
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float d = mq[j] > 0.f ? scr[r * 33 + cq + j] : 0.f;
                s0[j] += d;
                s1[j] = fmaf(d, x0[pass], s1[j]);
                s2[j] = fmaf(d, x1[pass], s2[j]);
              }
            }
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {                                   // sum over the 4 row groups of the warp
            s0[j] += __shfl_xor_sync(0xffffffffu, s0[j], 8);  s0[j] += __shfl_xor_sync(0xffffffffu, s0[j], 16);
            s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], 8);  s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], 16);
            s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 8);  s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 16);
          }
          if (lane < 8 && nq < 2) {
            float* a = racc + (size_t)nq * 3 * BN + c + cq;
#pragma unroll
            for (int j = 0; j < 4; ++j) { a[j] += s0[j]; a[BN + j] += s1[j]; a[2 * BN + j] += s2[j]; }
          }
          __syncwarp();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[buf]);
      }
      __syncwarp();
      for (int i = lane; i < 2 * 3 * BN; i += 32) {                       // my partial sums -> global
        const int nqq = i / (3 * BN), k = (i / BN) % 3, col = i % BN;
        const int64_t n = (int64_t)nqq * BN + col;
        if (n < N) ep.part[(((int64_t)blockIdx.x * EPI_WARPS + warp) * 3 + k) * N + n] = racc[i];
      }
    } else
    for (int64_t t = blockIdx.x; t < tm.total && ok; t += G, ++li) {
      const int buf = li & 1;
      const uint32_t aph = (uint32_t)(li >> 1) & 1u;
      ok = mbar_wait_abort(&acc_full[buf], aph, abortp);
      if (!ok) break;
      tc_fence_after();
      int64_t m0, nq, kb0; int zi, nkb;
      tm.decode(t, m0, nq, zi, kb0, nkb);
      const int64_t n0 = nq * BN;
      const int64_t m = m0 + warp * 32 + lane;                            // this lane's row of the tile (TMEM lane)
      const bool live = m < M && !(TM_DBGBITS & 1);
      RowStore<EP> rs;
      rs.open(ep, m < M ? m : M - 1, zi, N);
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(buf * BN);
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        if (n0 + c >= N) break;
        float v[32];
        tmem_ld32(trow + (uint32_t)c, v);                                 // (warp-collective: every lane takes part)
        if (live) rs.chunk(ep, n0 + c, N, v);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
    }
  }
  if (!ok) {
    abort_s = 1;
    if (err) atomicExch(err, 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(tmem_base, C::TMEM_COLS);
}

// N tile: as wide as the accumulator / staging budget allows, so the A operand is staged once
inline int pick_bn(int64_t N, int precision) {
  if (precision >= 3) return N > 64 ? 128 : (N > 32 ? 64 : 32);
  if (N > 128 && precision != 2) return 256;
  return N > 64 ? 128 : (N > 32 ? 64 : 32);
}

template <class AL, class BL, class EP, int BN, int SPLIT>
int launch_one(const AL& al, const BL& bl, const EP& ep, int64_t M, int64_t N, int64_t K, int splits,
               int64_t k_per_split, int* err, cudaStream_t st) {
  auto kern = tc_gemm_kernel<AL, BL, EP, BN, SPLIT>;
  constexpr size_t sm = Cfg<BN, SPLIT>::SMEM;
  static bool optin = false;
  if (!optin) {
    TM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    optin = true;
  }
  TileMap tm;
  tm.nt = (int)cdiv(N, BN);
  tm.z = splits < 1 ? 1 : splits;
  tm.total = cdiv(M, BM) * tm.nt * tm.z;
  tm.K = K;
  tm.k_per_split = k_per_split;
  static const int dbg = getenv("TM_TC_DEBUG") ? atoi(getenv("TM_TC_DEBUG")) : 0;
  tm.dbg = dbg;
  tm.trace = nullptr;
  static const bool trace_on = getenv("TM_TC_TRACE") != nullptr;
  static long long* trace_buf = nullptr;
  if (trace_on) {
    if (!trace_buf) cudaMalloc(&trace_buf, 1024 * sizeof(long long));
    cudaMemsetAsync(trace_buf, 0, 1024 * sizeof(long long), st);
    tm.trace = trace_buf;
  }
  const int64_t grid = tm.total < sm_count() ? tm.total : sm_count();
  kern<<<(unsigned)grid, THREADS, sm, st>>>(al, bl, ep, M, N, tm, err);
  if (trace_on) {
    static long long h[1024];
    cudaStreamSynchronize(st);
    cudaMemcpy(h, trace_buf, sizeof(h), cudaMemcpyDeviceToHost);
    long long t0 = h[0];
    fprintf(stderr, "[tc trace] BN=%d SPLIT=%d NS=%d tiles=%lld grid=%lld\n", BN, SPLIT, Cfg<BN, SPLIT>::NS, (long long)tm.total, (long long)grid);
    for (int i = 0; i < 40; ++i)
      fprintf(stderr, "  prod %2d: start %7lld  got-empty %7lld  stored %7lld  arrived %7lld | mma: wait %7lld full %7lld issued %7lld\n", i,
              h[i * 4] - t0, h[i * 4 + 1] - t0, h[i * 4 + 2] - t0, h[i * 4 + 3] - t0, h[256 + i * 4] - t0, h[256 + i * 4 + 1] - t0,
              h[256 + i * 4 + 2] - t0);
    for (int i = 0; i < 6; ++i)
      fprintf(stderr, "  epi %2d: wait %7lld full %7lld done %7lld\n", i, h[512 + i * 4] - t0, h[512 + i * 4 + 1] - t0, h[512 + i * 4 + 2] - t0);
  }
  return check_launch("tc_gemm");
}

inline int& tc_grid_cap() {
  static thread_local int cap = 0;
  return cap;
}

template <class AL, class BL, class EP, int BN, int PLANES>
int launch_tf(const AL& al, const BL& bl, const EP& ep, int64_t M, int64_t N, int64_t K, int splits,
              int64_t k_per_split, int* err, cudaStream_t st) {
  auto kern = tf_gemm_kernel<AL, BL, EP, BN, PLANES>;
  constexpr size_t sm = TfCfg<BN, PLANES>::SMEM + (IsReduce<EP>::value ? REDUCE_ACC_BYTES : 0);
  static bool optin = false;
  if (!optin) {
    TM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    optin = true;
  }
  TileMap tm;
  tm.nt = (int)cdiv(N, BN);
  tm.z = splits < 1 ? 1 : splits;
  tm.total = cdiv(M, BM) * tm.nt * tm.z;
  tm.K = K;
  tm.k_per_split = k_per_split;
  static const int dbg = getenv("TM_TC_DEBUG") ? atoi(getenv("TM_TC_DEBUG")) : 0;
  tm.dbg = dbg;
  tm.trace = nullptr;
  static const bool trace_on = getenv("TM_TC_TRACE") != nullptr;
  static long long* trace_buf = nullptr;
  if (trace_on) {
    if (!trace_buf) cudaMalloc(&trace_buf, 1024 * sizeof(long long));
    cudaMemsetAsync(trace_buf, 0, 1024 * sizeof(long long), st);
    tm.trace = trace_buf;
  }
  // tm_tc_set_grid_cap(n): at most n persistent CTAs for the launches of the calling thread (0 = one per SM) -- lets
  // a caller keep SMs free for a latency-critical kernel chain on another stream
  int64_t lim = sm_count();
  if (!IsReduce<EP>::value && tc_grid_cap() > 0 && tc_grid_cap() < lim) lim = tc_grid_cap();
  const int64_t grid = tm.total < lim ? tm.total : lim;
  kern<<<(unsigned)grid, TF_THREADS, sm, st>>>(al, bl, ep, M, N, tm, err);
  if (trace_on) {
    static long long h[1024];
    cudaStreamSynchronize(st);
    cudaMemcpy(h, trace_buf, sizeof(h), cudaMemcpyDeviceToHost);
    long long t0 = h[0];
    fprintf(stderr, "[tf trace] BN=%d PLANES=%d ND=%d tiles=%lld grid=%lld\n", BN, PLANES, TfCfg<BN, PLANES>::ND, (long long)tm.total, (long long)grid);
    for (int i = 0; i < 40; ++i)
      fprintf(stderr, "  prod %2d: start %7lld  landed %7lld  lo-done %7lld  arrived %7lld | mma: wait %7lld full %7lld issued %7lld\n", i,
              h[i * 4] - t0, h[i * 4 + 1] - t0, h[i * 4 + 2] - t0, h[i * 4 + 3] - t0, h[256 + i * 4] - t0, h[256 + i * 4 + 1] - t0,
              h[256 + i * 4 + 2] - t0);
  }
  return check_launch("tf_gemm");
}

template <class AL, class BL, class EP>
int launch(const AL& al, const BL& bl, const EP& ep, int64_t M, int64_t N, int64_t K, int splits,
           int64_t k_per_split, int precision, int* err, cudaStream_t st) {
  if (M <= 0 || N <= 0) return 0;
  const int bn = pick_bn(N, precision);
  if (precision >= 3) {
#define TM_TF_CASE(BN_)                                                                                  \
  return precision == 3 ? launch_tf<AL, BL, EP, BN_, 2>(al, bl, ep, M, N, K, splits, k_per_split, err, st) \
                        : launch_tf<AL, BL, EP, BN_, 1>(al, bl, ep, M, N, K, splits, k_per_split, err, st)
    switch (bn) {
      case 128: TM_TF_CASE(128);
      case 64: TM_TF_CASE(64);
      default: TM_TF_CASE(32);
    }
#undef TM_TF_CASE
  }
#define TM_TC_CASE(BN_)                                                                                 \
  return precision == 2   ? launch_one<AL, BL, EP, BN_, 6>(al, bl, ep, M, N, K, splits, k_per_split, err, st) \
         : precision == 1 ? launch_one<AL, BL, EP, BN_, 3>(al, bl, ep, M, N, K, splits, k_per_split, err, st) \
                          : launch_one<AL, BL, EP, BN_, 1>(al, bl, ep, M, N, K, splits, k_per_split, err, st)
  switch (bn) {
    case 256:
      return precision == 1 ? launch_one<AL, BL, EP, 256, 3>(al, bl, ep, M, N, K, splits, k_per_split, err, st)
                            : launch_one<AL, BL, EP, 256, 1>(al, bl, ep, M, N, K, splits, k_per_split, err, st);
    case 128: TM_TC_CASE(128);
    case 64: TM_TC_CASE(64);
    default: TM_TC_CASE(32);
  }
#undef TM_TC_CASE
}

// Y[m][0:N] (row stride ldy) = act(bias + sum_z P[z][m][0:N]): folds the fp32 partials of a K-split convolution in a
// fixed order (deterministic); N % 4 == 0.
int conv_split_fold(const float* part, int64_t M, int64_t N, int splits, const float* bias, int relu, float* y, int64_t ldy,
                    cudaStream_t st);

}  // namespace tc
}  // namespace tmk
