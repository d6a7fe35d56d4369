// G2/G3: level-wise timing propagation, forward and backward.
//
// Replaces PathConv.forward and its UDFs (src/model.py:88-116,138-153,158-213), which the reference
// runs as one DGL `pull` + several cuBLAS calls + a full (N,128) index_copy PER LEVEL, and the
// autograd backward through them (src/train.py:553).
//
// Data layout (HBM): H, S, G are [N][128] fp32 row-major indexed by pin id (one pin = one 512 B
// row = four full 128 B lines, so scattered rows still move at full sector efficiency); the
// buffers saved for backward (A, LSE, HID, GA, GHID, GZC) are compact [n_cell_rows][...] in
// schedule order, so each cell level owns a contiguous slab.
//
// Level schedule: pins sorted by (level, id); level l occupies order[level_ptr[l]..level_ptr[l+1]).
//   level 0        h[v] = relu(S[v])                                   (model.py:148-153,200-208)
//   odd  level     h[v] = relu(S[v] + mean_{u->v in net} h[u])         (model.py:103-108,186-187)
//   even level >0  a = sum_e m_e * softmax_e(m)_e (per channel), m_e = h[src e]   (model.py:113-116)
//                  h[v] = relu(S[v] + W2 relu(W1 a + b1) + b2)         (model.py:138-146)
// A warp owns a pin (lane = 4 channels, 128-bit loads); cell levels are processed in 16-pin tiles:
// the aggregated rows are staged in shared memory and pushed through the 128->256->128 MLP by the
// same CTA, so `a` and the hidden layer never round-trip through HBM on the forward critical path.
#include <cuda_fp16.h>
#include <stdlib.h>

#include "tm_common.cuh"
#include "tm_sm100.cuh"
#include "tm_split.cuh"

using namespace tmk;
using namespace tmk::sm100;

namespace {
constexpr int D = 128;     // out_feat_dim (model.py:43, options.py:10)
constexpr int HID = 256;   // MLP hidden width (model.py:48)
constexpr int TILE = 16;   // pins per CTA on a cell level
constexpr int CT = 256;    // threads per CTA on a cell level (8 warps: two per scheduler hide the ALU latency)

// Programmatic dependent launch: consecutive level kernels are chained so that a kernel's CTAs may
// start while the previous level is still running -- everything that does not read the previous
// level's output (weight-chunk prefetch, schedule lookups) overlaps it; pdl_wait() then blocks until
// the previous grid has completed and its writes are visible.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// forward, level 0 and odd (net) levels: one warp per pin
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gnn_net_fwd_kernel(const int* __restrict__ order, int p0, int cnt, const int* __restrict__ f_ptr,
                   const int* __restrict__ f_src, const float* __restrict__ S, float* H) {
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  pdl_launch_dependents();
  if (w >= cnt) { pdl_wait(); return; }
  const int p = p0 + w;
  const int v = order[p];
  const int s = f_ptr[p], e = f_ptr[p + 1];          // level 0: empty range
  const float4 sv = ld4_stream(S + (int64_t)v * D + lane * 4);
  pdl_wait();                                        // H rows of earlier levels are read from here on
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i = s; i < e; i += 4) {
    float4 m[4];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      m[q] = (i + q < e) ? ld4(H + (int64_t)f_src[i + q] * D + lane * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int q = 0; q < 4; ++q) acc = f4add(acc, m[q]);
  }
  if (e > s) acc = f4scale(acc, 1.f / (float)(e - s));
  st4(H + (int64_t)v * D + lane * 4, f4relu(f4add(sv, acc)));
}

// ---------------------------------------------------------------------------------------------
// tile MLP shared by forward and backward: out = (epi1(in @ Wa)) @ Wb for a 16-row tile,
//   Wa: [128][256] (k-major), Wb: [256][128].
// A level holds only a few thousand pins and the next level needs all of them, so the tile is 16
// rows and every SM gets one: the MLP runs on the warp-level tensor-core path (mma.sync m16n8k8,
// whose M = 16 is exactly the tile; tcgen05's M >= 64 would idle 3/4 of every instruction here) in
// 3xTF32: x = hi + lo with hi = x rounded to 11 bits, lo = x - hi (exact); lo*hi + hi*lo + hi*hi
// accumulated in fp32 keeps ~22 mantissa bits per product -- the fp32-class accuracy the 101-level
// recurrence needs.
//   * weights: re-packed once per call (gnn_pack_kernel) into padded rows, so the 256 KB stream
//     through shared memory as 16 contiguous chunks moved by ONE cp.async.bulk each.  The stream is
//     latency-bound (every CTA pulls the same lines out of L2), so the ring is 8 slots deep: all of
//     Wa is requested at kernel entry and lands while the tile is being gathered; Wb chunks follow
//     into the slots GEMM1 frees.  (Pre-splitting the weights into hi/lo rows would double this
//     L2 traffic -- 32 MB per level for config 2 -- for a few ALU ops per fragment; measured slower.)
//     B fragments are conflict-free LDS + an on-the-fly split;
//   * tiles: the input / hidden tiles are stored pre-split (hi and lo arrays), so A fragments are
//     plain LDS as well and every element is split exactly once.
// 256 threads = 8 warps; warp w owns hidden columns 32w..32w+31 in GEMM1 and output columns
// 16w..16w+15 in GEMM2.
// ---------------------------------------------------------------------------------------------
constexpr int NSTAGE = 8;
constexpr int NCHUNK = 16;
constexpr int IN_LD = D + 4;      // 132: bank(g*132 + t) = 4g + t   -> conflict-free A fragments
constexpr int MID_LD = HID + 4;   // 260
constexpr int WA_ROW = HID + 8;   // 264 floats per packed k-row of Wa: bank(t*264 + g) = 8t + g -> conflict-free B fragments
constexpr int WB_ROW = D + 8;     // 136
constexpr int CHUNK_A = 16 * WA_ROW;    // floats per chunk of Wa (16 k-rows)  = 4224
constexpr int CHUNK_B = 32 * WB_ROW;    // floats per chunk of Wb (32 k-rows)  = 4352
constexpr int SLOT = CHUNK_B > CHUNK_A ? CHUNK_B : CHUNK_A;
constexpr size_t PACK_FLOATS = (size_t)D * WA_ROW + (size_t)HID * WB_ROW;   // one (Wa, Wb) pair
constexpr int TILE_FLOATS = 3 * TILE * IN_LD + 2 * TILE * MID_LD;
constexpr int IN_LDH = D / 2 + 4;     // 68 half2 words per row:  bank(g*68 + t) = 4g + t  -> conflict-free A fragments (m16n8k16)
constexpr int MID_LDH = HID / 2 + 4;  // 132
static_assert(TILE * MID_LD + 2 * TILE * IN_LDH + 2 * TILE * MID_LDH + 2 * TILE <= 2 * TILE * IN_LD + 2 * TILE * MID_LD,
              "the fp16-split tiles must fit the area of the fp32 hi / lo tiles");
constexpr size_t CELL_SMEM = (size_t)(TILE_FLOATS + NSTAGE * SLOT) * sizeof(float) + TILE * sizeof(int) + 64;

struct Tiles {                    // shared-memory carve-up of one CTA
  float* scr;                     // [TILE][IN_LD]  fp32 scratch / raw GEMM2 output
  float* in_hi;                   // [TILE][IN_LD]
  float* in_lo;
  float* mid_hi;                  // [TILE][MID_LD]
  float* mid_lo;
  float* wbuf;                    // NSTAGE x SLOT
  int* v_s;                       // [TILE]
  uint64_t* wfull;                // [NSTAGE] mbarriers
  // fp16-split variant (H16): the same area behind scr holds the fp32 hidden tile, the half2 (hi, lo') planes of the
  // input / hidden tiles and the per-pin scales instead of the four fp32 hi / lo tiles
  float* hid_f;                   // [TILE][MID_LD] fp32 hidden (unscaled: what the backward needs)
  uint32_t* ah_hi;                // [TILE][IN_LDH] half2 words, k pairs
  uint32_t* ah_lo;
  uint32_t* mh_hi;                // [TILE][MID_LDH]
  uint32_t* mh_lo;
  float* sc_s;                    // [TILE] scale, [TILE] 1/scale
  float* inv_s;
  __device__ explicit Tiles(float* smem) {
    scr = smem;
    in_hi = scr + TILE * IN_LD;
    in_lo = in_hi + TILE * IN_LD;
    mid_hi = in_lo + TILE * IN_LD;
    mid_lo = mid_hi + TILE * MID_LD;
    hid_f = in_hi;
    ah_hi = reinterpret_cast<uint32_t*>(hid_f + TILE * MID_LD);
    ah_lo = ah_hi + TILE * IN_LDH;
    mh_hi = ah_lo + TILE * IN_LDH;
    mh_lo = mh_hi + TILE * MID_LDH;
    sc_s = reinterpret_cast<float*>(mh_lo + TILE * MID_LDH);
    inv_s = sc_s + TILE;
    wbuf = mid_lo + TILE * MID_LD;
    v_s = reinterpret_cast<int*>(wbuf + NSTAGE * SLOT);
    wfull = reinterpret_cast<uint64_t*>(v_s + TILE);
  }
};

// hi = x rounded to 11 significant bits (round half away: add half an ulp_tf32, clear the low 13
// bits -- two integer ops; cvt.rna.tf32 expands to a much longer sequence), lo = x - hi (exact)
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
  hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
  lo = x - hi;
}
__device__ __forceinline__ void split4(float4 x, float4& hi, float4& lo) {
  split_tf32(x.x, hi.x, lo.x); split_tf32(x.y, hi.y, lo.y); split_tf32(x.z, hi.z, lo.z); split_tf32(x.w, hi.w, lo.w);
}

// src [R][C] row-major -> dst [R][C + 8] (row padding only)
__global__ void gnn_pack_kernel(const float* __restrict__ src, int R, int C, float* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R * (C + 8)) return;
  const int r = i / (C + 8), c = i - r * (C + 8);
  dst[i] = (c < C) ? src[(size_t)r * C + c] : 0.f;
}

// one elected thread: chunk c of the packed weights -> ring slot c % NSTAGE, completion on wfull
__device__ __forceinline__ void issue_chunk(const Tiles& T, const float* __restrict__ Wa,
                                            const float* __restrict__ Wb, int c) {
  if (c >= NCHUNK) return;
  const float* src = (c < 8) ? Wa + (size_t)c * CHUNK_A : Wb + (size_t)(c - 8) * CHUNK_B;
  const uint32_t bytes = (uint32_t)((c < 8 ? CHUNK_A : CHUNK_B) * sizeof(float));
  mbar_expect_tx(&T.wfull[c % NSTAGE], bytes);
  bulk_copy_g2s(smem_u32(T.wbuf + (c % NSTAGE) * SLOT), src, bytes, &T.wfull[c % NSTAGE]);
}
// A lost bulk copy traps after 2^24 probes.  Unlike mbar_wait_trap, the bound is tested before the exit: with
// mbar_wait_trap's order the compiler reschedules the cell kernels, and the config-2 design step measured 1% slower
// (one B200 at 1000 W).
__device__ __forceinline__ void wait_chunk(const Tiles& T, int c) {
  const uint32_t bar = smem_u32(&T.wfull[c % NSTAGE]), parity = (uint32_t)(c / NSTAGE) & 1u;
  bool done = false;
  for (uint32_t spin = 0; !done; ++spin) {
    done = mbar_try_wait(bar, parity);
    if (spin > (1u << 24)) __trap();
  }
}

// Call order inside a kernel:  mlp_prologue() -> fill in_hi / in_lo -> mlp_tile()
__device__ __forceinline__ void mlp_prologue(const Tiles& T, const float* Wa, const float* Wb, int tid) {
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < NSTAGE; ++i) mbar_init(&T.wfull[i], 1);
    fence_mbarrier_init();
    fence_async_smem();
#pragma unroll
    for (int c = 0; c < NSTAGE - 1; ++c) issue_chunk(T, Wa, Wb, c);
  }
}

__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// one k-step (8) of a 16 x (8*NT) product: A fragments from the pre-split tile, B from a packed chunk
template <int NT>
__device__ __forceinline__ void mma_kstep(float (&acc)[NT][4], const float* a_hi, const float* a_lo, int a_ld, int ka,
                                          const float* w, int w_row, int kw, int n_base, int g, int t) {
  uint32_t ah[4], al[4];
  const int i0 = g * a_ld + ka + t, i1 = (g + 8) * a_ld + ka + t;
  ah[0] = __float_as_uint(a_hi[i0]); ah[1] = __float_as_uint(a_hi[i1]);
  ah[2] = __float_as_uint(a_hi[i0 + 4]); ah[3] = __float_as_uint(a_hi[i1 + 4]);
  al[0] = __float_as_uint(a_lo[i0]); al[1] = __float_as_uint(a_lo[i1]);
  al[2] = __float_as_uint(a_lo[i0 + 4]); al[3] = __float_as_uint(a_lo[i1 + 4]);
  const float* w0 = w + (kw + t) * w_row + n_base + g;
  const float* w1 = w0 + 4 * w_row;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    float h0, l0, h1, l1;
    split_tf32(w0[j * 8], h0, l0);
    split_tf32(w1[j * 8], h1, l1);
    const uint32_t bh0 = __float_as_uint(h0), bh1 = __float_as_uint(h1), bl0 = __float_as_uint(l0), bl1 = __float_as_uint(l1);
    mma_tf32(acc[j], al, bh0, bh1);        // small terms first
    mma_tf32(acc[j], ah, bl0, bl1);
    mma_tf32(acc[j], ah, bh0, bh1);
  }
}

// T.in_hi/in_lo: the pre-split input tile; T.mid_hi/mid_lo receive epi1 of the first product
// (epi1(row, col, v0, v1) -> float2 for columns col, col+1); T.scr receives the raw second product.
// Ends with a __syncthreads(): mid and scr are complete and visible to the whole CTA.
template <class Epi1>
__device__ __forceinline__ void mlp_tile(const Tiles& T, const float* Wa, const float* Wb, int tid, Epi1 epi1) {
  const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  constexpr int NT1 = HID / 8 / (CT / 32), NT2 = D / 8 / (CT / 32);   // n-tiles per warp: 4 and 2
  float acc1[NT1][4], acc2[NT2][4];
#pragma unroll
  for (int j = 0; j < NT1; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc1[j][c] = 0.f;
#pragma unroll
  for (int j = 0; j < NT2; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc2[j][c] = 0.f;

  for (int c = 0; c < NCHUNK; ++c) {
    __syncthreads();                      // everybody is done with chunk c-1 (its slot is free); tiles visible
    if (tid == 0) issue_chunk(T, Wa, Wb, c + NSTAGE - 1);
    wait_chunk(T, c);
    const float* w = T.wbuf + (c % NSTAGE) * SLOT;
    if (c < 8) {                          // GEMM1: k rows 16c .. 16c+15 of Wa
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        mma_kstep<NT1>(acc1, T.in_hi, T.in_lo, IN_LD, c * 16 + ks * 8, w, WA_ROW, ks * 8, warp * NT1 * 8, g, t);
      if (c == 7) {
#pragma unroll
        for (int j = 0; j < NT1; ++j) {
          const int col = warp * NT1 * 8 + j * 8 + 2 * t;
          float2 h0, l0, h1, l1;
          const float2 e0 = epi1(g, col, acc1[j][0], acc1[j][1]), e1 = epi1(g + 8, col, acc1[j][2], acc1[j][3]);
          split_tf32(e0.x, h0.x, l0.x); split_tf32(e0.y, h0.y, l0.y);
          split_tf32(e1.x, h1.x, l1.x); split_tf32(e1.y, h1.y, l1.y);
          *reinterpret_cast<float2*>(&T.mid_hi[g * MID_LD + col]) = h0;
          *reinterpret_cast<float2*>(&T.mid_lo[g * MID_LD + col]) = l0;
          *reinterpret_cast<float2*>(&T.mid_hi[(g + 8) * MID_LD + col]) = h1;
          *reinterpret_cast<float2*>(&T.mid_lo[(g + 8) * MID_LD + col]) = l1;
        }
      }
    } else {                              // GEMM2: k rows 32(c-8) .. +31 of Wb
#pragma unroll
      for (int ks = 0; ks < 4; ++ks)
        mma_kstep<NT2>(acc2, T.mid_hi, T.mid_lo, MID_LD, (c - 8) * 32 + ks * 8, w, WB_ROW, ks * 8, warp * NT2 * 8, g, t);
    }
  }
#pragma unroll
  for (int j = 0; j < NT2; ++j) {
    const int col = warp * NT2 * 8 + j * 8 + 2 * t;
    *reinterpret_cast<float2*>(&T.scr[g * IN_LD + col]) = make_float2(acc2[j][0], acc2[j][1]);
    *reinterpret_cast<float2*>(&T.scr[(g + 8) * IN_LD + col]) = make_float2(acc2[j][2], acc2[j][3]);
  }
  __syncthreads();
}

// =============================================================================================
// fp16 two-term split variant of the tile MLP (TM_GNN_CELL_MATH=h16, round 2): the split of tm_split.cuh, per-pin scale,
// on mma.sync.m16n8k16 (f16 operands, fp32 accumulate): 3 tensor instructions per k16 step and n-tile instead of the 6 of
// 3xTF32 (m16n8k8), and the operand fragments are single 32-bit shared-memory words (half2 k-pairs), no on-the-fly split.
// The weights are packed ONCE per call into the same chunk geometry as the fp32 path (so the cp.async.bulk ring is
// unchanged): chunk c < 8 = k16 step c of Wa as [plane hi | lo'][8 k-pairs][264 words], chunk 8 + c = two k16 steps of
// Wb as [plane][16 k-pairs][136 words].
// =============================================================================================
// one tile row (this lane: channels 4 lane .. 4 lane + 3) -> scale, split, half2 planes
__device__ __forceinline__ void store_row_h(const Tiles& T, int row, int lane, float4 x, int emin) {
  const float rm = warp_max(fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
  float sc, inv;
  row_scale(rm, emin, sc, inv);
  __half h0, h1, h2, h3, l0, l1, l2, l3;
  split_h(x.x * sc, h0, l0); split_h(x.y * sc, h1, l1); split_h(x.z * sc, h2, l2); split_h(x.w * sc, h3, l3);
  *reinterpret_cast<uint2*>(&T.ah_hi[row * IN_LDH + 2 * lane]) = make_uint2(pack_h2(h0, h1), pack_h2(h2, h3));
  *reinterpret_cast<uint2*>(&T.ah_lo[row * IN_LDH + 2 * lane]) = make_uint2(pack_h2(l0, l1), pack_h2(l2, l3));
  if (lane == 0) { T.sc_s[row] = sc; T.inv_s[row] = inv; }
}
// (Wa [128][256], Wb [256][128]) fp32 -> the chunked half2 planes described above.  One thread per (k pair, n).
__global__ void gnn_pack_h_kernel(const float* __restrict__ Wa, const float* __restrict__ Wb, uint32_t* __restrict__ dst) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (D / 2) * HID) {                                   // Wa: k pair kq < 64, n < 256
    const int kq = i / HID, n = i - kq * HID;
    __half h0, l0, h1, l1;
    split_h(Wa[(size_t)(2 * kq) * HID + n], h0, l0);
    split_h(Wa[(size_t)(2 * kq + 1) * HID + n], h1, l1);
    uint32_t* c = dst + (size_t)(kq >> 3) * CHUNK_A + (kq & 7) * WA_ROW + n;
    c[0] = pack_h2(h0, h1);
    c[8 * WA_ROW] = pack_h2(l0, l1);
  } else if (i < (D / 2) * HID + (HID / 2) * D) {            // Wb: k pair kq < 128, n < 128
    const int j = i - (D / 2) * HID;
    const int kq = j / D, n = j - kq * D;
    __half h0, l0, h1, l1;
    split_h(Wb[(size_t)(2 * kq) * D + n], h0, l0);
    split_h(Wb[(size_t)(2 * kq + 1) * D + n], h1, l1);
    uint32_t* c = dst + (size_t)8 * CHUNK_A + (size_t)(kq >> 4) * CHUNK_B + (kq & 15) * WB_ROW + n;
    c[0] = pack_h2(h0, h1);
    c[16 * WB_ROW] = pack_h2(l0, l1);
  }
}
__device__ __forceinline__ void mma_f16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// one k16 step of a 16 x (8*NT) product: A words from the tile planes (row stride a_ld words, k-pair offset kp0),
// B words from a chunk's planes (w_hi / w_lo, k-pair row kpw0, row stride w_row words)
template <int NT>
__device__ __forceinline__ void mma_kstep_h(float (&am)[NT][4], float (&ac)[NT][4], const uint32_t* a_hi, const uint32_t* a_lo,
                                            int a_ld, int kp0, const uint32_t* w_hi, const uint32_t* w_lo, int w_row, int kpw0,
                                            int n_base, int g, int t) {
  uint32_t ah[4], al[4];
  const int i0 = g * a_ld + kp0 + t, i1 = (g + 8) * a_ld + kp0 + t;
  ah[0] = a_hi[i0]; ah[1] = a_hi[i1]; ah[2] = a_hi[i0 + 4]; ah[3] = a_hi[i1 + 4];
  al[0] = a_lo[i0]; al[1] = a_lo[i1]; al[2] = a_lo[i0 + 4]; al[3] = a_lo[i1 + 4];
  const int o0 = (kpw0 + t) * w_row + n_base + g, o1 = o0 + 4 * w_row;
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const uint32_t bh0 = w_hi[o0 + j * 8], bh1 = w_hi[o1 + j * 8], bl0 = w_lo[o0 + j * 8], bl1 = w_lo[o1 + j * 8];
    mma_f16(ac[j], al, bh0, bh1);          // small terms
    mma_f16(ac[j], ah, bl0, bl1);
    mma_f16(am[j], ah, bh0, bh1);
  }
}
// The fp16-split tile MLP.  T.ah_hi / ah_lo: the scaled, split input tile (store_row_h); epi1(row, col, v0, v1) maps the
// first product's (still scaled) values of columns col, col+1 to the scaled hidden values; T.hid_f receives the UNSCALED
// hidden tile, T.scr the unscaled second product.  Ends with a __syncthreads().
template <class Epi1>
__device__ __forceinline__ void mlp_tile_h(const Tiles& T, const float* Wa, const float* Wb, int tid, Epi1 epi1) {
  const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  constexpr int NT1 = HID / 8 / (CT / 32), NT2 = D / 8 / (CT / 32);   // n-tiles per warp: 4 and 2
  float m1[NT1][4], c1[NT1][4], m2[NT2][4], c2[NT2][4];
#pragma unroll
  for (int j = 0; j < NT1; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) { m1[j][c] = 0.f; c1[j][c] = 0.f; }
#pragma unroll
  for (int j = 0; j < NT2; ++j)
#pragma unroll
    for (int c = 0; c < 4; ++c) { m2[j][c] = 0.f; c2[j][c] = 0.f; }
  for (int c = 0; c < NCHUNK; ++c) {
    __syncthreads();                      // everybody is done with chunk c-1 (its slot is free); tiles visible
    if (tid == 0) issue_chunk(T, Wa, Wb, c + NSTAGE - 1);         // (one barrier per TWO chunks measured the same: not kept)
    wait_chunk(T, c);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(T.wbuf + (c % NSTAGE) * SLOT);
    if (c < 8) {                          // GEMM1: k16 step c of Wa
      mma_kstep_h<NT1>(m1, c1, T.ah_hi, T.ah_lo, IN_LDH, c * 8, w, w + 8 * WA_ROW, WA_ROW, 0, warp * NT1 * 8, g, t);
      if (c == 7) {
#pragma unroll
        for (int j = 0; j < NT1; ++j) {
          const int col = warp * NT1 * 8 + j * 8 + 2 * t;
          const float2 e0 = epi1(g, col, fmaf(c1[j][0], LO_INV, m1[j][0]), fmaf(c1[j][1], LO_INV, m1[j][1]));
          const float2 e1 = epi1(g + 8, col, fmaf(c1[j][2], LO_INV, m1[j][2]), fmaf(c1[j][3], LO_INV, m1[j][3]));
          const float i0 = T.inv_s[g], i1 = T.inv_s[g + 8];
          *reinterpret_cast<float2*>(&T.hid_f[g * MID_LD + col]) = make_float2(e0.x * i0, e0.y * i0);
          *reinterpret_cast<float2*>(&T.hid_f[(g + 8) * MID_LD + col]) = make_float2(e1.x * i1, e1.y * i1);
          __half h0, l0, h1, l1;
          split_h(e0.x, h0, l0); split_h(e0.y, h1, l1);
          T.mh_hi[g * MID_LDH + (col >> 1)] = pack_h2(h0, h1);
          T.mh_lo[g * MID_LDH + (col >> 1)] = pack_h2(l0, l1);
          split_h(e1.x, h0, l0); split_h(e1.y, h1, l1);
          T.mh_hi[(g + 8) * MID_LDH + (col >> 1)] = pack_h2(h0, h1);
          T.mh_lo[(g + 8) * MID_LDH + (col >> 1)] = pack_h2(l0, l1);
        }
      }
    } else {                              // GEMM2: two k16 steps of Wb
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
        mma_kstep_h<NT2>(m2, c2, T.mh_hi, T.mh_lo, MID_LDH, (c - 8) * 16 + ks * 8, w, w + 16 * WB_ROW, WB_ROW, ks * 8,
                         warp * NT2 * 8, g, t);
    }
  }
#pragma unroll
  for (int j = 0; j < NT2; ++j) {
    const int col = warp * NT2 * 8 + j * 8 + 2 * t;
    const float i0 = T.inv_s[g], i1 = T.inv_s[g + 8];
    *reinterpret_cast<float2*>(&T.scr[g * IN_LD + col]) =
        make_float2(fmaf(c2[j][0], LO_INV, m2[j][0]) * i0, fmaf(c2[j][1], LO_INV, m2[j][1]) * i0);
    *reinterpret_cast<float2*>(&T.scr[(g + 8) * IN_LD + col]) =
        make_float2(fmaf(c2[j][2], LO_INV, m2[j][2]) * i1, fmaf(c2[j][3], LO_INV, m2[j][3]) * i1);
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// forward, even level > 0: gather + per-channel softmax-weighted sum + MLP, 16 pins per CTA
// ---------------------------------------------------------------------------------------------
template <bool H16>
__global__ void __launch_bounds__(CT)
gnn_cell_fwd_kernel(const int* __restrict__ order, int p0, int cnt, int crow0,
                    const int* __restrict__ f_ptr, const int* __restrict__ f_src,
                    const float* __restrict__ S, float* H, const float* __restrict__ W1t,
                    const float* __restrict__ b1, const float* __restrict__ W2t,
                    const float* __restrict__ b2, float* __restrict__ A, float* __restrict__ LSE,
                    float* __restrict__ HIDb) {
  extern __shared__ __align__(16) float smem[];
  const Tiles T(smem);
  int* v_s = T.v_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t0 = blockIdx.x * TILE;
  mlp_prologue(T, W1t, W2t, tid);
  pdl_wait();                                        // (the weight prefetch above overlaps the previous level)

  // phase 1: each warp aggregates PPW consecutive pins.  Their in-edges are one contiguous range of
  // the level-ordered edge list, walked once with warp-uniform pin boundaries; eight source rows
  // are in flight per step (online softmax per channel, lane = 4 channels).
  constexpr int PPW = TILE / (CT / 32);
  {
    const int r0 = warp * PPW;
    const int npin = min(PPW, cnt - (t0 + r0));                  // may be <= 0 on the tail tile
    const int pb = p0 + t0 + r0;
    int ptrs = 0, vv = -1;
    if (npin > 0) {
      if (lane <= npin) ptrs = f_ptr[pb + lane];
      if (lane < npin) vv = order[pb + lane];
    }
    if (lane < PPW) v_s[r0 + lane] = vv;
    int q = 0;
    float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    float sm[4] = {0.f, 0.f, 0.f, 0.f}, tw[4] = {0.f, 0.f, 0.f, 0.f};
    auto finish_pin = [&]() {                                    // writes pin q, resets the state
      float4 av = make_float4(0.f, 0.f, 0.f, 0.f), lse = av;
      if (sm[0] > 0.f) {                                         // at least one in-edge
        av = make_float4(tw[0] / sm[0], tw[1] / sm[1], tw[2] / sm[2], tw[3] / sm[3]);
        lse = make_float4(mx[0] + logf(sm[0]), mx[1] + logf(sm[1]), mx[2] + logf(sm[2]), mx[3] + logf(sm[3]));
      }
      if constexpr (H16) {
        store_row_h(T, r0 + q, lane, av, -4);
      } else {
        float4 avh, avl;
        split4(av, avh, avl);
        *reinterpret_cast<float4*>(&T.in_hi[(r0 + q) * IN_LD + lane * 4]) = avh;
        *reinterpret_cast<float4*>(&T.in_lo[(r0 + q) * IN_LD + lane * 4]) = avl;
      }
      if (A) {
        st4(A + (int64_t)(crow0 + t0 + r0 + q) * D + lane * 4, av);
        st4(LSE + (int64_t)(crow0 + t0 + r0 + q) * D + lane * 4, lse);
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) { mx[c] = -INFINITY; sm[c] = 0.f; tw[c] = 0.f; }
      ++q;
    };
    if (npin > 0) {
      const int E0 = __shfl_sync(0xffffffffu, ptrs, 0), E1 = __shfl_sync(0xffffffffu, ptrs, npin);
      int bnd = __shfl_sync(0xffffffffu, ptrs, 1);               // end of pin q's range
      for (int i = E0; i < E1; i += 8) {
        const int idx = (i + (lane & 7) < E1) ? f_src[i + (lane & 7)] : 0;
        float4 m[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int src = __shfl_sync(0xffffffffu, idx, u);
          if (i + u < E1) m[u] = ld4(H + (int64_t)src * D + lane * 4);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (i + u < E1) {
            while (i + u >= bnd) { finish_pin(); bnd = __shfl_sync(0xffffffffu, ptrs, q + 1); }
            const float mv[4] = {m[u].x, m[u].y, m[u].z, m[u].w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float nm = fmaxf(mx[c], mv[c]);
              const float sc = expf(mx[c] - nm);                 // exp(-inf) = 0 on the first edge
              const float ex = expf(mv[c] - nm);
              sm[c] = sm[c] * sc + ex;
              tw[c] = tw[c] * sc + mv[c] * ex;
              mx[c] = nm;
            }
          }
        }
      }
      while (q < npin) finish_pin();
    }
    for (int r = max(npin, 0); r < PPW; ++r) {                   // rows past the end of the level
      if constexpr (H16) {
        store_row_h(T, r0 + r, lane, make_float4(0.f, 0.f, 0.f, 0.f), -4);
      } else {
        *reinterpret_cast<float4*>(&T.in_hi[(r0 + r) * IN_LD + lane * 4]) = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(&T.in_lo[(r0 + r) * IN_LD + lane * 4]) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }

  // phases 2+3: hidden = relu(a @ W1t + b1);  h = relu(S + hidden @ W2t + b2)
  if constexpr (H16) {
    auto epi1 = [&](int row, int col, float v0, float v1) {      // v = sc[row] (a @ W1t): add the scaled bias
      const float2 bb = __ldg(reinterpret_cast<const float2*>(b1 + col));
      const float sc = T.sc_s[row];
      return make_float2(fmaxf(fmaf(bb.x, sc, v0), 0.f), fmaxf(fmaf(bb.y, sc, v1), 0.f));
    };
    mlp_tile_h(T, W1t, W2t, tid, epi1);
  } else {
    auto epi1 = [&](int row, int col, float v0, float v1) {
      const float2 bb = __ldg(reinterpret_cast<const float2*>(b1 + col));
      return make_float2(fmaxf(v0 + bb.x, 0.f), fmaxf(v1 + bb.y, 0.f));
    };
    mlp_tile(T, W1t, W2t, tid, epi1);
  }
  pdl_launch_dependents();                           // the next level may be scheduled while the epilogue drains
  // coalesced epilogues from shared memory: hidden rows (saved for backward; hi + lo is exact), then h rows
  if (HIDb) {
#pragma unroll
    for (int i = 0; i < TILE * HID / 4 / CT; ++i) {
      const int q = tid + i * CT, row = q >> 6, c4 = (q & 63) * 4;
      if (t0 + row < cnt) {
        if constexpr (H16)
          st4(HIDb + (int64_t)(crow0 + t0 + row) * HID + c4, *reinterpret_cast<const float4*>(&T.hid_f[row * MID_LD + c4]));
        else
          st4(HIDb + (int64_t)(crow0 + t0 + row) * HID + c4,
              f4add(*reinterpret_cast<const float4*>(&T.mid_hi[row * MID_LD + c4]), *reinterpret_cast<const float4*>(&T.mid_lo[row * MID_LD + c4])));
      }
    }
  }
#pragma unroll
  for (int i = 0; i < TILE * D / 4 / CT; ++i) {
    const int q = tid + i * CT, row = q >> 5, c4 = (q & 31) * 4;
    const int v = v_s[row];
    if (v >= 0) {
      const float4 acc = *reinterpret_cast<const float4*>(&T.scr[row * IN_LD + c4]);
      const float4 bb = __ldg(reinterpret_cast<const float4*>(b2 + c4));
      const float4 sv = ld4_stream(S + (int64_t)v * D + c4);
      st4(H + (int64_t)v * D + c4,
          f4relu(make_float4(acc.x + bb.x + sv.x, acc.y + bb.y + sv.y, acc.z + bb.z + sv.z, acc.w + bb.w + sv.w)));
    }
  }
}

// ---------------------------------------------------------------------------------------------
// backward: every pin PULLS its gradient from its successors over the out-edge CSRs (no atomics,
// deterministic).  Appendix B of SURVEY.md:
//   net  edge v->u (u odd level):   g_h[v] += g_z[u] / indeg_net(u)
//   cell edge v->u (u even level):  g_h[v] += g_a[u] * w_e * (1 + h[v] - a[u]),  w_e = exp(h[v]-lse[u])
// then g_z[v] = g_h[v] * (h[v] > 0) is written back into G[v].
// ---------------------------------------------------------------------------------------------
struct SchedDev {
  const int* order;
  const int* bn_ptr;
  const int* bn_dst;
  const float* bn_w;
  const int* bc_ptr;
  const int* bc_row;
};

__device__ __forceinline__ float4 cell_edge_grad(float4 hv, float4 ga, float4 ls, float4 aa) {
  return make_float4(ga.x * expf(hv.x - ls.x) * (1.f + hv.x - aa.x), ga.y * expf(hv.y - ls.y) * (1.f + hv.y - aa.y),
                     ga.z * expf(hv.z - ls.z) * (1.f + hv.z - aa.z), ga.w * expf(hv.w - ls.w) * (1.f + hv.w - aa.w));
}
__device__ __forceinline__ float4 relu_mask(float4 hv, float4 g) {
  return make_float4(hv.x > 0.f ? g.x : 0.f, hv.y > 0.f ? g.y : 0.f, hv.z > 0.f ? g.z : 0.f, hv.w > 0.f ? g.w : 0.f);
}

// one warp per pin (level 0 and odd levels)
__global__ void __launch_bounds__(256)
gnn_net_bwd_kernel(SchedDev s, int p0, int cnt, const float* __restrict__ H, float* G,
                   const float* __restrict__ GA, const float* __restrict__ A,
                   const float* __restrict__ LSE) {
  const int lane = threadIdx.x & 31;
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  pdl_launch_dependents();
  if (w >= cnt) { pdl_wait(); return; }
  const int p = p0 + w;
  const int v = s.order[p];
  const int ns = s.bn_ptr[p], ne = s.bn_ptr[p + 1], cs = s.bc_ptr[p], ce = s.bc_ptr[p + 1];
  pdl_wait();
  const int64_t off = (int64_t)v * D + lane * 4;
  float4 g = ld4(G + off);
  const float4 hv = ld4(H + off);
  for (int i = ns; i < ne; i += 4) {
    float4 m[4];
    float wq[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      wq[q] = 0.f;
      m[q] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i + q < ne) { wq[q] = s.bn_w[i + q]; m[q] = ld4(G + (int64_t)s.bn_dst[i + q] * D + lane * 4); }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) g = f4add(g, f4scale(m[q], wq[q]));
  }
  for (int i = cs; i < ce; i += 2) {
    float4 ga[2], ls[2], aa[2];
#pragma unroll
    for (int q = 0; q < 2; ++q)
      if (i + q < ce) {
        const int64_t co = (int64_t)s.bc_row[i + q] * D + lane * 4;
        ga[q] = ld4(GA + co); ls[q] = ld4(LSE + co); aa[q] = ld4(A + co);
      }
#pragma unroll
    for (int q = 0; q < 2; ++q)
      if (i + q < ce) g = f4add(g, cell_edge_grad(hv, ga[q], ls[q], aa[q]));
  }
  st4(G + off, relu_mask(hv, g));
}

// WG == false: G and GA only -- the operands of the hoisted weight-gradient GEMMs (GZC, GHID) are not stored
template <bool H16, bool WG>
__global__ void __launch_bounds__(CT)
gnn_cell_bwd_kernel(SchedDev s, int p0, int cnt, int crow0, const float* __restrict__ H, float* G,
                    const float* __restrict__ W1, const float* __restrict__ W2, float* GA,
                    const float* __restrict__ A, const float* __restrict__ LSE,
                    const float* __restrict__ HIDb, float* __restrict__ GHID, float* __restrict__ GZC) {
  extern __shared__ __align__(16) float smem[];
  const Tiles T(smem);
  float (*gz_s)[IN_LD] = reinterpret_cast<float (*)[IN_LD]>(T.scr);          // gradient accumulation scratch
  float (*gh_s)[MID_LD] = reinterpret_cast<float (*)[MID_LD]>(H16 ? T.hid_f : T.mid_hi);   // the pins' own h rows until the MLP runs
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int t0 = blockIdx.x * TILE;
  // g_hid = (g_z @ W2) * (hid > 0): W2 is [128][256] as stored by nn.Linear(256,128)  -> "Wa"
  // g_a   =  g_hid @ W1:            W1 is [256][128] as stored by nn.Linear(128,256)  -> "Wb"
  mlp_prologue(T, W2, W1, tid);
  pdl_wait();

  // phase 1: each warp pulls the gradient of PPW consecutive pins.  gz_s accumulates, the first
  // 128 columns of gh_s hold the pins' own h rows until the MLP overwrites them.
  constexpr int PPW = TILE / (CT / 32);
  {
    const int r0 = warp * PPW;
    const int npin = min(PPW, cnt - (t0 + r0));
    const int pb = p0 + t0 + r0;
    int nptr = 0, cptr = 0, vv = 0;
    if (npin > 0) {
      if (lane <= npin) { nptr = s.bn_ptr[pb + lane]; cptr = s.bc_ptr[pb + lane]; }
      if (lane < npin) vv = s.order[pb + lane];
    }
#pragma unroll
    for (int r = 0; r < PPW; ++r) {
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f), hv = g;
      if (r < npin) {
        const int64_t off = (int64_t)__shfl_sync(0xffffffffu, vv, r) * D + lane * 4;
        g = ld4(G + off);
        hv = ld4(H + off);
      }
      *reinterpret_cast<float4*>(&gz_s[r0 + r][lane * 4]) = g;
      *reinterpret_cast<float4*>(&gh_s[r0 + r][lane * 4]) = hv;
    }
    if (npin > 0) {
      {  // net out-edges: one contiguous range for the warp's pins
        const int E0 = __shfl_sync(0xffffffffu, nptr, 0), E1 = __shfl_sync(0xffffffffu, nptr, npin);
        int q = 0, bnd = __shfl_sync(0xffffffffu, nptr, 1);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        auto flush = [&]() {
          float4* dst = reinterpret_cast<float4*>(&gz_s[r0 + q][lane * 4]);
          *dst = f4add(*dst, acc);
          acc = make_float4(0.f, 0.f, 0.f, 0.f);
          ++q;
        };
        for (int i = E0; i < E1; i += 8) {
          const bool ok = i + (lane & 7) < E1;
          const int idx = ok ? s.bn_dst[i + (lane & 7)] : 0;
          const float wt = ok ? s.bn_w[i + (lane & 7)] : 0.f;
          float4 m[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int dst = __shfl_sync(0xffffffffu, idx, u);
            if (i + u < E1) m[u] = ld4(G + (int64_t)dst * D + lane * 4);
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float wu = __shfl_sync(0xffffffffu, wt, u);
            if (i + u < E1) {
              while (i + u >= bnd) { flush(); bnd = __shfl_sync(0xffffffffu, nptr, q + 1); }
              acc = f4add(acc, f4scale(m[u], wu));
            }
          }
        }
        if (q < npin) flush();
      }
      {  // cell out-edges (rare on cell levels)
        const int E0 = __shfl_sync(0xffffffffu, cptr, 0), E1 = __shfl_sync(0xffffffffu, cptr, npin);
        int q = 0, bnd = __shfl_sync(0xffffffffu, cptr, 1);
        for (int i = E0; i < E1; ++i) {
          while (i >= bnd) { ++q; bnd = __shfl_sync(0xffffffffu, cptr, q + 1); }
          const int64_t co = (int64_t)s.bc_row[i] * D + lane * 4;
          const float4 hv = *reinterpret_cast<const float4*>(&gh_s[r0 + q][lane * 4]);
          float4* dst = reinterpret_cast<float4*>(&gz_s[r0 + q][lane * 4]);
          *dst = f4add(*dst, cell_edge_grad(hv, ld4(GA + co), ld4(LSE + co), ld4(A + co)));
        }
      }
    }
#pragma unroll
    for (int r = 0; r < PPW; ++r) {
      if (r < npin) {
        const float4 hv = *reinterpret_cast<const float4*>(&gh_s[r0 + r][lane * 4]);
        const float4 gz = relu_mask(hv, *reinterpret_cast<const float4*>(&gz_s[r0 + r][lane * 4]));
        if constexpr (H16) {
          store_row_h(T, r0 + r, lane, gz, -100);
        } else {
          float4 gzh, gzl;
          split4(gz, gzh, gzl);
          *reinterpret_cast<float4*>(&T.in_hi[(r0 + r) * IN_LD + lane * 4]) = gzh;
          *reinterpret_cast<float4*>(&T.in_lo[(r0 + r) * IN_LD + lane * 4]) = gzl;
        }
        st4(G + (int64_t)__shfl_sync(0xffffffffu, vv, r) * D + lane * 4, gz);
        if constexpr (WG) st4(GZC + (int64_t)(crow0 + t0 + r0 + r) * D + lane * 4, gz);
      } else if constexpr (H16) {
        store_row_h(T, r0 + r, lane, make_float4(0.f, 0.f, 0.f, 0.f), -100);
      } else {
        *reinterpret_cast<float4*>(&T.in_hi[(r0 + r) * IN_LD + lane * 4]) = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(&T.in_lo[(r0 + r) * IN_LD + lane * 4]) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  }
  // g_hid = (g_z @ W2) * (hid > 0);  g_a = g_hid @ W1
  auto epi1 = [&](int row, int col, float v0, float v1) {
    const int p = t0 + row;
    float2 o = make_float2(0.f, 0.f);
    if (p < cnt) {
      const float2 hd = *reinterpret_cast<const float2*>(HIDb + (int64_t)(crow0 + p) * HID + col);
      o = make_float2(hd.x > 0.f ? v0 : 0.f, hd.y > 0.f ? v1 : 0.f);
    }
    return o;
  };
  if constexpr (H16) mlp_tile_h(T, W2, W1, tid, epi1);       // (the ReLU mask commutes with the per-pin scale)
  else mlp_tile(T, W2, W1, tid, epi1);
  pdl_launch_dependents();
#pragma unroll
  for (int i = 0; i < TILE * HID / 4 / CT; ++i) {
    const int q = tid + i * CT, row = q >> 6, c4 = (q & 63) * 4;
    if (WG && t0 + row < cnt) {
      if constexpr (H16)
        st4(GHID + (int64_t)(crow0 + t0 + row) * HID + c4, *reinterpret_cast<const float4*>(&T.hid_f[row * MID_LD + c4]));
      else
        st4(GHID + (int64_t)(crow0 + t0 + row) * HID + c4,
            f4add(*reinterpret_cast<const float4*>(&T.mid_hi[row * MID_LD + c4]), *reinterpret_cast<const float4*>(&T.mid_lo[row * MID_LD + c4])));
    }
  }
#pragma unroll
  for (int i = 0; i < TILE * D / 4 / CT; ++i) {
    const int q = tid + i * CT, row = q >> 5, c4 = (q & 31) * 4;
    if (t0 + row < cnt) st4(GA + (int64_t)(crow0 + t0 + row) * D + c4, *reinterpret_cast<const float4*>(&gz_s[row][c4]));
  }
}

// launch with programmatic stream serialization (the kernel calls griddepcontrol.wait itself)
template <class... KArgs, class... Args>
int launch_pdl(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, const char* what, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (e != cudaSuccess) return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
  return 0;
}

int cell_smem_optin() {
  // the attribute is per function AND per device: set it on every call (cheap), so a second device works
  TM_CUDA(cudaFuncSetAttribute(gnn_cell_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CELL_SMEM));
  TM_CUDA(cudaFuncSetAttribute(gnn_cell_bwd_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CELL_SMEM));
  TM_CUDA(cudaFuncSetAttribute(gnn_cell_bwd_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CELL_SMEM));
  TM_CUDA(cudaFuncSetAttribute(gnn_cell_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CELL_SMEM));
  TM_CUDA(cudaFuncSetAttribute(gnn_cell_bwd_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CELL_SMEM));
  TM_CUDA(cudaFuncSetAttribute(gnn_cell_bwd_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CELL_SMEM));
  return 0;
}

int cell_base_of(const tm_schedule* s, int level) {
  int acc = 0;
  for (int l = 2; l < level; l += 2) acc += s->h_level_ptr[l + 1] - s->h_level_ptr[l];
  return acc;
}
}  // namespace

namespace tmk {
size_t gnn_persist_ws_bytes();
void gnn_persist_set_profile(long long* p);
int gnn_persist_profile_slots();
int gnn_persist_forward(const tm_schedule* s, int lb, int le, float* H, const float* S, const float* W1t, const float* b1,
                        const float* W2t, const float* b2, float* A, float* LSE, float* HIDb, void* ws, cudaStream_t st);
int gnn_persist_backward(const tm_schedule* s, const float* H, float* G, const float* W1, const float* W2, const float* A,
                         const float* LSE, const float* HIDb, float* GA, float* GHID, float* GZC, void* ws, cudaStream_t st,
                         int lb, int le);
int gnn_persist_save(const tm_schedule* s, const float* H, const float* W1t, const float* b1, const float* W2t, float* A,
                     float* LSE, float* HIDb, void* ws, cudaStream_t st);
}  // namespace tmk

namespace {
constexpr int IMPL_BITS = 1 | 2 | 4 | 16;     // the tm_gnn_set_impl bits that select something
std::atomic<int> g_impl{-1};
thread_local int g_last_barriers = 0;
int gnn_impl() {
  int v = g_impl.load(std::memory_order_relaxed);
  if (v < 0) {
    // bit 0: forward persistent, bit 1: backward persistent.  Default 1: measured on B200 the persistent
    // forward beats the per-level chain (config 2: 0.89 vs 1.01 ms, config 3: 1.92 vs 2.64 ms) while the
    // persistent backward does not (1.24 vs 1.00 ms, 2.61 vs 2.59 ms).
    //   C3: 2.31 vs 2.61 ms in favour of the persistent backward).  Bit 2 = "auto" (default): persistent forward;
    //   persistent backward only on wide schedules (>= 6 000 pins per level on average).
    const char* e = getenv("TM_GNN_IMPL");
    //   Bit 4 (16): the per-level cell kernels run the fp16 two-term split (mma.sync.m16n8k16) instead of 3xTF32.
    v = !e ? 20 : (e[0] == 'l' ? 0 : (e[0] == 'p' ? 3 : (atoi(e) & IMPL_BITS)));
    g_impl.store(v, std::memory_order_relaxed);
  }
  return v;
}
int count_levels(const tm_schedule* s, int lb, int le) {
  int k = 0;
  for (int l = lb; l < le; ++l) k += (s->h_level_ptr[l + 1] > s->h_level_ptr[l]);
  return k;
}
}  // namespace

extern "C" int tm_gnn_set_impl(int impl) {
  const int prev = gnn_impl();
  if (impl >= 0) g_impl.store(impl & IMPL_BITS, std::memory_order_relaxed);
  return prev;
}
extern "C" int tm_gnn_last_barriers() { return g_last_barriers; }
extern "C" int tm_gnn_set_profile(void* clocks) {
  tmk::gnn_persist_set_profile(reinterpret_cast<long long*>(clocks));
  return 0;
}

extern "C" size_t tm_gnn_ws_bytes() { return PACK_FLOATS * sizeof(float) + 256 + tmk::gnn_persist_ws_bytes(); }

namespace {
// (Wa [128][256], Wb [256][128]) -> padded, hi/lo pre-split rows in the caller's workspace
int pack_pair(const float* Wa, const float* Wb, void* ws, size_t ws_bytes, const float** pa, const float** pb, cudaStream_t st,
              bool h16) {
  TM_REQUIRE(ws && ws_bytes >= tm_gnn_ws_bytes(), "tm_gnn: workspace too small (tm_gnn_ws_bytes)");
  float* a = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  float* b = a + (size_t)D * WA_ROW;
  *pa = a;
  *pb = b;
  if (h16) {                               // same chunk geometry, half2 (hi | lo') planes inside each chunk
    gnn_pack_h_kernel<<<(D * HID + 255) / 256, 256, 0, st>>>(Wa, Wb, reinterpret_cast<uint32_t*>(a));
    return check_launch("gnn_pack_h");
  }
  gnn_pack_kernel<<<(D * WA_ROW + 255) / 256, 256, 0, st>>>(Wa, D, HID, a);
  TM_TRY(check_launch("gnn_pack(Wa)"));
  gnn_pack_kernel<<<(HID * WB_ROW + 255) / 256, 256, 0, st>>>(Wb, HID, D, b);
  TM_TRY(check_launch("gnn_pack(Wb)"));
  *pa = a;
  *pb = b;
  return 0;
}
}  // namespace

extern "C" int tm_gnn_forward(const tm_schedule* s, int32_t lb, int32_t le, float* H, const float* S,
                              const float* W1t_in, const float* b1, const float* W2t_in, const float* b2,
                              float* A, float* LSE, float* HIDb, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(s && s->f_ptr && s->f_src, "tm_gnn_forward: schedule lacks the level-ordered edge lists");
  TM_REQUIRE(s && s->h_level_ptr && lb >= 0 && le <= s->num_levels && lb <= le, "tm_gnn_forward: bad level range");
  TM_REQUIRE((A == nullptr) == (LSE == nullptr) && (A == nullptr) == (HIDb == nullptr),
             "tm_gnn_forward: A, LSE, HID must be all set or all NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (gnn_impl() & 5) {
    TM_REQUIRE(ws && ws_bytes >= tm_gnn_ws_bytes(), "tm_gnn_forward: workspace too small (tm_gnn_ws_bytes)");
    g_last_barriers = count_levels(s, lb, le);
    return tmk::gnn_persist_forward(s, lb, le, H, S, W1t_in, b1, W2t_in, b2, A, LSE, HIDb, ws, st);
  }
  g_last_barriers = 0;
  TM_TRY(cell_smem_optin());
  const float *W1t = nullptr, *W2t = nullptr;
  const bool h16 = gnn_impl() & 16;
  TM_TRY(pack_pair(W1t_in, W2t_in, ws, ws_bytes, &W1t, &W2t, st, h16));
  int crow0 = cell_base_of(s, lb + (lb & 1));
  for (int l = lb; l < le; ++l) {
    const int p0 = s->h_level_ptr[l], cnt = s->h_level_ptr[l + 1] - p0;
    const bool cell = (l > 0) && !(l & 1);
    if (cnt > 0) {
      if (!cell) {
        TM_TRY(launch_pdl(gnn_net_fwd_kernel, (unsigned)cdiv(cnt, 8), 256, 0, st, "gnn_net_fwd", s->order, p0, cnt, s->f_ptr,
                          s->f_src, S, H));
      } else {
        TM_TRY(launch_pdl(h16 ? gnn_cell_fwd_kernel<true> : gnn_cell_fwd_kernel<false>, (unsigned)cdiv(cnt, TILE), CT, CELL_SMEM, st, "gnn_cell_fwd", s->order, p0, cnt,
                          crow0, s->f_ptr, s->f_src, S, H, W1t, b1, W2t, b2, A, LSE, HIDb));
      }
    }
    if (cell) crow0 += cnt;
  }
  return 0;
}

extern "C" int tm_gnn_backward(const tm_schedule* s, const float* H, float* G, const float* W1_in,
                               const float* W2_in, const float* A, const float* LSE, const float* HIDb,
                               float* GA, float* GHID, float* GZC, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(s && s->h_level_ptr && s->bn_ptr && s->bc_ptr, "tm_gnn_backward: bad schedule");
  TM_REQUIRE((GHID == nullptr) == (GZC == nullptr), "tm_gnn_backward: GHID and GZC must be both set or both NULL");
  const bool wg = GHID != nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  const bool wide = s->num_levels > 0 && s->h_level_ptr[s->num_levels] / s->num_levels >= 6000;
  if ((gnn_impl() & 2) || ((gnn_impl() & 4) && wide)) {
    TM_REQUIRE(ws && ws_bytes >= tm_gnn_ws_bytes(), "tm_gnn_backward: workspace too small (tm_gnn_ws_bytes)");
    g_last_barriers = count_levels(s, 0, s->num_levels);
    return tmk::gnn_persist_backward(s, H, G, W1_in, W2_in, A, LSE, HIDb, GA, GHID, GZC, ws, st, 0, s->num_levels);
  }
  g_last_barriers = 0;
  TM_TRY(cell_smem_optin());
  // backward products: g_hid = g_z @ W2 (W2 [128][256] is "Wa"), g_a = g_hid @ W1 (W1 [256][128] is "Wb")
  const float *W2 = nullptr, *W1 = nullptr;
  const bool h16 = gnn_impl() & 16;
  TM_TRY(pack_pair(W2_in, W1_in, ws, ws_bytes, &W2, &W1, st, h16));
  SchedDev d{s->order, s->bn_ptr, s->bn_dst, s->bn_w, s->bc_ptr, s->bc_row};
  int crow_end = cell_base_of(s, s->num_levels + (s->num_levels & 1));  // total cell rows
  for (int l = s->num_levels - 1; l >= 0; --l) {
    const int p0 = s->h_level_ptr[l], cnt = s->h_level_ptr[l + 1] - p0;
    const bool cell = (l > 0) && !(l & 1);
    if (cell) crow_end -= cnt;
    if (cnt <= 0) continue;
    if (!cell) {
      TM_TRY(launch_pdl(gnn_net_bwd_kernel, (unsigned)cdiv(cnt, 8), 256, 0, st, "gnn_net_bwd", d, p0, cnt, H, G, (const float*)GA, A, LSE));
    } else {
      auto kern = h16 ? (wg ? gnn_cell_bwd_kernel<true, true> : gnn_cell_bwd_kernel<true, false>)
                      : (wg ? gnn_cell_bwd_kernel<false, true> : gnn_cell_bwd_kernel<false, false>);
      TM_TRY(launch_pdl(kern, (unsigned)cdiv(cnt, TILE), CT, CELL_SMEM, st, "gnn_cell_bwd", d, p0, cnt, crow_end, H,
                        G, W1, W2, GA, A, LSE, HIDb, GHID, GZC));
    }
  }
  return 0;
}

extern "C" int tm_gnn_forward_cone(const tm_schedule* cone, float* H, const float* S, const float* W1t, const float* b1,
                                   const float* W2t, const float* b2, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(cone && cone->order && cone->f_ptr && cone->f_src && cone->level_ptr && cone->cell_base,
             "tm_gnn_forward_cone: schedule lacks the device arrays (order, f_ptr, f_src, level_ptr, cell_base)");
  TM_REQUIRE(cone->num_levels >= 0, "tm_gnn_forward_cone: bad level count");
  TM_REQUIRE(H && S && W1t && b1 && W2t && b2, "tm_gnn_forward_cone: NULL operand");
  TM_REQUIRE(ws && ws_bytes >= tm_gnn_ws_bytes(), "tm_gnn_forward_cone: workspace too small (tm_gnn_ws_bytes)");
  // the persistent kernel skips empty levels on the device, so the cone's sizes never reach the host
  return tmk::gnn_persist_forward(cone, 0, cone->num_levels, H, S, W1t, b1, W2t, b2, nullptr, nullptr, nullptr, ws,
                                  (cudaStream_t)stream);
}

extern "C" int tm_gnn_save_cone(const tm_schedule* cone, const float* H, const float* W1t, const float* b1,
                                const float* W2t, float* A, float* LSE, float* HID, void* ws, size_t ws_bytes,
                                void* stream) {
  TM_REQUIRE(cone && cone->order && cone->f_ptr && cone->f_src && cone->level_ptr && cone->cell_base,
             "tm_gnn_save_cone: schedule lacks the device arrays (order, f_ptr, f_src, level_ptr, cell_base)");
  TM_REQUIRE(cone->num_levels >= 0, "tm_gnn_save_cone: bad level count");
  TM_REQUIRE(H && W1t && b1 && W2t && A && LSE && HID, "tm_gnn_save_cone: NULL operand");
  TM_REQUIRE(ws && ws_bytes >= tm_gnn_ws_bytes(), "tm_gnn_save_cone: workspace too small (tm_gnn_ws_bytes)");
  return tmk::gnn_persist_save(cone, H, W1t, b1, W2t, A, LSE, HID, ws, (cudaStream_t)stream);
}

extern "C" int tm_gnn_backward_cone(const tm_schedule* cone, const float* H, float* G, const float* W1, const float* W2,
                                    const float* A, const float* LSE, const float* HID, float* GA, void* ws,
                                    size_t ws_bytes, void* stream) {
  TM_REQUIRE(cone && cone->order && cone->level_ptr && cone->cell_base && cone->bn_ptr && cone->bn_dst && cone->bn_w &&
                 cone->bc_ptr && cone->bc_row,
             "tm_gnn_backward_cone: schedule lacks the device arrays (order, level_ptr, cell_base, bn_ptr, bn_dst, "
             "bn_w, bc_ptr, bc_row)");
  TM_REQUIRE(cone->num_levels >= 0, "tm_gnn_backward_cone: bad level count");
  TM_REQUIRE(H && G && W1 && W2 && A && LSE && HID && GA, "tm_gnn_backward_cone: NULL operand");
  TM_REQUIRE(ws && ws_bytes >= tm_gnn_ws_bytes(), "tm_gnn_backward_cone: workspace too small (tm_gnn_ws_bytes)");
  // the persistent sweep skips empty levels on the device, so the cone's sizes never reach the host
  return tmk::gnn_persist_backward(cone, H, G, W1, W2, A, LSE, HID, GA, nullptr, nullptr, ws, (cudaStream_t)stream, 0,
                                   cone->num_levels);
}
