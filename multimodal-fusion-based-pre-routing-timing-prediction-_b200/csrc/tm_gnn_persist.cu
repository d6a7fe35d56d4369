// G2/G3, persistent form: the WHOLE level-wise propagation (forward) or its reverse sweep (backward)
// is ONE kernel -- 74 two-CTA clusters, one CTA per SM, each looping over the levels -- instead of
// one launch per level.  Levels are ordered by a grid-wide barrier per level on a monotonic counter
// (one release-add per CTA, one warp polls), with the next level's static inputs prefetched into L2
// between arrive and wait.  (Dataflow orderings without a barrier, net-level push fusion and one launch
// per cell level were all measured slower on B200: DESIGN.md section 4.)  Replaces PathConv.forward
// and its UDFs (src/model.py:88-116,138-153,158-213, one DGL `pull` + cuBLAS calls + an (N,128)
// index_copy PER LEVEL) and the autograd backward (src/train.py:553).
//
// Why a cluster pair: the 128->256->128 MLP of fc_cell_neigh (model.py:48,138-146) sits inside the
// level recurrence and every cell pin needs all of its weights.  They stay RESIDENT in shared
// memory for the whole kernel, split over the pair: CTA r holds hidden units 128r..128r+127 of both
// layers as fp16 (hi, lo) planes (4 x 32 KB).  The MLP runs TRANSPOSED on tcgen05:
//     hid^T[128r.., pins] = W1[128r.., :] . a^T          M = 128 hidden units, N = pins, K = 128
//     out^T[:, pins]     += W2[:, 128r..] . hid^T[128r..] M = 128 channels,     N = pins, K = 128
// so the pin tile is the MMA's N dimension (32 / 64 / 96 pins) and a level of only ~2 000 pins
// still spreads over every SM.  The two partial out^T tiles are exchanged through distributed shared
// memory (each CTA finalises half of the tile's pins).
//
// Arithmetic: the fp16 two-term split (tm_split.cuh), the exact analogue of 3xTF32 at half the bytes,
// with a per-pin scale, so gradients of any size keep 22 significant bits; acc_main and acc_corr are
// both fp32 in TMEM.
//
// Net levels / level 0 (mean over net in-edges) are processed by sub-warp groups (8 / 16 / 32 lanes
// per pin, chosen per level so that every pin gets its own group when the level fits).
// Everything static (schedule pointers, edge indices, S rows) is fetched BEFORE the barrier wait.
#include <cuda_fp16.h>

#include "tm_common.cuh"
#include "tm_sm100.cuh"
#include "tm_split.cuh"

using namespace tmk;
using namespace tmk::sm100;

namespace {
constexpr int D = 128;
constexpr int HID = 256;
constexpr int THREADS = 512;
constexpr int WARPS = THREADS / 32;
constexpr int NMAX = 96;                       // pins per tile (MMA N): 32, 64 or 96

// shared-memory operand layouts: K-major, SWIZZLE_NONE core matrices (8 rows x 16 bytes)
//   off(row, k) = (row / 8) * SBO + (k / 8) * LBO + (row % 8) * 16 + (k % 8) * 2          [bytes, fp16]
constexpr uint32_t W_LBO = 128, W_SBO = 2048, W_PLANE = 128 * 128 * 2;
// pin operand: the k-group stride is padded by 16 bytes so that the 16 k-groups a warp writes for
// one pin fall into different banks
constexpr uint32_t B_LBO = 144, B_SBO = 16 * B_LBO, B_PLANE = (NMAX / 8) * B_SBO;
constexpr uint32_t X_BYTES = (NMAX / 2) * D * 4;
constexpr uint32_t OFF_W = 0;                  // A1hi, A1lo, A2hi, A2lo
constexpr uint32_t OFF_B = OFF_W + 4 * W_PLANE;    // Bhi, Blo   (also fp32 [N][128] scratch in the backward gather)
constexpr uint32_t OFF_X = OFF_B + 2 * B_PLANE;    // partial sums received from the peer CTA
constexpr uint32_t OFF_MISC = OFF_X + X_BYTES;     // scale[NMAX], inv[NMAX], pin[NMAX], mbarrier, tmem slot
constexpr uint32_t SMEM_BYTES = OFF_MISC + 3 * NMAX * 4 + 48;
static_assert(2 * B_PLANE >= NMAX * D * 4, "backward scratch must fit the operand planes");
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

constexpr uint32_t TM_MAIN1 = 0, TM_CORR1 = 128, TM_MAIN2 = 256, TM_CORR2 = 384, TM_COLS = 512;
constexpr uint32_t MBAR_SPINS = 1u << 22;         // mbarrier waits trap after this many probes

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4fma(float4 a, float s, float4 c) { return make_float4(fmaf(a.x, s, c.x), fmaf(a.y, s, c.y), fmaf(a.z, s, c.z), fmaf(a.w, s, c.w)); }
__device__ __forceinline__ float4 relu_mask(float4 hv, float4 g) {
  return make_float4(hv.x > 0.f ? g.x : 0.f, hv.y > 0.f ? g.y : 0.f, hv.z > 0.f ? g.z : 0.f, hv.w > 0.f ? g.w : 0.f);
}
// SURVEY.md Appendix B: d a / d m_e = w_e (1 + m_e - a), w_e = exp(m_e - lse)
__device__ __forceinline__ float4 cell_edge_grad(float4 hv, float4 ga, float4 ls, float4 aa) {
  return make_float4(ga.x * __expf(hv.x - ls.x) * (1.f + hv.x - aa.x), ga.y * __expf(hv.y - ls.y) * (1.f + hv.y - aa.y),
                     ga.z * __expf(hv.z - ls.z) * (1.f + hv.z - aa.z), ga.w * __expf(hv.w - ls.w) * (1.f + hv.w - aa.w));
}

// ---------------------------------------------------------------------------------------------
// synchronisation
// ---------------------------------------------------------------------------------------------
// Grid-wide barrier on a monotonic counter (zeroed by the host before the launch): every CTA adds one
// per level; level k is complete when the counter reaches k * gridDim.x.  Split into arrive / wait so
// that static fetches sit between them; the last warp polls.  Bounded: a lost CTA traps.
struct GridBar {
  unsigned int* ctr;
  unsigned int nblk;
  unsigned int narr;
  __device__ __forceinline__ void arrive() {
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
    ++narr;
  }
  __device__ __forceinline__ void wait() const {
    if (narr != 0 && threadIdx.x == THREADS - 32) {
      const unsigned int target = narr * nblk;
      unsigned int v = 0;
      for (uint32_t spin = 0;; ++spin) {
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
        if (v >= target) break;
        if (spin > (1u << 23)) __trap();
      }
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
    }
    __syncthreads();
  }
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f32(uint32_t addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// one product  acc = W (128 x 128, resident planes) . tile^T (N x 128, pin planes):  8 k-steps of
// 16, three MMAs each (hi*hi -> main; hi*lo' + lo'*hi -> corr), then one commit.  One thread.
__device__ __forceinline__ void issue_gemm(uint32_t w_hi, uint32_t w_lo, uint32_t b_hi, uint32_t b_lo, uint32_t t_main,
                                           uint32_t t_corr, uint32_t idesc, uint64_t* bar) {
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    const uint64_t ah = smem_desc(w_hi + ks * 2 * W_LBO, W_LBO, W_SBO), al = smem_desc(w_lo + ks * 2 * W_LBO, W_LBO, W_SBO);
    const uint64_t bh = smem_desc(b_hi + ks * 2 * B_LBO, B_LBO, B_SBO), bl = smem_desc(b_lo + ks * 2 * B_LBO, B_LBO, B_SBO);
    umma_f16(t_main, ah, bh, idesc, ks > 0);
    umma_f16(t_corr, ah, bl, idesc, ks > 0);
    umma_f16(t_corr, al, bh, idesc, 1u);
  }
  umma_commit(bar);
}

__device__ __forceinline__ uint32_t pin_off(int row, int k) {       // byte offset inside a pin plane
  return (uint32_t)(row >> 3) * B_SBO + (uint32_t)(k >> 3) * B_LBO + (uint32_t)(row & 7) * 16 + (uint32_t)(k & 7) * 2;
}

// Resident weight planes.  A pre-kernel writes, per CTA rank, the exact shared-memory image of the
// four planes (A1hi, A1lo, A2hi, A2lo; plane[m][k] = src[k * cs + m], m contiguous in HBM) into the
// caller's workspace; every CTA then pulls its 128 KB with four bulk copies (cp.async.bulk).
__global__ void gnn_pack_planes_kernel(const float* __restrict__ Wa, const float* __restrict__ Wb, uint8_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;          // [rank 2][matrix 2][k 128][m 128]
  if (i >= 2 * 2 * 128 * 128) return;
  const int m = i & 127, k = (i >> 7) & 127, mat = (i >> 14) & 1, rank = i >> 15;
  // Wa: first product, [k = 128][256] with this CTA's 128 result rows contiguous at 128 * rank;
  // Wb: second product, [256][128]: this CTA contracts over rows 128 * rank .. +127
  const float w = mat == 0 ? Wa[(size_t)k * 256 + rank * 128 + m] : Wb[(size_t)(rank * 128 + k) * 128 + m];
  __half h, l;
  split_h(w, h, l);
  const uint32_t off = (uint32_t)(m >> 3) * W_SBO + (uint32_t)(k >> 3) * W_LBO + (uint32_t)(m & 7) * 16 + (uint32_t)(k & 7) * 2;
  uint8_t* base = out + (size_t)rank * 4 * W_PLANE + (size_t)mat * 2 * W_PLANE;
  *reinterpret_cast<__half*>(base + off) = h;
  *reinterpret_cast<__half*>(base + W_PLANE + off) = l;
}

// the per-pin row written by a gather warp: scale, split, store into the pin planes
__device__ __forceinline__ void store_pin_row(uint8_t* smem, int row, int lane, float4 x, int emin, int pin) {
  const float rm = warp_max(fmaxf(fmaxf(fabsf(x.x), fabsf(x.y)), fmaxf(fabsf(x.z), fabsf(x.w))));
  float s, inv;
  row_scale(rm, emin, s, inv);
  uint2 hi, lo;
  split_h4(f4scale(x, s), hi, lo);
  const uint32_t off = pin_off(row, lane * 4);
  *reinterpret_cast<uint2*>(smem + OFF_B + off) = hi;
  *reinterpret_cast<uint2*>(smem + OFF_B + B_PLANE + off) = lo;
  if (lane == 0) {
    reinterpret_cast<float*>(smem + OFF_MISC)[row] = s;
    reinterpret_cast<float*>(smem + OFF_MISC)[NMAX + row] = inv;
    reinterpret_cast<int*>(smem + OFF_MISC)[2 * NMAX + row] = pin;
  }
}

struct Ctx {                       // per-CTA state shared by forward and backward
  uint8_t* smem;
  float* scale_s;
  float* inv_s;
  int* pin_s;
  uint64_t* mbar;
  uint32_t tmem;
  uint32_t rank;
  uint32_t mphase;
  bool pend_b;                     // a cluster "X consumed" arrive is outstanding
  long long* prof;                 // optional per-CTA phase clocks (tm_gnn_set_profile), NULL in production
  long long last;
  // phase clocks: thread 0 adds the cycles since the previous stamp to prof[phase]
  __device__ __forceinline__ void stamp(int phase) {
    if (prof && threadIdx.x == 0) {
      const long long t = clock64();
      prof[phase] += t - last;
      last = t;
    }
  }
};
enum { PH_SETUP = 0, PH_CPRE, PH_GATHER, PH_MMA1, PH_EPI1, PH_MMA2, PH_EXCH, PH_CPUB, PH_NPRE, PH_NBODY, PH_NTAIL, PH_COUNT = 16 };

// tile width for a cell level: as few pins as keeps every cluster busy once, 32 <= N <= 96
__device__ __forceinline__ int tile_width(int cnt, int nclusters) {
  int n = ((cnt + nclusters - 1) / nclusters + 31) & ~31;
  return min(max(n, 32), NMAX);
}

// both products of the resident MLP over the tile currently in the pin planes; epi1(n0, m, main, corr)
// turns 8 accumulator columns of row m into the (scaled) input of the second product
// pre1 / pre2 run between the issue of a product and the wait for it (global loads for the epilogues).
template <class Pre1, class Epi1, class Pre2>
__device__ __forceinline__ void mlp_tile(Ctx& c, int N, Pre1 pre1, Epi1 epi1, Pre2 pre2) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t sW = smem_u32(c.smem + OFF_W), sB = smem_u32(c.smem + OFF_B);
  const uint32_t idesc = make_idesc(Fmt::F16, N);
  const int qd = warp & 3, cg = warp >> 2, m = qd * 32 + lane, nper = N >> 2;
  const uint32_t tl = c.tmem + ((uint32_t)(qd * 32) << 16);
  fence_async_smem();                    // the pin planes were written through the generic proxy
  tc_fence_before();
  __syncthreads();
  c.stamp(PH_GATHER);
  if (tid == 0) {
    tc_fence_after();
    issue_gemm(sW, sW + W_PLANE, sB, sB + B_PLANE, c.tmem + TM_MAIN1, c.tmem + TM_CORR1, idesc, c.mbar);
  }
  pre1();
  mbar_wait_trap<MBAR_SPINS>(c.mbar, c.mphase);
  c.mphase ^= 1u;
  tc_fence_after();
  c.stamp(PH_MMA1);
  // epilogue 1: accumulator row m = hidden unit 128*rank + m; columns = pins.  The second product's
  // pin planes alias the first one's (its MMAs are complete).
#pragma unroll
  for (int cc = 0; cc < NMAX / 4 / 8; ++cc) {
    if (cc * 8 < nper) {
      const int n0 = cg * nper + cc * 8;
      float vm[8], vc[8];
      tmem_ld8(tl + TM_MAIN1 + n0, vm);
      tmem_ld8(tl + TM_CORR1 + n0, vc);
      epi1(n0, m, vm, vc);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        __half h, l;
        split_h(vm[j], h, l);
        const uint32_t off = pin_off(n0 + j, m);
        *reinterpret_cast<__half*>(c.smem + OFF_B + off) = h;
        *reinterpret_cast<__half*>(c.smem + OFF_B + B_PLANE + off) = l;
      }
    }
  }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  c.stamp(PH_EPI1);
  if (tid == 0) {
    tc_fence_after();
    issue_gemm(sW + 2 * W_PLANE, sW + 3 * W_PLANE, sB, sB + B_PLANE, c.tmem + TM_MAIN2, c.tmem + TM_CORR2, idesc, c.mbar);
  }
  pre2();
  mbar_wait_trap<MBAR_SPINS>(c.mbar, c.mphase);
  c.mphase ^= 1u;
  tc_fence_after();
  c.stamp(PH_MMA2);
}

// epilogue 2: accumulator row m = output channel, columns = pins.  Each CTA holds a partial sum over
// its 128 hidden units; pins of the tile's first half are finalised by CTA 0, the others by CTA 1.
// Column groups 0,1 (warps 0..7) cover the first half, 2,3 the second: a warp either keeps its
// values or ships them to the peer's X buffer.  fin(n, m, slot, value) receives the complete sums
// (slot = compile-time index of the pin inside the warp's column group).
template <class Fin>
__device__ __forceinline__ void exchange_tile(Ctx& c, int N, Fin fin) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int qd = warp & 3, cg = warp >> 2, m = qd * 32 + lane, nper = N >> 2, half = N >> 1;
  const uint32_t tl = c.tmem + ((uint32_t)(qd * 32) << 16);
  const bool mine = ((uint32_t)(cg >> 1) == c.rank);
  float* Xl = reinterpret_cast<float*>(c.smem + OFF_X);
  const uint32_t Xpeer = mapa(smem_u32(Xl), c.rank ^ 1u);
  float keep[NMAX / 4];
  if (c.pend_b) cluster_wait();          // the peer has consumed what we sent for the previous tile
#pragma unroll
  for (int cc = 0; cc < NMAX / 4 / 8; ++cc) {
    if (cc * 8 < nper) {
      const int n0 = cg * nper + cc * 8;
      float vm[8], vc[8];
      tmem_ld8(tl + TM_MAIN2 + n0, vm);
      tmem_ld8(tl + TM_CORR2 + n0, vc);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float val = fmaf(vc[j], LO_INV, vm[j]) * c.inv_s[n0 + j];
        if (mine) keep[cc * 8 + j] = val;
        else st_cluster_f32(Xpeer + (uint32_t)(((n0 + j) - (int)(c.rank ^ 1u) * half) * D + m) * 4u, val);
      }
    }
  }
  tc_fence_before();
  cluster_arrive();
  cluster_wait();
  if (mine) {
#pragma unroll
    for (int cc = 0; cc < NMAX / 4 / 8; ++cc) {
      if (cc * 8 < nper) {
        const int n0 = cg * nper + cc * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) fin(n0 + j, m, cc * 8 + j, keep[cc * 8 + j] + Xl[((n0 + j) - (int)c.rank * half) * D + m]);
      }
    }
  }
  cluster_arrive();                      // X consumed
  c.pend_b = true;
  c.stamp(PH_EXCH);
}

__device__ __forceinline__ void ctx_setup(Ctx& c, uint8_t* smem, const uint8_t* __restrict__ planes, long long* prof) {
  const int tid = threadIdx.x, warp = tid >> 5;
  c.smem = smem;
  c.prof = prof ? prof + (size_t)blockIdx.x * PH_COUNT : nullptr;
  c.last = clock64();
  c.scale_s = reinterpret_cast<float*>(smem + OFF_MISC);
  c.inv_s = c.scale_s + NMAX;
  c.pin_s = reinterpret_cast<int*>(c.inv_s + NMAX);
  c.mbar = reinterpret_cast<uint64_t*>(c.pin_s + NMAX);
  uint32_t* slot = reinterpret_cast<uint32_t*>(c.mbar + 1);
  c.rank = cluster_ctarank();
  c.mphase = 0;
  c.pend_b = false;
  uint64_t* wbar = reinterpret_cast<uint64_t*>(slot + 2);
  if (warp == 0) tmem_alloc(slot, TM_COLS);
  if (tid == 32) {
    mbar_init(c.mbar, 1);
    fence_mbarrier_init();
    mbar_init(wbar, 1);
    fence_mbarrier_init();
    fence_async_smem();
    mbar_expect_tx(wbar, 4u * W_PLANE);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      bulk_copy_g2s(smem_u32(smem + OFF_W + i * W_PLANE), planes + (size_t)c.rank * 4 * W_PLANE + (size_t)i * W_PLANE, W_PLANE, wbar);
  }
  __syncthreads();                       // the barriers are initialised
  mbar_wait_trap<MBAR_SPINS>(wbar, 0);   // the weights have landed (async proxy: what the MMAs read through)
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  c.tmem = *slot;
  cluster_arrive();                      // both CTAs of the pair are running before any DSMEM traffic
  cluster_wait();
  c.stamp(PH_SETUP);
}
__device__ __forceinline__ void ctx_teardown(Ctx& c) {
  if (c.pend_b) cluster_wait();
  tc_fence_before();
  __syncthreads();
  if ((threadIdx.x >> 5) == 0) {
    tc_fence_after();
    tmem_dealloc(c.tmem, TM_COLS);
  }
}


// ---------------------------------------------------------------------------------------------
// next-level prefetch.  A level's static inputs (schedule pointers, edge indices, S / H / HID rows) are
// cold in HBM and two dependent loads deep; the window between a CTA's barrier arrive and the barrier's
// completion is too short to hide that.  So, while waiting for level l, every CTA also pulls into L2
// what IT will read on level l+-1 (its pin ranges are contiguous in the schedule), and the pointer
// lines of the level after that; the per-thread fetch before the next wait then hits L2.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pf_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// lines covering elements [e0, e1) of a 4-byte array, spread over the CTA's threads
__device__ __forceinline__ void pf_range4(const void* base, int e0, int e1) {
  const char* b = reinterpret_cast<const char*>(base);
  for (int i = e0 + (int)threadIdx.x * 32; i < e1; i += THREADS * 32) pf_l2(b + (size_t)i * 4);
  if (threadIdx.x == 0 && e1 > e0) pf_l2(b + (size_t)(e1 - 1) * 4);
}
// schedule positions (relative to the level) this CTA processes in its k-th pass over level l
__device__ __forceinline__ void cta_range(int l, int cnt, int k, int& q0, int& qn) {
  const int nclusters = gridDim.x >> 1;
  if (l == 0 || (l & 1)) {
    const int nw = gridDim.x * WARPS;
    const int nv = cnt <= nw ? 1 : (cnt <= 2 * nw ? 2 : 4);
    q0 = ((int)blockIdx.x + k * (int)gridDim.x) * WARPS * nv;
    qn = WARPS * nv;
  } else {
    const int n = tile_width(cnt, nclusters);
    q0 = ((int)(blockIdx.x >> 1) + k * nclusters) * n;
    qn = n;
  }
  qn = max(0, min(qn, cnt - q0));
}
struct PfState { int v, e0, e1, c0, c1, qn, row0; };

// =============================================================================================
// forward
// =============================================================================================
struct FwdArgs {
  const int* level_ptr; const int* cell_base; const int* order; const int* f_ptr; const int* f_src;
  const float* S; float* H;
  const uint8_t* planes; const float* b1; const float* b2;                // packed fc_cell_neigh weights (gnn_pack_planes_kernel)
  float* A; float* LSE; float* HIDb;
  unsigned int* bar;               // grid-barrier counter (zeroed by gnn_persist_begin)
  long long* prof;
  int lb, le;
};

// issue the loads the prefetch of level l1 depends on (pass k); consumed by pf_end_fwd
__device__ __forceinline__ PfState pf_begin_fwd(const FwdArgs& a, int l1, int k) {
  PfState st{};
  if (l1 >= a.le) return st;
  const int p0 = __ldg(a.level_ptr + l1), cnt = __ldg(a.level_ptr + l1 + 1) - p0;
  int q0, qn;
  cta_range(l1, cnt, k, q0, qn);
  if (qn > 0) {
    if ((int)threadIdx.x < qn) st.v = __ldg(a.order + p0 + q0 + threadIdx.x);
    st.e0 = __ldg(a.f_ptr + p0 + q0);
    st.e1 = __ldg(a.f_ptr + p0 + q0 + qn);
    st.qn = qn;
  }
  const int l2 = l1 + 1;
  if (k == 0 && l2 < a.le) {                   // pointer lines of the level after
    const int p2 = __ldg(a.level_ptr + l2), cnt2 = __ldg(a.level_ptr + l2 + 1) - p2;
    int r0, rn;
    cta_range(l2, cnt2, 0, r0, rn);
    const int t = threadIdx.x;
    if (rn > 0 && t < 8 && (t & 3) * 32 <= rn) pf_l2((t < 4 ? a.f_ptr : a.order) + p2 + r0 + (t & 3) * 32);
  }
  return st;
}
__device__ __forceinline__ void pf_end_fwd(const FwdArgs& a, const PfState& st) {
  if (st.qn <= 0) return;
  pf_range4(a.f_src, st.e0, st.e1);
  if ((int)threadIdx.x < st.qn) {
#pragma unroll
    for (int j = 0; j < 4; ++j) pf_l2(a.S + (int64_t)st.v * D + j * 32);
  }
}

// level 0 and odd levels: h[v] = relu(S[v] + mean_{u->v in net} h[u])  (model.py:103-108,148-153,186-187)
// NV float4 per lane, 32/NV lanes per pin.
template <int NV>
__device__ __forceinline__ void fwd_net_level(const FwdArgs& a, int p0, int cnt, Ctx& c, const GridBar& gb) {
  constexpr int G = 32 / NV, UN = (NV == 4) ? 2 : 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G;
  const int ngroups = gridDim.x * WARPS * NV;
  int p = (blockIdx.x * WARPS + warp) * NV + grp;
  int s = 0, e = 0, v = 0, idx[UN];
  float4 sv[NV];
  auto fetch = [&]() {
    s = __ldg(a.f_ptr + p0 + p);
    e = __ldg(a.f_ptr + p0 + p + 1);
    v = __ldg(a.order + p0 + p);
#pragma unroll
    for (int q = 0; q < UN; ++q) idx[q] = (s + q < e) ? __ldg(a.f_src + s + q) : 0;
#pragma unroll
    for (int j = 0; j < NV; ++j) sv[j] = ldg4(a.S + (int64_t)v * D + (j * G + lg) * 4);
  };
  if (p < cnt) fetch();
  gb.wait();
  c.stamp(PH_NPRE);
  while (p < cnt) {
    float4 acc[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) acc[j] = f4zero();
    for (int i = s; i < e; i += UN) {
      if (i > s) {
#pragma unroll
        for (int q = 0; q < UN; ++q) idx[q] = (i + q < e) ? __ldg(a.f_src + i + q) : 0;
      }
      float4 m[UN][NV];
#pragma unroll
      for (int q = 0; q < UN; ++q)
#pragma unroll
        for (int j = 0; j < NV; ++j)
          m[q][j] = (i + q < e) ? ldcg4(a.H + (int64_t)idx[q] * D + (j * G + lg) * 4) : f4zero();
#pragma unroll
      for (int q = 0; q < UN; ++q)
#pragma unroll
        for (int j = 0; j < NV; ++j) acc[j] = f4add(acc[j], m[q][j]);
    }
    const float rdeg = (e > s) ? 1.f / (float)(e - s) : 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j)
      *reinterpret_cast<float4*>(a.H + (int64_t)v * D + (j * G + lg) * 4) = f4relu(f4fma(acc[j], rdeg, sv[j]));
    p += ngroups;
    if (p < cnt) fetch();
  }
  c.stamp(PH_NBODY);
}

__global__ void __launch_bounds__(THREADS, 1) gnn_persist_fwd_kernel(const FwdArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  Ctx c;
  ctx_setup(c, smem, a.planes, a.prof);
  const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;
  GridBar gb{a.bar, gridDim.x, 0u};
  const bool save = a.A != nullptr;
  const int qd = warp & 3;
  const float b1m = __ldg(a.b1 + c.rank * 128 + qd * 32 + lane), b2m = __ldg(a.b2 + qd * 32 + lane);

  for (int l = a.lb; l < a.le; ++l) {
    const int p0 = __ldg(a.level_ptr + l), cnt = __ldg(a.level_ptr + l + 1) - p0;
    if (cnt <= 0) continue;
    {
      const PfState pf0 = pf_begin_fwd(a, l + 1, 0), pf1 = pf_begin_fwd(a, l + 1, 1);
      pf_end_fwd(a, pf0);
      pf_end_fwd(a, pf1);
    }
    if (l == 0 || (l & 1)) {
      const int nw = gridDim.x * WARPS;
      if (cnt <= nw) fwd_net_level<1>(a, p0, cnt, c, gb);
      else if (cnt <= 2 * nw) fwd_net_level<2>(a, p0, cnt, c, gb);
      else fwd_net_level<4>(a, p0, cnt, c, gb);
      gb.arrive();
      continue;
    }
    // even level > 0:  a = sum_e m_e softmax_e(m)_e per channel (model.py:113-116);
    //                  h = relu(S + W2 relu(W1 a + b1) + b2)     (model.py:138-146)
    const int crow0 = __ldg(a.cell_base + l);
    const int N = tile_width(cnt, nclusters), ntiles = (cnt + N - 1) / N;
    const int PPW = N >> 4;
    bool waited = false;
    for (int tile = cluster_id; tile < ntiles; tile += nclusters) {
      const int t0 = tile * N;
      const int r0 = warp * PPW;
      const int npin = min(PPW, cnt - (t0 + r0));            // <= 0 past the end of the level
      const int pb = p0 + t0 + r0;
      const bool owner = ((uint32_t)(warp >> 3) == c.rank);  // rows of the first half belong to CTA 0
      int ptrs = 0, vv = -1;
      if (npin > 0) {
        if (lane <= npin) ptrs = __ldg(a.f_ptr + pb + lane);
        if (lane < npin) vv = __ldg(a.order + pb + lane);
      }
      const int E0 = __shfl_sync(0xffffffffu, ptrs, 0), E1 = __shfl_sync(0xffffffffu, ptrs, max(npin, 0));
      int idx = (E0 + (lane & 7) < E1) ? __ldg(a.f_src + E0 + (lane & 7)) : 0;
      if (!waited) gb.wait();                                // ends with a CTA barrier
      else __syncthreads();                                  // the previous tile's epilogue still reads pin_s
      waited = true;
      c.stamp(PH_CPRE);

      // gather: online softmax over the warp's contiguous edge range (eight source rows in flight)
      int q = 0;
      float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      float sm[4] = {0.f, 0.f, 0.f, 0.f}, tw[4] = {0.f, 0.f, 0.f, 0.f};
      auto finish_pin = [&]() {
        float4 av = f4zero(), lse = av;
        if (sm[0] > 0.f) {
          av = make_float4(__fdividef(tw[0], sm[0]), __fdividef(tw[1], sm[1]), __fdividef(tw[2], sm[2]), __fdividef(tw[3], sm[3]));
          lse = make_float4(mx[0] + __logf(sm[0]), mx[1] + __logf(sm[1]), mx[2] + __logf(sm[2]), mx[3] + __logf(sm[3]));
        }
        if (save && owner) {
          const int64_t o = (int64_t)(crow0 + t0 + r0 + q) * D + lane * 4;
          *reinterpret_cast<float4*>(a.A + o) = av;
          *reinterpret_cast<float4*>(a.LSE + o) = lse;
        }
        store_pin_row(smem, r0 + q, lane, av, -4, __shfl_sync(0xffffffffu, vv, q));
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) { mx[ch] = -INFINITY; sm[ch] = 0.f; tw[ch] = 0.f; }
        ++q;
      };
      if (npin > 0) {
        int bnd = __shfl_sync(0xffffffffu, ptrs, 1);
        for (int i = E0; i < E1; i += 8) {
          if (i > E0) idx = (i + (lane & 7) < E1) ? __ldg(a.f_src + i + (lane & 7)) : 0;
          float4 m[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int src = __shfl_sync(0xffffffffu, idx, u);
            m[u] = (i + u < E1) ? ldcg4(a.H + (int64_t)src * D + lane * 4) : f4zero();
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            if (i + u < E1) {
              while (i + u >= bnd) { finish_pin(); bnd = __shfl_sync(0xffffffffu, ptrs, q + 1); }
              const float mv[4] = {m[u].x, m[u].y, m[u].z, m[u].w};
#pragma unroll
              for (int ch = 0; ch < 4; ++ch) {
                const float nm = fmaxf(mx[ch], mv[ch]);
                const float sc = __expf(mx[ch] - nm);        // exp(-inf) = 0 on the first edge
                const float ex = __expf(mv[ch] - nm);
                sm[ch] = sm[ch] * sc + ex;
                tw[ch] = tw[ch] * sc + mv[ch] * ex;
                mx[ch] = nm;
              }
            }
          }
        }
        while (q < npin) finish_pin();
      }
      for (int r = max(npin, 0); r < PPW; ++r) store_pin_row(smem, r0 + r, lane, f4zero(), -4, -1);

      // hidden = relu(W1 a + b1) in units of the pin's scale (s > 0 commutes with the ReLU)
      auto epi1 = [&](int n0, int m, float (&vm)[8], const float (&vc)[8]) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float hv = fmaxf(fmaf(vc[j], LO_INV, vm[j]) + b1m * c.scale_s[n0 + j], 0.f);
          vm[j] = hv;
          if (save && t0 + n0 + j < cnt) a.HIDb[(int64_t)(crow0 + t0 + n0 + j) * HID + c.rank * 128 + m] = hv * c.inv_s[n0 + j];
        }
      };
      const int cg = warp >> 2, nper = N >> 2;
      float sreg[NMAX / 4];
      auto pre2 = [&]() {                                    // S rows of the pins this warp finalises
        if ((uint32_t)(cg >> 1) == c.rank) {
#pragma unroll
          for (int j = 0; j < NMAX / 4; ++j) {
            sreg[j] = 0.f;
            if (j < nper) {
              const int v = c.pin_s[cg * nper + j];
              if (v >= 0) sreg[j] = __ldg(a.S + (int64_t)v * D + qd * 32 + lane);
            }
          }
        }
      };
      mlp_tile(c, N, [] {}, epi1, pre2);
      auto fin = [&](int n, int m, int slot, float val) {
        const int v = c.pin_s[n];
        if (v >= 0) a.H[(int64_t)v * D + m] = fmaxf(val + b2m + sreg[slot], 0.f);
      };
      exchange_tile(c, N, fin);
      c.stamp(PH_CPUB);
    }
    if (!waited) gb.wait();
    gb.arrive();
  }
  ctx_teardown(c);
}

// =============================================================================================
// backward: every pin PULLS its gradient over the out-edge lists (no atomics, deterministic)
//   net  edge v->u:  g_h[v] += g_z[u] / indeg_net(u)
//   cell edge v->u:  g_h[v] += g_a[u] * w_e * (1 + h[v] - a[u]),  w_e = exp(h[v] - lse[u])
//   g_z[v] = g_h[v] * (h[v] > 0)  -> G[v];  cell pins: g_hid = (W2^T g_z) * (hid > 0), g_a = W1^T g_hid
// =============================================================================================
struct BwdArgs {
  const int* level_ptr; const int* cell_base; const int* order;
  const int* bn_ptr; const int* bn_dst; const float* bn_w; const int* bc_ptr; const int* bc_row;
  const float* H; float* G;
  const uint8_t* planes;                                 // packed W2 [128][256], W1 [256][128] (gnn_pack_planes_kernel)
  const float* A; const float* LSE; const float* HIDb;
  float* GA; float* GHID; float* GZC;
  unsigned int* bar;               // grid-barrier counter (zeroed by gnn_persist_begin)
  long long* prof;
  int lb, le;                      // levels [lb, le) are processed (downwards)
};

__device__ __forceinline__ PfState pf_begin_bwd(const BwdArgs& a, int l1, int k) {
  PfState st{};
  if (l1 < 0) return st;
  const int p0 = __ldg(a.level_ptr + l1), cnt = __ldg(a.level_ptr + l1 + 1) - p0;
  int q0, qn;
  cta_range(l1, cnt, k, q0, qn);
  if (qn > 0) {
    if ((int)threadIdx.x < qn) st.v = __ldg(a.order + p0 + q0 + threadIdx.x);
    st.e0 = __ldg(a.bn_ptr + p0 + q0);
    st.e1 = __ldg(a.bn_ptr + p0 + q0 + qn);
    st.c0 = __ldg(a.bc_ptr + p0 + q0);
    st.c1 = __ldg(a.bc_ptr + p0 + q0 + qn);
    st.qn = qn;
    st.row0 = (l1 > 0 && !(l1 & 1)) ? __ldg(a.cell_base + l1) + q0 : -1;
  }
  if (k == 0 && l1 - 1 >= 0) {
    const int p2 = __ldg(a.level_ptr + l1 - 1), cnt2 = __ldg(a.level_ptr + l1) - p2;
    int r0, rn;
    cta_range(l1 - 1, cnt2, 0, r0, rn);
    const int t = threadIdx.x;
    if (rn > 0 && t < 12 && (t & 3) * 32 <= rn)
      pf_l2((t < 4 ? a.bn_ptr : (t < 8 ? a.bc_ptr : a.order)) + p2 + r0 + (t & 3) * 32);
  }
  return st;
}
__device__ __forceinline__ void pf_end_bwd(const BwdArgs& a, const PfState& st, uint32_t rank) {
  if (st.qn <= 0) return;
  pf_range4(a.bn_dst, st.e0, st.e1);
  pf_range4(a.bn_w, st.e0, st.e1);
  pf_range4(a.bc_row, st.c0, st.c1);
  if ((int)threadIdx.x < st.qn) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      pf_l2(a.H + (int64_t)st.v * D + j * 32);
      pf_l2(a.G + (int64_t)st.v * D + j * 32);
      if (st.row0 >= 0) pf_l2(a.HIDb + (int64_t)(st.row0 + (int)threadIdx.x) * HID + rank * 128 + j * 32);
    }
  }
}

// hraw[k] with a k that is a compile-time constant after unrolling for each of the three 8-column chunks
__device__ __forceinline__ float hsel(const float (&h)[NMAX / 4], int k) {
  float r = 0.f;
#pragma unroll
  for (int i = 0; i < NMAX / 4; ++i) r = (i == k) ? h[i] : r;
  return r;
}

template <int NV>
__device__ __forceinline__ void bwd_net_level(const BwdArgs& a, int p0, int cnt, Ctx& c, const GridBar& gb) {
  constexpr int G = 32 / NV, UN = (NV == 4) ? 2 : 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int lg = lane % G, grp = lane / G;
  const int ngroups = gridDim.x * WARPS * NV;
  int p = (blockIdx.x * WARPS + warp) * NV + grp;
  int ns = 0, ne = 0, cs = 0, ce = 0, v = 0, ndst[UN], crow[2];
  float nw[UN];
  float4 hv[NV], g[NV];
  auto fetch = [&]() {
    ns = __ldg(a.bn_ptr + p0 + p); ne = __ldg(a.bn_ptr + p0 + p + 1);
    cs = __ldg(a.bc_ptr + p0 + p); ce = __ldg(a.bc_ptr + p0 + p + 1);
    v = __ldg(a.order + p0 + p);
#pragma unroll
    for (int q = 0; q < UN; ++q) {
      ndst[q] = (ns + q < ne) ? __ldg(a.bn_dst + ns + q) : 0;
      nw[q] = (ns + q < ne) ? __ldg(a.bn_w + ns + q) : 0.f;
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) crow[q] = (cs + q < ce) ? __ldg(a.bc_row + cs + q) : 0;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      hv[j] = ldg4(a.H + (int64_t)v * D + (j * G + lg) * 4);
      g[j] = ldcg4(a.G + (int64_t)v * D + (j * G + lg) * 4);     // the head's gradient: written before the launch
    }
  };
  if (p < cnt) fetch();
  gb.wait();
  c.stamp(PH_NPRE);
  while (p < cnt) {
    for (int i = ns; i < ne; i += UN) {
      if (i > ns) {
#pragma unroll
        for (int q = 0; q < UN; ++q) {
          ndst[q] = (i + q < ne) ? __ldg(a.bn_dst + i + q) : 0;
          nw[q] = (i + q < ne) ? __ldg(a.bn_w + i + q) : 0.f;
        }
      }
      float4 m[UN][NV];
#pragma unroll
      for (int q = 0; q < UN; ++q)
#pragma unroll
        for (int j = 0; j < NV; ++j)
          m[q][j] = (i + q < ne) ? ldcg4(a.G + (int64_t)ndst[q] * D + (j * G + lg) * 4) : f4zero();
#pragma unroll
      for (int q = 0; q < UN; ++q)
#pragma unroll
        for (int j = 0; j < NV; ++j) g[j] = f4fma(m[q][j], nw[q], g[j]);
    }
    for (int i = cs; i < ce; i += 2) {
      if (i > cs) {
#pragma unroll
        for (int q = 0; q < 2; ++q) crow[q] = (i + q < ce) ? __ldg(a.bc_row + i + q) : 0;
      }
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        if (i + q < ce) {
          float4 ls[NV], aa[NV];
#pragma unroll
          for (int j = 0; j < NV; ++j) {
            const int64_t co = (int64_t)crow[q] * D + (j * G + lg) * 4;
            ls[j] = ldg4(a.LSE + co);
            aa[j] = ldg4(a.A + co);
          }
#pragma unroll
          for (int j = 0; j < NV; ++j)
            g[j] = f4add(g[j], cell_edge_grad(hv[j], ldcg4(a.GA + (int64_t)crow[q] * D + (j * G + lg) * 4), ls[j], aa[j]));
        }
      }
    }
#pragma unroll
    for (int j = 0; j < NV; ++j)
      *reinterpret_cast<float4*>(a.G + (int64_t)v * D + (j * G + lg) * 4) = relu_mask(hv[j], g[j]);
    p += ngroups;
    if (p < cnt) fetch();
  }
  c.stamp(PH_NBODY);
}

// WG == false: G and GA only.  GHID / GZC (the operands of the hoisted weight-gradient GEMMs) are not stored; g_z stays
// in registers until the pair's exchange barrier instead of being staged in GZC.
template <bool WG>
__global__ void __launch_bounds__(THREADS, 1) gnn_persist_bwd_kernel(const BwdArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  Ctx c;
  ctx_setup(c, smem, a.planes, a.prof);
  const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;
  float* scratch = reinterpret_cast<float*>(smem + OFF_B);      // [N][128] fp32 gradient accumulators during the gather
  GridBar gb{a.bar, gridDim.x, 0u};

  for (int l = a.le - 1; l >= a.lb; --l) {
    const int p0 = __ldg(a.level_ptr + l), cnt = __ldg(a.level_ptr + l + 1) - p0;
    if (cnt <= 0) continue;
    {
      const PfState pf0 = pf_begin_bwd(a, l - 1, 0), pf1 = pf_begin_bwd(a, l - 1, 1);
      pf_end_bwd(a, pf0, c.rank);
      pf_end_bwd(a, pf1, c.rank);
    }
    if (l == 0 || (l & 1)) {
      const int nw = gridDim.x * WARPS;
      if (cnt <= nw) bwd_net_level<1>(a, p0, cnt, c, gb);
      else if (cnt <= 2 * nw) bwd_net_level<2>(a, p0, cnt, c, gb);
      else bwd_net_level<4>(a, p0, cnt, c, gb);
      gb.arrive();
      continue;
    }
    const int crow0 = __ldg(a.cell_base + l);
    const int N = tile_width(cnt, nclusters), ntiles = (cnt + N - 1) / N;
    const int PPW = N >> 4;
    bool waited = false;
    for (int tile = cluster_id; tile < ntiles; tile += nclusters) {
      const int t0 = tile * N;
      const int r0 = warp * PPW;
      const int npin = min(PPW, cnt - (t0 + r0));
      const int pb = p0 + t0 + r0;
      const bool owner = ((uint32_t)(warp >> 3) == c.rank);
      int nptr = 0, cptr = 0, vv = -1;
      if (npin > 0) {
        if (lane <= npin) { nptr = __ldg(a.bn_ptr + pb + lane); cptr = __ldg(a.bc_ptr + pb + lane); }
        if (lane < npin) vv = __ldg(a.order + pb + lane);
      }
      const int E0 = __shfl_sync(0xffffffffu, nptr, 0), E1 = __shfl_sync(0xffffffffu, nptr, max(npin, 0));
      int idx = 0;
      float wt = 0.f;
      if (E0 + (lane & 7) < E1) { idx = __ldg(a.bn_dst + E0 + (lane & 7)); wt = __ldg(a.bn_w + E0 + (lane & 7)); }
      if (!waited) gb.wait();                                // ends with a CTA barrier
      else __syncthreads();                                  // the previous tile's epilogue still reads the scales
      waited = true;
      c.stamp(PH_CPRE);

      // gather (both CTAs of the pair, redundantly): accumulators live in the fp32 scratch rows
#pragma unroll
      for (int r = 0; r < NMAX / 16; ++r) {
        if (r < PPW) {
          float4 g = f4zero();
          if (r < npin) g = ldcg4(a.G + (int64_t)__shfl_sync(0xffffffffu, vv, r) * D + lane * 4);
          *reinterpret_cast<float4*>(scratch + (r0 + r) * D + lane * 4) = g;
        }
      }
      if (npin > 0) {
        {  // net out-edges: one contiguous range for the warp's pins
          int q = 0, bnd = __shfl_sync(0xffffffffu, nptr, 1);
          float4 acc = f4zero();
          auto flush = [&]() {
            float4* dst = reinterpret_cast<float4*>(scratch + (r0 + q) * D + lane * 4);
            *dst = f4add(*dst, acc);
            acc = f4zero();
            ++q;
          };
          for (int i = E0; i < E1; i += 8) {
            if (i > E0) {
              const bool ok = i + (lane & 7) < E1;
              idx = ok ? __ldg(a.bn_dst + i + (lane & 7)) : 0;
              wt = ok ? __ldg(a.bn_w + i + (lane & 7)) : 0.f;
            }
            float4 m[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const int dst = __shfl_sync(0xffffffffu, idx, u);
              m[u] = (i + u < E1) ? ldcg4(a.G + (int64_t)dst * D + lane * 4) : f4zero();
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const float wu = __shfl_sync(0xffffffffu, wt, u);
              if (i + u < E1) {
                while (i + u >= bnd) { flush(); bnd = __shfl_sync(0xffffffffu, nptr, q + 1); }
                acc = f4fma(m[u], wu, acc);
              }
            }
          }
          if (q < npin) flush();
        }
        {  // cell out-edges (rare on cell levels)
          const int C0 = __shfl_sync(0xffffffffu, cptr, 0), C1 = __shfl_sync(0xffffffffu, cptr, npin);
          int q = 0, bnd = __shfl_sync(0xffffffffu, cptr, 1);
          for (int i = C0; i < C1; ++i) {
            while (i >= bnd) { ++q; bnd = __shfl_sync(0xffffffffu, cptr, q + 1); }
            const int row = __ldg(a.bc_row + i);
            const int64_t co = (int64_t)row * D + lane * 4;
            const float4 hv = ldg4(a.H + (int64_t)__shfl_sync(0xffffffffu, vv, q) * D + lane * 4);
            float4* dst = reinterpret_cast<float4*>(scratch + (r0 + q) * D + lane * 4);
            *dst = f4add(*dst, cell_edge_grad(hv, ldcg4(a.GA + co), ldg4(a.LSE + co), ldg4(a.A + co)));
          }
        }
      }
      // g_z = g_h * (h > 0): into registers; the owner CTA publishes it as GZC (G[v] itself is
      // rewritten only after the pair's barrier: the peer gathers the same pins from G)
      float4 gz[NMAX / 16];
#pragma unroll
      for (int r = 0; r < NMAX / 16; ++r) {
        gz[r] = f4zero();
        if (r < PPW && r < npin) {
          const float4 hv = ldg4(a.H + (int64_t)__shfl_sync(0xffffffffu, vv, r) * D + lane * 4);
          gz[r] = relu_mask(hv, *reinterpret_cast<const float4*>(scratch + (r0 + r) * D + lane * 4));
          if (WG && owner) *reinterpret_cast<float4*>(a.GZC + (int64_t)(crow0 + t0 + r0 + r) * D + lane * 4) = gz[r];
        }
      }
      __syncthreads();                                       // every warp is done with the scratch rows
#pragma unroll
      for (int r = 0; r < NMAX / 16; ++r)
        if (r < PPW) store_pin_row(smem, r0 + r, lane, gz[r], -100, r < npin ? __shfl_sync(0xffffffffu, vv, r) : -1);

      // g_hid = (W2^T g_z) * (hid > 0), in units of the pin's scale.  The ReLU mask of this thread's hidden unit
      // for the warp's pins is fetched (one bit per pin) while the first product runs.
      const int cg = warp >> 2, nper = N >> 2, qd = warp & 3;
      float hraw[NMAX / 4];                                  // raw loads: consumed only in the epilogue, after the MMA wait
      auto pre1 = [&]() {
#pragma unroll
        for (int j = 0; j < NMAX / 4; ++j) {
          hraw[j] = 0.f;
          if (j < nper && t0 + cg * nper + j < cnt)
            hraw[j] = __ldg(a.HIDb + (int64_t)(crow0 + t0 + cg * nper + j) * HID + c.rank * 128 + qd * 32 + lane);
        }
      };
      auto epi1 = [&](int n0, int m, float (&vm)[8], const float (&vc)[8]) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float gh = 0.f;
          if (t0 + n0 + j < cnt) {
            gh = hsel(hraw, n0 - cg * nper + j) > 0.f ? fmaf(vc[j], LO_INV, vm[j]) : 0.f;
            if constexpr (WG) a.GHID[(int64_t)(crow0 + t0 + n0 + j) * HID + c.rank * 128 + m] = gh * c.inv_s[n0 + j];
          }
          vm[j] = gh;
        }
      };
      mlp_tile(c, N, pre1, epi1, [] {});
      auto fin = [&](int n, int m, int, float val) {
        if (t0 + n < cnt) a.GA[(int64_t)(crow0 + t0 + n) * D + m] = val;
      };
      exchange_tile(c, N, fin);
      // the peer has finished gathering (it passed the exchange barrier): G[v] = g_z
      if (owner) {
#pragma unroll
        for (int r = 0; r < NMAX / 16; ++r)
          if (r < PPW && r < npin)
            *reinterpret_cast<float4*>(a.G + (int64_t)__shfl_sync(0xffffffffu, vv, r) * D + lane * 4) =
                WG ? *reinterpret_cast<const float4*>(a.GZC + (int64_t)(crow0 + t0 + r0 + r) * D + lane * 4) : gz[r];
      }
      c.stamp(PH_CPUB);
    }
    if (!waited) gb.wait();
    gb.arrive();
  }
  ctx_teardown(c);
}

// =============================================================================================
// save-only forward (tm_gnn_save_cone): what the forward saves for the backward -- A, LSE and HID -- recomputed over the
// cell levels of a sub-schedule whose in-edge sources are all final in H.  Per tile: the gather's online softmax and
// MMA 1 with its per-pin scale; no MMA 2, no exchange, no H store.  No level waits for another, so there is no grid
// barrier and the tiles of all levels are dealt to the clusters round-robin.  The gather and epilogue 1 repeat
// gnn_persist_fwd_kernel's expressions one for one: a pin's rows depend only on its own sources, its scale and the
// weights (not on the tile it shares), so they are the same bits the full forward saves.
// =============================================================================================
struct SaveArgs {
  const int* level_ptr; const int* cell_base; const int* order; const int* f_ptr; const int* f_src;
  const float* H;
  const uint8_t* planes; const float* b1;                                 // packed fc_cell_neigh weights
  float* A; float* LSE; float* HIDb;
  long long* prof;
  int L;
};

__global__ void __launch_bounds__(THREADS, 1) gnn_persist_save_kernel(const SaveArgs a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  Ctx c;
  ctx_setup(c, smem, a.planes, a.prof);
  const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;
  const int qd = warp & 3, cg = warp >> 2, m = qd * 32 + lane;
  const float b1m = __ldg(a.b1 + c.rank * 128 + qd * 32 + lane);
  const uint32_t sW = smem_u32(c.smem + OFF_W), sB = smem_u32(c.smem + OFF_B);
  const uint32_t tl = c.tmem + ((uint32_t)(qd * 32) << 16);
  int dealt = 0;                                             // tiles of the levels before this one
  for (int l = 2; l < a.L; l += 2) {
    const int p0 = __ldg(a.level_ptr + l), cnt = __ldg(a.level_ptr + l + 1) - p0;
    if (cnt <= 0) continue;
    const int crow0 = __ldg(a.cell_base + l);
    const int N = tile_width(cnt, nclusters), ntiles = (cnt + N - 1) / N;
    const int PPW = N >> 4, nper = N >> 2;
    const int first = (cluster_id - dealt % nclusters + nclusters) % nclusters;
    dealt += ntiles;
    for (int tile = first; tile < ntiles; tile += nclusters) {
      const int t0 = tile * N;
      const int r0 = warp * PPW;
      const int npin = min(PPW, cnt - (t0 + r0));
      const int pb = p0 + t0 + r0;
      const bool owner = ((uint32_t)(warp >> 3) == c.rank);
      int ptrs = 0, vv = -1;
      if (npin > 0) {
        if (lane <= npin) ptrs = __ldg(a.f_ptr + pb + lane);
        if (lane < npin) vv = __ldg(a.order + pb + lane);
      }
      const int E0 = __shfl_sync(0xffffffffu, ptrs, 0), E1 = __shfl_sync(0xffffffffu, ptrs, max(npin, 0));
      int idx = (E0 + (lane & 7) < E1) ? __ldg(a.f_src + E0 + (lane & 7)) : 0;
      tc_fence_before();
      __syncthreads();                                       // the previous tile's epilogue still reads the scales
      c.stamp(PH_CPRE);

      int q = 0;
      float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      float sm[4] = {0.f, 0.f, 0.f, 0.f}, tw[4] = {0.f, 0.f, 0.f, 0.f};
      auto finish_pin = [&]() {
        float4 av = f4zero(), lse = av;
        if (sm[0] > 0.f) {
          av = make_float4(__fdividef(tw[0], sm[0]), __fdividef(tw[1], sm[1]), __fdividef(tw[2], sm[2]), __fdividef(tw[3], sm[3]));
          lse = make_float4(mx[0] + __logf(sm[0]), mx[1] + __logf(sm[1]), mx[2] + __logf(sm[2]), mx[3] + __logf(sm[3]));
        }
        if (owner) {
          const int64_t o = (int64_t)(crow0 + t0 + r0 + q) * D + lane * 4;
          *reinterpret_cast<float4*>(a.A + o) = av;
          *reinterpret_cast<float4*>(a.LSE + o) = lse;
        }
        store_pin_row(smem, r0 + q, lane, av, -4, __shfl_sync(0xffffffffu, vv, q));
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) { mx[ch] = -INFINITY; sm[ch] = 0.f; tw[ch] = 0.f; }
        ++q;
      };
      if (npin > 0) {
        int bnd = __shfl_sync(0xffffffffu, ptrs, 1);
        for (int i = E0; i < E1; i += 8) {
          if (i > E0) idx = (i + (lane & 7) < E1) ? __ldg(a.f_src + i + (lane & 7)) : 0;
          float4 mv8[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int src = __shfl_sync(0xffffffffu, idx, u);
            mv8[u] = (i + u < E1) ? ldcg4(a.H + (int64_t)src * D + lane * 4) : f4zero();
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            if (i + u < E1) {
              while (i + u >= bnd) { finish_pin(); bnd = __shfl_sync(0xffffffffu, ptrs, q + 1); }
              const float mv[4] = {mv8[u].x, mv8[u].y, mv8[u].z, mv8[u].w};
#pragma unroll
              for (int ch = 0; ch < 4; ++ch) {
                const float nm = fmaxf(mx[ch], mv[ch]);
                const float sc = __expf(mx[ch] - nm);
                const float ex = __expf(mv[ch] - nm);
                sm[ch] = sm[ch] * sc + ex;
                tw[ch] = tw[ch] * sc + mv[ch] * ex;
                mx[ch] = nm;
              }
            }
          }
        }
        while (q < npin) finish_pin();
      }
      for (int r = max(npin, 0); r < PPW; ++r) store_pin_row(smem, r0 + r, lane, f4zero(), -4, -1);

      // MMA 1 and its epilogue: hidden = relu(W1 a + b1), stored unscaled
      fence_async_smem();
      tc_fence_before();
      __syncthreads();
      c.stamp(PH_GATHER);
      if (tid == 0) {
        tc_fence_after();
        issue_gemm(sW, sW + W_PLANE, sB, sB + B_PLANE, c.tmem + TM_MAIN1, c.tmem + TM_CORR1, make_idesc(Fmt::F16, N), c.mbar);
      }
      mbar_wait_trap<MBAR_SPINS>(c.mbar, c.mphase);
      c.mphase ^= 1u;
      tc_fence_after();
      c.stamp(PH_MMA1);
#pragma unroll
      for (int cc = 0; cc < NMAX / 4 / 8; ++cc) {
        if (cc * 8 < nper) {
          const int n0 = cg * nper + cc * 8;
          float vm[8], vc[8];
          tmem_ld8(tl + TM_MAIN1 + n0, vm);
          tmem_ld8(tl + TM_CORR1 + n0, vc);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float hv = fmaxf(fmaf(vc[j], LO_INV, vm[j]) + b1m * c.scale_s[n0 + j], 0.f);
            if (t0 + n0 + j < cnt) a.HIDb[(int64_t)(crow0 + t0 + n0 + j) * HID + c.rank * 128 + m] = hv * c.inv_s[n0 + j];
          }
        }
      }
      c.stamp(PH_EPI1);
    }
  }
  ctx_teardown(c);
}

// ---------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------
template <class Args>
int launch_persist(void (*kern)(const Args), const Args& args, cudaStream_t st, const char* what) {
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // every CTA must be resident at once (the grid barrier waits for all of them): size the grid by what the
  // device can hold, one CTA per SM
  cfg.gridDim = dim3((unsigned)(sm_count() & ~1));
  int ncl = 0;
  // Inside a stream capture the attribute and occupancy calls are skipped when an eager launch on this device already
  // made them (the attribute persists; the cluster count is cached): a captured launch then makes no driver query.
  static std::atomic<int> ncl_cache[64];
  int dev = 0;
  TM_CUDA(cudaGetDevice(&dev));
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  TM_CUDA(cudaStreamIsCapturing(st, &cap));
  if (cap != cudaStreamCaptureStatusNone && dev < 64) ncl = ncl_cache[dev].load(std::memory_order_relaxed);
  if (ncl == 0) {
    TM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    TM_CUDA(cudaOccupancyMaxActiveClusters(&ncl, kern, &cfg));
    if (dev < 64 && ncl >= 1) ncl_cache[dev].store(ncl, std::memory_order_relaxed);
  }
  TM_REQUIRE(ncl >= 1, "%s: no 2-CTA cluster with %u bytes of shared memory fits this device", what, SMEM_BYTES);
  cfg.gridDim = dim3((unsigned)(2 * std::min(ncl, sm_count() / 2)));
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (e != cudaSuccess) return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
  return 0;
}

// workspace: the packed weight planes of both CTA ranks (256-byte aligned), then the grid-barrier counter on a
// 256-byte slot of its own
constexpr size_t WS_PLANES = 2 * 4 * W_PLANE, WS_BAR = 256;
uint8_t* ws_planes(void* ws) { return reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255); }
unsigned int* ws_bar(void* ws) { return reinterpret_cast<unsigned int*>(ws_planes(ws) + WS_PLANES); }
}  // namespace

namespace tmk {
size_t gnn_persist_ws_bytes() { return 256 + WS_PLANES + WS_BAR; }
static long long* g_prof = nullptr;
void gnn_persist_set_profile(long long* p) { g_prof = p; }
int gnn_persist_profile_slots() { return PH_COUNT; }

// pack the fc_cell_neigh planes and clear the barrier counter: once per pass
int gnn_persist_begin(const tm_schedule* s, const float* Wa, const float* Wb, void* ws, cudaStream_t st) {
  TM_REQUIRE(s->level_ptr && s->cell_base, "tm_gnn: schedule lacks the device level_ptr / cell_base arrays");
  TM_CUDA(cudaMemsetAsync(ws_bar(ws), 0, WS_BAR, st));
  gnn_pack_planes_kernel<<<2 * 2 * 128 * 128 / 256, 256, 0, st>>>(Wa, Wb, ws_planes(ws));
  return check_launch("gnn_pack_planes");
}

int gnn_persist_forward(const tm_schedule* s, int lb, int le, float* H, const float* S, const float* W1t, const float* b1,
                        const float* W2t, const float* b2, float* A, float* LSE, float* HIDb, void* ws, cudaStream_t st) {
  TM_TRY(gnn_persist_begin(s, W1t, W2t, ws, st));
  FwdArgs a{s->level_ptr, s->cell_base, s->order, s->f_ptr, s->f_src, S, H, ws_planes(ws), b1, b2, A, LSE, HIDb,
            ws_bar(ws), g_prof, lb, le};
  return launch_persist(gnn_persist_fwd_kernel, a, st, "gnn_persist_fwd");
}

int gnn_persist_backward(const tm_schedule* s, const float* H, float* G, const float* W1, const float* W2, const float* A,
                         const float* LSE, const float* HIDb, float* GA, float* GHID, float* GZC, void* ws, cudaStream_t st,
                         int lb, int le) {
  TM_TRY(gnn_persist_begin(s, W2, W1, ws, st));
  BwdArgs a{s->level_ptr, s->cell_base, s->order, s->bn_ptr, s->bn_dst, s->bn_w, s->bc_ptr, s->bc_row, H, G, ws_planes(ws),
            A, LSE, HIDb, GA, GHID, GZC, ws_bar(ws), g_prof, lb, le};
  if (GHID) return launch_persist(gnn_persist_bwd_kernel<true>, a, st, "gnn_persist_bwd");
  return launch_persist(gnn_persist_bwd_kernel<false>, a, st, "gnn_persist_bwd");
}

int gnn_persist_save(const tm_schedule* s, const float* H, const float* W1t, const float* b1, const float* W2t, float* A,
                     float* LSE, float* HIDb, void* ws, cudaStream_t st) {
  TM_TRY(gnn_persist_begin(s, W1t, W2t, ws, st));
  SaveArgs a{s->level_ptr, s->cell_base, s->order, s->f_ptr, s->f_src, H, ws_planes(ws), b1, A, LSE, HIDb, g_prof,
             s->num_levels};
  return launch_persist(gnn_persist_save_kernel, a, st, "gnn_persist_save");
}
}  // namespace tmk
