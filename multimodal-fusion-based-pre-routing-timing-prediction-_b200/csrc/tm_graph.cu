// G1: graph structure kernels -- CSR build, level construction, level schedule.
//
// Replaces (reference call sites): dgl.heterograph + DGL's lazy in-edge CSR used by graph.pull
// (src/dataset.py:274-278, src/model.py:186-204) and Parser.cal_topo_level
// (src/verilog_parser_asap7.py:1452-1517).  All integer work, bit-exact against
// oracle/levelize.py.  HBM-bound byte/integer kernels: coalesced grid-stride loops, no tensor cores.
#include <cooperative_groups.h>

#include "tm_common.cuh"

namespace cg = cooperative_groups;

using namespace tmk;

// ------------------------------------------------------------------------------------------
// exclusive scan (3 kernels).  Logical element i lives at physical index phys(i); with
// transposed != 0 the input is a [W][L] matrix scanned in column-major (l-major) order.
// ------------------------------------------------------------------------------------------
namespace {
constexpr int SCAN_T = 256;
constexpr int SCAN_E = 8;
constexpr int SCAN_B = SCAN_T * SCAN_E;

__device__ __forceinline__ int64_t scan_phys(int64_t i, int64_t W, int64_t L, int transposed) {
  if (!transposed || i >= W * L) return i;
  return (i % W) * L + (i / W);
}

__global__ void scan_local_kernel(const int* __restrict__ in, int* __restrict__ out,
                                  int* __restrict__ bsum, int64_t n, int64_t W, int64_t L,
                                  int transposed) {
  __shared__ int wsum[SCAN_T / 32];
  const int64_t base = (int64_t)blockIdx.x * SCAN_B + (int64_t)threadIdx.x * SCAN_E;
  int v[SCAN_E];
  int run = 0;
#pragma unroll
  for (int i = 0; i < SCAN_E; ++i) {
    int64_t g = base + i;
    int x = (g < n) ? in[scan_phys(g, W, L, transposed)] : 0;
    v[i] = run;
    run += x;
  }
  int incl = run;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  int woff = 0;
  for (int w = 0; w < warp; ++w) woff += wsum[w];
  const int off = woff + incl - run;
#pragma unroll
  for (int i = 0; i < SCAN_E; ++i) {
    int64_t g = base + i;
    if (g < n) out[scan_phys(g, W, L, transposed)] = v[i] + off;
  }
  if (threadIdx.x == SCAN_T - 1) bsum[blockIdx.x] = off + run;
}

__global__ void scan_bsum_kernel(int* __restrict__ bsum, int64_t nb) {
  // single block, sequential over chunks of blockDim.x
  __shared__ int wsum[32];
  __shared__ int carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t base = 0; base < nb; base += blockDim.x) {
    int64_t g = base + threadIdx.x;
    int x = (g < nb) ? bsum[g] : 0;
    int incl = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += wsum[w];
    int carry = carry_s;
    if (g < nb) bsum[g] = carry + woff + incl - x;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = carry + woff + incl;
    __syncthreads();
  }
}

__global__ void scan_add_kernel(int* __restrict__ out, const int* __restrict__ bsum, int64_t n,
                                int64_t W, int64_t L, int transposed) {
  int64_t g = (int64_t)blockIdx.x * SCAN_B + threadIdx.x;
  const int add = bsum[blockIdx.x];
#pragma unroll
  for (int i = 0; i < SCAN_E; ++i, g += SCAN_T)
    if (g < n) out[scan_phys(g, W, L, transposed)] += add;
}

inline size_t scan_ws_ints(int64_t n) { return (size_t)cdiv(n, SCAN_B) + 1; }

int exclusive_scan(const int* in, int* out, int64_t n, int* bsum, int64_t W, int64_t L,
                   int transposed, cudaStream_t st) {
  if (n <= 0) return 0;
  const int64_t nb = cdiv(n, SCAN_B);
  scan_local_kernel<<<(unsigned)nb, SCAN_T, 0, st>>>(in, out, bsum, n, W, L, transposed);
  TM_TRY(check_launch("scan_local"));
  if (nb > 1) {
    scan_bsum_kernel<<<1, 1024, 0, st>>>(bsum, nb);
    TM_TRY(check_launch("scan_bsum"));
    scan_add_kernel<<<(unsigned)nb, SCAN_T, 0, st>>>(out, bsum, n, W, L, transposed);
    TM_TRY(check_launch("scan_add"));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// CSR build
// ------------------------------------------------------------------------------------------
__global__ void csr_count_kernel(const int64_t* __restrict__ key, int64_t e, int* __restrict__ cnt) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < e;
       i += (int64_t)gridDim.x * blockDim.x)
    atomicAdd(&cnt[key[i]], 1);
}

__global__ void csr_fill_kernel(const int64_t* __restrict__ key, const int64_t* __restrict__ val,
                                int64_t e, int* __restrict__ cursor, int* __restrict__ indices) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < e;
       i += (int64_t)gridDim.x * blockDim.x) {
    int pos = atomicAdd(&cursor[key[i]], 1);
    indices[pos] = (int)val[i];
  }
}

// one warp per row; ascending, duplicates kept.  All comparators ascending ("flip" bitonic
// network) so that +inf padding never moves real elements past the end of a long row.
__global__ void csr_rowsort_kernel(const int* __restrict__ indptr, int* __restrict__ indices,
                                   int64_t n) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = wid; r < n; r += nw) {
    const int s = indptr[r], deg = indptr[r + 1] - s;
    if (deg <= 1) continue;
    if (deg <= 32) {
      int x = lane < deg ? indices[s + lane] : INT_MAX;
#pragma unroll
      for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
          int y = __shfl_xor_sync(0xffffffffu, x, j);
          bool keep_min = ((lane & j) == 0) == ((lane & k) == 0);
          x = keep_min ? min(x, y) : max(x, y);
        }
      }
      if (lane < deg) indices[s + lane] = x;
    } else {
      int P = 64;
      while (P < deg) P <<= 1;
      int* v = indices + s;
      for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
          const bool flip = (j == (k >> 1));
          for (int t = lane; t < P; t += 32) {
            int l = flip ? (t ^ (k - 1)) : (t ^ j);
            if (l > t && l < deg) {
              int a = v[t], b = v[l];
              if (a > b) { v[t] = b; v[l] = a; }
            }
          }
          __syncwarp();
        }
      }
    }
  }
}

inline unsigned grid_for(int64_t work, int threads, int per_sm = 8) {
  int64_t want = cdiv(work, threads);
  int64_t cap = (int64_t)sm_count() * per_sm;
  if (want < 1) want = 1;
  return (unsigned)(want < cap ? want : cap);
}
}  // namespace

extern "C" size_t tm_csr_build_ws(int64_t n, int64_t e) {
  (void)e;
  return (size_t)(2 * (n + 1) + (int64_t)scan_ws_ints(n + 1)) * sizeof(int) + 3 * 256;
}

extern "C" int tm_csr_build(int64_t n, int64_t e, const int64_t* key, const int64_t* val,
                            int32_t* indptr, int32_t* indices, void* ws, size_t ws_bytes,
                            void* stream) {
  TM_REQUIRE(n >= 0 && e >= 0 && n < INT32_MAX && e < INT32_MAX, "tm_csr_build: bad sizes");
  TM_REQUIRE(ws_bytes >= tm_csr_build_ws(n, e), "tm_csr_build: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  Carver c(ws);
  int* cnt = c.take<int>(n + 1);
  int* cursor = c.take<int>(n + 1);
  int* bsum = c.take<int>(scan_ws_ints(n + 1));
  TM_CUDA(cudaMemsetAsync(cnt, 0, (size_t)(n + 1) * sizeof(int), st));
  if (e > 0) {
    csr_count_kernel<<<grid_for(e, 256), 256, 0, st>>>(key, e, cnt);
    TM_TRY(check_launch("csr_count"));
  }
  TM_TRY(exclusive_scan(cnt, indptr, n + 1, bsum, 0, 0, 0, st));
  if (e > 0) {
    TM_CUDA(cudaMemcpyAsync(cursor, indptr, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToDevice, st));
    csr_fill_kernel<<<grid_for(e, 256), 256, 0, st>>>(key, val, e, cursor, indices);
    TM_TRY(check_launch("csr_fill"));
    csr_rowsort_kernel<<<grid_for(n * 32, 256), 256, 0, st>>>(indptr, indices, n);
    TM_TRY(check_launch("csr_rowsort"));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// level construction: one cooperative persistent kernel
//   pass 1  frontier BFS from the PI set: reach[] and in-degree inside the reachable sub-graph
//   pass 2  Kahn peeling: iteration k assigns level k to every pin whose reachable
//           predecessors are all done  ==  longest walk from the PI set  ==  the last frontier
//           the pin appears in (verilog_parser_asap7.py:1494-1511)
// ------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256)
levelize_kernel(int n, const int* __restrict__ optr, const int* __restrict__ oidx,
                const int64_t* __restrict__ pis, int n_pi, int* __restrict__ level,
                int* __restrict__ num_levels, int* __restrict__ reach, int* __restrict__ indeg,
                int* qa, int* qb, int* cnt) {
  cg::grid_group grid = cg::this_grid();
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const int nth = gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  const int wid = tid >> 5, nw = nth >> 5;
  volatile int* vcnt = cnt;

  for (int i = tid; i < n; i += nth) { reach[i] = 0; indeg[i] = 0; level[i] = -1; }
  if (tid == 0) { cnt[0] = 0; cnt[1] = 0; cnt[2] = 0; }
  grid.sync();
  for (int i = tid; i < n_pi; i += nth) {
    int64_t p = pis[i];
    if (p >= 0 && p < n && atomicExch(&reach[(int)p], 1) == 0) qa[atomicAdd(&cnt[0], 1)] = (int)p;
  }
  grid.sync();
  int* qin = qa;
  int* qout = qb;
  int it = 0;
  while (true) {
    const int nf = vcnt[it % 3];
    if (nf == 0) break;
    if (tid == 0) cnt[(it + 2) % 3] = 0;
    int* oc = &cnt[(it + 1) % 3];
    for (int w = wid; w < nf; w += nw) {
      const int u = qin[w];
      const int e1 = optr[u + 1];
      for (int e = optr[u] + lane; e < e1; e += 32) {
        const int v = oidx[e];
        atomicAdd(&indeg[v], 1);
        if (atomicExch(&reach[v], 1) == 0) qout[atomicAdd(oc, 1)] = v;
      }
    }
    grid.sync();
    int* t = qin; qin = qout; qout = t;
    ++it;
  }
  grid.sync();
  if (tid == 0) { cnt[0] = 0; cnt[1] = 0; cnt[2] = 0; }
  grid.sync();
  for (int i = tid; i < n; i += nth)
    if (reach[i] && indeg[i] == 0) qa[atomicAdd(&cnt[0], 1)] = i;
  grid.sync();
  qin = qa; qout = qb; it = 0;
  while (true) {
    const int nf = vcnt[it % 3];
    if (nf == 0) break;
    if (tid == 0) cnt[(it + 2) % 3] = 0;
    int* oc = &cnt[(it + 1) % 3];
    for (int w = wid; w < nf; w += nw) {
      const int u = qin[w];
      if (lane == 0) level[u] = it;
      const int e1 = optr[u + 1];
      for (int e = optr[u] + lane; e < e1; e += 32) {
        const int v = oidx[e];
        if (atomicSub(&indeg[v], 1) == 1) qout[atomicAdd(oc, 1)] = v;
      }
    }
    grid.sync();
    int* t = qin; qin = qout; qout = t;
    ++it;
  }
  if (tid == 0) *num_levels = it;
}
}  // namespace

extern "C" size_t tm_levelize_ws(int64_t n) { return (size_t)(4 * n + 16) * sizeof(int) + 6 * 256; }

extern "C" int tm_levelize(int64_t n, const int32_t* optr, const int32_t* oidx, const int64_t* pis,
                           int64_t n_pi, int32_t* level, int32_t* num_levels, void* ws,
                           size_t ws_bytes, void* stream) {
  TM_REQUIRE(n > 0 && n < INT32_MAX && n_pi >= 0 && n_pi < INT32_MAX, "tm_levelize: bad sizes");
  TM_REQUIRE(ws_bytes >= tm_levelize_ws(n), "tm_levelize: workspace too small");
  Carver c(ws);
  int* reach = c.take<int>(n);
  int* indeg = c.take<int>(n);
  int* qa = c.take<int>(n);
  int* qb = c.take<int>(n);
  int* cnt = c.take<int>(16);
  int per_sm = 0;
  TM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, levelize_kernel, 256, 0));
  TM_REQUIRE(per_sm >= 1, "tm_levelize: kernel does not fit an SM");
  if (per_sm > 4) per_sm = 4;
  int ni = (int)n, npi = (int)n_pi;
  void* args[] = {&ni, (void*)&optr, (void*)&oidx, (void*)&pis, &npi, &level, &num_levels,
                  &reach, &indeg, &qa, &qb, &cnt};
  TM_CUDA(cudaLaunchCooperativeKernel((void*)levelize_kernel, dim3(sm_count() * per_sm), dim3(256),
                                      args, 0, (cudaStream_t)stream));
  return check_launch("levelize");
}

// ------------------------------------------------------------------------------------------
// level order: stable counting sort of pins by level (ascending pin id inside a level)
// ------------------------------------------------------------------------------------------
namespace {
constexpr int LO_CHUNK = 1024;  // pins per warp

__global__ void lvl_hist_kernel(const int* __restrict__ level, int64_t n, int L, int* __restrict__ hist) {
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t base = w * LO_CHUNK;
  if (base >= n) return;
  int* row = hist + w * L;
  for (int i = lane; i < LO_CHUNK; i += 32) {
    int64_t v = base + i;
    if (v < n) {
      int l = level[v];
      if (l >= 0) atomicAdd(&row[l], 1);
    }
  }
}

__global__ void lvl_ptr_kernel(const int* __restrict__ base, int64_t W, int L, int* __restrict__ level_ptr) {
  int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < L) level_ptr[l] = base[l];                // chunk 0 holds the first slot of each level
  if (l == L) level_ptr[L] = base[W * (int64_t)L];  // total
}

__global__ void lvl_scatter_kernel(const int* __restrict__ level, int64_t n, int L, int* base,
                                   int* __restrict__ order) {
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t b0 = w * LO_CHUNK;
  if (b0 >= n) return;
  volatile int* row = base + w * L;
  for (int i = 0; i < LO_CHUNK; i += 32) {
    int64_t v = b0 + i + lane;
    int l = (v < n) ? level[v] : -1;
    unsigned same = __match_any_sync(0xffffffffu, l);
    if (l >= 0) {
      int rank = __popc(same & ((1u << lane) - 1u));
      int start = row[l];
      order[start + rank] = (int)v;
    }
    __syncwarp();
    if (l >= 0 && lane == (__ffs(same) - 1)) row[l] = row[l] + __popc(same);
    __syncwarp();
  }
}

__global__ void sched_aux_kernel(int L, const int* __restrict__ level,
                                 const int* __restrict__ order, const int* __restrict__ level_ptr,
                                 const int* __restrict__ cell_base, const int* __restrict__ net_iptr,
                                 const int* __restrict__ net_isrc, const int* __restrict__ cell_iptr,
                                 const int* __restrict__ cell_isrc, int* __restrict__ crow,
                                 int* __restrict__ n_viol) {
  int bad = 0;
  const int64_t n_sched = level_ptr[L];
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_sched;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int v = order[p];
    const int l = level[v];
    const bool is_cell = (l > 0) && ((l & 1) == 0);
    crow[v] = is_cell ? cell_base[l] + (int)(p - level_ptr[l]) : -1;
    if (l & 1) {
      for (int e = net_iptr[v]; e < net_iptr[v + 1]; ++e) bad += (level[net_isrc[e]] >= l);
    } else if (l > 0) {
      for (int e = cell_iptr[v]; e < cell_iptr[v + 1]; ++e) bad += (level[cell_isrc[e]] >= l);
    }
  }
  if (bad) atomicAdd(n_viol, bad);
}

__global__ void cell_base_kernel(const int* __restrict__ level_ptr, int L, int* __restrict__ cell_base) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int acc = 0;
    for (int l = 0; l <= L; ++l) {
      cell_base[l] = acc;
      if (l < L && l > 0 && (l & 1) == 0) acc += level_ptr[l + 1] - level_ptr[l];
    }
  }
}
}  // namespace

extern "C" size_t tm_level_order_ws(int64_t n, int32_t L) {
  int64_t W = cdiv(n, LO_CHUNK);
  int64_t cells = W * (int64_t)L + 1;
  return (size_t)(cells + (int64_t)scan_ws_ints(cells)) * sizeof(int) + 2 * 256;
}

extern "C" int tm_level_order(int64_t n, int32_t L, const int32_t* level, int32_t* order,
                              int32_t* level_ptr, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(n > 0 && L > 0, "tm_level_order: bad sizes");
  TM_REQUIRE(ws_bytes >= tm_level_order_ws(n, L), "tm_level_order: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t W = cdiv(n, LO_CHUNK);
  const int64_t cells = W * (int64_t)L + 1;
  Carver c(ws);
  int* hist = c.take<int>(cells);
  int* bsum = c.take<int>(scan_ws_ints(cells));
  TM_CUDA(cudaMemsetAsync(hist, 0, (size_t)cells * sizeof(int), st));
  const unsigned blocks = (unsigned)cdiv(W * 32, 128);
  lvl_hist_kernel<<<blocks, 128, 0, st>>>(level, n, L, hist);
  TM_TRY(check_launch("lvl_hist"));
  TM_TRY(exclusive_scan(hist, hist, cells, bsum, W, L, 1, st));
  lvl_ptr_kernel<<<(unsigned)cdiv(L + 1, 128), 128, 0, st>>>(hist, W, L, level_ptr);
  TM_TRY(check_launch("lvl_ptr"));
  lvl_scatter_kernel<<<blocks, 128, 0, st>>>(level, n, L, hist, order);
  return check_launch("lvl_scatter");
}

extern "C" int tm_schedule_aux(int64_t n, int32_t L, const int32_t* level, const int32_t* order,
                               const int32_t* level_ptr, const int32_t* net_iptr,
                               const int32_t* net_isrc, const int32_t* cell_iptr,
                               const int32_t* cell_isrc, int32_t* crow, int32_t* cell_base,
                               int32_t* n_violations, void* stream) {
  TM_REQUIRE(n > 0 && L > 0, "tm_schedule_aux: bad sizes");
  cudaStream_t st = (cudaStream_t)stream;
  TM_CUDA(cudaMemsetAsync(crow, 0xFF, (size_t)n * sizeof(int), st));
  cell_base_kernel<<<1, 32, 0, st>>>(level_ptr, L, cell_base);
  TM_TRY(check_launch("cell_base"));
  sched_aux_kernel<<<grid_for(n, 256), 256, 0, st>>>(L, level, order, level_ptr, cell_base, net_iptr,
                                                     net_isrc, cell_iptr, cell_isrc, crow, n_violations);
  return check_launch("sched_aux");
}

// ------------------------------------------------------------------------------------------
// level-ordered edge lists: the gather structures of the propagation kernels.
// For schedule position p (pin v = order[p], level l):
//   forward   f_ptr/f_src : sources of the in-edges pulled on v's level (net if l odd, cell if
//                           l even > 0, none on level 0);
//   backward  bn_ptr/bn_dst/bn_w : net out-edges v->u that carry gradient (u on a later odd
//                           level) with weight 1/indeg_net(u);
//             bc_ptr/bc_row : cell out-edges v->u that carry gradient (u on a later even level),
//                           stored as the compact row crow[u].
// Positions are contiguous per level, so a warp that owns consecutive pins reads one contiguous
// edge range: the dependent-load chain of a gather is ptr -> src -> row (3 deep).
// ------------------------------------------------------------------------------------------
namespace {
struct EdgeIn {
  const int* order; const int* level; const int* crow;
  const int* net_iptr; const int* net_isrc; const int* cell_iptr; const int* cell_isrc;
  const int* net_optr; const int* net_odst; const int* cell_optr; const int* cell_odst;
};

__global__ void sched_edges_count_kernel(EdgeIn g, int64_t n_sched, int* __restrict__ cf,
                                         int* __restrict__ cbn, int* __restrict__ cbc) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p > n_sched) return;
  if (p == n_sched) { cf[p] = 0; cbn[p] = 0; cbc[p] = 0; return; }
  const int v = g.order[p], l = g.level[v];
  cf[p] = (l & 1) ? g.net_iptr[v + 1] - g.net_iptr[v] : (l > 0 ? g.cell_iptr[v + 1] - g.cell_iptr[v] : 0);
  int a = 0, b = 0;
  for (int e = g.net_optr[v]; e < g.net_optr[v + 1]; ++e) { const int lu = g.level[g.net_odst[e]]; a += ((lu & 1) && lu > l); }
  for (int e = g.cell_optr[v]; e < g.cell_optr[v + 1]; ++e) { const int lu = g.level[g.cell_odst[e]]; b += (lu > 0 && !(lu & 1) && lu > l); }
  cbn[p] = a;
  cbc[p] = b;
}

__global__ void sched_edges_fill_kernel(EdgeIn g, int64_t n_sched, const int* __restrict__ f_ptr,
                                        int* __restrict__ f_src, const int* __restrict__ bn_ptr,
                                        int* __restrict__ bn_dst, float* __restrict__ bn_w,
                                        const int* __restrict__ bc_ptr, int* __restrict__ bc_row) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_sched) return;
  const int v = g.order[p], l = g.level[v];
  int o = f_ptr[p];
  if (l & 1) { for (int e = g.net_iptr[v]; e < g.net_iptr[v + 1]; ++e) f_src[o++] = g.net_isrc[e]; }
  else if (l > 0) { for (int e = g.cell_iptr[v]; e < g.cell_iptr[v + 1]; ++e) f_src[o++] = g.cell_isrc[e]; }
  o = bn_ptr[p];
  for (int e = g.net_optr[v]; e < g.net_optr[v + 1]; ++e) {
    const int u = g.net_odst[e], lu = g.level[u];
    if ((lu & 1) && lu > l) { bn_dst[o] = u; bn_w[o] = 1.f / (float)(g.net_iptr[u + 1] - g.net_iptr[u]); ++o; }
  }
  o = bc_ptr[p];
  for (int e = g.cell_optr[v]; e < g.cell_optr[v + 1]; ++e) {
    const int u = g.cell_odst[e], lu = g.level[u];
    if (lu > 0 && !(lu & 1) && lu > l) bc_row[o++] = g.crow[u];
  }
}
}  // namespace

extern "C" size_t tm_schedule_edges_ws(int64_t n_sched) {
  return (size_t)(3 * (n_sched + 1) + 3 * (int64_t)scan_ws_ints(n_sched + 1)) * sizeof(int) + 8 * 256;
}

extern "C" int tm_schedule_edges(const tm_schedule* s, int64_t n_sched, int32_t* f_ptr, int32_t* f_src,
                                 int32_t* bn_ptr, int32_t* bn_dst, float* bn_w, int32_t* bc_ptr,
                                 int32_t* bc_row, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(s && n_sched > 0, "tm_schedule_edges: bad schedule");
  TM_REQUIRE(ws_bytes >= tm_schedule_edges_ws(n_sched), "tm_schedule_edges: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  Carver c(ws);
  int* cf = c.take<int>(n_sched + 1);
  int* cbn = c.take<int>(n_sched + 1);
  int* cbc = c.take<int>(n_sched + 1);
  int* b0 = c.take<int>(scan_ws_ints(n_sched + 1));
  int* b1 = c.take<int>(scan_ws_ints(n_sched + 1));
  int* b2 = c.take<int>(scan_ws_ints(n_sched + 1));
  EdgeIn g{s->order, s->level, s->crow, s->net_iptr, s->net_isrc, s->cell_iptr, s->cell_isrc,
           s->net_optr, s->net_odst, s->cell_optr, s->cell_odst};
  const unsigned blocks = (unsigned)cdiv(n_sched + 1, 256);
  sched_edges_count_kernel<<<blocks, 256, 0, st>>>(g, n_sched, cf, cbn, cbc);
  TM_TRY(check_launch("sched_edges_count"));
  TM_TRY(exclusive_scan(cf, f_ptr, n_sched + 1, b0, 0, 0, 0, st));
  TM_TRY(exclusive_scan(cbn, bn_ptr, n_sched + 1, b1, 0, 0, 0, st));
  TM_TRY(exclusive_scan(cbc, bc_ptr, n_sched + 1, b2, 0, 0, 0, st));
  sched_edges_fill_kernel<<<blocks, 256, 0, st>>>(g, n_sched, f_ptr, f_src, bn_ptr, bn_dst, bn_w, bc_ptr, bc_row);
  return check_launch("sched_edges_fill");
}

// ------------------------------------------------------------------------------------------
// forward cone: the sub-schedule of the pins whose H row can change after the self terms S of
// some seed pins changed -- every scheduled pin reachable from a seed along the in-edges the
// propagation reads (the f_ptr / f_src lists), the seeds included.
//
// ONE thread block sweeps the levels from the lowest seed's level upwards, PULLING: a pin is in
// the cone when it is a seed or one of its f_src sources is.  Sources sit on earlier levels, so
// a level depends only on the levels below it, and the level boundary is a __syncthreads, not a
// grid-wide barrier (a whole-GPU barrier per level would cost about what the propagation over a
// small cone does).  Membership is one bit per pin, in shared memory when it fits, else in the
// workspace.  The same pass compacts the cone: a block scan of (in-cone, in-degree) per chunk of
// positions gives each member its cone position and edge offset, so order / f_ptr / f_src are
// written in the parent's order, and level_ptr and the count fall out of the running totals.
// Work: every schedule position from the lowest seed's level on (one read of order / f_ptr /
// f_src there), in L - lmin dependent steps; the next level's arrays are prefetched into L2 while
// the current one is processed.
//
// The sweep itself only needs "is any source of this position marked", so a backward cone (the
// pins an endpoint batch reads) is the same loop run downwards over out-edge lists.
// ------------------------------------------------------------------------------------------
namespace {
constexpr int CONE_T = 1024;
constexpr int CONE_V = 4;                          // consecutive schedule positions per thread per chunk
constexpr int CONE_CHUNK = CONE_T * CONE_V;
constexpr size_t CONE_SMEM_MAX = 192 * 1024;       // membership bitmap in shared memory up to 1.5M pins

struct ConeArgs {
  int n, L;
  const int* level; const int* level_ptr; const int* order; const int* f_ptr; const int* f_src;
  const int* seeds; int n_seeds;
  uint32_t* gbits;                                 // NULL: the bitmap lives in dynamic shared memory
  int* c_order; int* c_level_ptr; int* c_f_ptr; int* c_f_src; int* c_count;
};

__device__ __forceinline__ void pf_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ bool cone_bit(const volatile uint32_t* bits, int v) {
  return (bits[v >> 5] >> (v & 31)) & 1u;
}

__global__ void __launch_bounds__(CONE_T, 1) fwd_cone_kernel(const ConeArgs a) {
  extern __shared__ uint32_t sbits[];
  __shared__ int wsum_c[CONE_T / 32], wsum_e[CONE_T / 32];
  __shared__ int s_lmin;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t* bits = a.gbits ? a.gbits : sbits;      // generic: shared or global
  const volatile uint32_t* vbits = bits;
  if (!a.gbits)
    for (int i = tid; i < ((a.n + 31) >> 5); i += CONE_T) sbits[i] = 0u;
  if (tid == 0) s_lmin = a.L;
  __syncthreads();
  for (int i = tid; i < a.n_seeds; i += CONE_T) {
    const int v = a.seeds[i];
    if (v < 0 || v >= a.n) continue;
    const int l = a.level[v];
    if (l < 0 || l >= a.L) continue;               // outside the schedule: changes nothing
    atomicOr(bits + (v >> 5), 1u << (v & 31));
    atomicMin(&s_lmin, l);
  }
  __syncthreads();
  const int lmin = s_lmin;
  for (int l = tid; l < lmin; l += CONE_T) a.c_level_ptr[l] = 0;
  int run_c = 0, run_e = 0;                        // cone pins / edges so far (block-uniform)
  for (int l = lmin; l < a.L; ++l) {
    const int p0 = __ldg(a.level_ptr + l), p1 = __ldg(a.level_ptr + l + 1);
    if (tid == 0) a.c_level_ptr[l] = run_c;
    int p2 = p1, fa = 0, fb = 0;
    if (l + 1 < a.L) {
      p2 = __ldg(a.level_ptr + l + 2);
      fa = __ldg(a.f_ptr + p1);
      fb = __ldg(a.f_ptr + p2);
    }
    for (int c0 = p0; c0 < p1; c0 += CONE_CHUNK) {
      const int q = c0 + tid * CONE_V;
      const int nq = max(0, min(CONE_V, p1 - q));
      int ptr[CONE_V + 1], v[CONE_V];
      bool in[CONE_V];
#pragma unroll
      for (int j = 0; j <= CONE_V; ++j) ptr[j] = (j <= nq && nq > 0) ? __ldg(a.f_ptr + q + j) : 0;
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) v[j] = j < nq ? __ldg(a.order + q + j) : 0;
      if (c0 == p0) {                              // the next level's static arrays into L2
        for (int i = p1 + tid * 32; i < p2; i += CONE_T * 32) {
          pf_l2(a.order + i);
          pf_l2(a.f_ptr + i);
        }
        for (int i = fa + tid * 32; i < fb; i += CONE_T * 32) pf_l2(a.f_src + i);
      }
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) in[j] = j < nq && cone_bit(vbits, v[j]);
      int e1 = ptr[0];                             // ptr[nq] without a dynamic register index
#pragma unroll
      for (int j = 1; j <= CONE_V; ++j) e1 = j == nq ? ptr[j] : e1;
      const int e0 = ptr[0];
      for (int e = e0; e < e1; e += 8) {
        int src[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) src[u] = e + u < e1 ? __ldg(a.f_src + e + u) : -1;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (src[u] >= 0 && cone_bit(vbits, src[u])) {
#pragma unroll
            for (int j = 0; j < CONE_V; ++j) in[j] |= (e + u >= ptr[j] && e + u < ptr[j + 1]);
          }
        }
      }
      int cnt = 0, edg = 0;
#pragma unroll
      for (int j = 0; j < CONE_V; ++j)
        if (in[j]) { ++cnt; edg += ptr[j + 1] - ptr[j]; }
      // block-wide exclusive scan of (cnt, edg)
      int ic = cnt, ie = edg;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int yc = __shfl_up_sync(0xffffffffu, ic, o), ye = __shfl_up_sync(0xffffffffu, ie, o);
        if (lane >= o) { ic += yc; ie += ye; }
      }
      if (lane == 31) { wsum_c[warp] = ic; wsum_e[warp] = ie; }
      __syncthreads();
      int oc = 0, oe = 0, tc = 0, te = 0;
#pragma unroll 8
      for (int w = 0; w < CONE_T / 32; ++w) {
        const int xc = wsum_c[w], xe = wsum_e[w];
        if (w < warp) { oc += xc; oe += xe; }
        tc += xc;
        te += xe;
      }
      int pos = run_c + oc + ic - cnt, eo = run_e + oe + ie - edg;
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) {
        if (in[j]) {
          a.c_order[pos] = v[j];
          a.c_f_ptr[pos] = eo;
          for (int e = ptr[j]; e < ptr[j + 1]; ++e) a.c_f_src[eo++] = __ldg(a.f_src + e);
          ++pos;
          atomicOr(bits + (v[j] >> 5), 1u << (v[j] & 31));
        }
      }
      run_c += tc;
      run_e += te;
      __syncthreads();                             // bits of this level are set; wsum may be reused
    }
  }
  if (tid == 0) {
    a.c_level_ptr[a.L] = run_c;
    a.c_f_ptr[run_c] = run_e;
    *a.c_count = run_c;
  }
}
}  // namespace

extern "C" size_t tm_forward_cone_ws(int64_t n) { return (size_t)cdiv(n, 32) * sizeof(uint32_t) + 256; }

extern "C" int tm_forward_cone(const tm_schedule* s, int64_t n_seeds, const int32_t* seeds, int32_t* order,
                               int32_t* level_ptr, int32_t* f_ptr, int32_t* f_src, int32_t* count, void* ws,
                               size_t ws_bytes, void* stream) {
  TM_REQUIRE(s && s->order && s->level && s->level_ptr && s->f_ptr && s->f_src,
             "tm_forward_cone: the parent schedule lacks its device arrays (order, level, level_ptr, f_ptr, f_src)");
  TM_REQUIRE(s->n > 0 && s->n < INT32_MAX && s->num_levels > 0, "tm_forward_cone: bad schedule sizes");
  TM_REQUIRE(n_seeds >= 0 && n_seeds < INT32_MAX && (n_seeds == 0 || seeds), "tm_forward_cone: bad seed list");
  TM_REQUIRE(order && level_ptr && f_ptr && f_src && count, "tm_forward_cone: NULL output buffer");
  TM_REQUIRE(ws && ws_bytes >= tm_forward_cone_ws(s->n), "tm_forward_cone: workspace too small (tm_forward_cone_ws)");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t bit_bytes = (size_t)cdiv(s->n, 32) * sizeof(uint32_t);
  const bool in_smem = bit_bytes <= CONE_SMEM_MAX;
  uint32_t* gbits = nullptr;
  if (!in_smem) {
    gbits = reinterpret_cast<uint32_t*>(ws);
    TM_CUDA(cudaMemsetAsync(gbits, 0, bit_bytes, st));
  }
  TM_CUDA(cudaFuncSetAttribute(fwd_cone_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CONE_SMEM_MAX));
  ConeArgs a{(int)s->n, s->num_levels, s->level, s->level_ptr, s->order, s->f_ptr, s->f_src, seeds, (int)n_seeds,
             gbits, order, level_ptr, f_ptr, f_src, count};
  fwd_cone_kernel<<<1, CONE_T, in_smem ? bit_bytes : 0, st>>>(a);
  return check_launch("fwd_cone");
}

// ------------------------------------------------------------------------------------------
// fan-in cone: the sub-schedule a backward pass seeded on some endpoints reads -- every scheduled pin from which a
// seeded endpoint is reachable along the out-edges that carry gradient (bn_dst, and the cell out-edges bc_row), the
// seeded endpoints included.  Every other pin's gradient is exactly zero in the full backward, so the edges into such
// pins are dropped: no sum changes except possibly the sign of a zero.  Every in-edge source of a cone pin is in the
// cone (the source's out-edge to it carries gradient), so the in-edge lists are copied unchanged.
//
// fwd_cone_kernel's loop run downwards: ONE block sweeps from the highest seeded level to level 0, and a position is in
// the cone when its pin is a seeded endpoint or one of its carrying out-edges leads into the cone.  Destinations sit on
// later levels, so a level depends only on the levels above it.  Pins are marked in the same bitmap; a cell out-edge
// names its destination's compact cell row, so row_map[row] (-1 outside the cone) is both the membership test of that
// destination and its cone row.
// The cone is laid out from the END of the buffers (positions, edges and cell rows): each chunk of positions takes the
// block just below what the chunks above it took, and the chunks of a level are visited from the top, so the layout is
// the parent's order with ascending levels, and no second pass is needed.  The class lists (fc_cell_self /
// fc_net_self rows of the self-MLP data gradients) start at index 0 in the sweep's (descending) order.
// ------------------------------------------------------------------------------------------
namespace {
struct FaninArgs {
  int n, L, T;
  const int* level; const int* level_ptr; const int* cell_base; const int* order; const int* f_ptr; const int* f_src;
  const int* bn_ptr; const int* bn_dst; const float* bn_w; const int* bc_ptr; const int* bc_row;
  const int* endpoints; const float* seed;
  uint32_t* gbits;                                 // NULL: the bitmap lives in dynamic shared memory
  int* row_map;                                    // parent cell row -> cone cell row, -1 outside the cone
  int* c_order; int* c_level_ptr; int* c_cell_base; int* c_f_ptr; int* c_f_src;
  int* c_bn_ptr; int* c_bn_dst; float* c_bn_w; int* c_bc_ptr; int* c_bc_row;
  int* c_cell_pins; int* c_net_pins; int* c_counts;
};

// exclusive block scan of four ints over CONE_T threads; tot receives the block totals.  The caller syncs before wsum
// is reused.
__device__ __forceinline__ void block_scan4(int (&x)[4], int (&tot)[4], int (*wsum)[32]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) inc[k] = x[k];
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int y = __shfl_up_sync(0xffffffffu, inc[k], o);
      if (lane >= o) inc[k] += y;
    }
  }
  if (lane == 31) {
#pragma unroll
    for (int k = 0; k < 4; ++k) wsum[k][warp] = inc[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int off = 0, t = 0;
#pragma unroll 8
    for (int w = 0; w < CONE_T / 32; ++w) {
      const int xv = wsum[k][w];
      if (w < warp) off += xv;
      t += xv;
    }
    x[k] = off + inc[k] - x[k];
    tot[k] = t;
  }
}

__global__ void __launch_bounds__(CONE_T, 1) fanin_cone_kernel(const FaninArgs a) {
  extern __shared__ uint32_t sbits[];
  __shared__ int wsum[4][32];
  __shared__ int s_lmax;
  const int tid = threadIdx.x;
  uint32_t* bits = a.gbits ? a.gbits : sbits;      // generic: shared or global
  const volatile uint32_t* vbits = bits;
  const volatile int* vrow = a.row_map;            // written by this block on the levels above
  if (!a.gbits)
    for (int i = tid; i < ((a.n + 31) >> 5); i += CONE_T) sbits[i] = 0u;
  if (tid == 0) s_lmax = -1;
  __syncthreads();
  for (int t = tid; t < a.T; t += CONE_T) {
    if (a.seed[t] == 0.f) continue;                // an unseeded endpoint: its gradient is exactly zero
    const int v = a.endpoints[t];
    if (v < 0 || v >= a.n) continue;
    const int l = a.level[v];
    if (l < 0 || l >= a.L) continue;               // outside the schedule: reads nothing
    atomicOr(bits + (v >> 5), 1u << (v & 31));
    atomicMax(&s_lmax, l);
  }
  __syncthreads();
  const int lmax = s_lmax;
  const int ns = __ldg(a.level_ptr + a.L);
  int top = ns, ftop = __ldg(a.f_ptr + ns), ntop = __ldg(a.bn_ptr + ns), ctop = __ldg(a.bc_ptr + ns);
  int rtop = __ldg(a.cell_base + a.L), ncell = 0, nnet = 0;   // block-uniform running totals
  for (int l = lmax + 1 + tid; l <= a.L; l += CONE_T) {
    a.c_level_ptr[l] = ns;
    a.c_cell_base[l] = rtop;
  }
  if (tid == 0) {
    a.c_f_ptr[ns] = ftop;
    a.c_bn_ptr[ns] = ntop;
    a.c_bc_ptr[ns] = ctop;
  }
  for (int l = lmax; l >= 0; --l) {
    const int p0 = __ldg(a.level_ptr + l), p1 = __ldg(a.level_ptr + l + 1);
    const bool cell_rows = l > 0 && !(l & 1);
    const int crow0 = cell_rows ? __ldg(a.cell_base + l) : 0;
    if (l > 0) {                                   // the next level's static arrays into L2
      const int pm = __ldg(a.level_ptr + l - 1);
      for (int i = pm + tid * 32; i < p0; i += CONE_T * 32) {
        pf_l2(a.order + i);
        pf_l2(a.bn_ptr + i);
        pf_l2(a.bc_ptr + i);
      }
      for (int i = __ldg(a.bn_ptr + pm) + tid * 32; i < __ldg(a.bn_ptr + p0); i += CONE_T * 32) pf_l2(a.bn_dst + i);
      for (int i = __ldg(a.bc_ptr + pm) + tid * 32; i < __ldg(a.bc_ptr + p0); i += CONE_T * 32) pf_l2(a.bc_row + i);
    }
    for (int c0 = p1 > p0 ? p0 + (p1 - p0 - 1) / CONE_CHUNK * CONE_CHUNK : p0 - 1; c0 >= p0; c0 -= CONE_CHUNK) {
      const int q = c0 + tid * CONE_V;
      const int nq = max(0, min(CONE_V, p1 - q));
      int nptr[CONE_V + 1], cptr[CONE_V + 1], v[CONE_V];
      bool in[CONE_V];
      // pins, in-edges, net out-edges kept, cell out-edges kept; a pin outside the cone has no kept out-edge, so the
      // kept edges are counted over all of the thread's positions
      int x[4] = {0, 0, 0, 0}, tot[4];
#pragma unroll
      for (int j = 0; j <= CONE_V; ++j) {
        nptr[j] = (j <= nq && nq > 0) ? __ldg(a.bn_ptr + q + j) : 0;
        cptr[j] = (j <= nq && nq > 0) ? __ldg(a.bc_ptr + q + j) : 0;
      }
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) {
        v[j] = j < nq ? __ldg(a.order + q + j) : 0;
        in[j] = false;
      }
      int ne1 = nptr[0], ce1 = cptr[0];            // ptr[nq] without a dynamic register index
#pragma unroll
      for (int j = 1; j <= CONE_V; ++j) {
        ne1 = j == nq ? nptr[j] : ne1;
        ce1 = j == nq ? cptr[j] : ce1;
      }
      for (int e = nptr[0]; e < ne1; e += 8) {     // net out-edges into the cone
        int dst[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) dst[u] = e + u < ne1 ? __ldg(a.bn_dst + e + u) : -1;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (dst[u] >= 0 && cone_bit(vbits, dst[u])) {
            ++x[2];
#pragma unroll
            for (int j = 0; j < CONE_V; ++j) in[j] |= (e + u >= nptr[j] && e + u < nptr[j + 1]);
          }
        }
      }
      for (int e = cptr[0]; e < ce1; e += 8) {     // cell out-edges into the cone
        int row[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) row[u] = e + u < ce1 ? __ldg(a.bc_row + e + u) : -1;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (row[u] >= 0 && vrow[row[u]] >= 0) {
            ++x[3];
#pragma unroll
            for (int j = 0; j < CONE_V; ++j) in[j] |= (e + u >= cptr[j] && e + u < cptr[j + 1]);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) {
        in[j] = j < nq && (in[j] || cone_bit(vbits, v[j]));
        if (in[j]) {
          ++x[0];
          x[1] += __ldg(a.f_ptr + q + j + 1) - __ldg(a.f_ptr + q + j);
        }
      }
      block_scan4(x, tot, wsum);
      int rank = x[0];                             // cone pins of this chunk before this thread's first
      int pos = top - tot[0] + x[0], fo = ftop - tot[1] + x[1], no = ntop - tot[2] + x[2], co = ctop - tot[3] + x[3];
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) {
        if (in[j]) {
          a.c_order[pos] = v[j];
          a.c_f_ptr[pos] = fo;
          for (int e = __ldg(a.f_ptr + q + j); e < __ldg(a.f_ptr + q + j + 1); ++e) a.c_f_src[fo++] = __ldg(a.f_src + e);
          a.c_bn_ptr[pos] = no;
          for (int e = nptr[j]; e < nptr[j + 1]; ++e) {
            const int u = __ldg(a.bn_dst + e);
            if (cone_bit(vbits, u)) {
              a.c_bn_dst[no] = u;
              a.c_bn_w[no] = __ldg(a.bn_w + e);
              ++no;
            }
          }
          a.c_bc_ptr[pos] = co;
          for (int e = cptr[j]; e < cptr[j + 1]; ++e) {
            const int r = vrow[__ldg(a.bc_row + e)];
            if (r >= 0) a.c_bc_row[co++] = r;
          }
          if (cell_rows) a.row_map[crow0 + (q + j - p0)] = rtop - tot[0] + rank;
          if (l & 1) a.c_net_pins[nnet + tot[0] - 1 - rank] = v[j];
          else a.c_cell_pins[ncell + tot[0] - 1 - rank] = v[j];
          atomicOr(bits + (v[j] >> 5), 1u << (v[j] & 31));
          ++pos;
          ++rank;
        }
      }
      top -= tot[0];
      ftop -= tot[1];
      ntop -= tot[2];
      ctop -= tot[3];
      if (cell_rows) rtop -= tot[0];
      if (l & 1) nnet += tot[0];
      else ncell += tot[0];
      __syncthreads();                             // bits / row_map of this chunk are set; wsum may be reused
    }
    if (tid == 0) {
      a.c_level_ptr[l] = top;
      a.c_cell_base[l] = rtop;
    }
  }
  if (tid == 0) {
    a.c_counts[0] = ns - top;
    a.c_counts[1] = ncell;
    a.c_counts[2] = nnet;
  }
}

size_t fanin_bits_bytes(int64_t n) { return ((size_t)cdiv(n, 32) * sizeof(uint32_t) + 255) & ~(size_t)255; }
}  // namespace

extern "C" size_t tm_fanin_cone_ws(int64_t n, int32_t n_cell_rows) {
  return fanin_bits_bytes(n) + (size_t)(n_cell_rows > 0 ? n_cell_rows : 0) * sizeof(int) + 256;
}

// bits_out NULL: the bitmap lives in shared memory (or the workspace over 1.5M pins) and dies with the build; else the
// same kernel keeps it in bits_out, which outlives the build (tm_fanin_cone_bits)
static int fanin_cone_launch(const tm_schedule* s, int64_t n_endpoints, const int32_t* endpoints, const float* seed,
                             int32_t* order, int32_t* level_ptr, int32_t* cell_base, int32_t* f_ptr, int32_t* f_src,
                             int32_t* bn_ptr, int32_t* bn_dst, float* bn_w, int32_t* bc_ptr, int32_t* bc_row,
                             int32_t* cell_pins, int32_t* net_pins, int32_t* counts, uint32_t* bits_out, void* ws,
                             size_t ws_bytes, void* stream) {
  TM_REQUIRE(s && s->order && s->level && s->level_ptr && s->cell_base && s->f_ptr && s->f_src && s->bn_ptr &&
                 s->bn_dst && s->bn_w && s->bc_ptr && s->bc_row,
             "tm_fanin_cone: the parent schedule lacks its device arrays (order, level, level_ptr, cell_base, f_ptr, "
             "f_src, bn_ptr, bn_dst, bn_w, bc_ptr, bc_row)");
  TM_REQUIRE(s->n > 0 && s->n < INT32_MAX && s->num_levels > 0 && s->n_cell_rows >= 0,
             "tm_fanin_cone: bad schedule sizes");
  TM_REQUIRE(n_endpoints >= 0 && n_endpoints < INT32_MAX && (n_endpoints == 0 || (endpoints && seed)),
             "tm_fanin_cone: bad endpoint list or seed");
  TM_REQUIRE(order && level_ptr && cell_base && f_ptr && f_src && bn_ptr && bn_dst && bn_w && bc_ptr && bc_row &&
                 cell_pins && net_pins && counts,
             "tm_fanin_cone: NULL output buffer");
  TM_REQUIRE(ws && ws_bytes >= tm_fanin_cone_ws(s->n, s->n_cell_rows),
             "tm_fanin_cone: workspace too small (tm_fanin_cone_ws)");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t bit_bytes = (size_t)cdiv(s->n, 32) * sizeof(uint32_t);
  const bool in_smem = !bits_out && bit_bytes <= CONE_SMEM_MAX;
  uint8_t* p = reinterpret_cast<uint8_t*>(ws);
  uint32_t* gbits = nullptr;
  if (!in_smem) {
    gbits = bits_out ? bits_out : reinterpret_cast<uint32_t*>(p);
    TM_CUDA(cudaMemsetAsync(gbits, 0, bit_bytes, st));
  }
  int* row_map = reinterpret_cast<int*>(p + fanin_bits_bytes(s->n));
  if (s->n_cell_rows > 0) TM_CUDA(cudaMemsetAsync(row_map, 0xff, (size_t)s->n_cell_rows * sizeof(int), st));
  TM_CUDA(cudaFuncSetAttribute(fanin_cone_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CONE_SMEM_MAX));
  FaninArgs a{(int)s->n, s->num_levels, (int)n_endpoints, s->level, s->level_ptr, s->cell_base, s->order, s->f_ptr,
              s->f_src, s->bn_ptr, s->bn_dst, s->bn_w, s->bc_ptr, s->bc_row, endpoints, seed, gbits, row_map,
              order, level_ptr, cell_base, f_ptr, f_src, bn_ptr, bn_dst, bn_w, bc_ptr, bc_row, cell_pins, net_pins,
              counts};
  fanin_cone_kernel<<<1, CONE_T, in_smem ? bit_bytes : 0, st>>>(a);
  return check_launch("fanin_cone");
}

extern "C" int tm_fanin_cone(const tm_schedule* s, int64_t n_endpoints, const int32_t* endpoints, const float* seed,
                             int32_t* order, int32_t* level_ptr, int32_t* cell_base, int32_t* f_ptr, int32_t* f_src,
                             int32_t* bn_ptr, int32_t* bn_dst, float* bn_w, int32_t* bc_ptr, int32_t* bc_row,
                             int32_t* cell_pins, int32_t* net_pins, int32_t* counts, void* ws, size_t ws_bytes,
                             void* stream) {
  return fanin_cone_launch(s, n_endpoints, endpoints, seed, order, level_ptr, cell_base, f_ptr, f_src, bn_ptr, bn_dst,
                           bn_w, bc_ptr, bc_row, cell_pins, net_pins, counts, nullptr, ws, ws_bytes, stream);
}

extern "C" int tm_fanin_cone_bits(const tm_schedule* s, int64_t n_endpoints, const int32_t* endpoints,
                                  const float* seed, int32_t* order, int32_t* level_ptr, int32_t* cell_base,
                                  int32_t* f_ptr, int32_t* f_src, int32_t* bn_ptr, int32_t* bn_dst, float* bn_w,
                                  int32_t* bc_ptr, int32_t* bc_row, int32_t* cell_pins, int32_t* net_pins,
                                  int32_t* counts, uint32_t* bits, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(bits, "tm_fanin_cone_bits: NULL bitmap");
  return fanin_cone_launch(s, n_endpoints, endpoints, seed, order, level_ptr, cell_base, f_ptr, f_src, bn_ptr, bn_dst,
                           bn_w, bc_ptr, bc_row, cell_pins, net_pins, counts, bits, ws, ws_bytes, stream);
}

// ------------------------------------------------------------------------------------------
// forward cones of K candidate edits, joined into one sub-schedule over private virtual rows
// (what-if evaluation: score many alternative edits of one design in one propagation).
//
// mark:  grid K, one 1024-thread block per candidate.  fwd_cone_kernel's pull sweep from the
//        candidate's lowest seed level, without compaction: a pin is in the cone when it is a seed
//        or one of its f_src sources is.  Sources sit on earlier levels, so bits set during a level
//        are never read in it and one block barrier per level suffices.  Per-level pin / edge
//        counts are summed in shared memory (double-buffered by level parity).  At the end the
//        block writes its bitmap to the workspace (when it lived in shared memory) and a rank
//        directory: dir[w] = set bits in words < w, so rank(u) = dir[u>>5] + popc(lower bits).
// plan:  one block.  Admission in index order, the joined level_ptr (level l = the admitted
//        candidates' cone pins of level l, candidate by candidate), per-(candidate, level) pin and
//        edge offsets inside the level, the edge offset of every level, the count.
// emit:  blocks over (candidate, level); the extra level index L does the candidate's seed and
//        endpoint rows.  A block scan of (in cone, in-degree) over the parent's level compacts the
//        cone in the parent's order, as fwd_cone_kernel does; sources in the cone are remapped to
//        their virtual rows; the cone pins' S rows are copied to their virtual rows, a warp a row.
// ------------------------------------------------------------------------------------------
namespace {
constexpr int EMIT_T = 256;

struct ConesArgs {
  int n, L, K, R;
  long long ecap;
  int W;                                           // bitmap words per candidate
  bool in_smem;                                    // mark keeps its bitmap in shared memory
  const int* level; const int* level_ptr; const int* order; const int* f_ptr; const int* f_src;
  const int* seed_ptr; const int* seeds; const int* seed_slot;
  int T; const int* endpoints;
  float* S;
  int* c_order; int* c_level_ptr; int* c_f_ptr; int* c_f_src; int* c_count;
  int* vpin; int* seed_rows; int* head_rows; int* fitted; int* sizes; int* row_base;
  // workspace
  uint32_t* bits; int* dir;                        // [K][W] each
  int* cnt; int* edg; int* posoff; int* eoff;      // [K][L] each
  int* lmin; int* etot;                            // [K]
  int* lev_e;                                      // [L+1]: edges before level l in the joined schedule
};

// exclusive block scan of two ints; wsum: 64 ints of shared memory.  The caller syncs before wsum is reused.
__device__ __forceinline__ void block_scan2(int& c, int& e, int& tc, int& te, int* wsum) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int ic = c, ie = e;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int yc = __shfl_up_sync(0xffffffffu, ic, o), ye = __shfl_up_sync(0xffffffffu, ie, o);
    if (lane >= o) { ic += yc; ie += ye; }
  }
  if (lane == 31) { wsum[warp] = ic; wsum[32 + warp] = ie; }
  __syncthreads();
  int oc = 0, oe = 0;
  tc = 0;
  te = 0;
  for (int w = 0; w < nw; ++w) {
    const int xc = wsum[w], xe = wsum[32 + w];
    if (w < warp) { oc += xc; oe += xe; }
    tc += xc;
    te += xe;
  }
  c = oc + ic - c;
  e = oe + ie - e;
}

__device__ __forceinline__ int warp_sum(int x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

__global__ void __launch_bounds__(CONE_T, 1) cones_mark_kernel(const ConesArgs a) {
  extern __shared__ uint32_t sbits[];
  __shared__ int s_lmin, s_c[2], s_e[2];
  __shared__ int wsum[64];
  const int k = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  uint32_t* gbits = a.bits + (size_t)k * a.W;
  uint32_t* bits = a.in_smem ? sbits : gbits;
  const volatile uint32_t* vbits = bits;
  if (a.in_smem)
    for (int i = tid; i < a.W; i += CONE_T) sbits[i] = 0u;
  if (tid == 0) { s_lmin = a.L; s_c[0] = s_c[1] = 0; s_e[0] = s_e[1] = 0; }
  __syncthreads();
  const int s0 = __ldg(a.seed_ptr + k), s1 = __ldg(a.seed_ptr + k + 1);
  for (int i = s0 + tid; i < s1; i += CONE_T) {
    const int v = a.seeds[i];
    if (v < 0 || v >= a.n) continue;
    const int l = a.level[v];
    if (l < 0 || l >= a.L) continue;               // outside the schedule: changes nothing
    atomicOr(bits + (v >> 5), 1u << (v & 31));
    atomicMin(&s_lmin, l);
  }
  __syncthreads();
  const int lmin = s_lmin;
  int* cnt = a.cnt + (size_t)k * a.L;
  int* edg = a.edg + (size_t)k * a.L;
  for (int l = tid; l < lmin; l += CONE_T) { cnt[l] = 0; edg[l] = 0; }
  for (int l = lmin; l < a.L; ++l) {
    const int p0 = __ldg(a.level_ptr + l), p1 = __ldg(a.level_ptr + l + 1);
    int p2 = p1, fa = 0, fb = 0;
    if (l + 1 < a.L) {
      p2 = __ldg(a.level_ptr + l + 2);
      fa = __ldg(a.f_ptr + p1);
      fb = __ldg(a.f_ptr + p2);
    }
    for (int i = p1 + tid * 32; i < p2; i += CONE_T * 32) {   // the next level's static arrays into L2
      pf_l2(a.order + i);
      pf_l2(a.f_ptr + i);
    }
    for (int i = fa + tid * 32; i < fb; i += CONE_T * 32) pf_l2(a.f_src + i);
    int my_c = 0, my_e = 0;
    for (int c0 = p0; c0 < p1; c0 += CONE_CHUNK) {
      const int q = c0 + tid * CONE_V;
      const int nq = max(0, min(CONE_V, p1 - q));
      if (nq == 0) continue;
      int ptr[CONE_V + 1], v[CONE_V];
      bool in[CONE_V];
#pragma unroll
      for (int j = 0; j <= CONE_V; ++j) ptr[j] = j <= nq ? __ldg(a.f_ptr + q + j) : 0;
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) v[j] = j < nq ? __ldg(a.order + q + j) : 0;
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) in[j] = j < nq && cone_bit(vbits, v[j]);
      int e1 = ptr[0];                             // ptr[nq] without a dynamic register index
#pragma unroll
      for (int j = 1; j <= CONE_V; ++j) e1 = j == nq ? ptr[j] : e1;
      for (int e = ptr[0]; e < e1; e += 8) {
        int src[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) src[u] = e + u < e1 ? __ldg(a.f_src + e + u) : -1;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (src[u] >= 0 && cone_bit(vbits, src[u])) {
#pragma unroll
            for (int j = 0; j < CONE_V; ++j) in[j] |= (e + u >= ptr[j] && e + u < ptr[j + 1]);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < CONE_V; ++j) {
        if (in[j]) {
          ++my_c;
          my_e += ptr[j + 1] - ptr[j];
          atomicOr(bits + (v[j] >> 5), 1u << (v[j] & 31));
        }
      }
    }
    my_c = warp_sum(my_c);
    my_e = warp_sum(my_e);
    if (lane == 0 && (my_c | my_e)) { atomicAdd(&s_c[l & 1], my_c); atomicAdd(&s_e[l & 1], my_e); }
    __syncthreads();                               // bits and counts of level l are complete
    if (tid == 0) {
      cnt[l] = s_c[l & 1];
      edg[l] = s_e[l & 1];
      s_c[l & 1] = 0;                              // reused by level l + 2, after the next barrier
      s_e[l & 1] = 0;
    }
  }
  if (a.in_smem) {
    for (int i = tid; i < a.W; i += CONE_T) gbits[i] = sbits[i];
  }
  // rank directory: exclusive scan of the words' popcounts
  int* dir = a.dir + (size_t)k * a.W;
  int run = 0;
  for (int w0 = 0; w0 < a.W; w0 += CONE_T) {
    const int w = w0 + tid;
    int c = w < a.W ? __popc(vbits[w]) : 0, e = 0, tc, te;
    block_scan2(c, e, tc, te, wsum);
    if (w < a.W) dir[w] = run + c;
    run += tc;
    __syncthreads();
  }
  if (tid == 0) {
    a.sizes[k] = run;
    a.lmin[k] = lmin;
  }
}

__global__ void __launch_bounds__(CONE_T, 1) cones_plan_kernel(const ConesArgs a) {
  __shared__ int wsum[64];
  const int tid = threadIdx.x, K = a.K, L = a.L;
  for (int k = tid; k < K; k += CONE_T) {
    int e = 0;
    for (int l = 0; l < L; ++l) e += a.edg[(size_t)k * L + l];
    a.etot[k] = e;
  }
  __syncthreads();
  if (tid == 0) {                                  // admission: the longest prefix that fits
    long long rc = 0, re = 0;
    bool open = true;
    for (int k = 0; k < K; ++k) {
      const int c = a.sizes[k], e = a.etot[k];
      open = open && rc + c <= a.R && re + e <= a.ecap;
      a.fitted[k] = open ? 1 : 0;
      a.row_base[k] = open ? (int)rc : 0;
      if (open) { rc += c; re += e; }
    }
  }
  __syncthreads();
  int run_c = 0, run_e = 0;
  for (int l0 = 0; l0 < L; l0 += CONE_T) {
    const int l = l0 + tid;
    int c = 0, e = 0, tc, te;
    if (l < L) {
      for (int k = 0; k < K; ++k) {
        if (!a.fitted[k]) break;                   // admitted candidates form a prefix
        const size_t i = (size_t)k * L + l;
        a.posoff[i] = c;
        a.eoff[i] = e;
        c += a.cnt[i];
        e += a.edg[i];
      }
    }
    block_scan2(c, e, tc, te, wsum);
    if (l < L) {
      a.c_level_ptr[l] = run_c + c;
      a.lev_e[l] = run_e + e;
    }
    run_c += tc;
    run_e += te;
    __syncthreads();
  }
  if (tid == 0) {
    a.c_level_ptr[L] = run_c;
    a.lev_e[L] = run_e;
    a.c_f_ptr[run_c] = run_e;
    *a.c_count = run_c;
  }
}

__device__ __forceinline__ int cone_vrow(const ConesArgs& a, const uint32_t* bits, const int* dir, int base, int u) {
  return a.n + base + __ldg(dir + (u >> 5)) + __popc(__ldg(bits + (u >> 5)) & ((1u << (u & 31)) - 1u));
}

__global__ void __launch_bounds__(EMIT_T) cones_emit_kernel(const ConesArgs a) {
  __shared__ int wsum[64];
  __shared__ int s_vr[EMIT_T], s_pin[EMIT_T];
  const int k = blockIdx.x, l = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t* bits = a.bits + (size_t)k * a.W;
  const int* dir = a.dir + (size_t)k * a.W;
  const bool admitted = a.fitted[k] != 0;
  const int base = a.row_base[k];
  auto in_cone = [&](int u) { return (__ldg(bits + (u >> 5)) >> (u & 31)) & 1u; };
  if (l == a.L) {                                  // the candidate's seed rows and endpoint head rows
    const int sink = a.n + a.R;
    const int s0 = a.seed_ptr[k], s1 = a.seed_ptr[k + 1];
    for (int i = s0 + tid; i < s1; i += EMIT_T) {
      const int u = a.seeds[i];
      int row = sink;
      if (admitted && u >= 0 && u < a.n) {
        const int lu = a.level[u];
        if (lu >= 0 && lu < a.L) row = cone_vrow(a, bits, dir, base, u);
      }
      a.seed_rows[a.seed_slot ? a.seed_slot[i] : i] = row;
    }
    for (int t = tid; t < a.T; t += EMIT_T) {
      const int u = a.endpoints[t];
      a.head_rows[(size_t)k * a.T + t] = (admitted && in_cone(u)) ? cone_vrow(a, bits, dir, base, u) : u;
    }
    return;
  }
  if (!admitted || l < a.lmin[k]) return;
  const size_t kl = (size_t)k * a.L + l;
  if (a.cnt[kl] == 0) return;
  int pos = a.c_level_ptr[l] + a.posoff[kl];
  int eo = a.lev_e[l] + a.eoff[kl];
  const int p0 = __ldg(a.level_ptr + l), p1 = __ldg(a.level_ptr + l + 1);
  for (int c0 = p0; c0 < p1; c0 += EMIT_T) {
    const int p = c0 + tid;
    int v = 0, e0 = 0, e1 = 0;
    bool in = false;
    if (p < p1) {
      v = __ldg(a.order + p);
      in = in_cone(v);
      if (in) { e0 = __ldg(a.f_ptr + p); e1 = __ldg(a.f_ptr + p + 1); }
    }
    int oc = in ? 1 : 0, oe = e1 - e0, tc, te;
    block_scan2(oc, oe, tc, te, wsum);
    if (in) {
      const int vr = cone_vrow(a, bits, dir, base, v);
      a.c_order[pos + oc] = vr;
      a.c_f_ptr[pos + oc] = eo + oe;
      int o = eo + oe;
      for (int e = e0; e < e1; ++e) {
        const int src = __ldg(a.f_src + e);
        a.c_f_src[o++] = in_cone(src) ? cone_vrow(a, bits, dir, base, src) : src;
      }
      a.vpin[vr - a.n] = v;
      s_vr[oc] = vr;
      s_pin[oc] = v;
    }
    __syncthreads();
    for (int i = warp; i < tc; i += EMIT_T / 32) {  // S[virtual row] = S[pin], a warp a 512-byte row
      const float4* src = reinterpret_cast<const float4*>(a.S + (size_t)s_pin[i] * 128);
      float4* dst = reinterpret_cast<float4*>(a.S + (size_t)s_vr[i] * 128);
      dst[lane] = src[lane];
    }
    pos += tc;
    eo += te;
    __syncthreads();                               // wsum / s_vr / s_pin are reused
  }
}

__global__ void what_if_commit_kernel(int n, int k, const int* fitted, const int* sizes, const int* row_base,
                                      const int* vpin, float4* H, float4* S) {
  if (!fitted[k]) return;
  const int r0 = row_base[k], cnt = sizes[k];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (int64_t)cnt * 32;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int r = r0 + (int)(i >> 5), c = (int)(i & 31);
    const int64_t from = (int64_t)(n + r) * 32 + c, to = (int64_t)vpin[r] * 32 + c;
    H[to] = H[from];
    S[to] = S[from];
  }
}

__global__ void what_if_mask_kernel(int K, int64_t T, const int* fitted, float* pred) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)K * T && !fitted[i / T]) pred[i] = __int_as_float(0x7fc00000);
}

// a seed outside the restriction becomes -1, which the mark and emit kernels treat as a seed outside the schedule
__global__ void seeds_within_kernel(int n, int m, const int* seeds, const uint32_t* within, int* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const int v = seeds[i];
  out[i] = (v >= 0 && v < n && ((within[v >> 5] >> (v & 31)) & 1u)) ? v : -1;
}

struct ConesWs {
  size_t bits, dir, kl, k, lev, total;
};
ConesWs cones_ws_layout(int64_t n, int64_t K, int64_t L) {
  auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
  ConesWs w{};
  w.bits = up((size_t)K * cdiv(n, 32) * sizeof(uint32_t));
  w.dir = w.bits;
  w.kl = up((size_t)K * L * sizeof(int));
  w.k = up((size_t)K * sizeof(int));
  w.lev = up((size_t)(L + 1) * sizeof(int));
  w.total = w.bits + w.dir + 4 * w.kl + 2 * w.k + w.lev;
  return w;
}
}  // namespace

extern "C" size_t tm_forward_cones_ws(int64_t n, int32_t n_cand, int32_t num_levels) {
  return cones_ws_layout(n, n_cand > 0 ? n_cand : 1, num_levels > 0 ? num_levels : 1).total;
}

extern "C" int tm_forward_cones(const tm_schedule* s, int32_t n_cand, const int32_t* seed_ptr, const int32_t* seeds,
                                const int32_t* seed_slot, int64_t rows, int64_t edge_cap, int64_t n_endpoints,
                                const int32_t* endpoints, float* S, int32_t* order, int32_t* level_ptr, int32_t* f_ptr,
                                int32_t* f_src, int32_t* count, int32_t* vpin, int32_t* seed_rows, int32_t* head_rows,
                                int32_t* fitted, int32_t* sizes, int32_t* row_base, void* ws, size_t ws_bytes,
                                void* stream) {
  TM_REQUIRE(s && s->order && s->level && s->level_ptr && s->f_ptr && s->f_src,
             "tm_forward_cones: the parent schedule lacks its device arrays (order, level, level_ptr, f_ptr, f_src)");
  TM_REQUIRE(s->n > 0 && s->num_levels > 0 && s->num_levels < 65535, "tm_forward_cones: bad schedule sizes");
  TM_REQUIRE(n_cand > 0 && n_cand < 65536 && seed_ptr, "tm_forward_cones: bad candidate list");
  TM_REQUIRE(rows > 0 && s->n + rows + 1 < INT32_MAX && edge_cap >= 0 && edge_cap < INT32_MAX,
             "tm_forward_cones: bad capacity (rows, edge_cap)");
  TM_REQUIRE(n_endpoints >= 0 && (int64_t)n_cand * n_endpoints < INT32_MAX && (n_endpoints == 0 || endpoints),
             "tm_forward_cones: bad endpoint list");
  TM_REQUIRE(S && order && level_ptr && f_ptr && f_src && count && vpin && seed_rows && head_rows && fitted && sizes &&
                 row_base,
             "tm_forward_cones: NULL output buffer");
  TM_REQUIRE(ws && ws_bytes >= tm_forward_cones_ws(s->n, n_cand, s->num_levels),
             "tm_forward_cones: workspace too small (tm_forward_cones_ws)");
  cudaStream_t st = (cudaStream_t)stream;
  const int K = n_cand, L = s->num_levels;
  const ConesWs w = cones_ws_layout(s->n, K, L);
  uint8_t* p = reinterpret_cast<uint8_t*>(ws);
  ConesArgs a{};
  a.n = (int)s->n; a.L = L; a.K = K; a.R = (int)rows; a.ecap = edge_cap;
  a.W = (int)cdiv(s->n, 32);
  const size_t bit_bytes = (size_t)a.W * sizeof(uint32_t);
  a.in_smem = bit_bytes <= CONE_SMEM_MAX;
  a.level = s->level; a.level_ptr = s->level_ptr; a.order = s->order; a.f_ptr = s->f_ptr; a.f_src = s->f_src;
  a.seed_ptr = seed_ptr; a.seeds = seeds; a.seed_slot = seed_slot;
  a.T = (int)n_endpoints; a.endpoints = endpoints; a.S = S;
  a.c_order = order; a.c_level_ptr = level_ptr; a.c_f_ptr = f_ptr; a.c_f_src = f_src; a.c_count = count;
  a.vpin = vpin; a.seed_rows = seed_rows; a.head_rows = head_rows; a.fitted = fitted; a.sizes = sizes;
  a.row_base = row_base;
  a.bits = reinterpret_cast<uint32_t*>(p); p += w.bits;
  a.dir = reinterpret_cast<int*>(p); p += w.dir;
  a.cnt = reinterpret_cast<int*>(p); p += w.kl;
  a.edg = reinterpret_cast<int*>(p); p += w.kl;
  a.posoff = reinterpret_cast<int*>(p); p += w.kl;
  a.eoff = reinterpret_cast<int*>(p); p += w.kl;
  a.lmin = reinterpret_cast<int*>(p); p += w.k;
  a.etot = reinterpret_cast<int*>(p); p += w.k;
  a.lev_e = reinterpret_cast<int*>(p);
  if (!a.in_smem) TM_CUDA(cudaMemsetAsync(a.bits, 0, (size_t)K * bit_bytes, st));
  TM_CUDA(cudaFuncSetAttribute(cones_mark_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CONE_SMEM_MAX));
  cones_mark_kernel<<<K, CONE_T, a.in_smem ? bit_bytes : 0, st>>>(a);
  if (int rc = check_launch("cones_mark")) return rc;
  cones_plan_kernel<<<1, CONE_T, 0, st>>>(a);
  if (int rc = check_launch("cones_plan")) return rc;
  cones_emit_kernel<<<dim3((unsigned)K, (unsigned)(L + 1)), EMIT_T, 0, st>>>(a);
  return check_launch("cones_emit");
}

// The cones restricted to a fan-in cone R(E): the same three kernels over R(E)'s sub-schedule (their sweeps only walk
// level_ptr / order / f_ptr / f_src), after the seeds outside R(E) are replaced by -1.  R(E) holds every in-edge
// source of its pins, so a candidate's restricted cone is exactly its forward cone intersected with R(E).
extern "C" size_t tm_forward_cones_within_ws(int64_t n, int32_t n_cand, int32_t num_levels, int64_t n_seeds) {
  return tm_forward_cones_ws(n, n_cand, num_levels) + (((size_t)(n_seeds > 0 ? n_seeds : 0) * sizeof(int) + 255) &
                                                       ~(size_t)255);
}

extern "C" int tm_forward_cones_within(const tm_schedule* s, const uint32_t* within, int32_t n_cand,
                                       const int32_t* seed_ptr, const int32_t* seeds, const int32_t* seed_slot,
                                       int64_t n_seeds, int64_t rows, int64_t edge_cap, int64_t n_endpoints,
                                       const int32_t* endpoints, float* S, int32_t* order, int32_t* level_ptr,
                                       int32_t* f_ptr, int32_t* f_src, int32_t* count, int32_t* vpin,
                                       int32_t* seed_rows, int32_t* head_rows, int32_t* fitted, int32_t* sizes,
                                       int32_t* row_base, void* ws, size_t ws_bytes, void* stream) {
  TM_REQUIRE(s && s->n > 0 && s->num_levels > 0 && within, "tm_forward_cones_within: bad schedule or bitmap");
  TM_REQUIRE(n_seeds >= 0 && n_seeds < INT32_MAX && (n_seeds == 0 || seeds),
             "tm_forward_cones_within: bad seed list");
  TM_REQUIRE(ws && ws_bytes >= tm_forward_cones_within_ws(s->n, n_cand, s->num_levels, n_seeds),
             "tm_forward_cones_within: workspace too small (tm_forward_cones_within_ws)");
  const size_t cones_bytes = tm_forward_cones_ws(s->n, n_cand, s->num_levels);
  int* kept = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(ws) + cones_bytes);
  if (n_seeds > 0) {
    seeds_within_kernel<<<(unsigned)cdiv(n_seeds, 256), 256, 0, (cudaStream_t)stream>>>((int)s->n, (int)n_seeds, seeds,
                                                                                         within, kept);
    if (int rc = check_launch("seeds_within")) return rc;
  }
  return tm_forward_cones(s, n_cand, seed_ptr, n_seeds > 0 ? kept : seeds, seed_slot, rows, edge_cap, n_endpoints,
                          endpoints, S, order, level_ptr, f_ptr, f_src, count, vpin, seed_rows, head_rows, fitted,
                          sizes, row_base, ws, cones_bytes, stream);
}

extern "C" int tm_what_if_commit(int64_t n, int32_t k, const int32_t* fitted, const int32_t* sizes,
                                 const int32_t* row_base, const int32_t* vpin, float* H, float* S, void* stream) {
  TM_REQUIRE(n > 0 && n < INT32_MAX && k >= 0, "tm_what_if_commit: bad sizes");
  TM_REQUIRE(fitted && sizes && row_base && vpin && H && S, "tm_what_if_commit: NULL operand");
  what_if_commit_kernel<<<296, 256, 0, (cudaStream_t)stream>>>((int)n, k, fitted, sizes, row_base, vpin,
                                                              reinterpret_cast<float4*>(H), reinterpret_cast<float4*>(S));
  return check_launch("what_if_commit");
}

extern "C" int tm_what_if_mask(int32_t n_cand, int64_t T, const int32_t* fitted, float* pred, void* stream) {
  TM_REQUIRE(n_cand >= 0 && T >= 0 && (n_cand == 0 || T == 0 || (fitted && pred)), "tm_what_if_mask: bad operands");
  const int64_t m = (int64_t)n_cand * T;
  if (m == 0) return 0;
  what_if_mask_kernel<<<(unsigned)cdiv(m, 256), 256, 0, (cudaStream_t)stream>>>(n_cand, T, fitted, pred);
  return check_launch("what_if_mask");
}
