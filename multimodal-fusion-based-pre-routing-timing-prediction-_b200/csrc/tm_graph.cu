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
