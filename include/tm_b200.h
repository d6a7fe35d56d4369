/*
 * tm_b200.h -- C ABI of libtm_b200.so: the B200 (sm_100a) hot path of the multimodal
 * pre-routing timing predictor (level-wise netlist GNN + layout U-Net + mask fusion).
 *
 * The reference (ZeayW/Multimodal-fusion-based-Pre-routing-Timing-Prediction-) has no
 * FFI/plugin layer: its hot path is Python calling DGL and ATen.  Each entry point below
 * therefore cites the reference *call site* (src/<file>:<line>) whose library work it
 * replaces.  Conventions:
 *   - every pointer is a DEVICE pointer unless its name starts with h_ (host);
 *   - no allocation and no ownership transfer inside: the caller passes workspaces;
 *   - all launches go to the given cudaStream_t (passed as void*), nothing synchronises
 *     unless stated;
 *   - return 0 on success, a negative TM_E* for argument errors or a positive cudaError_t;
 *     tm_last_error() returns a thread-local message for the last failure.
 * Python binding: multimodal-fusion-based-pre-routing-timing-prediction-_b200/tm_lib.py (ctypes).
 */
#ifndef TM_B200_H
#define TM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TM_OK 0
#define TM_EINVAL (-1)   /* bad argument                      */
#define TM_EWORKSPACE (-2) /* workspace too small             */
#define TM_EUNSUPPORTED (-3)

int tm_version(void);
const char* tm_last_error(void);
/* Number of kernels this library has launched since load (bench.py "gpu_launches"). */
long long tm_launch_count(void);
int tm_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* The level schedule of one graph (all device arrays int32 unless noted).  Built by the G1
 * entry points below, consumed by the G2/G3 propagation kernels. */
typedef struct {
  int64_t n;                 /* pins                                                   */
  int32_t num_levels;
  int32_t n_cell_rows;       /* pins on even levels > 0                                */
  const int32_t* h_level_ptr;/* HOST copy of level_ptr[num_levels+1]                   */
  const int32_t* order;      /* scheduled pins by (level, id)                          */
  const int32_t* level;      /* pin -> level                                           */
  const int32_t* crow;       /* pin -> compact cell row or -1                          */
  const int32_t* net_iptr;  const int32_t* net_isrc;   /* in-edge CSRs                 */
  const int32_t* cell_iptr; const int32_t* cell_isrc;
  const int32_t* net_optr;  const int32_t* net_odst;   /* out-edge CSRs                */
  const int32_t* cell_optr; const int32_t* cell_odst;
  /* level-ordered edge lists (tm_schedule_edges), indexed by schedule position            */
  const int32_t* f_ptr;  const int32_t* f_src;         /* forward gather sources           */
  const int32_t* bn_ptr; const int32_t* bn_dst; const float* bn_w;   /* backward, net edges */
  const int32_t* bc_ptr; const int32_t* bc_row;        /* backward, cell edges (compact row) */
  /* device copies the persistent propagation kernels read (one launch loops over all levels) */
  const int32_t* level_ptr;  /* [num_levels+1] first schedule position of each level       */
  const int32_t* cell_base;  /* [num_levels+1] first compact cell row of each level        */
} tm_schedule;

/* ------------------------------------------------------------------------------------
 * G1  graph structure: CSR build and level schedule
 *     replaces dgl.heterograph(...) + the lazy in-edge CSR DGL builds inside graph.pull
 *     (src/dataset.py:274-278, src/model.py:186-204) and Parser.cal_topo_level
 *     (src/verilog_parser_asap7.py:1452-1517).
 * ---------------------------------------------------------------------------------- */

/* Bytes of workspace tm_csr_build needs. */
size_t tm_csr_build_ws(int64_t n, int64_t e);
/* CSR keyed on `key` (dst for an in-edge CSR, src for an out-edge CSR):
 * indptr[n+1], indices[e] = `val` of every edge, ascending inside each row (duplicates kept).
 * key/val are the int64 edge lists of one edge type as DGL stores them. */
int tm_csr_build(int64_t n, int64_t e, const int64_t* key, const int64_t* val,
                 int32_t* indptr, int32_t* indices, void* ws, size_t ws_bytes, void* stream);

size_t tm_levelize_ws(int64_t n);
/* level[v] = length of the longest walk from the PI set to v (pins not reachable from a PI:
 * -1), i.e. the last frontier v appears in (verilog_parser_asap7.py:1494-1511).
 * optr/oidx: out-edge CSR over the union of both edge types.  num_levels: device int32.
 * Cooperative persistent kernel (frontier BFS + Kahn peeling with grid-wide barriers). */
int tm_levelize(int64_t n, const int32_t* optr, const int32_t* oidx, const int64_t* pis,
                int64_t n_pi, int32_t* level, int32_t* num_levels, void* ws, size_t ws_bytes,
                void* stream);

size_t tm_level_order_ws(int64_t n, int32_t num_levels);
/* order[] = scheduled pins sorted by (level, pin id); level_ptr[num_levels+1].
 * Deterministic stable counting sort. */
int tm_level_order(int64_t n, int32_t num_levels, const int32_t* level, int32_t* order,
                   int32_t* level_ptr, void* ws, size_t ws_bytes, void* stream);

/* Per-pin auxiliaries of a schedule:
 * crow[v]   = row of pin v in the compact "cell pin" buffers (pins on even levels > 0), else -1,
 *             numbered in schedule order;
 * cell_base[num_levels+1] = first compact row of each level (cell_base[num_levels] = row count);
 * n_violations (device int32) += number of in-edges whose source is not on an earlier level
 *             (such a schedule is not a topological one; the caller must refuse it). */
int tm_schedule_aux(int64_t n, int32_t num_levels, const int32_t* level, const int32_t* order,
                    const int32_t* level_ptr, const int32_t* net_iptr, const int32_t* net_isrc,
                    const int32_t* cell_iptr, const int32_t* cell_isrc, int32_t* crow,
                    int32_t* cell_base, int32_t* n_violations, void* stream);

size_t tm_schedule_edges_ws(int64_t n_sched);
/* Level-ordered edge lists for the propagation kernels (see tm_schedule): f_ptr/bn_ptr/bc_ptr
 * [n_sched+1]; f_src [E_net+E_cell]; bn_dst, bn_w [E_net]; bc_row [E_cell] (upper bounds).
 * `s` needs order, level, crow and the four CSRs filled in. */
int tm_schedule_edges(const tm_schedule* s, int64_t n_sched, int32_t* f_ptr, int32_t* f_src,
                      int32_t* bn_ptr, int32_t* bn_dst, float* bn_w, int32_t* bc_ptr,
                      int32_t* bc_row, void* ws, size_t ws_bytes, void* stream);

size_t tm_forward_cone_ws(int64_t n);
/* Forward cone of `n_seeds` seed pins (device int32; duplicates, pins outside the schedule and n_seeds = 0 are
 * valid): every scheduled pin reachable from a scheduled seed along the in-edges the propagation reads (s->f_src),
 * the seeds included -- the pins whose H row can change when the seeds' self terms S change.  Written as a
 * sub-schedule into caller buffers sized by the parent: order[n_sched] (the stable subsequence of s->order),
 * level_ptr[num_levels+1], f_ptr[n_sched+1] and f_src[len(s->f_src)] (the parent's in-edge lists of the cone's pins,
 * in the parent's edge order), count (device int32: the cone's pin count).  No host synchronisation: one block
 * sweeps the levels from the lowest seed's level on.  `s` needs order, level, level_ptr, f_ptr and f_src. */
int tm_forward_cone(const tm_schedule* s, int64_t n_seeds, const int32_t* seeds, int32_t* order,
                    int32_t* level_ptr, int32_t* f_ptr, int32_t* f_src, int32_t* count, void* ws,
                    size_t ws_bytes, void* stream);

size_t tm_fanin_cone_ws(int64_t n, int32_t n_cell_rows);
/* Fan-in cone of the endpoints whose seed is non-zero (endpoints: device int32 [n_endpoints], seed: device float32
 * [n_endpoints], both read on the device; duplicates and endpoints outside the schedule are valid): every scheduled
 * pin from which a seeded endpoint is reachable along the out-edges a backward pass reads (s->bn_dst and the cell
 * out-edges s->bc_row), the seeded endpoints included -- the pins whose gradient can be non-zero.  Written as a
 * sub-schedule for tm_gnn_save_cone / tm_gnn_backward_cone into caller buffers sized by the parent, laid out from their
 * END: positions [n_sched - count, n_sched) of order[n_sched] (the stable subsequence of s->order), level_ptr and
 * cell_base [num_levels+1] (cell rows [n_cell_rows - cone cell rows, n_cell_rows), one per cone pin on an even level
 * > 0, in schedule order), f_ptr / bn_ptr / bc_ptr [n_sched+1] with f_src [len(s->f_src)] (the parent's in-edge lists,
 * unchanged), bn_dst / bn_w [len(s->bn_dst)] and bc_row [len(s->bc_row)] (out-edges whose destination is in the
 * cone, in the parent's order, bc_row as cone cell rows).  cell_pins / net_pins (capacity: the pins on even / odd
 * levels) list the cone's pins on even / odd levels from index 0; counts (device int32 [3]) = cone pins, cell_pins
 * entries, net_pins entries.  No host synchronisation: one block sweeps from the highest seeded level down.  ws:
 * tm_fanin_cone_ws(s->n, s->n_cell_rows) -- the membership bitmap when it exceeds shared memory (over 1.5M pins) and
 * one int per cell row. */
int tm_fanin_cone(const tm_schedule* s, int64_t n_endpoints, const int32_t* endpoints, const float* seed,
                  int32_t* order, int32_t* level_ptr, int32_t* cell_base, int32_t* f_ptr, int32_t* f_src,
                  int32_t* bn_ptr, int32_t* bn_dst, float* bn_w, int32_t* bc_ptr, int32_t* bc_row, int32_t* cell_pins,
                  int32_t* net_pins, int32_t* counts, void* ws, size_t ws_bytes, void* stream);

/* tm_fanin_cone that also keeps the cone's membership bitmap: bits[ceil(n/32)] (device, caller's), bit v of word
 * v / 32 set for every cone pin.  The same kernel, with the bitmap in bits instead of shared memory; ws as for
 * tm_fanin_cone.  For tm_forward_cones_within. */
int tm_fanin_cone_bits(const tm_schedule* s, int64_t n_endpoints, const int32_t* endpoints, const float* seed,
                       int32_t* order, int32_t* level_ptr, int32_t* cell_base, int32_t* f_ptr, int32_t* f_src,
                       int32_t* bn_ptr, int32_t* bn_dst, float* bn_w, int32_t* bc_ptr, int32_t* bc_row,
                       int32_t* cell_pins, int32_t* net_pins, int32_t* counts, uint32_t* bits, void* ws,
                       size_t ws_bytes, void* stream);

size_t tm_forward_cones_ws(int64_t n, int32_t n_cand, int32_t num_levels);
/* Forward cones of `n_cand` candidate edits, joined into ONE sub-schedule over private virtual rows, for scoring
 * alternative edits of the same design without touching the rows of its pins (what-if evaluation).
 *
 * Candidate k's seeds are seeds[seed_ptr[k] : seed_ptr[k+1]] (seed_ptr: device int32 [n_cand+1]; seeds as in
 * tm_forward_cone).  Its cone pins get the virtual rows n + row_base[k] + rank, rank = the pin's rank by id among the
 * cone's pins, so H / S are (n + rows + 1)-row buffers; row n + rows is a sink row.  Candidates are admitted in index
 * order while the running totals of cone pins fit in `rows` and of cone in-edges in `edge_cap`; the first that does
 * not fit and every later one is not admitted (fitted[k] = 0) and writes nothing outside the buffers.
 *
 * Outputs (caller buffers): order[rows], level_ptr[num_levels+1], f_ptr[rows+1], f_src[edge_cap], count -- a
 * sub-schedule for tm_gnn_forward_cone whose level l holds candidate 0's cone pins of level l, then candidate 1's, and
 * so on (admitted candidates only), each in the parent's order, with order[pos] the virtual row and every in-edge
 * source inside the candidate's cone replaced by its virtual row (sources outside it keep their pin id); vpin[rows]
 * (the pin of each virtual row); S[virtual row] = S[pin] for every cone pin; seed_rows[seed_slot ? seed_slot[i] : i] =
 * the virtual row of seed i, or the sink row for a seed outside the schedule or of a non-admitted candidate (where a
 * caller writes the seeds' new self terms); head_rows[k * n_endpoints + t] = the virtual row of endpoints[t] when it
 * is in candidate k's admitted cone, else endpoints[t]; fitted[n_cand] (1 = admitted), sizes[n_cand] (cone pins, also
 * of non-admitted candidates), row_base[n_cand].
 *
 * Three launches, no host synchronisation (capturable): one 1024-thread block per candidate sweeps its levels pulling
 * membership (bitmap in shared memory up to 1.5M pins, else in the workspace) and writes its bitmap, a rank directory
 * and per-level pin / edge counts; one block admits and lays out the joined levels; blocks over (candidate, level)
 * compact the cones into the joined arrays.  ws: tm_forward_cones_ws(s->n, n_cand, s->num_levels) -- two n/8-byte
 * bitmaps per candidate plus 16 bytes per (candidate, level).  `s` needs order, level, level_ptr, f_ptr and f_src. */
int tm_forward_cones(const tm_schedule* s, int32_t n_cand, const int32_t* seed_ptr, const int32_t* seeds,
                     const int32_t* seed_slot, int64_t rows, int64_t edge_cap, int64_t n_endpoints,
                     const int32_t* endpoints, float* S, int32_t* order, int32_t* level_ptr, int32_t* f_ptr,
                     int32_t* f_src, int32_t* count, int32_t* vpin, int32_t* seed_rows, int32_t* head_rows,
                     int32_t* fitted, int32_t* sizes, int32_t* row_base, void* ws, size_t ws_bytes, void* stream);

size_t tm_forward_cones_within_ws(int64_t n, int32_t n_cand, int32_t num_levels, int64_t n_seeds);
/* tm_forward_cones restricted to a fan-in cone R(E) (what-if evaluation of an objective that reads only the endpoints
 * E): `s` is R(E)'s sub-schedule as tm_fanin_cone_bits wrote it and `within` its bitmap.  Candidate k's cone is its
 * forward cone intersected with R(E), exactly: every in-edge source of a pin of R(E) is in R(E), so the pins of R(E)
 * that candidate k can change are reached from its seeds inside R(E) through R(E) only.  A seed outside R(E) is
 * treated as one outside the schedule: not marked, not counted, the sink row in seed_rows.  The outputs are those of
 * tm_forward_cones (the endpoints passed are normally E).  seeds[n_seeds] with seed_ptr[n_cand] <= n_seeds.  One more
 * launch than tm_forward_cones (the seed filter), no host synchronisation.  ws: tm_forward_cones_within_ws(s->n, n_cand,
 * s->num_levels, n_seeds). */
int tm_forward_cones_within(const tm_schedule* s, const uint32_t* within, int32_t n_cand, const int32_t* seed_ptr,
                            const int32_t* seeds, const int32_t* seed_slot, int64_t n_seeds, int64_t rows,
                            int64_t edge_cap, int64_t n_endpoints, const int32_t* endpoints, float* S, int32_t* order,
                            int32_t* level_ptr, int32_t* f_ptr, int32_t* f_src, int32_t* count, int32_t* vpin,
                            int32_t* seed_rows, int32_t* head_rows, int32_t* fitted, int32_t* sizes,
                            int32_t* row_base, void* ws, size_t ws_bytes, void* stream);

/* Apply candidate k of a tm_forward_cones layout: H[vpin[r]] = H[n + r] and S[vpin[r]] = S[n + r] (128 floats a
 * row) for r in [row_base[k], row_base[k] + sizes[k]); nothing when fitted[k] == 0. */
int tm_what_if_commit(int64_t n, int32_t k, const int32_t* fitted, const int32_t* sizes, const int32_t* row_base,
                      const int32_t* vpin, float* H, float* S, void* stream);

/* pred[k * T + t] = NaN for every candidate k with fitted[k] == 0 (the rows of candidates not admitted). */
int tm_what_if_mask(int32_t n_cand, int64_t T, const int32_t* fitted, float* pred, void* stream);

/* ------------------------------------------------------------------------------------
 * dense fp32 building blocks (replace the cuBLAS SGEMMs behind nn.Linear,
 * src/model.py:15,23 and every MLP call site model.py:104,141-142,151,272,280,292)
 * ---------------------------------------------------------------------------------- */

/* epilogue flags for tm_gemm_nn */
#define TM_EPI_BIAS 1      /* C += bias[col]                                    */
#define TM_EPI_RELU 2      /* C = max(C,0)                                      */
#define TM_EPI_MASK 4      /* C *= (mask[row][col] > 0)   (ReLU backward)       */
#define TM_EPI_ACCUM 8     /* C += old C                                        */

/* C[M,N] = epi( A[M,K] @ B[K,N] ).  Row-major, leading dimensions in elements.
 * a_rows (optional, int32[M]): gather  A row i from A[a_rows[i]];
 * c_rows (optional, int32[M]): scatter C row i to   C[c_rows[i]] (mask is indexed like C). */
int tm_gemm_nn(int64_t M, int64_t N, int64_t K, const float* A, int64_t lda, const int32_t* a_rows,
               const float* B, int64_t ldb, float* C, int64_t ldc, const int32_t* c_rows,
               const float* bias, const float* mask, int64_t ldmask, int flags, void* stream);

size_t tm_gemm_tn_ws(int64_t M, int64_t N, int64_t R);
/* C[M,N] (+)= A[R,M]^T @ B[R,N]  (weight gradients; reduction over the R rows, deterministic
 * split + fixed-order second pass).  a_rows/b_rows optional row gathers.  Optional bias
 * gradients: colsum_a[M] (+)= sum_r A[r,:], colsum_b[N] (+)= sum_r B[r,:].
 * accumulate != 0 adds to C / colsum_*. */
int tm_gemm_tn(int64_t M, int64_t N, int64_t R, const float* A, int64_t lda, const int32_t* a_rows,
               const float* B, int64_t ldb, const int32_t* b_rows, float* C, int64_t ldc,
               float* colsum_a, float* colsum_b, int accumulate, void* ws, size_t ws_bytes,
               void* stream);

/* out[c][r] = in[r][c]  (weight re-layout; in is rows x cols row-major) */
int tm_transpose(int64_t rows, int64_t cols, const float* in, float* out, void* stream);

/* ------------------------------------------------------------------------------------
 * G2/G3  level-wise timing propagation (replaces PathConv.forward, src/model.py:158-213,
 *        its UDFs :88-116,:138-153 and the autograd backward train.py:553)
 * ---------------------------------------------------------------------------------- */

/* Forward over levels [level_begin, level_end).  D = 128, hidden = 256 (model.py:48).
 *   H[n,128]   in/out: rows of the processed levels are written, sources are read
 *              (caller zero-fills before level 0, like train.py:342,559);
 *   S[n,128]   hoisted self terms fc_cell_self(cell_feat) / fc_net_self(net_feat) incl. bias;
 *   W1t[128,256], b1[256], W2t[256,128], b2[128]: fc_cell_neigh, weights TRANSPOSED;
 *   A[n_cell_rows,128], LSE[n_cell_rows,128], HID[n_cell_rows,256]: saved for backward
 *              (may be NULL for inference). */
size_t tm_gnn_ws_bytes(void);   /* workspace of tm_gnn_forward / tm_gnn_backward: the packed weights and the grid-barrier
                                 * counter of the persistent kernels (default) / the re-packed weights of the per-level
                                 * kernels */
/* Implementation selector (process-wide; also env TM_GNN_IMPL=<bits>|persist|levels).  Bit 0 selects the forward
 * pass, bit 1 the backward pass; 4 (default) = auto: persistent forward, persistent backward only when the schedule
 * is wide (>= 6 000 pins per level on average) -- what measures fastest on config 2 and config 3:
 *   bit set   = ONE persistent kernel for the whole pass: 2-CTA clusters, fc_cell_neigh resident in shared memory,
 *               the tile MLP transposed on tcgen05 (fp16 two-term split, fp32 accumulate in TMEM), one grid-wide
 *               barrier per level;
 *   bit clear = one launch per level (mma.sync 3xTF32 tile MLP, weights streamed per level, PDL-chained);
 *   16        = the per-level cell kernels run the fp16 two-term split (mma.sync.m16n8k16) instead of 3xTF32.
 * Other bits are ignored.  Returns the previous value; impl < 0 only queries. */
int tm_gnn_set_impl(int impl);
/* Grid-wide barriers inside the last tm_gnn_forward / tm_gnn_backward call of this thread (persistent kernel:
 * one per non-empty level; per-level kernels: 0, they synchronise by kernel boundaries). */
int tm_gnn_last_barriers(void);
/* Diagnostics: with clocks != NULL (device int64 [grid CTAs <= 148][slots], zero-filled by the caller) thread 0 of
 * every CTA of the persistent kernels adds the SM cycles it spent per phase (setup, barrier wait, gather, MMA 1,
 * epilogue 1, MMA 2, exchange, tail; net-level wait / body / tail; slots = 16).  NULL disables. */
int tm_gnn_set_profile(void* clocks);
int tm_gnn_forward(const tm_schedule* s, int32_t level_begin, int32_t level_end, float* H,
                   const float* S, const float* W1t, const float* b1, const float* W2t,
                   const float* b2, float* A, float* LSE, float* HID, void* ws, size_t ws_bytes,
                   void* stream);

/* Backward over all levels in reverse.
 *   G[n,128]   in: dLoss/dH contributions from the head (zero elsewhere);
 *              out: dLoss/d(pre-activation) of every scheduled pin == dLoss/dS;
 *   W1[256,128], W2[128,256]: fc_cell_neigh weights as stored by nn.Linear;
 *   GA[n_cell_rows,128] scratch; GHID[n_cell_rows,256], GZC[n_cell_rows,128] out: operands of
 *   the hoisted weight-gradient GEMMs (dW1 = GHID^T A, dW2 = GZC^T HID).  GHID = GZC = NULL (both or neither): the
 *   data gradient alone, a compile-time variant of either back end that stores neither; G is the same bits. */
int tm_gnn_backward(const tm_schedule* s, const float* H, float* G, const float* W1,
                    const float* W2, const float* A, const float* LSE, const float* HID,
                    float* GA, float* GHID, float* GZC, void* ws, size_t ws_bytes, void* stream);

/* Forward over a sub-schedule built by tm_forward_cone (or any schedule with the device arrays order, f_ptr, f_src,
 * level_ptr, cell_base): the persistent kernel over levels [0, num_levels), empty levels skipped on the device,
 * nothing saved for a backward.  Never reads h_level_ptr.  H rows of the schedule's pins are rewritten, every other
 * row is read only; a pin's row is the same bits tm_gnn_forward's persistent back end writes for the same inputs.
 * ws: tm_gnn_ws_bytes(). */
int tm_gnn_forward_cone(const tm_schedule* cone, float* H, const float* S, const float* W1t, const float* b1,
                        const float* W2t, const float* b2, void* ws, size_t ws_bytes, void* stream);

/* What tm_gnn_forward saves for the backward (A, LSE, HID), recomputed over the cell levels of a sub-schedule built by
 * tm_fanin_cone whose in-edge sources are all final in H: per cell pin the gather's online softmax and the first
 * fc_cell_neigh product with its per-pin scale, written at the sub-schedule's cell rows (cell_base).  No second product,
 * no H store, no grid barrier.  The rows are the same bits tm_gnn_forward's persistent back end saves for those pins.
 * Never reads h_level_ptr.  ws: tm_gnn_ws_bytes(). */
int tm_gnn_save_cone(const tm_schedule* cone, const float* H, const float* W1t, const float* b1, const float* W2t,
                     float* A, float* LSE, float* HID, void* ws, size_t ws_bytes, void* stream);
/* tm_gnn_backward's data-gradient sweep (GHID = GZC = NULL) on the persistent back end over a sub-schedule built by
 * tm_fanin_cone, empty levels skipped on the device: G rows of the sub-schedule's pins are read (the head's gradient)
 * and rewritten with dLoss/dS; A / LSE / HID / GA are indexed by the sub-schedule's cell rows (tm_gnn_save_cone).  Never
 * reads h_level_ptr.  ws: tm_gnn_ws_bytes(). */
int tm_gnn_backward_cone(const tm_schedule* cone, const float* H, float* G, const float* W1, const float* W2,
                         const float* A, const float* LSE, const float* HID, float* GA, void* ws, size_t ws_bytes,
                         void* stream);

/* ------------------------------------------------------------------------------------
 * G5  mask fusion (replaces  path_mask.to_dense()*feat_map  and  fcn(path_map),
 *     src/train.py:500-501 + src/model.py:272)
 * ---------------------------------------------------------------------------------- */
/* out[t,0:D] = bias + sum_{j in mask row rows[t]} F[j] * Wt[j,:]     (Wt = fcn.weight^T, [J,D])
 * rows: optional int32[T] selecting mask rows (NULL = identity). D must be 128.
 * ld_out: row stride of out (lets the result land inside cat(h_gnn,h_cnn,h_global)). */
int tm_fuse_forward(int64_t T, int64_t J, int64_t D, const int32_t* mask_indptr,
                    const int32_t* mask_cols, const int32_t* rows, const float* F,
                    const float* Wt, const float* bias, float* out, int64_t ld_out, void* stream);
/* The same forward from the RUN-LENGTH form of the selected mask rows: endpoint t owns runs
 * run_ptr[t]..run_ptr[t+1], run r covers columns [run_lo[r], run_hi[r]).  Builds the fp64 prefix table
 * P[j] = sum_{i<j} F[i]*Wt[i,:] in ws (tm_fuse_runs_ws(J) bytes) and sums P[hi]-P[lo] per run:
 * 2 table rows per run instead of one weight row per column. */
size_t tm_fuse_runs_ws(int64_t J);
int tm_fuse_forward_runs(int64_t T, int64_t J, int64_t D, const int32_t* run_ptr, const int32_t* run_lo,
                         const int32_t* run_hi, const float* F, const float* Wt, const float* bias,
                         float* out, int64_t ld_out, void* ws, size_t ws_bytes, void* stream);
/* Column-major pull (deterministic, no atomics): csc_ptr[J+1], csc_t[nnz] list the positions t
 * (0..T-1) whose mask contains column j.
 *   dWt[j,:] = F[j] * sum_t g[t,:];   dF[j] = sum_t sum_c g[t,c] * Wt[j,c].
 * dWt = NULL (here and in tm_fuse_backward_multi): dF alone, the same bits. */
int tm_fuse_backward(int64_t T, int64_t J, int64_t D, const int32_t* csc_ptr, const int32_t* csc_t,
                     const float* g, int64_t ld_g, const float* F, const float* Wt, float* dWt,
                     float* dF, void* stream);
/* Several designs per step (the reference's per-design loop, src/train.py:461, taken K designs at a time):
 * design k owns rows ep_off[k]..ep_off[k+1] of out / g (int32 ep_off[K+1] on the device), its feature map F + k*J
 * and its own selected mask rows, named by design_tab: a device array of K records of five device pointers
 * {run_ptr, run_lo, run_hi, csc_ptr, csc_t} (the MaskRows buffers of tm_mask_select).
 * Forward: the K prefix tables are built in one launch (ws: tm_fuse_runs_multi_ws(K, J) bytes); design k's rows are
 * bit-identical to tm_fuse_forward_runs on design k.
 * Backward: dF [K][J], dF_k bit-identical to tm_fuse_backward on design k; dWt[j,:] = sum_k F_k[j] * sum_t g[t,:]
 * over design k's positions t, summed in design order (one [J][D] result, not K). */
size_t tm_fuse_runs_multi_ws(int64_t K, int64_t J);
int tm_fuse_forward_runs_multi(int64_t K, int64_t T, int64_t J, int64_t D, const void* design_tab,
                               const int32_t* ep_off, const float* F, const float* Wt, const float* bias,
                               float* out, int64_t ld_out, void* ws, size_t ws_bytes, void* stream);
int tm_fuse_backward_multi(int64_t K, int64_t J, int64_t D, const void* design_tab, const int32_t* ep_off,
                           const float* g, int64_t ld_g, const float* F, const float* Wt, float* dWt, float* dF,
                           void* stream);

/* ------------------------------------------------------------------------------------
 * N2  path-mask rasteriser (replaces the host code that builds `path_masks`:
 *     find_critical_path, verilog_parser_asap7.py:1433-1450, and the bounding-box rasterisation,
 *     :1302-1369).  src/dst: ALL pin-graph edges in insertion order (the order networkx iterates
 *     predecessors in); level: longest-path levels (tm_levelize / cal_topo_level); pin_xy: int32 [n][2]
 *     bins; endpoints: int32 [T].  Row t of the result = ascending columns x*map_size+y covered by the
 *     union of the bounding boxes of consecutive pins on endpoint t's critical path.
 *     tm_mask_count -> counts[t] (-1: a pin on the path has no predecessor one level below, where the
 *     reference would loop forever); the caller builds indptr = exclusive scan(counts) and sizes cols;
 *     tm_mask_fill writes cols.  Both use the same workspace (tm_mask_ws_bytes), untouched in between.
 * ---------------------------------------------------------------------------------- */
size_t tm_mask_ws_bytes(int64_t n, int64_t T, int64_t map_size);
int tm_mask_count(int64_t n, int64_t E, const int32_t* src, const int32_t* dst, const int32_t* level,
                  int64_t T, const int32_t* endpoints, const int32_t* pin_xy, int64_t map_size,
                  int32_t* counts, void* ws, size_t ws_bytes, void* stream);
int tm_mask_fill(int64_t n, int64_t T, int64_t map_size, const int32_t* indptr, int32_t* cols, void* ws,
                 size_t ws_bytes, void* stream);

/* Row selection of a path-mask CSR for one endpoint batch -- th.index_select(path_masks, 0, th.tensor(paths)),
 * src/train.py:500 (and :213, test.py:201) -- entirely on the device: no host round trip, every size a bound the
 * host already has, so it can be replayed inside a CUDA graph with `rows` as an input.
 *   rows[T]: mask row (path id) of every endpoint of the batch, repeats allowed (oversampled paths, train.py:377-380);
 *   run_ptr[T+1], run_lo / run_hi [cap]: run-length form of the selected rows (tm_fuse_forward_runs);
 *   csc_ptr[J+1], csc_t[cap]: column-major transpose, t ascending inside a column (tm_fuse_backward), built as a
 *            stable counting sort: deterministic without sorting;
 *   cap >= sum of the selected rows' lengths (e.g. T * longest row), J * 4 bytes <= 200 KB of shared memory. */
size_t tm_mask_select_ws(int64_t T, int64_t J);
int tm_mask_select(int64_t T, int64_t J, const int32_t* indptr, const int32_t* cols, const int32_t* rows,
                   int32_t* run_ptr, int32_t* run_lo, int32_t* run_hi, int32_t* csc_ptr, int32_t* csc_t,
                   void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * G6  head helpers (src/model.py:280-292, src/train.py:513-522)
 * ---------------------------------------------------------------------------------- */
/* dst[i, col0:col0+w] = src[rows ? rows[i] : i, 0:w]   (builds cat(h_gnn,h_cnn,h_global)) */
int tm_gather_cols(int64_t T, int64_t w, const float* src, int64_t lds, const int32_t* rows,
                   float* dst, int64_t ldd, int64_t col0, void* stream);
/* dst[rows[i], 0:w] += src[i, col0:col0+w]  (atomic: rows may repeat) */
int tm_scatter_add_cols(int64_t T, int64_t w, const float* src, int64_t lds, int64_t col0,
                        const int32_t* rows, float* dst, int64_t ldd, void* stream);
/* out[c] (+)= sum_r X[rows ? rows[r] : r, c]  (bias gradients; fixed reduction order) */
size_t tm_colsum_ws(int64_t R, int64_t C);
int tm_colsum(int64_t R, int64_t C, const float* X, int64_t ld, const int32_t* rows, float* out,
              int accumulate, void* ws, size_t ws_bytes, void* stream);
/* out[c_rows[m] * ldo] = act(X[a_rows[m], 0:K] . w + bias[0]): nn.Linear(K, 1) (mlp_fuse's last layer, model.py:292),
 * one warp per row. */
int tm_rowdot(int64_t M, int64_t K, const float* X, int64_t ldx, const int32_t* a_rows, const float* w,
              const float* bias, float* out, int64_t ldo, const int32_t* c_rows, int relu, void* stream);
/* tm_colsum (accumulate = 0) that also returns max |X[rows]| in absmax[0] (C % 4 == 0, 16-byte aligned rows). */
int tm_colsum_absmax(int64_t R, int64_t C, const float* X, int64_t ld, const int32_t* rows, float* out,
                     float* absmax, void* ws, size_t ws_bytes, void* stream);
/* loss[0] = mean((pred-y)^2); grad[i] = 2*(pred[i]-y[i])/T * grad_scale  (nn.MSELoss) */
int tm_mse(int64_t T, const float* pred, const float* y, float* loss, float* grad,
           float grad_scale, void* stream);
/* K designs' losses in one step (src/train.py:513-522 per design, averaged over the K designs): design k owns
 * positions ep_off[k]..ep_off[k+1] (int32 ep_off[K+1] on the device); loss_k[k] and grad on those positions are what
 * tm_mse computes for them with grad_scale / K; loss[0] = mean of loss_k in design order.  K = 1 equals tm_mse. */
int tm_mse_multi(int64_t K, const int32_t* ep_off, const float* pred, const float* y, float* loss_k, float* loss,
                 float* grad, float grad_scale, void* stream);
/* N4: the per-batch statistics the reference reads back one .item() at a time (train.py:513-549):
 * out8 = [mse, R2 (torchmetrics R2Score), correct, tp, fn, tn, fp, T] with predicted critical <=>
 * required - pred < 0 (judge_critical, train.py:391-395) against label (int64, 0 = non-critical).
 * required / label may be NULL (regression statistics only). */
int tm_step_metrics(int64_t T, const float* pred, const float* arrival, const float* required,
                    const int64_t* label, float* out8, void* stream);
/* The same statistics per segment, for validate() (train.py:137-291) and test.py's per-design / per-level report:
 * segment s is the endpoint list seg_idx[seg_ptr[s] .. seg_ptr[s+1]) (int32 on the device; segments may overlap or be
 * empty).  out (n_seg, 9) float32, row s = [mse, r2, correct, tp, fn, tn, fp, count, mape]: the first eight as out8 of
 * tm_step_metrics, mape = mean(|pred - y| / max(|y|, 1.17e-6)) (torchmetrics MeanAbsolutePercentageError).  r2 is NaN
 * for count < 2 or a zero total sum of squares; an empty segment gives count 0, NaN mse / r2 / mape and zero counts.
 * One CTA per segment, fp64 sums in a fixed order: the same bits on every launch.  No synchronisation (capturable).
 * required / label may be NULL. */
int tm_eval_metrics(int32_t n_seg, const int32_t* seg_ptr, const int32_t* seg_idx, const float* pred,
                    const float* arrival, const float* required, const int64_t* label, float* out, void* stream);

/* ------------------------------------------------------------------------------------
 * G4  U-Net / LayoutNet image branch, fp32 NHWC (replaces the cuDNN/ATen calls behind
 *     src/Unet.py:16-21,53,75-77 and src/model.py:227-243)
 *     Activations are NHWC with an explicit pixel stride `ld` (elements) so that a tensor may
 *     live inside a wider concat buffer (Unet.py:67 torch.cat becomes free).
 * ---------------------------------------------------------------------------------- */
int tm_nchw_to_nhwc(int64_t B, int64_t C, int64_t H, int64_t W, const float* in, float* out,
                    int64_t ld, void* stream);
int tm_nhwc_to_nchw(int64_t B, int64_t C, int64_t H, int64_t W, const float* in, int64_t ld,
                    float* out, void* stream);
/* Conv2d weight (Cout,Cin,k,k) -> fprop layout wf[k*k][Cin][Cout] and dgrad layout
 * wb[k*k][Cout][Cin] with flipped taps (either may be NULL). */
int tm_conv_pack_weight(int64_t Cout, int64_t Cin, int64_t k, const float* w, float* wf, float* wb,
                        void* stream);
/* inverse of the fprop layout: dw (Cout,Cin,k,k) = unpack(dwf[k*k][Cin][Cout]) */
int tm_conv_unpack_wgrad(int64_t Cout, int64_t Cin, int64_t k, const float* dwf, float* dw,
                         void* stream);
/* y[b,y,x,co] = bias[co] + sum_{tap,ci} x[b,y+dy,x+dx,ci] * wf[tap][ci][co]; stride 1, pad k/2.
 * flags: TM_EPI_RELU optional.  The same call with wb computes the data gradient. */
int tm_conv2d_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                   const float* x, int64_t ldx, const float* wf, const float* bias, float* y,
                   int64_t ldy, int flags, void* stream);
size_t tm_conv2d_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k);
/* dwf[tap][ci][co] = sum_{b,y,x} x[b,y+dy,x+dx,ci] * dy[b,y,x,co];  dbias[co] = sum dy (optional) */
int tm_conv2d_wgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                         const float* x, int64_t ldx, const float* dy, int64_t lddy, float* dwf,
                         float* dbias, void* ws, size_t ws_bytes, void* stream);

/* ConvTranspose2d(k=2,s=2) weight (Cin,Cout,2,2) -> wt[Cin][4*Cout] ((dy,dx,co) fastest) and
 * its transpose wtT[4*Cout][Cin]. */
int tm_convt_pack_weight(int64_t Cin, int64_t Cout, const float* w, float* wt, float* wtT,
                         void* stream);
int tm_convt_unpack_wgrad(int64_t Cin, int64_t Cout, const float* dwt, float* dw, void* stream);
/* y[b,2y+dy+oy,2x+dx+ox,co] = bias[co] + sum_ci x[b,y,x,ci]*wt[ci][(dy,dx,co)]  (Unet.py:53,57-63)
 * y is (B,Hy,Wy,*) with pixel stride ldy; (oy,ox) is the F.pad offset. */
int tm_convt2x2_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* x,
                     int64_t ldx, const float* wt, const float* bias, float* y, int64_t ldy,
                     int64_t Hy, int64_t Wy, int64_t oy, int64_t ox, void* stream);
/* dx[b,y,x,ci] = sum_{dy,dx,co} dyo[b,2y+dy+oy,2x+dx+ox,co] * wtT[(dy,dx,co)][ci] */
int tm_convt2x2_dgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout,
                           const float* dyo, int64_t lddy, int64_t Hy, int64_t Wy, int64_t oy,
                           int64_t ox, const float* wtT, float* dx, int64_t lddx, void* stream);
size_t tm_convt2x2_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
/* dwt[ci][(dy,dx,co)] = sum x*dyo ; dbias[co] = sum over the 2H x 2W window of dyo */
int tm_convt2x2_wgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout,
                           const float* x, int64_t ldx, const float* dyo, int64_t lddy, int64_t Hy,
                           int64_t Wy, int64_t oy, int64_t ox, float* dwt, float* dbias, void* ws,
                           size_t ws_bytes, void* stream);

size_t tm_bn_ws(int64_t npix, int64_t C);
/* Train-mode BatchNorm2d + ReLU (Unet.py:17-18,20-21): batch statistics over B*H*W,
 * y = relu(gamma*(x-mean)*invstd+beta); running stats updated with `momentum`, unbiased var.
 * save_mean/save_invstd [C] kept for backward.  y_bf16 (optional): compact bf16 copy [npix][C] of y written by
 * the same pass (the TMA operand of the next convolution in bf16 mode); dx_bf16 likewise for the backward.
 * stats_part (optional): nparts fp64 partials [nparts][C][2] (sum, sum of squares) already produced by the
 * convolution's epilogue (tm_conv3x3_bf16 stats): the statistics pass over x is skipped. */
int tm_bn_relu_forward(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* gamma,
                       const float* beta, float* running_mean, float* running_var, float momentum,
                       float eps, float* y, int64_t ldy, float* save_mean, float* save_invstd,
                       void* y_bf16, const void* stats_part, int64_t nparts, void* ws, size_t ws_bytes, void* stream);
/* The same pair with nn.BatchNorm2d in EVAL mode (module.eval()): y = relu(gamma * (x - running_mean) *
 * rsqrt(running_var + eps) + beta); save_mean / save_invstd receive the statistics used (inference only). */
int tm_bn_relu_eval(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* gamma, const float* beta,
                    const float* running_mean, const float* running_var, float eps, float* y, int64_t ldy,
                    float* save_mean, float* save_invstd, void* y_bf16, void* stream);
/* Backward of the pair: dy is the gradient w.r.t. the ReLU output y.
 * dx = BN'( dy * (y>0) ), dgamma, dbeta [C].  dx may be NULL when only dx_bf16 is wanted; y may be NULL:
 * the ReLU mask is then rebuilt bit-for-bit from x, the saved statistics, gamma and beta (one tensor less to
 * read, and the forward need not store y: tm_bn_relu_forward accepts y = NULL when y_bf16 is given). */
int tm_bn_relu_backward(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* y,
                        int64_t ldy, const float* dy, int64_t lddy, const float* gamma, const float* beta,
                        const float* save_mean, const float* save_invstd, float* dx, int64_t lddx,
                        float* dgamma, float* dbeta, void* dx_bf16, void* ws, size_t ws_bytes, void* stream);
/* The same pair over nseg images of npix pixels each, with each image's OWN statistics: what the reference's
 * batch-of-one cnn(cnn_inputs) (src/train.py:465) computes for every design of a multi-design step.  Image k's rows
 * start at x + k*npix*ldx (likewise y, dy, dx; y_bf16 / dx_bf16 compact [nseg*npix][C]); save_mean / save_invstd are
 * [nseg][C].  Each image uses the block partition and fold order of a single-image call, so its y, statistics and dx
 * are bit-identical to tm_bn_relu_forward / tm_bn_relu_backward on that image.  The running statistics are updated
 * nseg times, image 0 first; dgamma / dbeta [C] are the per-image values summed in image order.
 * ws: tm_bn_seg_ws(nseg, npix, C) bytes. */
size_t tm_bn_seg_ws(int64_t nseg, int64_t npix, int64_t C);
int tm_bn_relu_forward_seg(int64_t nseg, int64_t npix, int64_t C, const float* x, int64_t ldx, const float* gamma,
                           const float* beta, float* running_mean, float* running_var, float momentum, float eps,
                           float* y, int64_t ldy, float* save_mean, float* save_invstd, void* y_bf16, void* ws,
                           size_t ws_bytes, void* stream);
int tm_bn_relu_backward_seg(int64_t nseg, int64_t npix, int64_t C, const float* x, int64_t ldx, const float* y,
                            int64_t ldy, const float* dy, int64_t lddy, const float* gamma, const float* beta,
                            const float* save_mean, const float* save_invstd, float* dx, int64_t lddx, float* dgamma,
                            float* dbeta, void* dx_bf16, void* ws, size_t ws_bytes, void* stream);

/* OutConv (Unet.py:74-75): nn.Conv2d(C, 1, kernel_size=1) as streaming kernels, exact fp32.
 * forward y[p] = x[p,:] . w + bias; dgrad dx[p,c] = dy[p] * w[c]; wgrad dw[c] = sum_p x[p,c] dy[p], dbias = sum_p dy[p]. */
int tm_conv1x1_c1_forward(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* w, const float* bias,
                          float* y, int64_t ldy, void* stream);
int tm_conv1x1_c1_dgrad(int64_t npix, int64_t C, const float* dy, int64_t lddy, const float* w, float* dx, int64_t lddx,
                        void* stream);
size_t tm_conv1x1_c1_wgrad_ws(int64_t C);
int tm_conv1x1_c1_wgrad(int64_t npix, int64_t C, const float* x, int64_t ldx, const float* dy, int64_t lddy, float* dw,
                        float* dbias, void* ws, size_t ws_bytes, void* stream);

/* Gradient w.r.t. the input image of the first convolution of each image network (U-Net inc.double_conv.0: k = 3,
 * 16 -> 3; LayoutNet encode.0: k = 9, 32 -> 2): dx = conv_transpose2d(dy, w) for nn.Conv2d(Cin, Cout, k, stride 1,
 * padding k/2).  dy: NHWC [B][H][W], pixel stride lddy, Cout channels, fp32 (dy_bf16 = 0) or bf16 (dy_bf16 = 1);
 * w: the nn.Conv2d weight [Cout][Cin][k][k] fp32; dx: NCHW fp32 [B][Cin][H][W], every element written.
 * k in {3, 9}, 1 <= Cin <= 4, Cout % 8 == 0, lddy % 8 == 0, dy 16-byte aligned.  Direct convolution on the CUDA
 * cores (fp32 products and accumulation in a fixed order: deterministic, fp32-class for fp32 dy). */
int tm_conv_dgrad_narrow(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k, const void* dy,
                         int64_t lddy, int dy_bf16, const float* w, float* dx, void* stream);

/* 2x2 stride-2 pooling (Unet.py:89-91, model.py:222-224). mode 0 = max (idx: uint8 argmax
 * saved for backward, first maximum in row-major window order), 1 = avg (idx unused).
 * flags: TM_EPI_RELU applies ReLU after pooling (OutConv, Unet.py:76-77). */
int tm_pool2x2_forward(int64_t B, int64_t H, int64_t W, int64_t C, int mode, const float* x,
                       int64_t ldx, float* y, int64_t ldy, uint8_t* idx, int flags, void* stream);
/* dx (B,H,W,C) fully written (zeros where no gradient flows; odd trailing row/col get 0).
 * With TM_EPI_RELU, dy is first masked by (y>0).  add (optional, pixel stride ldadd): a second gradient of the
 * pooled tensor's source (the U-Net skip connection, Unet.py:67) summed into dx by the same pass. */
int tm_pool2x2_backward(int64_t B, int64_t H, int64_t W, int64_t C, int mode, const float* dy,
                        int64_t lddy, const float* y, int64_t ldy, const uint8_t* idx, float* dx,
                        int64_t lddx, int flags, const float* add, int64_t ldadd, void* stream);
/* dx = dy * (y > 0) * (slope where y <= 0)   elementwise helper for bare ReLU / LeakyReLU layers
 * (LayoutNet, model.py:219-220).  y is the activation OUTPUT. n elements, contiguous. */
int tm_leaky_relu_backward(int64_t n, const float* y, const float* dy, float slope, float* dx,
                           void* stream);
int tm_leaky_relu_forward(int64_t n, const float* x, float slope, float* y, void* stream);
/* dst[i*ldd + c] += src[i*lds + c]  for c < C  (adds a gradient living in a strided buffer) */
int tm_add_strided(int64_t npix, int64_t C, const float* src, int64_t lds, float* dst, int64_t ldd,
                   void* stream);

/* ------------------------------------------------------------------------------------
 * Tensor-core variants (tcgen05.mma kind::f16, accumulator in TMEM) of the dense contractions.
 * Same meaning as tm_gemm_nn / tm_gemm_tn / tm_conv2d_nhwc / tm_conv2d_wgrad_nhwc above.
 *   precision 0: operands rounded to bf16 (fp32 accumulate)            -- rtol 2e-2 class
 *   precision 1: operands split into two bf16 terms, three MMAs        -- ~16-bit products
 *   precision 2: operands split into three bf16 terms (24 bits), six MMAs -- fp32-class
 *   precision 3: 3xTF32 -- kind::tf32 on the raw fp32 words (hi) plus the residual x - trunc_tf32(x) (lo),
 *                hi*hi + hi*lo + lo*hi, ~21-bit products -- fp32-class, the default rtol 1e-3 path
 *   precision 4: single-pass TF32
 *   err: optional device int32, set to 1 if a tensor-core barrier timed out (never expected).
 * tm_tc_gemm_nn: b_is_nk != 0 means B is given as [N,K] row-major (an nn.Linear weight as
 * stored), otherwise [K,N] row-major like tm_gemm_nn.
 * ---------------------------------------------------------------------------------- */
int tm_tc_gemm_nn(int64_t M, int64_t N, int64_t K, const float* A, int64_t lda, const int32_t* a_rows,
                  const float* B, int64_t ldb, int b_is_nk, float* C, int64_t ldc,
                  const int32_t* c_rows, const float* bias, const float* mask, int64_t ldmask,
                  int flags, int precision, int* err, void* stream);
/* Backward of the FIRST layer of an MLP whose input has 1 or 2 columns (fc_net_self.layers.0 = Linear(2,256),
 * model.py:50), fused into the data-gradient GEMM of the second layer: with dh = (G[g_rows] @ W2) * (H > 0)
 * (never written) it returns db1[n] = sum_m dh[m,n] and dW1[n,c] = sum_m dh[m,n] * X[x_rows[m], c].
 * W2t: the second layer's weight transposed to [N,K] row-major (N = hidden width <= 256, K = its outputs);
 * H: [M,N] hidden activations; 3xTF32; deterministic (fixed-order partial sums in ws). */
size_t tm_tc_mlp1_bwd_ws(int64_t N);
int tm_tc_mlp1_bwd_fused(int64_t M, int64_t N, int64_t K, const float* G, int64_t ldg, const int32_t* g_rows,
                         const float* W2t, const float* H, int64_t ldh, const float* X, int64_t ldx,
                         const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, float* dW1,
                         float* db1, void* ws, size_t ws_bytes, int* err, void* stream);
/* The same MLP (first layer Linear(kx <= 2, K)) with the hidden layer GENERATED inside the operand loaders
 * instead of stored (2 FMAs per element; H = NULL above then regenerates the ReLU mask from W1, b1):
 *   forward:  out[out_rows[m], 0:N] = relu(X[x_rows[m]] @ W1^T + b1) @ W2^T + b2     (W2: [N,K] as stored)
 *   wgrad2:   dW2[Mo, hid] = G[g_rows]^T @ relu(X[x_rows] @ W1^T + b1)               (ws: tm_tc_gemm_tn_ws) */
/* The forward of that MLP for the reference's sizes (hidden 256, 128 outputs: fc_net_self, model.py:46,151) as ONE
 * fused kernel: generator warps write the hidden tile straight into fp16 two-term-split operand planes, W2 is split
 * once and stays resident in shared memory, tcgen05.mma with the accumulators in TMEM (csrc/tm_selfmlp.cu).
 * ws: tm_selfmlp_ws_bytes(). */
size_t tm_selfmlp_ws_bytes(void);
/* Its second-layer weight gradient dW2[128][256] = G[g_rows]^T relu(W1 X[x_rows] + b1) as ONE fused kernel of the same
 * kind (the hidden layer generated as the B operand, G transposed into the A operand on the way in, contraction over
 * the rows on tcgen05 with the accumulators resident in TMEM for the whole kernel).  A contraction over rows cannot
 * use per-row scales: `gmax` = device scalar holding max|G| over the rows (tm_colsum_absmax computes it in the pass
 * that takes the bias gradient).  ws: tm_selfmlp_wgrad2_ws_bytes(). */
/* ... and its first-layer gradients db1[256], dW1[256][kx] = reductions of dh = (G[g_rows] W2) * (W1 x + b1 > 0) over
 * the rows; dh is never written (per-lane column accumulators in registers).  W2: [128][256] as stored.
 * ws: tm_selfmlp_bwd1_ws_bytes(). */
size_t tm_selfmlp_bwd1_ws_bytes(void);
int tm_selfmlp_gen_bwd1(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* X, int64_t ldx,
                        const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, const float* W2,
                        float* dW1, float* db1, void* ws, size_t ws_bytes, void* stream);
/* The same kernel with the input's data gradient as well: dX[r, 0:kx] = dh W1 for row m, r = x_rows ? x_rows[m] : m
 * (the row the forward read), summed over the 256 hidden units in a fixed order: deterministic.  dW1 / db1 are bitwise
 * those of tm_selfmlp_gen_bwd1.  The rows r must be distinct (each row of dX is written by one thread, never
 * accumulated); rows of dX that no m maps to are left untouched.  dW1 = db1 = NULL: dX alone (the column accumulators and
 * their reduction are compiled out), the same bits.  ws: tm_selfmlp_bwd1_ws_bytes(). */
int tm_selfmlp_gen_bwd1_dx(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* X, int64_t ldx,
                           const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, const float* W2,
                           float* dW1, float* db1, float* dX, int64_t lddx, void* ws, size_t ws_bytes, void* stream);
/* The same product for an MLP whose hidden activations H were STORED (fc_cell_self, 36 inputs): the hidden-layer
 * gradient DH[r] = (G[g_rows[m]] @ W2) * (H[r] > 0), r = h_rows ? h_rows[m] : m, written out (it feeds the first-layer
 * weight gradient).  Replaces the masked data-gradient GEMM of the general MLP backward. */
/* First layer of such an MLP: HID[m, 0:256] = relu(X[x_rows[m], 0:kin] @ W1^T + b1), kin % 4 == 0, kin <= 48;
 * rowmax (optional, [M]): max of row m's outputs.  Second layer: out[out_rows[m], 0:128] = HID[h_rows[m]] @ W2^T + b2
 * with the per-row operand scale taken from rowmax (ws: tm_selfmlp_ws_bytes()). */
size_t tm_selfmlp_lin1_ws_bytes(void);
int tm_selfmlp_lin1_relu(int64_t M, const float* X, int64_t ldx, const int32_t* x_rows, int64_t kin, const float* W1,
                         const float* b1, float* HID, int64_t ldh, float* rowmax, void* ws, size_t ws_bytes,
                         void* stream);
int tm_selfmlp_rows_forward(int64_t M, const float* H, int64_t ldh, const int32_t* h_rows, const float* rowmax,
                            const float* W2, const float* b2, float* out, int64_t ldo, const int32_t* out_rows,
                            void* ws, size_t ws_bytes, void* stream);
size_t tm_selfmlp_rows_dh_ws_bytes(void);
int tm_selfmlp_rows_dh(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* W2, const float* H,
                       int64_t ldh, const int32_t* h_rows, float* DH, int64_t lddh, void* ws, size_t ws_bytes,
                       void* stream);
/* The data gradient of that MLP in one pass: dX[r, 0:kin] = ((G[g_rows[m]] @ W2) * (H[h_rows[m]] > 0)) @ W1,
 * r = x_rows ? x_rows[m] : m (distinct), W1 [256][kin] as stored, kin % 4 == 0, kin <= 48.  The first product runs as in
 * tm_selfmlp_rows_dh (the same ReLU gates); the hidden gradient is never written: the lane that owns a row multiplies it
 * into W1 in hidden-unit order, so the result is deterministic.  ws: tm_selfmlp_rows_dh_ws_bytes(). */
int tm_selfmlp_rows_dx(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* W2, const float* H,
                       int64_t ldh, const int32_t* h_rows, const float* W1, int64_t kin, float* dX, int64_t lddx,
                       const int32_t* x_rows, void* ws, size_t ws_bytes, void* stream);
/* tm_selfmlp_lin1_relu (without rowmax), tm_selfmlp_rows_dx and tm_selfmlp_gen_bwd1_dx (dW1 = db1 = NULL) over a row
 * count that exists only on the device: m_dev (device int32) holds it, at most `cap`, the host capacity the grid is sized
 * by; CTAs past the count do nothing.  Row m's results are the same bits as with the host count (a fan-in cone's class
 * lists, tm_fanin_cone). */
int tm_selfmlp_lin1_relu_dcount(int64_t cap, const int32_t* m_dev, const float* X, int64_t ldx, const int32_t* x_rows,
                                int64_t kin, const float* W1, const float* b1, float* HID, int64_t ldh, void* ws,
                                size_t ws_bytes, void* stream);
int tm_selfmlp_rows_dx_dcount(int64_t cap, const int32_t* m_dev, const float* G, int64_t ldg, const int32_t* g_rows,
                              const float* W2, const float* H, int64_t ldh, const int32_t* h_rows, const float* W1,
                              int64_t kin, float* dX, int64_t lddx, const int32_t* x_rows, void* ws, size_t ws_bytes,
                              void* stream);
int tm_selfmlp_gen_bwd1_dx_dcount(int64_t cap, const int32_t* m_dev, const float* G, int64_t ldg, const int32_t* g_rows,
                                  const float* X, int64_t ldx, const int32_t* x_rows, int64_t kx, const float* W1,
                                  const float* b1, const float* W2, float* dX, int64_t lddx, void* ws, size_t ws_bytes,
                                  void* stream);
size_t tm_selfmlp_wgrad2_ws_bytes(void);
int tm_selfmlp_gen_wgrad2(int64_t M, const float* G, int64_t ldg, const int32_t* g_rows, const float* X, int64_t ldx,
                          const int32_t* x_rows, int64_t kx, const float* W1, const float* b1, const float* gmax,
                          float* dW2, void* ws, size_t ws_bytes, void* stream);
int tm_selfmlp_gen_forward(int64_t M, const float* X, int64_t ldx, const int32_t* x_rows, int64_t kx,
                           const float* W1, const float* b1, const float* W2, const float* b2, float* out,
                           int64_t ldo, const int32_t* out_rows, void* ws, size_t ws_bytes, void* stream);
int tm_tc_mlp2_smallk_forward(int64_t M, int64_t K, int64_t N, const float* X, int64_t ldx, const int32_t* x_rows,
                              int64_t kx, const float* W1, const float* b1, const float* W2, const float* b2,
                              float* out, int64_t ldo, const int32_t* out_rows, int precision, int* err,
                              void* stream);
int tm_tc_mlp2_smallk_wgrad2(int64_t Mo, int64_t hid, int64_t R, const float* G, int64_t ldg, const int32_t* g_rows,
                             const float* X, int64_t ldx, const int32_t* x_rows, int64_t kx, const float* W1,
                             const float* b1, float* dW2, int precision, void* ws, size_t ws_bytes, int* err,
                             void* stream);
/* At most `cap` persistent CTAs for the tcgen05 GEMM / convolution launches of the calling thread (0 = one per SM);
 * returns the previous value.  Lets a caller keep SMs free for a latency-critical kernel chain on another stream. */
int tm_tc_set_grid_cap(int cap);
size_t tm_tc_gemm_tn_ws(int64_t M, int64_t N, int64_t R);
int tm_tc_gemm_tn(int64_t M, int64_t N, int64_t R, const float* A, int64_t lda, const int32_t* a_rows,
                  const float* B, int64_t ldb, const int32_t* b_rows, float* C, int64_t ldc,
                  int accumulate, int precision, void* ws, size_t ws_bytes, int* err, void* stream);
int tm_tc_conv2d_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                      const float* x, int64_t ldx, const float* wf, const float* bias, float* y,
                      int64_t ldy, int flags, int precision, int* err, void* stream);
/* The same convolution with the K = k*k*Cin range split over CTAs when the layer has too few 128-pixel tiles to
 * fill the GPU (the 64 x 64 and 32 x 32 maps of one 256 x 256 design); partial tiles in `ws`, folded in a fixed
 * order.  Falls through to tm_tc_conv2d_nhwc when no split pays (ws may then be NULL / 0 bytes). */
size_t tm_tc_conv2d_splitk_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k, int precision);
int tm_tc_conv2d_nhwc_splitk(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                             const float* x, int64_t ldx, const float* wf, const float* bias, float* y,
                             int64_t ldy, int flags, int precision, void* ws, size_t ws_bytes, int* err,
                             void* stream);
size_t tm_tc_conv2d_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k);
int tm_tc_conv2d_wgrad_nhwc(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k,
                            const float* x, int64_t ldx, const float* dy, int64_t lddy, float* dwf,
                            int precision, void* ws, size_t ws_bytes, int* err, void* stream);

/* ------------------------------------------------------------------------------------
 * A6 (bf16 mode)  TMA-fed tcgen05 3x3 convolutions on bf16 NHWC activations
 * Replaces nn.Conv2d(k=3, padding=1, bias=False) of DoubleConv (src/Unet.py:15-22) and its
 * autograd (data + weight gradients) when the image branch runs with bf16 tensor-core operands
 * (BASELINE config 4).  Activations are compact bf16 [B][H][W][C], C a multiple of 16; H and W
 * powers of two.  One cp.async.bulk.tensor box per (128-pixel tile, tap): the box shifted by the
 * tap offset, out-of-bounds zero fill = the convolution's padding.  fp32 accumulate in TMEM,
 * fp32 outputs (they feed the batch-norm statistics).
 * ---------------------------------------------------------------------------------- */
int tm_conv3x3_bf16_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
/* fp32 rows (stride ldx, C channels) -> compact bf16 rows of Cp >= C channels (zero padded) */
int tm_to_bf16_rows(int64_t npix, int64_t C, const float* x, int64_t ldx, void* out, int64_t Cp, void* stream);
/* Narrow layers run as 64-channel layers over rows of P horizontally adjacent pixels (every TMA row a full
 * 128-byte line; the packed weights are block sparse).  P for a convolution reading Cin and producing Cout
 * channels per pixel on images W wide: */
int tm_conv3x3_bf16_pack(int64_t W, int64_t Cin, int64_t Cout);
/* nn.Conv2d weight w [Cout][Cin][3][3] fp32 -> bf16 operand q [9][P*Nc][P*KcP] of tm_conv3x3_bf16:
 * dgrad = 0: forward (Nc = Cout, K = Cin padded to KcP); dgrad = 1: data gradient (Nc = Cin, K = Cout padded
 * to KcP, taps reversed).  P = tm_conv3x3_bf16_pack(W, K padded, Nc). */
int tm_conv3x3_pack_bf16(int64_t Cout, int64_t Cin, const float* w, void* q, int64_t P, int64_t KcP, int dgrad,
                         void* stream);
/* y[pix, 0:N] (fp32, row stride ldy) = sum_{tap,c} xb[pix + tap, c] * W[tap][n][c]; bias optional,
 * flags: TM_EPI_RELU.  The data gradient is the same call on bf16(dy) with the dgrad operand. */
/* stats (optional; tm_conv3x3_bf16_stats_bytes(N, P) bytes; bias must be NULL, P * N <= 128): the batch-norm
 * statistics of the output, taken from the fp32 accumulators by the epilogue -- fp64 partial sums / sums of squares,
 * layout [slots = SMs * 4][P][N][2], consumed by tm_bn_relu_forward(stats_part, nparts = slots * P). */
size_t tm_conv3x3_bf16_stats_bytes(int64_t N, int64_t P);
int tm_conv3x3_bf16(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t P, const void* xb, const void* wq,
                    const float* bias, float* y, int64_t ldy, int flags, void* stats, int* err, void* stream);
/* nn.ConvTranspose2d(k=2, s=2) (Unet.py:53) on the same TMA path.  Weight w [Cin][Cout][2][2] fp32 ->
 * wf bf16 [4*Cout][Cin] (forward operand) and wd bf16 [4][Cin][Cout] (data-gradient operand; either may be NULL).
 * forward: y[b,2y+dy,2x+dx,co] = bias[co] + sum_ci xb[b,y,x,ci] w[ci][co][dy][dx]: ONE tap, the accumulator row of
 *   an input pixel is its 2x2 output window, scattered by the epilogue into (B,2H,2W,*) rows of stride ldy;
 * dgrad: dx[b,y,x,ci] = sum dyb[b,2y+dy,2x+dx,co] w[ci][co][dy][dx]: four taps, each reading every other pixel of
 *   the compact bf16 gradient [B][2H][2W][Cout] through a tensor map with element strides (1,2,2,1). */
int tm_convt2x2_bf16_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
int tm_convt2x2_pack_bf16(int64_t Cin, int64_t Cout, const float* w, void* wf, void* wd, void* stream);
int tm_convt2x2_bf16(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const void* xb, const void* wf,
                     const float* bias, float* y, int64_t ldy, int* err, void* stream);
int tm_convt2x2_bf16_dgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const void* dyb, const void* wd,
                           float* dx, int64_t lddx, int* err, void* stream);
/* dw[ci][co][dy][dx] (torch layout) = sum xb[b,y,x,ci] * dyb[b,2y+dy,2x+dx,co]; the bias gradient is tm_colsum of dy */
size_t tm_convt2x2_bf16_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
int tm_convt2x2_bf16_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const void* xb, const void* dyb,
                           float* dw, void* ws, size_t ws_bytes, int* err, void* stream);
/* dw[co][ci][ky][kx] (torch layout, ci < Cin_real) = sum_pix dyb[pix, co] * xb[pix + (ky-1,kx-1), ci] */
size_t tm_conv3x3_bf16_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
int tm_conv3x3_bf16_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cin_real, int64_t Cout,
                          const void* xb, const void* dyb, float* dw, void* ws, size_t ws_bytes, int* err,
                          void* stream);

/* ------------------------------------------------------------------------------------
 * A6' (tf32x3 mode)  The A6 kernels with fp32-class operands: 3xTF32 products (hi*hi + hi*lo + lo*hi,
 * lo = x - trunc_tf32(x)), the arithmetic of precision 3.  The operands are the fp32 activations read in
 * place by TMA through their pixel stride (16-byte aligned rows; packed rows, P > 1, need compact rows);
 * the lo planes are formed in shared memory, so no operand copy exists.  Weights packed in fp32.  Layers
 * whose tiles leave SMs idle split K over taps and channel steps; the fp32 partials (workspace) are folded
 * in a fixed order, so every call is deterministic.
 * ---------------------------------------------------------------------------------- */
/* 1 when forward and weight gradient take the shape (Cin -> Cout; the data gradient is the Cout -> Cin forward) */
int tm_conv3x3_tf32_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
/* pixels per packed row (rows of 32 fp32 channels); pack weights with it as for tm_conv3x3_bf16_pack */
int tm_conv3x3_tf32_pack(int64_t W, int64_t Cin, int64_t Cout);
/* the operand of tm_conv3x3_pack_bf16, fp32: q [9][P*Nc][P*KcP] */
int tm_conv3x3_pack_f32(int64_t Cout, int64_t Cin, const float* w, float* q, int64_t P, int64_t KcP, int dgrad,
                        void* stream);
/* workspace of tm_conv3x3_tf32 (0: the launch is not split; only then may it take stats) */
size_t tm_conv3x3_tf32_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t P);
/* y[pix, 0:N] (row stride ldy) = act(bias + sum_{tap,c} x[pix + tap, c] * W[tap][n][c]); x fp32 rows of stride ldx.
 * stats as for tm_conv3x3_bf16 (unsplit launches only). */
int tm_conv3x3_tf32(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t P, const float* x, int64_t ldx,
                    const float* wq, const float* bias, float* y, int64_t ldy, int flags, void* stats, void* ws,
                    size_t ws_bytes, int* err, void* stream);
size_t tm_conv3x3_tf32_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
/* dw[co][ci][ky][kx] (ci < Cin_real) = sum_pix dy[pix, co] * x[pix + (ky-1,kx-1), ci] */
int tm_conv3x3_tf32_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cin_real, int64_t Cout,
                          const float* x, int64_t ldx, const float* dy, int64_t lddy, float* dw, void* ws,
                          size_t ws_bytes, int* err, void* stream);
/* nn.ConvTranspose2d(k=2, s=2) as tm_convt2x2_bf16*: forward and data gradient take every convt2x2 shape; the
 * weight gradient needs Cin, Cout multiples of 32 (Cin <= 128, Cout <= 64).  One workspace size for all three. */
int tm_convt2x2_tf32_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
int tm_convt2x2_tf32_wgrad_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
int tm_convt2x2_pack_f32(int64_t Cin, int64_t Cout, const float* w, float* wf, float* wd, void* stream);
size_t tm_convt2x2_tf32_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout);
int tm_convt2x2_tf32(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* x, int64_t ldx,
                     const float* wf, const float* bias, float* y, int64_t ldy, void* ws, size_t ws_bytes, int* err,
                     void* stream);
int tm_convt2x2_tf32_dgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* dy, int64_t lddy,
                           const float* wd, float* dx, int64_t lddx, void* ws, size_t ws_bytes, int* err, void* stream);
int tm_convt2x2_tf32_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, const float* x, int64_t ldx,
                           const float* dy, int64_t lddy, float* dw, void* ws, size_t ws_bytes, int* err, void* stream);

/* ------------------------------------------------------------------------------------
 * A7 (bf16 mode)  TMA-fed tcgen05 k x k convolutions (odd k <= 9, stride 1, zero padding k/2)
 * Replaces nn.Conv2d(32, 64, 7, 1, 3) and nn.Conv2d(64, 32, 9, 1, 4) of LayoutNet (src/model.py:227-243) and
 * their autograd (data + weight gradients) when the image branch runs with bf16 tensor-core operands.  The kernels
 * of A6 with k*k taps; operand rows are single pixels and the weights stream through the shared-memory ring.
 * Activations compact bf16 [B][H][W][C] (tm_to_bf16_rows); H and W powers of two; Cin in {16, 32, 64},
 * Cout in {16, 32, 64, 128}.
 * ---------------------------------------------------------------------------------- */
/* 1 when forward, data gradient and weight gradient all take the shape, else 0 */
int tm_convkxk_bf16_supported(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k);
/* nn.Conv2d weight w [Cout][Cin][k][k] fp32 -> bf16 operand q [k*k][Nc][KcP] of tm_convkxk_bf16: dgrad = 0: forward
 * (Nc = Cout, K = Cin padded to KcP); dgrad = 1: data gradient (Nc = Cin, K = Cout padded to KcP, taps reversed). */
int tm_convkxk_pack_bf16(int64_t Cout, int64_t Cin, int64_t k, const float* w, void* q, int64_t KcP, int dgrad,
                         void* stream);
/* y[pix, 0:N] (fp32, row stride ldy) = act(bias + sum_{tap,c} xb[pix + tap, c] * q[tap][n][c]); bias optional,
 * flags: TM_EPI_RELU.  The data gradient is the same call on bf16(dy) with the dgrad operand and no bias. */
int tm_convkxk_bf16(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t N, int64_t k, const void* xb, const void* wq,
                    const float* bias, float* y, int64_t ldy, int flags, int* err, void* stream);
/* dw[co][ci][ky][kx] (torch layout) = sum_pix dyb[pix, co] * xb[pix + (ky-k/2, kx-k/2), ci]; deterministic.
 * The bias gradient is tm_colsum of dy. */
size_t tm_convkxk_bf16_wgrad_ws(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k);
int tm_convkxk_bf16_wgrad(int64_t B, int64_t H, int64_t W, int64_t Cin, int64_t Cout, int64_t k, const void* xb,
                          const void* dyb, float* dw, void* ws, size_t ws_bytes, int* err, void* stream);

/* ------------------------------------------------------------------------------------
 * N4  fused Adam (torch.optim.Adam defaults, src/train.py:431-435,555)
 * ---------------------------------------------------------------------------------- */
int tm_adam_step(int64_t n, float* p, const float* g, float* m, float* v, float lr, float beta1,
                 float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                 void* stream);
/* The same update for EVERY parameter tensor in ONE launch.  table: device array of
 * {float* p; const float* g; float* m; float* v; int64 n} (40 bytes each); chunk c of tm_adam_chunk() elements
 * starts at element chunk_off[c] of tensor chunk_tensor[c]. */
int tm_adam_chunk(void);
int tm_adam_multi(int64_t n_chunks, const void* table, const int32_t* chunk_tensor, const int32_t* chunk_off, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                  void* stream);
/* loss[0] = NaN if the device flag *err (set by a tensor-core kernel whose mbarrier wait timed out) is non-zero:
 * a failed tile can then not pass silently into the optimizer; the host still clears / reports the flag. */
int tm_poison_on_error(float* loss, const int32_t* err, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TM_B200_H */
