/*
 * rgbmp.h -- C ABI of the B200-native message-passing library (librgbmp.so).
 *
 * This is the drop-in boundary for the ONE hot path of PolarisRisingWar/rgb-experiment:
 * the neighbourhood aggregation that its model files delegate to torch_geometric /
 * torch_scatter / torch_sparse (SURVEY.md section 8b).  The reference has no FFI of its own
 * (pure Python); each entry point below cites the reference call site whose third-party
 * operator it replaces.  The Python host side (rgb-experiment_b200/) binds these with ctypes
 * and exposes them under the PyG names the reference imports.
 *
 * Conventions
 *   - every pointer is a caller-owned DEVICE pointer unless the name ends in _host;
 *     the library never allocates, frees or retains pointers past the call;
 *   - scratch memory comes from a caller-provided workspace sized by the *_workspace_bytes query;
 *   - `device` is the CUDA ordinal, `stream` a cudaStream_t passed as void*; nothing here
 *     synchronises the device (only the *_host entry points wait, on their own stream);
 *   - return value: 0 ok; >0 a cudaError_t; <0 an argument error (RGBMP_E*);
 *     rgbmp_last_error() returns a per-thread message; nothing is printed, nothing throws;
 *   - all functions are re-entrant (autograd calls backward from its own worker thread);
 *   - features are row-major [rows, F] with an explicit leading dimension in ELEMENTS;
 *     dtype is RGBMP_F32 or RGBMP_BF16 (bf16 storage, fp32 accumulation);
 *   - node ids / column indices are int32 (N < 2^31), row pointers int64, edge ids int32
 *     (nnz < 2^31 per GPU partition).
 */
#ifndef RGBMP_H_
#define RGBMP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define RGBMP_VERSION 101

/* argument errors */
#define RGBMP_EINVAL   (-1)  /* null pointer / bad enum / negative size */
#define RGBMP_EALIGN   (-2)  /* pointer or leading dimension not aligned for the vector path */
#define RGBMP_ERANGE   (-3)  /* N, F or nnz out of the supported range (32-bit overflow) */
#define RGBMP_EWORKSPACE (-4) /* workspace too small */

/* dtypes */
#define RGBMP_F32  0
#define RGBMP_BF16 1

/* self-loop edit applied before aggregation (SURVEY.md Appendix A1-A3) */
#define RGBMP_LOOP_NONE            0  /* LabelPropagation / C&S: gcn_norm(add_self_loops=False)           */
#define RGBMP_LOOP_ADD             1  /* add_self_loops                    (graphsage.py:56)              */
#define RGBMP_LOOP_ADD_REMAINING   2  /* add_remaining_self_loops          (dagnn.py:22-23; GCNConv/APPNP/SGConv/FAConv) */
#define RGBMP_LOOP_REMOVE_THEN_ADD 3  /* remove_self_loops+add_self_loops  (graphsage.py:55-56; GATConv/SuperGATConv)    */

/* node-normalisation vectors derived from the row pointer */
#define RGBMP_NORM_INV_SQRT 0  /* deg^-1/2, inf -> 0   (dagnn.py:27-30 gcn_norm)                        */
#define RGBMP_NORM_INV_MEAN 1  /* 1/max(deg,1)                                                          */
#define RGBMP_NORM_COUNT    2  /* max(deg,1)           (aggr='mean', graphsage.py:39 -> scatter mean divides by it) */

int         rgbmp_version(void);
const char* rgbmp_last_error(void);

/* ------------------------------------------------------------------------------------------
 * (a) integer graph-build kernels -- bit-exact against oracle.pyg_restated.{edit_loops,csr_build}
 * ------------------------------------------------------------------------------------------ */

/* Replaces remove_self_loops / add_self_loops / add_remaining_self_loops
 * (reference call sites graphsage.py:55-56, dagnn.py:22-23; inside GCNConv gcn.py:18-21 etc.).
 * In : src,dst int64 [E] (= edge_index[0], edge_index[1]).
 * Out: e_src,e_dst int32 [E+N] -- kept edges in original order then loops 0..N-1;
 *      nnz_dev int64 [1] (device) -- number of valid entries written. */
size_t rgbmp_edge_edit_workspace_bytes(int64_t E, int64_t N);
int rgbmp_edge_edit(const int64_t* src, const int64_t* dst, int64_t E, int64_t N, int loop_mode,
                    int32_t* e_src, int32_t* e_dst, int64_t* nnz_dev,
                    void* ws, size_t ws_bytes, int device, void* stream);

/* Stable counting/radix sort of an edge list by `key` -> CSR.  No reference counterpart (PyG
 * stays COO and scatters with atomics, SURVEY.md 8a a12); definition = oracle csr_build:
 * perm = argsort(key, stable); rowptr = [0, cumsum(bincount(key))]; col = other[perm]; eid = perm.
 * Forward CSR: key = e_dst, other = e_src.  Transpose CSR (backward): key = e_src, other = e_dst. */
size_t rgbmp_csr_build_workspace_bytes(int64_t nnz, int64_t N);
int rgbmp_csr_build(const int32_t* key, const int32_t* other, int64_t nnz, int64_t N,
                    int64_t* rowptr, int32_t* col, int32_t* eid,
                    void* ws, size_t ws_bytes, int device, void* stream);

/* deg = rowptr[i+1]-rowptr[i] -> node vector (dagnn.py:27-30 / scatter-mean count clamp). */
int rgbmp_degree_norm(const int64_t* rowptr, int64_t N, int mode, float* out, int device, void* stream);

/* Per-edge symmetric weights in CSR order: val[k] = dinv_col[col[k]] * 1.0f * dinv_row[i]
 * (dagnn.py:31: deg_inv_sqrt[row] * edge_weight * deg_inv_sqrt[col], same multiplication order). */
int rgbmp_gcn_edge_weight(const int64_t* rowptr, const int32_t* col, int64_t n_rows,
                          const float* dinv_row, const float* dinv_col, float* val,
                          int device, void* stream);

/* Permute a per-edge array between edge order and CSR order: out[k] = in[eid[k]]  (gather)
 * or out[eid[k]] = in[k] (scatter).  H contiguous floats per edge. */
int rgbmp_edge_permute(const float* in, const int32_t* eid, int64_t nnz, int H, int scatter,
                       float* out, int device, void* stream);

/* Long-row split: rows with more than `chunk` edges are processed as work items of
 * `long_chunk` edges each.  Step 1 counts (results in counts_dev[0]=n_long, [1]=n_items),
 * step 2 fills the lists once the caller has allocated them. */
int rgbmp_longrow_count(const int64_t* rowptr, int64_t n_rows, int32_t chunk, int32_t long_chunk,
                        int64_t* counts_dev, int device, void* stream);
size_t rgbmp_longrow_fill_workspace_bytes(int64_t n_rows);
int rgbmp_longrow_fill(const int64_t* rowptr, int64_t n_rows, int32_t chunk, int32_t long_chunk,
                       int64_t n_long, int64_t n_items,
                       int32_t* long_rows, int32_t* long_item_ptr, int32_t* item_long, int64_t* item_start,
                       void* ws, size_t ws_bytes, int device, void* stream);

/* The same lists with the long rows taken in the order of a row schedule (order[p] = row at position p, or NULL
 * = natural order): the work items of one locality group are then adjacent in the long-row launch. */
int rgbmp_longrow_fill_ordered(const int64_t* rowptr, int64_t n_rows, int32_t chunk, int32_t long_chunk,
                               const int32_t* order, int64_t n_long, int64_t n_items,
                               int32_t* long_rows, int32_t* long_item_ptr, int32_t* item_long, int64_t* item_start,
                               void* ws, size_t ws_bytes, int device, void* stream);

/* Row schedule for the short-row SpMM kernel: rows sorted by degree (longest first) inside windows
 * of `window` consecutive rows, so that the rows sharing a warp have equal length (no divergence)
 * while coarse locality of neighbouring rows is kept.  order int32 [n_rows]. */
size_t rgbmp_row_order_workspace_bytes(int64_t n_rows);
int rgbmp_row_order(const int64_t* rowptr, int64_t n_rows, int64_t window, int32_t* order,
                    void* ws, size_t ws_bytes, int device, void* stream);
/* ... sorted by (group[row], -degree) instead: group int32 [n_rows] with values in [0, n_groups), n_groups <= 32768
 * (the locality groups of rgbmp_cluster_lpa, ranked by the host).  group == NULL: as rgbmp_row_order. */
int rgbmp_row_order_grouped(const int64_t* rowptr, int64_t n_rows, int64_t window, const int32_t* group,
                            int32_t n_groups, int32_t* order, void* ws, size_t ws_bytes, int device, void* stream);

/* Sort an edge list by (row, col) and drop duplicate pairs = torch_sparse.coalesce(index, None, m, n)
 * (rd2pd.py:93); with symmetrize = 1 the list is first extended by every reversed edge =
 * torch_geometric.utils.to_undirected (itexperiments.py:235-238).  Two stable radix sorts (col, then
 * row) + a flagged compaction; bit-exact against oracle.pyg_restated.coalesce / to_undirected.
 * In : src,dst int64 [E].  Out: out_src,out_dst int64 [E or 2E capacity]; count_dev int64 [1] =
 * number of pairs written, or -1 when an id falls outside [0, N). */
size_t rgbmp_coalesce_workspace_bytes(int64_t E, int64_t N, int symmetrize);
int rgbmp_coalesce(const int64_t* src, const int64_t* dst, int64_t E, int64_t N, int symmetrize,
                   int64_t* out_src, int64_t* out_dst, int64_t* count_dev,
                   void* ws, size_t ws_bytes, int device, void* stream);

/* Column popularity and hot tagging (no reference counterpart; it steers the L2 so that the
 * feature rows gathered most often stay resident while once-touched rows stream through).
 *   rgbmp_col_freq: freq[c] = number of entries with col[k] == c   (int32 [n_cols], zeroed here)
 *   rgbmp_col_tag : out[k] = col[k] | (freq[col[k]] >= thresh ? 1u<<31 : 0) */
int rgbmp_col_freq(const int32_t* col, int64_t nnz, int64_t n_cols, int32_t* freq, int device, void* stream);
int rgbmp_col_tag(const int32_t* col, int64_t nnz, const int32_t* freq, int32_t thresh, int32_t* out,
                  int device, void* stream);

/* ------------------------------------------------------------------------------------------
 * (b) aggregation kernels
 * ------------------------------------------------------------------------------------------ */

typedef struct rgbmp_graph {
  int64_t        n_rows;       /* rows of this CSR (targets i for forward, sources j for transpose) */
  int64_t        n_cols;       /* number of addressable feature rows (max col + 1)                  */
  int64_t        nnz;
  const int64_t* rowptr;       /* [n_rows+1]                                                        */
  const int32_t* col;          /* [nnz]                                                             */
  int32_t        chunk;        /* rows with deg > chunk are "long" (0 = no split information)       */
  int32_t        long_chunk;
  int64_t        n_long;
  int64_t        n_items;
  const int32_t* long_rows;    /* [n_long]                                                          */
  const int32_t* long_item_ptr;/* [n_long+1]                                                        */
  const int32_t* item_long;    /* [n_items]                                                         */
  const int64_t* item_start;   /* [n_items]                                                         */
  const int32_t* row_order;    /* [n_rows] schedule of the short-row kernel, or NULL = natural order */
  int32_t        col_tagged;   /* 1: bit 31 of col[k] marks a frequently gathered ("hot") column, see
                                  rgbmp_col_tag                                                     */
} rgbmp_graph_t;
/* Every entry point that takes an rgbmp_graph_t checks it before it selects a device:
 *   RGBMP_EINVAL  NULL descriptor or rowptr, n_rows < 0, nnz < 0, or col NULL with nnz > 0;
 *   RGBMP_EINVAL  n_items > 0 without chunk > 0, long_chunk > 0 and all four long-row lists (never run unsplit);
 *   RGBMP_ERANGE  n_cols >= 2^31;
 *   RGBMP_EINVAL  col_tagged = 1, except in rgbmp_spmm, rgbmp_khop and rgbmp_appnp_host, whose kernels strip the tag;
 *   RGBMP_EINVAL  n_rows != n_cols where the graph must be square: rgbmp_khop, rgbmp_appnp_host, RGBMP_ATT_SD's g,
 *                 rgbmp_cluster_lpa and rgbmp_cluster_connectivity.
 * n_items <= 0 means no long rows: the long-row fields are then ignored. */


/* Fused epilogue applied to every output row i after the segmented sum s_i (all optional):
 *   s_i = acc_in ? acc_in[i,:] + s_i : s_i                          (column-blocked accumulation)
 *   v = row_scale ? (row_div ? s_i / row_scale[i] : row_scale[i]*s_i) : s_i
 *   if reset_when==1 and reset_mask[i]: v = reset_val[i,:]          (PTA label_propagation,
 *                                                                    itexperiments.py:715-717)
 *   v = a*v + (T ? b*T[i,:] : 0)                                     (APPNP appnp_stack.py:22,
 *                                                                    PTA pta.py:83, LP A15)
 *   if clamp: v = min(max(v,lo),hi)                                  (C&S post_step, A15)
 *   if reset_when==2 and reset_mask[i]: v = reset_val[i,:]           (C&S autoscale=False)
 *   Y[row_map ? row_map[i] : i,:] = v (if Y)                         (row_map: the graph's nodes are renamed)
 *   Y2[i,:] = out2_scale[i]*v (if Y2)                                (pre-scaled copy for the next hop)
 *   peer_out[q][peer_row0+i,:] = out2_scale ? out2_scale[i]*v : v    (fused all-gather, see below)
 */
#define RGBMP_MAX_PEERS 8
typedef struct rgbmp_epilogue {
  const float*   row_scale;
  int32_t        row_div;      /* 1: divide by row_scale[i] (scatter-mean's true divide) */
  const uint8_t* reset_mask;
  const float*   reset_val;
  int64_t        ld_reset;
  int32_t        reset_when;
  float          a;
  float          b;
  const void*    T;            /* same dtype as X */
  int64_t        ldt;
  int32_t        clamp;
  float          lo, hi;
  const float*   out2_scale;
  void*          Y2;
  int64_t        ldy2;
  const void*    acc_in;       /* optional [n_rows, ld_acc], dtype of X: s_i = acc_in[i,:] + s_i before anything
                                  else (partial sums of the previous column block; may alias Y)             */
  int64_t        ld_acc;
  int32_t        skip_empty;   /* 1: rows without edges in this launch are left untouched                   */
  /* fused all-gather (row-partitioned multi-GPU propagation, SURVEY.md 8e): the finished row i is also
   * stored to peer_out[q] + (peer_row0 + i) * ld_peer for q < n_peers -- peer-mapped buffers of the
   * other GPUs of the NVSwitch box (rgbmp_peer_open), written with plain stores over NVLink while the
   * kernel is still aggregating other rows.  Same dtype as Y. */
  void*          peer_out[RGBMP_MAX_PEERS];
  int32_t        n_peers;
  int64_t        peer_row0;
  int64_t        ld_peer;
  /* optional int32 [n_rows]: row i of the graph is row row_map[i] of Y.  A graph whose nodes are renamed in schedule
   * order stores its result under the original names this way; only the Y store is redirected (Y2, T, row_scale
   * and out2_scale stay indexed by i).  rgbmp_khop applies it to the last hop only. */
  const int32_t* row_map;
} rgbmp_epilogue_t;
/* rgbmp_spmm and rgbmp_khop check the epilogue before they select a device; NULL stands for {a = 1}, nothing else set:
 *   RGBMP_EINVAL  reset_when not 0, 1 or 2; reset_when != 0 without reset_mask, reset_val and ld_reset >= F;
 *   RGBMP_EINVAL  T with ldt < F; Y2 without out2_scale or with ldy2 < F; acc_in with ld_acc < F;
 *   RGBMP_EINVAL  n_peers outside [0, RGBMP_MAX_PEERS], a NULL peer_out[q] for q < n_peers, or peers with ld_peer < F;
 *   RGBMP_EALIGN  a peer_out[q] that is not 16-byte aligned;
 *   RGBMP_EINVAL  row_map together with peers, acc_in or reset rows;
 *   RGBMP_EINVAL  rgbmp_spmm only: no output (Y NULL, no Y2 and no peers).
 * K-hop only (rgbmp_khop owns every hop's stores, and every hop rewrites every row):
 *   RGBMP_EINVAL  Y2, acc_in, skip_empty or peers;
 *   RGBMP_EINVAL  row_map together with `hops`. */

/* CSR SpMM  Y[i,:] = epilogue( sum_k val[k] * X[col[k],:] ), k in rowptr[i]..rowptr[i+1].
 * Replaces MessagePassing.propagate = index_select -> message -> scatter
 * (graphsage.py:58, dagnn.py:46,57-59; inside GCNConv gcn.py:27,29, SAGEConv, GINConv, ...).
 * val may be NULL (unweighted sum / mean via row_scale).  The same call on the transpose CSR is
 * the backward.  `tune` = 0 picks the launch shape heuristically; otherwise (G | V<<8 | U<<16),
 * G in {1,2,4,8,16,32} lanes per row, V in 1..4 vectors per lane, U in {2,4,8} edges in flight
 * (+16: software-pipelined loop).  RGBMP_TUNE_NO_STREAM (may be or-ed into 0 too) turns off the
 * evict-first cache policy on the once-touched streams (column ids, weights, teleport, output). */
#define RGBMP_TUNE_NO_STREAM (1 << 24)
/* L2 eviction priority of the gathered feature rows, for experiments: or RGBMP_TUNE_POLICY with
 * (cold << 25) | (hot << 27), each 0 = normal, 1 = evict-first, 2 = evict-last.  Default: hot ids
 * (bit 31 set by rgbmp_col_tag) evict-last and the rest evict-first on a tagged graph, normal otherwise. */
#define RGBMP_TUNE_POLICY    (1 << 29)
/* rgbmp_khop: never take the one-cluster shared-memory path (below), always one SpMM launch per hop (A/B, tests) */
#define RGBMP_TUNE_NO_CTA    (1 << 30)
/* Fused all-gather (epilogue peer_out[]): rows of the short-row kernel reach the peers as 16-byte stores per lane
 * (default) or as ONE bulk asynchronous copy per (row, peer) from a shared-memory image of the row (cp.async.bulk, TMA).
 * rgbmp_set_push_bulk(0 | 1) selects process-wide (environment RGBMP_PUSH_BULK=1: bulk) and returns the previous
 * setting; other values only query.  Same bytes in the same places either way; measured equally fast. */
int rgbmp_set_push_bulk(int on);
size_t rgbmp_spmm_workspace_bytes(const rgbmp_graph_t* g, int F);
int rgbmp_spmm(const rgbmp_graph_t* g, const float* val, const void* X, int64_t ldx,
               void* Y, int64_t ldy, int F, int dtype, const rgbmp_epilogue_t* ep, int tune,
               void* ws, size_t ws_bytes, int device, void* stream);

/* Fused K-hop propagation (APPNP appnp_stack.py:22; SGConv sgc.py:9-10; Prop dagnn.py:45-47;
 * PTA.inference pta.py:82-83; label_propagation itexperiments.py:714-718; LabelPropagation /
 * CorrectAndSmooth itexperiments.py:525-526).  Hop k reads the previous iterate and writes the
 * next through ping/pong; the epilogue (teleport, clamp, reset, re-scaling for the folded
 * D^-1/2 normalisation) is applied inside the SpMM kernel of every hop.
 *   X0         first-hop input (already multiplied by out2_scale when the normalisation is folded)
 *   ping,pong  [n_rows, ldp] intermediates (only touched when K > 1)
 *   out        final iterate (unscaled)
 *   hops       optional [K][n_rows, ld_hops] -- every hop's unscaled output (DAGNN keeps them) */
int rgbmp_khop(const rgbmp_graph_t* g, const float* val, const void* X0, int64_t ldx0,
               void* ping, void* pong, int64_t ldp, void* out, int64_t ldo,
               void* hops, int64_t ld_hops, int64_t hop_stride,
               int F, int dtype, int K, const rgbmp_epilogue_t* ep, int tune,
               void* ws, size_t ws_bytes, int device, void* stream);
/* Small graphs take ONE launch of ONE thread-block cluster (16 CTAs, 8 where 16 cannot be placed) for all K hops
 * (csrc/khop_cta.cu; hops separated by the hardware cluster barrier, the iterate stays in ping / pong, i.e. in L2): fp32,
 * 16-byte aligned padded rows, K >= 2, F <= 16, at most 8 MB gathered per hop, n_rows <= 200,000, no row_map in the
 * epilogue.  Same operator, same per-row summation order.  rgbmp_set_khop_cta(0 | 1) turns the path off / on process-wide
 * (default on; environment RGBMP_KHOP_CTA=0 turns it off) and returns the previous setting; other values only query. */
int rgbmp_set_khop_cta(int on);
/* number of rgbmp_khop calls of this process that took the one-cluster path */
long long rgbmp_khop_cta_calls(void);

/* Device-wide knob (the one call that touches device state): size of the L2 set-aside that
 * evict-last ("persisting") lines may occupy, clamped to the device maximum; *granted = new limit. */
int rgbmp_l2_persist(int device, size_t bytes, size_t* granted);

/* Y[i,:] = scale[i] * X[i,:]  (the D^-1/2 pre-scaling of the folded normalisation), or with
 * divide=1  Y[i,:] = X[i,:] / scale[i]  (backward of scatter-mean: grad / count). */
int rgbmp_row_scale(const void* X, int64_t ldx, const float* scale, int divide, void* Y, int64_t ldy,
                    int64_t n_rows, int F, int dtype, int device, void* stream);

/* Locality groups for the row schedule (csrc/cluster.cu; no reference counterpart -- PyG's scatter has no schedule).
 * Seeded, leaves-first label propagation over the CSR g (square): the n_seeds (<= 4096) highest-degree nodes --
 * the first entries of deg_order, a global rgbmp_row_order -- keep their own label; in round t < iters an
 * unlabelled node takes the most frequent label among its labelled in-neighbours (ties: smallest label) once at
 * least taus[t] (host array) of its neighbours carry one, and keeps it.  label int32 [n_rows] out, every value in
 * [0, n_seeds).  Integer work, deterministic.  rgbmp_cluster_connectivity: W[a*n_groups + b] = number of CSR
 * entries of rows labelled a whose column is labelled b (uint32 [n_groups^2], zeroed inside), counted over every
 * row_stride-th row (1 = exact; the host only needs relative magnitudes to order the groups). */
size_t rgbmp_cluster_workspace_bytes(int64_t n_rows);
int rgbmp_cluster_lpa(const rgbmp_graph_t* g, const int32_t* deg_order, int32_t n_seeds, int iters,
                      const float* taus, int32_t* label, void* ws, size_t ws_bytes, int device, void* stream);
int rgbmp_cluster_connectivity(const rgbmp_graph_t* g, const int32_t* label, int32_t n_groups, int row_stride,
                               uint32_t* W, int device, void* stream);

/* One pass that prepares a folded K-hop call from an unpadded input: Z0[i, 0:ld] = X[s, 0:F] zero-padded to the
 * 16-byte aligned leading dimension ld (the teleport term) and U0[i,:] = scale[i] * Z0[i,:] (what hop 1 gathers),
 * with s = src_map ? src_map[i] : i (src_map renames the input into a renamed graph's node order).  Z0 may be NULL
 * when no teleport term is needed.  fp32. */
int rgbmp_stage_rows(const float* X, int64_t ldx, const int32_t* src_map, const float* scale, float* Z0, float* U0,
                     int64_t ld, int64_t n_rows, int F, int device, void* stream);

/* ------------------------------------------------------------------------------------------
 * (b2) peer memory for the row-partitioned multi-GPU path (one process per GPU, NVLink P2P)
 * ------------------------------------------------------------------------------------------ */
#define RGBMP_IPC_HANDLE_BYTES 64
/* Allocate `bytes` of device memory that other processes of the box can map (cudaMalloc +
 * cudaIpcGetMemHandle).  The one place where the library owns memory: IPC needs a whole allocation. */
int rgbmp_peer_alloc(size_t bytes, void** ptr, unsigned char handle[RGBMP_IPC_HANDLE_BYTES], int device);
int rgbmp_peer_free(void* ptr, int device);
/* Map a peer process's allocation into this process (cudaIpcOpenMemHandle, enables peer access). */
int rgbmp_peer_open(const unsigned char handle[RGBMP_IPC_HANDLE_BYTES], void** ptr, int device);
int rgbmp_peer_close(void* ptr, int device);

/* ------------------------------------------------------------------------------------------
 * (c) attention kernels
 * ------------------------------------------------------------------------------------------ */

/* Fused edge-score attention + weighted aggregate, one kernel family for the layers of the reference whose
 * per-edge weight is a function of the two endpoints (csrc/att.cu).  For target row i over its in-edges j -> i:
 *   RGBMP_ATT_GAT  GATConv (gat.py:18-21,28-30; SURVEY.md A10/A11):
 *                  e = leaky_relu(a_nbr[j] + a_own[i]);  alpha = exp(e - max)/(sum + 1e-16);  out[i] = sum alpha*mask*X[j]
 *   RGBMP_ATT_MX   SuperGATConv, MX attention (supergat.py:15-21; A12):
 *                  e = leaky_relu((a_nbr[j] + a_own[i]) * sigmoid(<X[i,h,:], X[j,h,:]>)), then as GAT
 *   RGBMP_ATT_FA   FAConv (fagcn.py:15,31; A13), H = 1:
 *                  out[i] = sum tanh(a_nbr[j] + a_own[i]) * dinv[j]*dinv[i] * mask * X[j]        (no softmax)
 *   RGBMP_ATT_SD   SuperGATConv, SD attention (A12):
 *                  e = leaky_relu(logit_scale * <X[i,h,:], X[j,h,:]>), then as GAT
 * X [n_cols, H*C] (ldx), a_nbr [n_cols,H] (a_src / att_l side), a_own [n_rows,H] (a_dst / att_r side).
 * Shapes: H == 1 with any C <= 128 (padding columns of X up to roundup(C,4) must be ZERO), or C a power of two in
 * 8..128 with any H (heads are tiled over the grid) -- rgbmp_att_supported() says which; the host layer pads heads.
 * What each score reads:
 *   GAT, MX  a_nbr, a_own (the backward writes da_nbr, da_own);
 *   FA       a_nbr, a_own and dinv [n]; H == 1;
 *   SD       no a_*, dinv or da_* (pass NULL); g square (X holds both endpoints), gT its transpose, logit_scale
 *            finite -- 1/sqrt(C) of the UNPADDED head width when the caller pads heads to a supported C.
 *            logit_scale is ignored by the other scores.
 * Attention dropout: at most one of `drop` and `d` may be non-NULL.  drop is the explicit keep-mask in forward-CSR
 * order [nnz,H], already divided by (1-p); the backward also needs tpos[k'] = forward-CSR position of transpose entry
 * k'.  d generates the mask inside the kernels (rgbmp_dropout_t below): the forward reads d->eid, the backward
 * d->eid_t (MX and SD also d->eid) and streams eid_t in its transpose pass -- no tpos, no random gather.
 * Softmax scores save rowmax,rowsum [n_rows,H].  TRAINING mode = out2 != NULL: GAT and FA accumulate a second
 * aggregate next to out (GAT: P_i = sum alpha*leaky'*mask*X[j] into out2 and q_i = sum alpha*leaky' into rowq;
 * FA: Q_i = sum (1-tanh^2)*dinv*dinv*mask*X[j]) from which the backward gets the gradient of the per-TARGET score
 * term without atomics (da_own[i] = <dout_i, P_i> - S_i q_i); MX and SD need none (out2 must be NULL).
 * The backward: g = the forward CSR, gT = its transpose (rows = sources j).  It recomputes the edge weights from the
 * saved per-target statistics; `out`/`out2`/`rowq` are the training-mode forward's results.  It writes dX [n, H*C]
 * (lddx) and, but for SD, da_nbr [n_cols,H], da_own [n_rows,H].  MX and SD run one pass per orientation (the logit
 * <x_i,x_j> feeds both endpoints) and need the scratch dXf [n_rows, lddxf]; GAT and FA run one transpose pass.
 * An unsupported score / H / C is RGBMP_ERANGE; a NULL pointer a score reads, both dropout forms or a graph SD
 * cannot take is RGBMP_EINVAL.  Nothing edge-sized is written; the result is deterministic. */
#define RGBMP_ATT_GAT 0
#define RGBMP_ATT_MX  1
#define RGBMP_ATT_FA  2
#define RGBMP_ATT_SD  3

/* Attention dropout generated inside the kernels (csrc/philox.cuh): no mask tensor exists.  For edge e (its id in
 * the edited edge list) and head h (FA: h = 0):
 *   u = Philox4x32-10(counter = (e, h, 0, 0), key = (seed & 0xffffffff, seed >> 32)).word0
 *   multiplier = (u < thresh) ? 0 : scale,   thresh = floor(p * 2^32),  scale = float32(1 / (1 - p))
 * p == 1 is passed as thresh = 0xffffffff, scale = 0 (every multiplier 0).  The multiplier is applied where the
 * explicit `drop` mask is, with the same operands: a fused call is bit-identical to the explicit-mask call fed the
 * mask rgbmp_dropout_mask writes for the same seed.  `seed` is read on the device (no host synchronisation). */
typedef struct rgbmp_dropout {
  const int64_t* seed;    /* device pointer to one int64 */
  const int32_t* eid;     /* [nnz] edge id of every forward-CSR entry */
  const int32_t* eid_t;   /* [nnz] edge id of every transpose-CSR entry; backward only */
  uint32_t thresh;
  float    scale;
} rgbmp_dropout_t;

int rgbmp_att_supported(int score, int H, int C);
size_t rgbmp_att_forward_workspace_bytes(const rgbmp_graph_t* g, int H, int C);
int rgbmp_att_forward(const rgbmp_graph_t* g, int score, const float* X, int64_t ldx,
                      const float* a_nbr, const float* a_own, const float* dinv, int H, int C,
                      float slope, float logit_scale, const float* drop, const rgbmp_dropout_t* d,
                      float* out, int64_t ldo, float* rowmax, float* rowsum, float* out2, int64_t ldo2, float* rowq,
                      void* ws, size_t ws_bytes, int device, void* stream);
size_t rgbmp_att_backward_workspace_bytes(const rgbmp_graph_t* g, const rgbmp_graph_t* gT, int H, int C);
int rgbmp_att_backward(const rgbmp_graph_t* g, const rgbmp_graph_t* gT, int score, const float* X, int64_t ldx,
                       const float* a_nbr, const float* a_own, const float* dinv, int H, int C,
                       float slope, float logit_scale, const float* drop, const int32_t* tpos, const rgbmp_dropout_t* d,
                       const float* rowmax, const float* rowsum, const float* rowq,
                       const float* out, int64_t ldo, const float* out2, int64_t ldo2, const float* dout, int64_t ldd,
                       float* dX, int64_t lddx, float* dXf, int64_t lddxf, float* da_nbr, float* da_own,
                       void* ws, size_t ws_bytes, int device, void* stream);
/* out[e*H + h] = the multiplier of edge e, head h, in EDGE order [nnz, H] (the mask of the unfused paths). */
int rgbmp_dropout_mask(const rgbmp_dropout_t* d, int64_t nnz, int H, float* out, int device, void* stream);

/* SuperGAT's self-supervised attention loss (SuperGATConv.get_attention_loss, supergat.py:26,29; csrc/supergat_loss.cu).
 * Seeded sampling, keyed like attention dropout but on counter word 2 = 1 (positives) or 2 (negatives):
 *   positive edge e (its id in the edited edge list) is kept iff keep_thresh == 0 or
 *     Philox4x32-10(counter = (e, 0, 1, 0), key = (seed lo, seed hi)).word0 >= keep_thresh,
 *     keep_thresh = floor((1 - edge_sample_ratio) * 2^32) (64-bit: 2^32 drops every edge);
 *   negative candidate k of round r (r = 0, 1, 2): (w0..w3) = Philox4x32-10((k, r, 2, 0), key),
 *     (row, col) = (umulhi64(w1:w0, N), umulhi64(w3:w2, N))  (bias <= N / 2^64 per id).
 * `seed` is read on the device. */
typedef struct rgbmp_sgat_sample {
  const int64_t* seed;     /* device pointer to one int64 */
  const int32_t* eid;      /* [nnz] edge id of every forward-CSR entry (needed when keep_thresh != 0) */
  const int32_t* eid_t;    /* [nnz] edge id of every transpose-CSR entry; backward only */
  uint64_t keep_thresh;
} rgbmp_sgat_sample_t;

/* Negative sampling (torch_geometric.utils.negative_sampling as SuperGATConv calls it): candidates of round r are
 * rejected iff (row, col) is a pair of U, given as a CSR over rows with sorted columns (u_rowptr [N+1], u_col);
 * survivors are compacted stably in (round, k) order into neg_src / neg_dst (capacity num_neg) and cut to num_neg;
 * rounds after the one that reaches num_neg do nothing (decided on the device).  *count_dev = pairs written.
 * num_neg and sample_size come from the host (the oracle's float formulas); sample_size >= 2^31 is RGBMP_ERANGE. */
size_t rgbmp_sgat_negative_sampling_workspace_bytes(int64_t sample_size);
int rgbmp_sgat_negative_sampling(const int64_t* u_rowptr, const int32_t* u_col, int64_t N, const rgbmp_sgat_sample_t* s,
                                 int64_t num_neg, int64_t sample_size, int32_t* neg_src, int32_t* neg_dst,
                                 int64_t* count_dev, void* ws, size_t ws_bytes, int device, void* stream);
/* out[e] = 1 if positive edge e is kept, else 0, in EDGE order (uint8 [nnz]; unfused paths, tests). */
int rgbmp_sgat_keep_mask(const rgbmp_sgat_sample_t* s, int64_t nnz, uint8_t* out, int device, void* stream);

/* Pair-logit BCE over the kept positives (forward CSR g, rows = targets i, through s->eid) and the negatives
 * (CSR gneg over the same N rows; the columns are the other endpoints):
 *   s_ij = scale * <X[i,:], X[j,:]>,  loss = (sum_pos softplus(-s) + sum_neg softplus(s)) / P,  P = pairs
 * F <= 512, fp32, rows 16-byte aligned (ld % 4 == 0, zero padding up to roundup(F, 4)).  Per-row fp32 partials,
 * then a fixed-order fp64 reduction: *loss (float, device) and *npairs (int64, device) -- deterministic. */
size_t rgbmp_sgat_loss_workspace_bytes(int64_t n_rows);
int rgbmp_sgat_loss_forward(const rgbmp_graph_t* g, const rgbmp_graph_t* gneg, const rgbmp_sgat_sample_t* s,
                            const float* X, int64_t ldx, int F, float scale, float* loss, int64_t* npairs,
                            void* ws, size_t ws_bytes, int device, void* stream);
/* dX = d loss / dX * (*dloss): one pass over target rows (g, gneg) writes every row of dX, one over source rows
 * (gT with s->eid_t, gnegT) adds into its own rows.  No atomics: bit-reproducible. */
int rgbmp_sgat_loss_backward(const rgbmp_graph_t* g, const rgbmp_graph_t* gT, const rgbmp_graph_t* gneg,
                             const rgbmp_graph_t* gnegT, const rgbmp_sgat_sample_t* s, const float* X, int64_t ldx, int F,
                             float scale, const int64_t* npairs, const float* dloss, float* dX, int64_t lddx,
                             int device, void* stream);

/* S[i,h] = sum_c A[i,h*C+c]*B[i,h*C+c] */
int rgbmp_rowdot(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t n_rows,
                 int H, int C, float* S, int device, void* stream);

/* Generic edge-score kernels in CSR order (SuperGATConv supergat.py:15-21, FAConv fagcn.py:15):
 *  SDDMM      out[k,h] = <A[row_i,h,:], B[col[k],h,:]>
 *  u_add_v    out[k,h] = u[col[k],h] + v[row_i,h]
 *  seg_softmax per-row softmax over k (max-subtracted, /(sum+1e-16)), in place capable.
 *  seg_sum     out[i,h] = sum_k in[k,h]        (deterministic segmented reduce)               */
int rgbmp_sddmm(const rgbmp_graph_t* g, const float* A, int64_t lda, const float* B, int64_t ldb,
                int H, int C, float* out, int device, void* stream);
int rgbmp_u_add_v(const rgbmp_graph_t* g, const float* u, const float* v, int H, float* out,
                  int device, void* stream);
int rgbmp_seg_softmax(const rgbmp_graph_t* g, const float* in, int H, float* out,
                      int device, void* stream);
int rgbmp_seg_softmax_backward(const rgbmp_graph_t* g, const float* alpha, const float* dalpha,
                               int H, float* dlogit, int device, void* stream);
int rgbmp_seg_sum(const rgbmp_graph_t* g, const float* in, int H, float* out,
                  int device, void* stream);
/* weighted multi-head SpMM: out[i,h,:] = sum_k w[k,h] * X[col[k],h,:]  (w in CSR order) */
int rgbmp_spmm_heads(const rgbmp_graph_t* g, const float* w, const float* X, int64_t ldx,
                     int H, int C, float* out, int64_t ldo, int device, void* stream);

/* ------------------------------------------------------------------------------------------
 * (c2) measurement aid: random ROW-GATHER peak of the device (csrc/microbench.cu).  n_groups groups of
 * row_bytes/16 lanes each read `gathers_per_group` random rows of `table` [n_rows, row_bytes] with 16-byte loads
 * (8 rows in flight per lane, ids from a counter hash) and write one 16-byte checksum per group to `out`.
 * Bytes gathered = n_groups * gathers_per_group * row_bytes; timed by the caller.  The roofline denominator of
 * aggregation kernels whose feature matrix is L2-resident (bench.py --workload arxiv_sage / reddit_gat).
 * ------------------------------------------------------------------------------------------ */
int rgbmp_microbench_gather(const void* table, int64_t n_rows, int row_bytes, int64_t gathers_per_group,
                            uint32_t seed, void* out, int64_t n_groups, int device, void* stream);

/* ------------------------------------------------------------------------------------------
 * (d) host-buffer entry point (end-to-end form of the hot path: H2D -> K hops -> D2H)
 * ------------------------------------------------------------------------------------------ */

/* APPNP-style K-hop propagation with HOST input/output (pinned or pageable):
 *   z = z0; K x { z = (1-alpha) * D^-1/2 (A+I) D^-1/2 z + alpha * z0 }
 * The graph (g, dinv) is device-resident, like the reference keeps edge_index on the device
 * across epochs (itexperiments.py:258).  dev_* are caller-provided device scratch buffers
 * [n_rows, ld] each.  Copies and kernels are enqueued on `stream`, which is synchronised
 * before returning. */
int rgbmp_appnp_host(const rgbmp_graph_t* g, const float* dinv,
                     const float* z0_host, float* out_host, int F, int K, float alpha,
                     float* dev_z0, float* dev_ping, float* dev_pong, float* dev_out, int64_t ld,
                     void* ws, size_t ws_bytes, int device, void* stream);
/* The same on a graph whose nodes are renamed: row i of g (and dinv[i]) is node row_map[i] of z0_host and out_host
 * (int32 [n_rows], device).  The staging pass reads the input in the renamed order and the last hop stores the result
 * under the original names, so the hops read and write their rows in order.  row_map = NULL: rgbmp_appnp_host. */
int rgbmp_appnp_host_mapped(const rgbmp_graph_t* g, const int32_t* row_map, const float* dinv,
                            const float* z0_host, float* out_host, int F, int K, float alpha,
                            float* dev_z0, float* dev_ping, float* dev_pong, float* dev_out, int64_t ld,
                            void* ws, size_t ws_bytes, int device, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* RGBMP_H_ */
