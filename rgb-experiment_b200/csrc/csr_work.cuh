// The CSR descriptor rgbmp_graph_t as the library reads it: the rules every entry point checks it against, and the
// row-split schedule shared by the SpMM and the attention kernels.  Rows of at most `chunk` edges go to one group of
// G lanes each, in `row_order`; longer rows are cut into work items of at most `long_chunk` edges, one CTA per item,
// whose partial results a combine kernel merges in item order -- deterministic, no atomics.
#pragma once
#include "common.cuh"

namespace rgbmp {

// the graph half of a row-split pass's kernel parameters (first member of SpmmParams and AttParams)
struct CsrWork {
  const int64_t* rowptr;
  const int32_t* col;
  const int32_t* row_order;  // nullable: schedule of the short-row phase
  int64_t n_rows;
  int32_t chunk, long_chunk; // chunk = 0: the graph has no long rows
  const int32_t* long_rows;
  const int32_t* long_item_ptr;
  const int32_t* item_long;
  const int64_t* item_start;
  int64_t n_long, n_items;
};

enum : unsigned {
  GRAPH_TAGS_OK = 1,  // the caller's kernels strip the hot tag (bit 31 of a column id) before they gather
  GRAPH_SQUARE = 2,   // n_rows == n_cols
};

// The descriptor rules of include/rgbmp.h; runs before any device is selected.
inline int check_graph(const rgbmp_graph_t* g, const char* fn, unsigned rules = 0) {
  if (!g || !g->rowptr || g->n_rows < 0 || g->nnz < 0 || (g->nnz > 0 && !g->col))
    return fail(RGBMP_EINVAL, "%s: bad graph descriptor", fn);
  if (g->n_items > 0 && (!g->long_rows || !g->long_item_ptr || !g->item_long || !g->item_start || g->chunk <= 0 ||
                         g->long_chunk <= 0))
    return fail(RGBMP_EINVAL, "%s: incomplete long-row lists", fn);
  if (g->n_cols >= (1ll << 31)) return fail(RGBMP_ERANGE, "%s: n_cols exceeds int32", fn);
  if (g->col_tagged && !(rules & GRAPH_TAGS_OK))
    return fail(RGBMP_EINVAL, "%s: hot-tagged column ids are not accepted here", fn);
  if ((rules & GRAPH_SQUARE) && g->n_rows != g->n_cols) return fail(RGBMP_EINVAL, "%s: needs a square graph", fn);
  return 0;
}

// g passed check_graph
inline CsrWork csr_work(const rgbmp_graph_t* g) {
  const bool split = g->n_items > 0;
  return CsrWork{g->rowptr, g->col, g->row_order, g->n_rows, split ? g->chunk : 0, g->long_chunk, g->long_rows,
                 g->long_item_ptr, g->item_long, g->item_start, split ? g->n_long : 0, split ? g->n_items : 0};
}

// Short-row phase: the row of this thread's group of G lanes and its edges [k0, k1).  false (and k0 == k1) when the
// group has no row or its row is long: the group still runs the warp-uniform edge loop, with no edges.
template <int G, int THREADS>
__device__ __forceinline__ bool short_row(const CsrWork& w, int64_t& row, int64_t& k0, int64_t& k1) {
  const int64_t gid = (int64_t)blockIdx.x * (THREADS / G) + threadIdx.x / G;
  row = -1;
  k0 = k1 = 0;
  if (gid < w.n_rows) {
    row = w.row_order ? (int64_t)__ldg(w.row_order + gid) : gid;
    k0 = __ldg(w.rowptr + row);
    k1 = __ldg(w.rowptr + row + 1);
    if (w.chunk > 0 && k1 - k0 > w.chunk) row = -1;  // long row: the work items own it
  }
  if (row < 0) k1 = k0;
  return row >= 0;
}

// Work-item phase: item blockIdx.x covers at most long_chunk edges of one long row; the CTA's THREADS / G groups take
// contiguous sub-ranges of it, this thread's group [k0, k1).
template <int G, int THREADS>
__device__ __forceinline__ void long_item(const CsrWork& w, int64_t& row, int64_t& k0, int64_t& k1) {
  const int Q = THREADS / G;
  const int q = threadIdx.x / G;
  const int64_t item = blockIdx.x;
  row = w.long_rows[w.item_long[item]];
  const int64_t rs = w.item_start[item];
  const int64_t rend = __ldg(w.rowptr + row + 1);
  const int64_t re = (rs + w.long_chunk < rend) ? rs + w.long_chunk : rend;
  const int64_t per = (re - rs + Q - 1) / Q;
  k0 = rs + (int64_t)q * per;
  k1 = k0 + per;
  if (k0 > re) k0 = re;
  if (k1 > re) k1 = re;
}

// Launches the three phases of a row-split pass: rows(grid) over ceil(n_rows / groups_per_cta) x tiles; when the graph
// has long rows, items(grid) over n_items x tiles, then combine(blocks) with 256 threads per (long row, column) of a
// `width`-column output.
template <class Rows, class Items, class Combine>
int launch_phases(const CsrWork& w, int groups_per_cta, unsigned tiles, int64_t width, const char* what, Rows&& rows,
                  Items&& items, Combine&& combine) {
  if (w.n_rows > 0) {
    rows(dim3((unsigned)ceil_div(w.n_rows, groups_per_cta), tiles));
    RGBMP_LAUNCH_CHECK(what);
  }
  if (w.n_items > 0) {
    items(dim3((unsigned)w.n_items, tiles));
    RGBMP_LAUNCH_CHECK(what);
    combine((unsigned)ceil_div(w.n_long * width, 256));
    RGBMP_LAUNCH_CHECK(what);
  }
  return 0;
}

// Column ids of a batch reach the lanes of a group through shared memory: one STS per lane, then a broadcast LDS of
// the N ids of a step instead of one SHFL per edge -- a SHFL occupies the LSU data pipe for 4 wavefronts, the same
// pipe that serves the gathers (profiles/r02_spmm_l1_wavefronts.txt).
template <int N>
__device__ __forceinline__ void lds_ids(const int32_t* p, uint32_t (&c)[N]) {
  if constexpr (N == 8) {
    const int4 v = *reinterpret_cast<const int4*>(p), w = *reinterpret_cast<const int4*>(p + 4);
    c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w; c[4] = w.x; c[5] = w.y; c[6] = w.z; c[7] = w.w;
  } else if constexpr (N == 4) {
    const int4 v = *reinterpret_cast<const int4*>(p);
    c[0] = v.x; c[1] = v.y; c[2] = v.z; c[3] = v.w;
  } else if constexpr (N == 2) {
    const int2 v = *reinterpret_cast<const int2*>(p);
    c[0] = v.x; c[1] = v.y;
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) c[i] = p[i];
  }
}

}  // namespace rgbmp
