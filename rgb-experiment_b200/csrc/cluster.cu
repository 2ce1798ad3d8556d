// Locality groups for the row schedule (sm_100a): seeded, leaves-first label propagation over the CSR, and the
// group-to-group connectivity matrix the host chains into a linear order.
//
// Why: the aggregation kernels gather feature rows of a matrix several times the size of L2.  With rows scheduled by
// degree alone the rows in flight are unrelated and every low-degree source misses L2 on each of its ~16 gathers per
// hop (L2 hit rate 42 %, 15.6 GB of DRAM traffic per hop against 1.95 GB compulsory on the products-shaped graph).
// Real graphs -- and the synthetic ones here, whose edges keep the class of an endpoint with probability 0.8 -- have
// communities; if the rows in flight belong to one community most of their sources do too and that slice of the
// feature matrix stays L2-resident (hit rate 68 %, 6.5 GB; profiles/r02_spmm_schedule.txt).  Only the ORDER in which
// rows are processed changes: no node is relabelled, no result bit changes.
//
// Algorithm (integer work, deterministic, built once per graph like the CSR itself; nothing here knows how the graph
// was generated -- it sees rowptr / col only):
//   1. seeds = the S highest-degree nodes, label = rank;
//   2. round t: an UNLABELLED node takes the most frequent label among its labelled in-neighbours (ties: smallest)
//      once at least tau_t of its neighbours carry one, and keeps it.  tau decreasing (0.3, 0.15, 0.05, 0, ...):
//      leaves settle first, hubs wait for their own leaves instead of copying a bigger hub across a hub-hub edge;
//   3. W[a][b] = number of edges from group b into group a; the host orders the groups so that strongly connected
//      ones are adjacent (graph.py), rows are then sorted by (group rank, -degree) by rgbmp_row_order_grouped.
#include "csr_work.cuh"

namespace rgbmp {

constexpr int CL_THREADS = 256;
constexpr int CL_WARPS = CL_THREADS / 32;

__global__ void __launch_bounds__(256)
lpa_seed_kernel(const int32_t* __restrict__ deg_order, int64_t n, int32_t S, int32_t* __restrict__ label) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  // deg_order lists the rows by degree, longest first: position < S is a seed
  label[deg_order[i]] = i < S ? (int32_t)i : -1;
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long w = __shfl_xor_sync(0xffffffffu, v, o);
    v = w > v ? w : v;
  }
  return v;
}

// one warp per row; per-warp histogram of S counters in shared memory (touched entries are re-zeroed per row)
// MODE 0: vote (label_out = plurality of the labelled in-neighbours when enough of them are labelled)
// MODE 1: connectivity (W[label[row]][l] += number of in-neighbours labelled l)
template <int MODE>
__global__ void __launch_bounds__(CL_THREADS)
lpa_rows_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t n_rows, int32_t S,
                const int32_t* __restrict__ label_in, float tau, int32_t* __restrict__ label_out,
                unsigned int* __restrict__ W, int32_t* __restrict__ changed, int row_stride) {
  extern __shared__ unsigned int hist_all[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned int* hist = hist_all + (size_t)warp * S;
  for (int t = lane; t < S; t += 32) hist[t] = 0;
  __syncwarp();
  const int64_t nwarps = (int64_t)gridDim.x * CL_WARPS;
  int nchanged = 0;
  for (int64_t slot = (int64_t)blockIdx.x * CL_WARPS + warp; slot * row_stride < n_rows; slot += nwarps) {
    const int64_t row = slot * row_stride;                  // connectivity may sample every row_stride-th row
    const int32_t own = label_in[row];
    if (MODE == 0 && own >= 0) {
      if (lane == 0) label_out[row] = own;
      continue;
    }
    if (MODE == 1 && own < 0) continue;
    const int64_t k0 = rowptr[row], k1 = rowptr[row + 1];
    int nlab = 0;
    for (int64_t k = k0 + lane; k < k1; k += 32) {
      const int32_t l = __ldg(label_in + (col[k] & 0x7fffffff));
      if (l >= 0) {
        atomicAdd(hist + l, 1u);
        ++nlab;
      }
    }
    __syncwarp();
    if (MODE == 0) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) nlab += __shfl_xor_sync(0xffffffffu, nlab, o);
      unsigned long long best = 0;                 // (count << 32) | (S - 1 - label): max count, then smallest label
      for (int64_t k = k0 + lane; k < k1; k += 32) {
        const int32_t l = __ldg(label_in + (col[k] & 0x7fffffff));
        if (l >= 0) {
          const unsigned long long c = ((unsigned long long)hist[l] << 32) | (unsigned)(S - 1 - l);
          best = c > best ? c : best;
        }
      }
      best = warp_max_u64(best);
      __syncwarp();
      for (int64_t k = k0 + lane; k < k1; k += 32) {
        const int32_t l = __ldg(label_in + (col[k] & 0x7fffffff));
        if (l >= 0) hist[l] = 0;
      }
      __syncwarp();
      const bool adopt = nlab > 0 && (double)nlab >= (double)tau * (double)(k1 - k0);
      if (lane == 0) {
        label_out[row] = adopt ? (int32_t)(S - 1 - (int32_t)(best & 0xffffffffu)) : -1;
        nchanged += adopt ? 1 : 0;
      }
    } else {
      unsigned int* Wrow = W + (size_t)own * S;
      for (int64_t k = k0 + lane; k < k1; k += 32) {
        const int32_t l = __ldg(label_in + (col[k] & 0x7fffffff));
        if (l >= 0) {
          const unsigned int c = atomicExch(hist + l, 0u);     // the first lane to arrive flushes the whole count
          if (c) atomicAdd(Wrow + l, c);
        }
      }
      __syncwarp();
    }
  }
  if (MODE == 0 && lane == 0 && nchanged) atomicAdd(changed, nchanged);
}

__global__ void __launch_bounds__(256)
lpa_fill_unlabelled_kernel(int32_t* __restrict__ label, int64_t n, int32_t S) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && label[i] < 0) label[i] = (int32_t)(i % S);       // unreachable from every seed (isolated nodes)
}

}  // namespace rgbmp

using namespace rgbmp;

extern "C" {

size_t rgbmp_cluster_workspace_bytes(int64_t n_rows) {
  return align_up((size_t)(n_rows > 0 ? n_rows : 1) * sizeof(int32_t), 256) + 1024;
}

int rgbmp_cluster_lpa(const rgbmp_graph_t* g, const int32_t* deg_order, int32_t n_seeds, int iters, const float* taus,
                      int32_t* label, void* ws, size_t ws_bytes, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_cluster_lpa", GRAPH_SQUARE);
  if (rc) return rc;
  if (g->n_rows <= 0 || !deg_order || !label || !taus || iters < 1 || !ws)
    return fail(RGBMP_EINVAL, "rgbmp_cluster_lpa: bad argument");
  if (n_seeds < 1 || n_seeds > 4096 || n_seeds > g->n_rows) return fail(RGBMP_ERANGE, "rgbmp_cluster_lpa: n_seeds must be in 1..min(4096, n_rows)");
  if (ws_bytes < rgbmp_cluster_workspace_bytes(g->n_rows)) return fail(RGBMP_EWORKSPACE, "rgbmp_cluster_lpa: workspace");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_cluster_lpa: bad device");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = g->n_rows;
  Carver cv(ws, ws_bytes);
  int32_t* tmp = cv.take<int32_t>((size_t)n);
  int32_t* changed = cv.take<int32_t>(1);
  if (!cv.ok()) return fail(RGBMP_EWORKSPACE, "rgbmp_cluster_lpa: workspace carve");
  const size_t smem = (size_t)CL_WARPS * n_seeds * sizeof(unsigned int);
  auto kern = lpa_rows_kernel<0>;
  RGBMP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // ping-pong so that the LAST round writes `label`
  int32_t* bufs[2] = {label, tmp};
  int cur = iters & 1;
  lpa_seed_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(deg_order, n, n_seeds, bufs[cur]);
  RGBMP_LAUNCH_CHECK("lpa_seed_kernel");
  RGBMP_CUDA(cudaMemsetAsync(changed, 0, sizeof(int32_t), st));
  const unsigned grid = (unsigned)(kSMs * (smem > 64 * 1024 ? 1 : 3));
  for (int t = 0; t < iters; ++t) {
    kern<<<grid, CL_THREADS, smem, st>>>(g->rowptr, g->col, n, n_seeds, bufs[cur], taus[t], bufs[cur ^ 1], nullptr, changed, 1);
    RGBMP_LAUNCH_CHECK("lpa_rows_kernel");
    cur ^= 1;
  }
  lpa_fill_unlabelled_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, st>>>(label, n, n_seeds);
  RGBMP_LAUNCH_CHECK("lpa_fill_unlabelled_kernel");
  return 0;
}

int rgbmp_cluster_connectivity(const rgbmp_graph_t* g, const int32_t* label, int32_t n_groups, int row_stride, uint32_t* W,
                               int device, void* stream) {
  int rc = check_graph(g, "rgbmp_cluster_connectivity", GRAPH_SQUARE);
  if (rc) return rc;
  if (g->n_rows <= 0 || !label || !W || row_stride < 1) return fail(RGBMP_EINVAL, "rgbmp_cluster_connectivity: bad argument");
  if (n_groups < 1 || n_groups > 4096) return fail(RGBMP_ERANGE, "rgbmp_cluster_connectivity: n_groups must be in 1..4096");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_cluster_connectivity: bad device");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)CL_WARPS * n_groups * sizeof(unsigned int);
  auto kern = lpa_rows_kernel<1>;
  RGBMP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  RGBMP_CUDA(cudaMemsetAsync(W, 0, (size_t)n_groups * n_groups * sizeof(uint32_t), st));
  const unsigned grid = (unsigned)(kSMs * (smem > 64 * 1024 ? 1 : 3));
  kern<<<grid, CL_THREADS, smem, st>>>(g->rowptr, g->col, g->n_rows, n_groups, label, 0.f, nullptr, W, nullptr, row_stride);
  RGBMP_LAUNCH_CHECK("lpa_rows_kernel");
  return 0;
}

}  // extern "C"
