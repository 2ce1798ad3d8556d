// SuperGAT's self-supervised attention loss on the device (SuperGATConv.get_attention_loss, supergat.py:26,29):
// the seeded positive edge sampling, the negative sampler and a pair-logit BCE whose forward and backward gather
// feature rows per pair without materialising anything pair- or edge-sized.
//
//   pairs   the kept positive edges j -> i of the forward CSR (keep rule through eid, csrc/philox.cuh), then the
//           negatives (a, b), held as a CSR keyed by b (columns a) and its transpose
//   s       = scale * <x'_i, x'_j>   (MX: scale = 1/H, SD: 1/(H sqrt(C)); the mean over heads of per-head dots)
//   loss    = (sum_pos softplus(-s) + sum_neg softplus(s)) / P,  P = P_pos + P_neg
//   grad    c = dloss * (sigmoid(s) - y) * scale / P;  dx'_i += c x'_j,  dx'_j += c x'_i
//
// One lane group per row (the SpMM's G lanes x V float4 per lane), rows in the CSR's schedule.  The forward writes
// per-row fp32 partials which a fixed-shape two-stage fp64 reduction turns into the scalar; the backward is one pass
// over target rows (forward CSR + negatives' CSR) that writes dx' and one over source rows (transpose CSRs) that adds
// into its own rows.  No atomics anywhere: every result is bit-reproducible.
#include "csr_work.cuh"
#include "philox.cuh"

namespace rgbmp {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxVec = 4;             // float4 per lane: F <= 32 * 4 * 4 = 512
constexpr int kReduceRows = 4096;      // rows per block of the first reduction stage
constexpr int kScanThreads = 1024;

// ---------------------------------------------------------------------------------------------------------------
// negative sampler
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool u_contains(const int64_t* __restrict__ rp, const int32_t* __restrict__ col,
                                           uint32_t row, uint32_t c) {
  int64_t lo = __ldg(rp + row);
  const int64_t end = __ldg(rp + row + 1);
  int64_t hi = end;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((uint32_t)__ldg(col + mid) < c) lo = mid + 1;
    else hi = mid;
  }
  return lo < end && (uint32_t)__ldg(col + lo) == c;
}

// survivors of round r: flag[k] and per-block counts.  A round after the one that filled num_neg does nothing.
__global__ void __launch_bounds__(kThreads) sgat_neg_flags(const int64_t* __restrict__ urp, const int32_t* __restrict__ ucol,
                                                           uint64_t n, const int64_t* __restrict__ seed, uint32_t round,
                                                           int64_t S, int64_t num_neg, const int64_t* __restrict__ count,
                                                           uint8_t* __restrict__ flag, int32_t* __restrict__ blk_cnt) {
  if (*count >= num_neg) return;
  const PhiloxKey key = philox_key((uint64_t)*seed);
  const int64_t k = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  int keep = 0;
  if (k < S) {
    uint32_t row, col;
    neg_candidate(key, (uint32_t)k, round, n, row, col);
    keep = !u_contains(urp, ucol, row, col);
    flag[k] = (uint8_t)keep;
  }
  const int c = __syncthreads_count(keep);
  if (threadIdx.x == 0) blk_cnt[blockIdx.x] = c;
}

// one block: exclusive scan of the block counts from base = count; count <- min(count + survivors, num_neg).
// base_out = base, or -1 when the round is not needed (the scatter then does nothing).
__global__ void __launch_bounds__(kScanThreads) sgat_neg_scan(int32_t* __restrict__ blk_cnt, int64_t nb, int64_t num_neg,
                                                              int64_t* __restrict__ count, int64_t* __restrict__ base_out) {
  __shared__ int64_t sh[kScanThreads];
  const int64_t base = *count;
  __syncthreads();
  if (base >= num_neg) {
    if (threadIdx.x == 0) *base_out = -1;
    return;
  }
  const int64_t per = (nb + kScanThreads - 1) / kScanThreads;
  const int64_t b0 = threadIdx.x * per, b1 = min(nb, b0 + per);
  int64_t local = 0;
  for (int64_t b = b0; b < b1; ++b) local += blk_cnt[b];
  sh[threadIdx.x] = local;
  __syncthreads();
  for (int off = 1; off < kScanThreads; off <<= 1) {        // inclusive Hillis-Steele scan
    const int64_t v = threadIdx.x >= off ? sh[threadIdx.x - off] : 0;
    __syncthreads();
    sh[threadIdx.x] += v;
    __syncthreads();
  }
  int64_t run = base + sh[threadIdx.x] - local;
  for (int64_t b = b0; b < b1; ++b) {                        // block offsets, clamped: they are compared with num_neg
    const int32_t c = blk_cnt[b];
    blk_cnt[b] = (int32_t)min(run, num_neg);
    run += c;
  }
  if (threadIdx.x == kScanThreads - 1) {
    *count = min(base + sh[kScanThreads - 1], num_neg);
    *base_out = base;
  }
}

// stable compaction: survivor k goes to position blk_off[block] + (survivors before k in its block)
__global__ void __launch_bounds__(kThreads) sgat_neg_scatter(uint64_t n, const int64_t* __restrict__ seed, uint32_t round,
                                                             int64_t S, int64_t num_neg, const int64_t* __restrict__ base,
                                                             const uint8_t* __restrict__ flag,
                                                             const int32_t* __restrict__ blk_off,
                                                             int32_t* __restrict__ neg_src, int32_t* __restrict__ neg_dst) {
  __shared__ int warp_cnt[kThreads / 32];
  if (*base < 0) return;
  const int64_t k = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const bool keep = k < S && flag[k];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned ballot = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) warp_cnt[warp] = __popc(ballot);
  __syncthreads();
  int before = 0;
  for (unsigned w = 0; w < warp; ++w) before += warp_cnt[w];
  if (!keep) return;
  const int64_t pos = (int64_t)blk_off[blockIdx.x] + before + __popc(ballot & ((1u << lane) - 1u));
  if (pos >= num_neg) return;
  uint32_t row, col;
  neg_candidate(philox_key((uint64_t)*seed), (uint32_t)k, round, n, row, col);
  neg_src[pos] = (int32_t)row;
  neg_dst[pos] = (int32_t)col;
}

__global__ void sgat_keep_mask(const int64_t* __restrict__ seed, uint64_t thresh, int64_t nnz, uint8_t* __restrict__ out) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  out[e] = (uint8_t)edge_sample_keep(philox_key((uint64_t)*seed), (uint32_t)e, thresh);
}

// ---------------------------------------------------------------------------------------------------------------
// pair-logit BCE
// ---------------------------------------------------------------------------------------------------------------
struct Rows {                       // one CSR as the pair kernels read it
  const int64_t* rowptr;
  const int32_t* col;
  const int32_t* eid;               // positives with thresh != 0: edge id of every entry
};

struct PairParams {
  Rows pos, neg;
  const int32_t* order;             // schedule of the rows, or NULL
  int64_t n_rows;
  const float* X;
  int64_t ldx;
  int nvec, G;
  float scale;
  const int64_t* seed;
  uint64_t thresh;
};

__device__ __forceinline__ float softplus(float x) { return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoid(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float dot4(const float4& a, const float4& b, float acc) {
  acc = fmaf(a.x, b.x, acc);
  acc = fmaf(a.y, b.y, acc);
  acc = fmaf(a.z, b.z, acc);
  return fmaf(a.w, b.w, acc);
}

__device__ __forceinline__ void axpy4(float c, const float4& x, float4& y) {
  y.x = fmaf(c, x.x, y.x);
  y.y = fmaf(c, x.y, y.y);
  y.z = fmaf(c, x.z, y.z);
  y.w = fmaf(c, x.w, y.w);
}

struct Group {
  int G, lane;
  unsigned mask;
  __device__ __forceinline__ float sum(float v) const {
    for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, G);
    return v;
  }
};

// edges in flight per lane group: 4, and 2 from three vectors per lane on (no spills in the backward)
template <int V>
struct EdgesInFlight { static constexpr int value = V >= 3 ? 2 : 4; };

// Walks the pairs of one row in edges-in-flight batches and calls f(s, xj) for each kept pair; the sum over the
// group is in a fixed order, so every lane sees the same s.
template <int V, typename Fn>
__device__ __forceinline__ void for_pairs(const PairParams& p, const Group& g, const Rows& r, int64_t row, bool sample,
                                          PhiloxKey key, const float4 (&xi)[V], Fn&& f) {
  const int64_t k0 = __ldg(r.rowptr + row), k1 = __ldg(r.rowptr + row + 1);
  constexpr int U = EdgesInFlight<V>::value;
  for (int64_t kb = k0; kb < k1; kb += U) {
    float4 xj[U][V];
    bool use[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t k = kb + u;
      use[u] = k < k1;
      if (use[u] && sample) use[u] = edge_sample_keep(key, (uint32_t)__ldg(r.eid + k), p.thresh);
      const int32_t j = use[u] ? __ldg(r.col + k) : 0;
      const float4* xr = reinterpret_cast<const float4*>(p.X + (int64_t)j * p.ldx);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = g.lane + v * g.G;
        xj[u][v] = (use[u] && c < p.nvec) ? __ldg(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (!use[u]) continue;                           // uniform across the group: same k, same keep draw
      float d = 0.0f;
#pragma unroll
      for (int v = 0; v < V; ++v) d = dot4(xi[v], xj[u][v], d);
      f(p.scale * g.sum(d), xj[u]);
    }
  }
}

template <int V>
__device__ __forceinline__ bool setup(const PairParams& p, Group& g, int64_t& row, float4 (&xi)[V]) {
  const int64_t t = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const int64_t gid = t / p.G;
  g.G = p.G;
  g.lane = threadIdx.x & (p.G - 1);
  g.mask = p.G == 32 ? 0xffffffffu : (((1u << p.G) - 1u) << ((threadIdx.x & 31) & ~(p.G - 1)));
  if (gid >= p.n_rows) return false;                    // whole groups leave together
  row = p.order ? (int64_t)__ldg(p.order + gid) : gid;
  const float4* xr = reinterpret_cast<const float4*>(p.X + row * p.ldx);
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int c = g.lane + v * g.G;
    xi[v] = c < p.nvec ? __ldg(xr + c) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  return true;
}

template <int V>
__global__ void __launch_bounds__(kThreads) sgat_loss_fwd_rows(PairParams p, float* __restrict__ part,
                                                               int32_t* __restrict__ kept) {
  Group g;
  int64_t row;
  float4 xi[V];
  if (!setup<V>(p, g, row, xi)) return;
  const PhiloxKey key = philox_key(p.thresh ? (uint64_t)*p.seed : 0ull);
  float acc = 0.0f;
  int cnt = 0;
  for_pairs<V>(p, g, p.pos, row, p.thresh != 0, key, xi, [&](float s, const float4(&)[V]) {
    acc += softplus(-s);
    ++cnt;
  });
  for_pairs<V>(p, g, p.neg, row, false, key, xi, [&](float s, const float4(&)[V]) { acc += softplus(s); });
  if (g.lane == 0) {
    part[row] = acc;
    kept[row] = cnt;
  }
}

// stage 1: block b sums rows [b * kReduceRows, (b + 1) * kReduceRows) in fp64, in a fixed order
__global__ void __launch_bounds__(kThreads) sgat_reduce_blocks(const float* __restrict__ part, const int32_t* __restrict__ kept,
                                                               int64_t n, double* __restrict__ bsum, int64_t* __restrict__ bcnt) {
  __shared__ double ss[kThreads];
  __shared__ int64_t sc[kThreads];
  double s = 0.0;
  int64_t c = 0;
  const int64_t r0 = (int64_t)blockIdx.x * kReduceRows;
  for (int i = threadIdx.x; i < kReduceRows; i += kThreads) {
    const int64_t r = r0 + i;
    if (r < n) {
      s += (double)part[r];
      c += kept[r];
    }
  }
  ss[threadIdx.x] = s;
  sc[threadIdx.x] = c;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      ss[threadIdx.x] += ss[threadIdx.x + o];
      sc[threadIdx.x] += sc[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    bsum[blockIdx.x] = ss[0];
    bcnt[blockIdx.x] = sc[0];
  }
}

// stage 2 (one block): loss = sum / (P_pos + P_neg), P_neg = the negatives' rowptr[n]
__global__ void __launch_bounds__(kThreads) sgat_reduce_final(const double* __restrict__ bsum, const int64_t* __restrict__ bcnt,
                                                              int64_t nb, const int64_t* __restrict__ neg_rowptr, int64_t n,
                                                              float* __restrict__ loss, int64_t* __restrict__ npairs) {
  __shared__ double ss[kThreads];
  __shared__ int64_t sc[kThreads];
  double s = 0.0;
  int64_t c = 0;
  for (int64_t b = threadIdx.x; b < nb; b += kThreads) {
    s += bsum[b];
    c += bcnt[b];
  }
  ss[threadIdx.x] = s;
  sc[threadIdx.x] = c;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      ss[threadIdx.x] += ss[threadIdx.x + o];
      sc[threadIdx.x] += sc[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const int64_t P = sc[0] + neg_rowptr[n];
    *npairs = P;
    *loss = (float)(ss[0] / (double)P);                 // P == 0: NaN, as the mean of an empty BCE
  }
}

// PASS2 = false: rows are targets (forward CSR, negatives' CSR), dX[row] = acc.
// PASS2 = true : rows are sources (transpose CSRs), dX[row] += acc.
template <int V, bool PASS2>
__global__ void __launch_bounds__(kThreads) sgat_loss_bwd_rows(PairParams p, const int64_t* __restrict__ npairs,
                                                               const float* __restrict__ dloss, float* __restrict__ dX,
                                                               int64_t lddx) {
  Group g;
  int64_t row;
  float4 xi[V];
  if (!setup<V>(p, g, row, xi)) return;
  const PhiloxKey key = philox_key(p.thresh ? (uint64_t)*p.seed : 0ull);
  const float cf = (float)((double)*dloss * (double)p.scale / (double)*npairs);
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
  bool any = false;
  for_pairs<V>(p, g, p.pos, row, p.thresh != 0, key, xi, [&](float s, const float4(&xj)[V]) {
    const float c = cf * (sigmoid(s) - 1.0f);
#pragma unroll
    for (int v = 0; v < V; ++v) axpy4(c, xj[v], acc[v]);
    any = true;
  });
  for_pairs<V>(p, g, p.neg, row, false, key, xi, [&](float s, const float4(&xj)[V]) {
    const float c = cf * sigmoid(s);
#pragma unroll
    for (int v = 0; v < V; ++v) axpy4(c, xj[v], acc[v]);
    any = true;
  });
  if (PASS2 && !any) return;
  float4* out = reinterpret_cast<float4*>(dX + row * lddx);
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int c = g.lane + v * g.G;
    if (c >= p.nvec) continue;
    float4 r = acc[v];
    if (PASS2) {
      const float4 o = out[c];
      r = make_float4(o.x + r.x, o.y + r.y, o.z + r.z, o.w + r.w);
    }
    out[c] = r;
  }
}

// the SpMM's lane groups (csrc/spmm.cu choose_shape), widened to 3 and 4 vectors per lane beyond 64 vectors
void choose_groups(int nvec, int* G, int* V) {
  if (nvec > 64) { *G = 32; *V = (nvec + 31) / 32; return; }
  if (nvec > 32) { *G = 32; *V = 2; return; }
  if (nvec > 16) { *G = 16; *V = 2; return; }
  *V = 1;
  *G = nvec > 8 ? 16 : nvec > 4 ? 8 : 4;
}

int check_rows(const rgbmp_graph_t* g, int64_t n, const char* fn, const char* what) {
  if (int rc = check_graph(g, fn)) return rc;
  if (g->n_rows != n) return fail(RGBMP_EINVAL, "%s: bad %s descriptor (rows must equal the node count)", fn, what);
  return 0;
}

int check_features(const float* X, int64_t ldx, int F, const char* fn) {
  if (!X) return fail(RGBMP_EINVAL, "%s: X is NULL", fn);
  if (F <= 0 || F > 32 * 4 * kMaxVec) return fail(RGBMP_ERANGE, "%s: F = %d outside 1..%d", fn, F, 32 * 4 * kMaxVec);
  if (ldx < F || ldx % 4 != 0 || ((uintptr_t)X & 15u) != 0)
    return fail(RGBMP_EALIGN, "%s: rows must be 16-byte aligned with ld %% 4 == 0 and ld >= F", fn);
  return 0;
}

PairParams make_params(const rgbmp_graph_t* gp, const int32_t* eid, const rgbmp_graph_t* gn,
                       const rgbmp_sgat_sample_t* s, const float* X, int64_t ldx, int F, float scale) {
  PairParams p;
  p.pos = Rows{gp->rowptr, gp->col, eid};
  p.neg = Rows{gn->rowptr, gn->col, nullptr};
  p.order = gp->row_order;
  p.n_rows = gp->n_rows;
  p.X = X;
  p.ldx = ldx;
  p.nvec = (F + 3) / 4;
  int V;
  choose_groups(p.nvec, &p.G, &V);
  p.scale = scale;
  p.seed = s->seed;
  p.thresh = s->keep_thresh;
  return p;
}

int vec_of(const PairParams& p) { return (p.nvec + p.G - 1) / p.G; }

size_t reduce_blocks(int64_t n) { return (size_t)ceil_div(n < 1 ? 1 : n, kReduceRows); }

int check_sample(const rgbmp_sgat_sample_t* s, bool need_eid_t, const char* fn) {
  if (!s) return fail(RGBMP_EINVAL, "%s: sample descriptor is NULL", fn);
  if (s->keep_thresh > (1ull << 32)) return fail(RGBMP_EINVAL, "%s: keep_thresh exceeds 2^32", fn);
  if (s->keep_thresh != 0 && (!s->seed || !s->eid || (need_eid_t && !s->eid_t)))
    return fail(RGBMP_EINVAL, "%s: sampling positives needs the seed and the edge ids", fn);
  return 0;
}

}  // namespace
}  // namespace rgbmp

using namespace rgbmp;

extern "C" {

size_t rgbmp_sgat_negative_sampling_workspace_bytes(int64_t sample_size) {
  const int64_t S = sample_size < 1 ? 1 : sample_size;
  return align_up((size_t)S, 256) + align_up((size_t)ceil_div(S, kThreads) * 4, 256) + 256 + 3 * 256;
}

int rgbmp_sgat_negative_sampling(const int64_t* u_rowptr, const int32_t* u_col, int64_t N, const rgbmp_sgat_sample_t* s,
                                 int64_t num_neg, int64_t sample_size, int32_t* neg_src, int32_t* neg_dst,
                                 int64_t* count_dev, void* ws, size_t ws_bytes, int device, void* stream) {
  const char* fn = "rgbmp_sgat_negative_sampling";
  if (!count_dev || !s || !s->seed || N < 0) return fail(RGBMP_EINVAL, "%s: bad arguments", fn);
  if (N >= (1ll << 31)) return fail(RGBMP_ERANGE, "%s: N exceeds int32", fn);
  if (sample_size >= (1ll << 31)) return fail(RGBMP_ERANGE, "%s: sample_size %lld >= 2^31", fn, (long long)sample_size);
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "%s: cannot select device %d", fn, device);
  cudaStream_t st = (cudaStream_t)stream;
  RGBMP_CUDA(cudaMemsetAsync(count_dev, 0, sizeof(int64_t), st));
  if (num_neg <= 0 || sample_size <= 0 || N == 0) return 0;
  if (!u_rowptr || !neg_src || !neg_dst || !ws) return fail(RGBMP_EINVAL, "%s: NULL pointer", fn);
  if (ws_bytes < rgbmp_sgat_negative_sampling_workspace_bytes(sample_size))
    return fail(RGBMP_EWORKSPACE, "%s: workspace too small", fn);
  const int64_t nb = ceil_div(sample_size, kThreads);
  Carver cv(ws, ws_bytes);
  uint8_t* flag = cv.take<uint8_t>(sample_size);
  int32_t* blk = cv.take<int32_t>(nb);
  int64_t* base = cv.take<int64_t>(1);
  for (uint32_t r = 0; r < 3; ++r) {               // rounds after the one that fills num_neg return at once
    sgat_neg_flags<<<(unsigned)nb, kThreads, 0, st>>>(u_rowptr, u_col, (uint64_t)N, s->seed, r, sample_size, num_neg,
                                                     count_dev, flag, blk);
    sgat_neg_scan<<<1, kScanThreads, 0, st>>>(blk, nb, num_neg, count_dev, base);
    sgat_neg_scatter<<<(unsigned)nb, kThreads, 0, st>>>((uint64_t)N, s->seed, r, sample_size, num_neg, base, flag, blk,
                                                       neg_src, neg_dst);
  }
  RGBMP_LAUNCH_CHECK("sgat_negative_sampling");
  return 0;
}

int rgbmp_sgat_keep_mask(const rgbmp_sgat_sample_t* s, int64_t nnz, uint8_t* out, int device, void* stream) {
  const char* fn = "rgbmp_sgat_keep_mask";
  if (!s || !s->seed || nnz < 0 || (nnz > 0 && !out)) return fail(RGBMP_EINVAL, "%s: bad arguments", fn);
  if (s->keep_thresh > (1ull << 32)) return fail(RGBMP_EINVAL, "%s: keep_thresh exceeds 2^32", fn);
  if (nnz >= (1ll << 31)) return fail(RGBMP_ERANGE, "%s: nnz exceeds int32", fn);
  if (nnz == 0) return 0;
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "%s: cannot select device %d", fn, device);
  sgat_keep_mask<<<(unsigned)ceil_div(nnz, kThreads), kThreads, 0, (cudaStream_t)stream>>>(s->seed, s->keep_thresh, nnz, out);
  RGBMP_LAUNCH_CHECK("sgat_keep_mask");
  return 0;
}

size_t rgbmp_sgat_loss_workspace_bytes(int64_t n_rows) {
  const size_t n = (size_t)(n_rows < 1 ? 1 : n_rows), nb = reduce_blocks(n_rows);
  return align_up(n * 4, 256) + align_up(n * 4, 256) + align_up(nb * 8, 256) + align_up(nb * 8, 256) + 256;
}

int rgbmp_sgat_loss_forward(const rgbmp_graph_t* g, const rgbmp_graph_t* gneg, const rgbmp_sgat_sample_t* s,
                            const float* X, int64_t ldx, int F, float scale, float* loss, int64_t* npairs,
                            void* ws, size_t ws_bytes, int device, void* stream) {
  const char* fn = "rgbmp_sgat_loss_forward";
  int rc = check_graph(g, fn);
  if (rc) return rc;
  const int64_t n = g->n_rows;
  if ((rc = check_rows(gneg, n, fn, "negatives")) ||
      (rc = check_features(X, ldx, F, fn)) || (rc = check_sample(s, false, fn)))
    return rc;
  if (!loss || !npairs || !ws) return fail(RGBMP_EINVAL, "%s: NULL output or workspace", fn);
  if (ws_bytes < rgbmp_sgat_loss_workspace_bytes(n)) return fail(RGBMP_EWORKSPACE, "%s: workspace too small", fn);
  if (n >= (1ll << 31)) return fail(RGBMP_ERANGE, "%s: N exceeds int32", fn);
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "%s: cannot select device %d", fn, device);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t nb = (int64_t)reduce_blocks(n);
  Carver cv(ws, ws_bytes);
  float* part = cv.take<float>(n < 1 ? 1 : n);
  int32_t* kept = cv.take<int32_t>(n < 1 ? 1 : n);
  double* bsum = cv.take<double>(nb);
  int64_t* bcnt = cv.take<int64_t>(nb);
  if (n > 0) {
    const PairParams p = make_params(g, s->eid, gneg, s, X, ldx, F, scale);
    const unsigned grid = (unsigned)ceil_div(n * p.G, kThreads);
    switch (vec_of(p)) {
      case 1: sgat_loss_fwd_rows<1><<<grid, kThreads, 0, st>>>(p, part, kept); break;
      case 2: sgat_loss_fwd_rows<2><<<grid, kThreads, 0, st>>>(p, part, kept); break;
      case 3: sgat_loss_fwd_rows<3><<<grid, kThreads, 0, st>>>(p, part, kept); break;
      default: sgat_loss_fwd_rows<4><<<grid, kThreads, 0, st>>>(p, part, kept); break;
    }
    sgat_reduce_blocks<<<(unsigned)nb, kThreads, 0, st>>>(part, kept, n, bsum, bcnt);
  } else {
    RGBMP_CUDA(cudaMemsetAsync(bsum, 0, 8, st));
    RGBMP_CUDA(cudaMemsetAsync(bcnt, 0, 8, st));
  }
  sgat_reduce_final<<<1, kThreads, 0, st>>>(bsum, bcnt, nb, gneg->rowptr, n, loss, npairs);
  RGBMP_LAUNCH_CHECK("sgat_loss_forward");
  return 0;
}

int rgbmp_sgat_loss_backward(const rgbmp_graph_t* g, const rgbmp_graph_t* gT, const rgbmp_graph_t* gneg,
                             const rgbmp_graph_t* gnegT, const rgbmp_sgat_sample_t* s, const float* X, int64_t ldx, int F,
                             float scale, const int64_t* npairs, const float* dloss, float* dX, int64_t lddx,
                             int device, void* stream) {
  const char* fn = "rgbmp_sgat_loss_backward";
  int rc = check_graph(g, fn);
  if (rc) return rc;
  const int64_t n = g->n_rows;
  if ((rc = check_rows(gT, n, fn, "transpose graph")) ||
      (rc = check_rows(gneg, n, fn, "negatives")) || (rc = check_rows(gnegT, n, fn, "negatives' transpose")) ||
      (rc = check_features(X, ldx, F, fn)) || (rc = check_sample(s, true, fn)))
    return rc;
  if (!npairs || !dloss || !dX) return fail(RGBMP_EINVAL, "%s: NULL pointer", fn);
  if (lddx < F || lddx % 4 != 0 || ((uintptr_t)dX & 15u) != 0)
    return fail(RGBMP_EALIGN, "%s: dX rows must be 16-byte aligned with ld %% 4 == 0", fn);
  if (n >= (1ll << 31)) return fail(RGBMP_ERANGE, "%s: N exceeds int32", fn);
  if (n == 0) return 0;
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "%s: cannot select device %d", fn, device);
  cudaStream_t st = (cudaStream_t)stream;
  const PairParams p1 = make_params(g, s->eid, gneg, s, X, ldx, F, scale);
  const PairParams p2 = make_params(gT, s->eid_t, gnegT, s, X, ldx, F, scale);
  const unsigned grid = (unsigned)ceil_div(n * p1.G, kThreads);
  switch (vec_of(p1)) {
    case 1:
      sgat_loss_bwd_rows<1, false><<<grid, kThreads, 0, st>>>(p1, npairs, dloss, dX, lddx);
      sgat_loss_bwd_rows<1, true><<<grid, kThreads, 0, st>>>(p2, npairs, dloss, dX, lddx);
      break;
    case 2:
      sgat_loss_bwd_rows<2, false><<<grid, kThreads, 0, st>>>(p1, npairs, dloss, dX, lddx);
      sgat_loss_bwd_rows<2, true><<<grid, kThreads, 0, st>>>(p2, npairs, dloss, dX, lddx);
      break;
    case 3:
      sgat_loss_bwd_rows<3, false><<<grid, kThreads, 0, st>>>(p1, npairs, dloss, dX, lddx);
      sgat_loss_bwd_rows<3, true><<<grid, kThreads, 0, st>>>(p2, npairs, dloss, dX, lddx);
      break;
    default:
      sgat_loss_bwd_rows<4, false><<<grid, kThreads, 0, st>>>(p1, npairs, dloss, dX, lddx);
      sgat_loss_bwd_rows<4, true><<<grid, kThreads, 0, st>>>(p2, npairs, dloss, dX, lddx);
      break;
  }
  RGBMP_LAUNCH_CHECK("sgat_loss_backward");
  return 0;
}

}  // extern "C"
