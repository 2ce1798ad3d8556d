// Edge-score kernels (sm_100a): SDDMM, u_add_v, segmented softmax (+backward), segmented sum,
// multi-head weighted SpMM, row dot.  (The fused GATConv kernels live in gat.cu.)
//
// All are gather / segment-reduce kernels over CSR -- HBM/L2-bound, no tensor cores.  A row of the
// CSR (all in-edges of one target, or all out-edges of one source for the transpose) is owned by a
// warp; reductions over a row's edges are sequential per lane + warp shuffles, so results are
// deterministic.
#include "csr_work.cuh"

namespace rgbmp {

__device__ __forceinline__ float leaky(float x, float slope) { return x > 0.f ? x : x * slope; }

__global__ void __launch_bounds__(256)
rowdot_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, int64_t n_rows, int H,
              int C, float* __restrict__ S) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n_rows * H) return;
  const int64_t i = t / H;
  const int h = (int)(t - i * H);
  const float* a = A + i * lda + h * C;
  const float* b = B + i * ldb + h * C;
  float s = 0.f;
  for (int c = 0; c < C; ++c) s += a[c] * b[c];
  S[t] = s;
}

// ------------------------------------------------------------------------------------------
// warp-per-row edge-score kernels
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
sddmm_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t n_rows,
             const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, int H, int C,
             float* __restrict__ out) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t k0 = rowptr[row], k1 = rowptr[row + 1];
  const int64_t total = (k1 - k0) * H;
  const float* a_row = A + row * lda;
  for (int64_t idx = lane; idx < total; idx += 32) {
    const int64_t k = k0 + idx / H;
    const int h = (int)(idx % H);
    const float* a = a_row + h * C;
    const float* b = B + (int64_t)col[k] * ldb + h * C;
    float s = 0.f;
    for (int c = 0; c < C; ++c) s += __ldg(a + c) * __ldg(b + c);
    out[k * H + h] = s;
  }
}

__global__ void __launch_bounds__(256)
u_add_v_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t n_rows,
               const float* __restrict__ u, const float* __restrict__ v, int H, float* __restrict__ out) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t k0 = rowptr[row], k1 = rowptr[row + 1];
  const int64_t total = (k1 - k0) * H;
  for (int64_t idx = lane; idx < total; idx += 32) {
    const int64_t k = k0 + idx / H;
    const int h = (int)(idx % H);
    out[k * H + h] = __ldg(u + (int64_t)col[k] * H + h) + __ldg(v + row * H + h);
  }
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// out[k,h] = exp(in[k,h]-max_h) / (sum_h + 1e-16)   (SURVEY.md A11)
__global__ void __launch_bounds__(256)
seg_softmax_kernel(const int64_t* __restrict__ rowptr, int64_t n_rows, const float* __restrict__ in, int H,
                   float* __restrict__ out) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t k0 = rowptr[row], k1 = rowptr[row + 1];
  for (int h = 0; h < H; ++h) {
    float m = -INFINITY;
    for (int64_t k = k0 + lane; k < k1; k += 32) m = fmaxf(m, in[k * H + h]);
    m = warp_max(m);
    float s = 0.f;
    for (int64_t k = k0 + lane; k < k1; k += 32) s += expf(in[k * H + h] - m);
    s = warp_sum(s);
    const float den = s + 1e-16f;
    for (int64_t k = k0 + lane; k < k1; k += 32) out[k * H + h] = expf(in[k * H + h] - m) / den;
  }
}

// dlogit[k,h] = alpha[k,h] * (dalpha[k,h] - sum_k' alpha[k',h]*dalpha[k',h])
__global__ void __launch_bounds__(256)
seg_softmax_bwd_kernel(const int64_t* __restrict__ rowptr, int64_t n_rows, const float* __restrict__ alpha,
                       const float* __restrict__ dalpha, int H, float* __restrict__ dlogit) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t k0 = rowptr[row], k1 = rowptr[row + 1];
  for (int h = 0; h < H; ++h) {
    float s = 0.f;
    for (int64_t k = k0 + lane; k < k1; k += 32) s += alpha[k * H + h] * dalpha[k * H + h];
    s = warp_sum(s);
    for (int64_t k = k0 + lane; k < k1; k += 32) dlogit[k * H + h] = alpha[k * H + h] * (dalpha[k * H + h] - s);
  }
}

__global__ void __launch_bounds__(256)
seg_sum_kernel(const int64_t* __restrict__ rowptr, int64_t n_rows, const float* __restrict__ in, int H,
               float* __restrict__ out) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t k0 = rowptr[row], k1 = rowptr[row + 1];
  for (int h = 0; h < H; ++h) {
    float s = 0.f;
    for (int64_t k = k0 + lane; k < k1; k += 32) s += in[k * H + h];
    s = warp_sum(s);
    if (lane == 0) out[row * H + h] = s;
  }
}

// out[i,h,:] = sum_k w[k,h] * X[col[k],h,:]   warp per row, lanes over the H*C features
__global__ void __launch_bounds__(256)
spmm_heads_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t n_rows,
                  const float* __restrict__ w, const float* __restrict__ X, int64_t ldx, int H, int C,
                  float* __restrict__ out, int64_t ldo) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int64_t k0 = rowptr[row], k1 = rowptr[row + 1];
  const int HC = H * C;
  for (int fb = 0; fb < HC; fb += 32) {
    const int f = fb + lane;
    const bool act = f < HC;
    const int h = act ? f / C : 0;
    float acc = 0.f;
    for (int64_t k = k0; k < k1; ++k) {
      const int64_t j = col[k];
      if (act) acc = __fadd_rn(acc, __fmul_rn(__ldg(w + k * H + h), __ldg(X + j * ldx + f)));
    }
    if (act) out[row * ldo + f] = acc;
  }
}

}  // namespace rgbmp

using namespace rgbmp;

extern "C" {

int rgbmp_rowdot(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t n_rows, int H, int C, float* S,
                 int device, void* stream) {
  if (!A || !B || !S || n_rows < 0 || H <= 0 || C <= 0) return fail(RGBMP_EINVAL, "rgbmp_rowdot: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_rowdot: bad device");
  if (n_rows == 0) return 0;
  rowdot_kernel<<<(unsigned)ceil_div(n_rows * H, 256), 256, 0, (cudaStream_t)stream>>>(A, lda, B, ldb, n_rows, H, C, S);
  RGBMP_LAUNCH_CHECK("rowdot_kernel");
  return 0;
}

#define WARP_ROW_GRID(n) (unsigned)ceil_div((n) * 32, 256), 256, 0, (cudaStream_t)stream

int rgbmp_sddmm(const rgbmp_graph_t* g, const float* A, int64_t lda, const float* B, int64_t ldb, int H, int C,
                float* out, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_sddmm");
  if (rc) return rc;
  if (!A || !B || (g->nnz > 0 && !out) || H <= 0 || C <= 0) return fail(RGBMP_EINVAL, "rgbmp_sddmm: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_sddmm: bad device");
  if (g->n_rows == 0 || g->nnz == 0) return 0;
  sddmm_kernel<<<WARP_ROW_GRID(g->n_rows)>>>(g->rowptr, g->col, g->n_rows, A, lda, B, ldb, H, C, out);
  RGBMP_LAUNCH_CHECK("sddmm_kernel");
  return 0;
}

int rgbmp_u_add_v(const rgbmp_graph_t* g, const float* u, const float* v, int H, float* out, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_u_add_v");
  if (rc) return rc;
  if (!u || !v || (g->nnz > 0 && !out) || H <= 0) return fail(RGBMP_EINVAL, "rgbmp_u_add_v: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_u_add_v: bad device");
  if (g->n_rows == 0 || g->nnz == 0) return 0;
  u_add_v_kernel<<<WARP_ROW_GRID(g->n_rows)>>>(g->rowptr, g->col, g->n_rows, u, v, H, out);
  RGBMP_LAUNCH_CHECK("u_add_v_kernel");
  return 0;
}

int rgbmp_seg_softmax(const rgbmp_graph_t* g, const float* in, int H, float* out, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_seg_softmax");
  if (rc) return rc;
  if ((g->nnz > 0 && (!in || !out)) || H <= 0) return fail(RGBMP_EINVAL, "rgbmp_seg_softmax: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_seg_softmax: bad device");
  if (g->n_rows == 0 || g->nnz == 0) return 0;
  seg_softmax_kernel<<<WARP_ROW_GRID(g->n_rows)>>>(g->rowptr, g->n_rows, in, H, out);
  RGBMP_LAUNCH_CHECK("seg_softmax_kernel");
  return 0;
}

int rgbmp_seg_softmax_backward(const rgbmp_graph_t* g, const float* alpha, const float* dalpha, int H, float* dlogit,
                               int device, void* stream) {
  int rc = check_graph(g, "rgbmp_seg_softmax_backward");
  if (rc) return rc;
  if ((g->nnz > 0 && (!alpha || !dalpha || !dlogit)) || H <= 0)
    return fail(RGBMP_EINVAL, "rgbmp_seg_softmax_backward: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_seg_softmax_backward: bad device");
  if (g->n_rows == 0 || g->nnz == 0) return 0;
  seg_softmax_bwd_kernel<<<WARP_ROW_GRID(g->n_rows)>>>(g->rowptr, g->n_rows, alpha, dalpha, H, dlogit);
  RGBMP_LAUNCH_CHECK("seg_softmax_bwd_kernel");
  return 0;
}

int rgbmp_seg_sum(const rgbmp_graph_t* g, const float* in, int H, float* out, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_seg_sum");
  if (rc) return rc;
  if ((g->nnz > 0 && !in) || !out || H <= 0) return fail(RGBMP_EINVAL, "rgbmp_seg_sum: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_seg_sum: bad device");
  if (g->n_rows == 0) return 0;
  seg_sum_kernel<<<WARP_ROW_GRID(g->n_rows)>>>(g->rowptr, g->n_rows, in, H, out);
  RGBMP_LAUNCH_CHECK("seg_sum_kernel");
  return 0;
}

int rgbmp_spmm_heads(const rgbmp_graph_t* g, const float* w, const float* X, int64_t ldx, int H, int C, float* out,
                     int64_t ldo, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_spmm_heads");
  if (rc) return rc;
  if ((g->nnz > 0 && !w) || !X || !out || H <= 0 || C <= 0) return fail(RGBMP_EINVAL, "rgbmp_spmm_heads: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_spmm_heads: bad device");
  if (g->n_rows == 0) return 0;
  spmm_heads_kernel<<<WARP_ROW_GRID(g->n_rows)>>>(g->rowptr, g->col, g->n_rows, w, X, ldx, H, C, out, ldo);
  RGBMP_LAUNCH_CHECK("spmm_heads_kernel");
  return 0;
}

}  // extern "C"
