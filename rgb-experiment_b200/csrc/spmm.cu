// CSR SpMM host-side dispatch, K-hop driver, host-buffer entry point (sm_100a).
#include <stdlib.h>
#include <string.h>
#include "spmm_kernels.cuh"

namespace rgbmp {

int khop_cta_try(const rgbmp_graph_t* g, const float* val, const void* X0, int64_t ldx0, void* ping, void* pong, int64_t ldp,
                 void* out, int64_t ldo, void* hops, int64_t ld_hops, int64_t hop_stride, int F, int dtype, int K,
                 const rgbmp_epilogue_t& ep, cudaStream_t st, int device, int* handled);   // khop_cta.cu

// packed [n,F] -> pitched z0 [n,ld] (optional) and u0 = scale*z0 [n,ld]; row r reads X row src_map[r] when mapped
__global__ void __launch_bounds__(256)
stage_rows_kernel(const float* __restrict__ X, int64_t ldx, const int32_t* __restrict__ src_map, const float* __restrict__ scale,
                  float* __restrict__ Z0, float* __restrict__ U0, int64_t ld, int64_t n_rows, int F) {
  const int64_t total = n_rows * ld;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    const int64_t r = t / ld;
    const int f = (int)(t - r * ld);
    const int64_t sr = src_map ? (int64_t)src_map[r] : r;
    const float v = (f < F) ? X[sr * ldx + f] : 0.f;
    if (Z0) Z0[t] = v;
    U0[t] = __fmul_rn(scale[r], v);
  }
}

// pitched [n,ld] -> packed [n,F]
__global__ void __launch_bounds__(256)
pack_rows_kernel(const float* __restrict__ X, int64_t ld, float* __restrict__ Y, int64_t n_rows, int F) {
  const int64_t total = n_rows * F;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    const int64_t r = t / F;
    Y[t] = X[r * ld + (t - r * F)];
  }
}

// bulk (TMA) pushes of the fused all-gather: off unless RGBMP_PUSH_BULK=1 / rgbmp_set_push_bulk(1).  Measured on the
// products-shaped APPNP (profiles/r02_push_bulk.txt): 2 GPUs 75.0 GTEPS bulk vs 76.9 stores, 4 GPUs 4x1 125.1 vs 126.4,
// 2x2 123.7 vs 125.5 -- bit-identical results, no gain: the way a row leaves the SM is not what limits the partitioned hop.
static int g_push_bulk = -1;
static int push_bulk_default() {
  if (g_push_bulk < 0) {
    const char* e = getenv("RGBMP_PUSH_BULK");
    g_push_bulk = (e && e[0] == '1') ? 1 : 0;
  }
  return g_push_bulk;
}

// choose (G, V, U) for nvec 16-byte vectors per row.  Measured on B200 with the round-2 inner loop (column ids
// staged through shared memory, lanes beyond F issue no load; tools/sweep.py, profiles/r02_sweep.txt):
//   * one vector per lane with 8 plain (not software-pipelined) edges in flight wins wherever a row fits 16 lanes --
//     products F=47 3.03 ms (G16 V1 U8) vs 3.64 (round 1's G8 V2 pipelined), F=64 3.04 vs 3.84, arxiv F=40 0.116 vs
//     0.156, bf16 F=128 0.129 vs 0.165, reddit F=64 1.51 vs 1.89 -- both when the gathers come from HBM and when
//     they are L2-resident: with the id broadcast out of the LSU data pipe, fewer and fuller wavefronts per edge
//     beat deeper per-lane pipelines;
//   * wider rows take two vectors per lane with 4 edges in flight (F=100: G16 V2 U4 6.02 vs 7.05; F=256: G32 V2
//     U4 0.307 vs 0.459); rows wider than 64 vectors are tiled over blockIdx.y;
//   * narrow rows: 8 lanes x 8 edges for 5-8 vectors (F=24/32: 1.81 / 1.74 ms), 4 lanes below that -- pipelined
//     for 1-2 vectors, where two idle lanes still beat the 2-lane group (F=8: 0.86 vs 1.08 ms).
//   * rows of 9-16 vectors whose gathers come from HBM (feature matrix well beyond L2), with the round-4 loop (one plain
//     load per vector on untagged graphs; profiles/r04_spmm_untagged_gather.txt, bench.py on one B200 at 1000 W):
//     rows of 32 edges and more on average keep 8 edges in flight at 4 CTAs/SM (62 registers) -- products F=47
//     55.5 GTEPS vs 54.6 with 4 edges at 5 CTAs/SM (48 registers; 8 edges at 5 CTAs spill 224 bytes); shorter rows
//     (papers100M-shaped block, 29.5 edges per row on average, bf16 F=128) keep 4 at 5 CTAs/SM, 22.2 vs 21.9 GTEPS
//     with 8 (both with the two-loop weighted bf16 kernel, since replaced).  The cut-off of 32 only separates these two measured graphs (29.5 and 51.5 edges per row); it has not
//     been swept.  L2-resident matrices (arxiv F=40, bf16 F=128) keep 8.
static void choose_shape(int nvec, bool hbm_short_rows, int* G, int* V, int* U) {
  if (nvec > 32) { *G = 32; *V = 2; *U = 4; return; }
  if (nvec > 16) { *G = 16; *V = 2; *U = 4; return; }
  if (nvec > 8) { *G = 16; *V = 1; *U = hbm_short_rows ? 4 : 8; return; }
  if (nvec > 4) { *G = 8; *V = 1; *U = 8; return; }
  *G = 4;
  *V = 1;
  *U = nvec > 2 ? 4 : 20;
}

struct Prepared {
  SpmmParams p;
  int G, V, U, epv;
};

// ep passed check_epilogue
static int spmm_prepare(const rgbmp_graph_t* g, const float* val, const void* X, int64_t ldx, void* Y, int64_t ldy, int F,
                        int dtype, const rgbmp_epilogue_t& ep, int tune, void* ws, size_t ws_bytes, Prepared* out) {
  SpmmParams& p = out->p;
  p.w = csr_work(g);
  p.val = val;
  p.push_bulk = push_bulk_default();
  p.X = X;
  p.ldx = ldx;
  p.Y = Y;
  p.ldy = ldy;
  p.F = F;
  p.ep = ep;

  const int esz = dtype == RGBMP_BF16 ? 2 : 4;
  const int epv_vec = 16 / esz;
  auto aligned = [&](const void* ptr, int64_t ld) {
    return ptr == nullptr || ((((uintptr_t)ptr) & 15) == 0 && (ld % epv_vec) == 0 && ld >= align_up(F, epv_vec));
  };
  const bool vec_ok = aligned(X, ldx) && aligned(Y, ldy) && aligned(p.ep.T, p.ep.ldt) && aligned(p.ep.Y2, p.ep.ldy2) &&
                      aligned(p.ep.acc_in, p.ep.ld_acc) &&
                      (p.ep.n_peers == 0 || ((p.ep.ld_peer % epv_vec) == 0 && ((p.ep.peer_row0 * p.ep.ld_peer) % epv_vec) == 0));
  const int epv = vec_ok ? epv_vec : 1;
  if (dtype == RGBMP_BF16 && !vec_ok)
    return fail(RGBMP_EALIGN, "rgbmp_spmm: bf16 needs 16-byte aligned pointers and ld %% 8 == 0");

  p.partial = nullptr;
  p.ldpart = 0;
  if (p.w.n_items > 0) {
    p.ldpart = (int64_t)align_up(F, 4);
    const size_t need = (size_t)p.w.n_items * p.ldpart * sizeof(float);
    if (!ws || ws_bytes < need) return fail(RGBMP_EWORKSPACE, "rgbmp_spmm: workspace %zu < %zu", ws_bytes, need);
    p.partial = (float*)ws;
  }

  int G, V, U;
  const int nvec = (int)ceil_div(F, epv);
  // gathered rows mostly come from HBM once the feature matrix is well beyond the 126 MB L2
  const bool hbm_regime = (double)g->n_cols * (double)ldx * esz > 96e6;
  const bool short_rows = g->nnz < 32 * g->n_rows;   // mean row shorter than two 16-edge batches
  choose_shape(nvec, hbm_regime && short_rows, &G, &V, &U);
  p.stream = (tune & RGBMP_TUNE_NO_STREAM) ? 0 : 1;
  // gathered rows: ids tagged hot by rgbmp_col_tag stay in L2 (evict-last), the rest leave first
  p.hinted = (g->col_tagged || (tune & RGBMP_TUNE_POLICY)) ? 1 : 0;
  p.pol_hot = g->col_tagged ? 2 : 0;
  p.pol_cold = g->col_tagged ? 1 : 0;
  if (tune & RGBMP_TUNE_POLICY) {
    p.pol_cold = (tune >> 25) & 3;
    p.pol_hot = (tune >> 27) & 3;
    if (p.pol_cold > 2 || p.pol_hot > 2) return fail(RGBMP_EINVAL, "rgbmp_spmm: bad cache policy in tune word 0x%x", tune);
  }
  tune &= 0xFFFFFF;
  if (tune != 0) {
    G = tune & 0xFF;
    V = (tune >> 8) & 0xFF;
    U = (tune >> 16) & 0xFF;
    const bool pow2 = G > 0 && (G & (G - 1)) == 0 && G <= 32;
    if (!pow2 || V < 1 || V > 2 || (U != 2 && U != 4 && U != 8 && U != 18 && U != 20))
      return fail(RGBMP_EINVAL, "rgbmp_spmm: bad tune word 0x%x", tune);
  }
  out->G = G;
  out->V = V;
  out->U = U;
  out->epv = epv;
  return 0;
}

static int spmm_impl(const rgbmp_graph_t* g, const float* val, const void* X, int64_t ldx, void* Y, int64_t ldy, int F,
                     int dtype, const rgbmp_epilogue_t& ep, int tune, void* ws, size_t ws_bytes, cudaStream_t st) {
  Prepared pr;
  const int rc = spmm_prepare(g, val, X, ldx, Y, ldy, F, dtype, ep, tune, ws, ws_bytes, &pr);
  if (rc) return rc;
  if (dtype == RGBMP_BF16) return spmm_dispatch_bf16(pr.p, pr.G, pr.V, pr.U, st);
  if (pr.epv == 4) return spmm_dispatch_f32v(pr.p, pr.G, pr.V, pr.U, st);
  return spmm_dispatch_f32s(pr.p, pr.G, pr.V, pr.U, st);
}

}  // namespace rgbmp

using namespace rgbmp;

extern "C" {

size_t rgbmp_spmm_workspace_bytes(const rgbmp_graph_t* g, int F) {
  if (!g || g->n_items <= 0) return 256;
  return (size_t)g->n_items * align_up((size_t)F, 4) * sizeof(float) + 256;
}

int rgbmp_set_push_bulk(int on) {
  const int old = push_bulk_default();
  if (on == 0 || on == 1) g_push_bulk = on;
  return old;
}

int rgbmp_spmm(const rgbmp_graph_t* g, const float* val, const void* X, int64_t ldx, void* Y, int64_t ldy, int F,
               int dtype, const rgbmp_epilogue_t* ep, int tune, void* ws, size_t ws_bytes, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_spmm", GRAPH_TAGS_OK);
  if (rc) return rc;
  if (!X || F <= 0 || ldx < F || (Y && ldy < F)) return fail(RGBMP_EINVAL, "rgbmp_spmm: bad feature arguments");
  if (dtype != RGBMP_F32 && dtype != RGBMP_BF16) return fail(RGBMP_EINVAL, "rgbmp_spmm: bad dtype %d", dtype);
  rgbmp_epilogue_t e;
  rc = check_epilogue(ep, F, Y != nullptr, "rgbmp_spmm", 0, &e);
  if (rc) return rc;
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_spmm: bad device %d", device);
  return spmm_impl(g, val, X, ldx, Y, ldy, F, dtype, e, tune, ws, ws_bytes, (cudaStream_t)stream);
}

int rgbmp_khop(const rgbmp_graph_t* g, const float* val, const void* X0, int64_t ldx0, void* ping, void* pong,
               int64_t ldp, void* out, int64_t ldo, void* hops, int64_t ld_hops, int64_t hop_stride, int F, int dtype,
               int K, const rgbmp_epilogue_t* ep, int tune, void* ws, size_t ws_bytes, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_khop", GRAPH_TAGS_OK | GRAPH_SQUARE);
  if (rc) return rc;
  if (!X0 || (!out && !hops) || F <= 0 || K < 1 || ldx0 < F || (out && ldo < F))
    return fail(RGBMP_EINVAL, "rgbmp_khop: bad arguments");
  if (K > 1 && (!ping || !pong || ldp < F)) {
    const bool through_hops = hops != nullptr && !(ep && ep->out2_scale);
    if (!through_hops) return fail(RGBMP_EINVAL, "rgbmp_khop: K > 1 needs ping/pong buffers");
  }
  if (dtype != RGBMP_F32 && dtype != RGBMP_BF16) return fail(RGBMP_EINVAL, "rgbmp_khop: bad dtype %d", dtype);
  rgbmp_epilogue_t e;
  rc = check_epilogue(ep, F, true /* out or hops */, "rgbmp_khop", EP_KHOP | (hops ? EP_HOPS : 0), &e);
  if (rc) return rc;
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_khop: bad device %d", device);
  cudaStream_t st = (cudaStream_t)stream;
  if (!(tune & RGBMP_TUNE_NO_CTA)) {     // small graphs: all K hops in one launch of one thread-block cluster
    int handled = 0;
    rc = khop_cta_try(g, val, X0, ldx0, ping, pong, ldp, out, ldo, hops, ld_hops, hop_stride, F, dtype, K, e, st, device,
                      &handled);
    if (handled) return rc;
  }
  const size_t esz = dtype == RGBMP_BF16 ? 2 : 4;
  const bool folded = e.out2_scale != nullptr;  // iterate lives in the pre-scaled copy
  const void* in = X0;
  int64_t ldin = ldx0;
  for (int k = 0; k < K; ++k) {
    const bool last = (k == K - 1);
    void* buf = (k & 1) ? pong : ping;
    void* y = nullptr;
    int64_t ldy = 0;
    rgbmp_epilogue_t ek = e;
    ek.row_map = last ? e.row_map : nullptr;     // the iterate stays in the graph's own naming until the last store
    if (hops) { y = (char*)hops + (size_t)k * hop_stride * esz; ldy = ld_hops; }
    if (last && !hops) { y = out; ldy = ldo; }
    if (folded) {
      ek.Y2 = last ? nullptr : buf;
      ek.ldy2 = ldp;
    } else if (!y) {
      y = buf;
      ldy = ldp;
    }
    rc = spmm_impl(g, val, in, ldin, y, ldy, F, dtype, ek, tune, ws, ws_bytes, st);
    if (rc) return rc;
    if (folded) { in = buf; ldin = ldp; }
    else { in = y; ldin = ldy; }
  }
  if (hops && out) {  // final iterate also requested in `out`
    const void* lastp = (const char*)hops + (size_t)(K - 1) * hop_stride * esz;
    if (lastp != out)
      RGBMP_CUDA(cudaMemcpy2DAsync(out, ldo * esz, lastp, ld_hops * esz, F * esz, g->n_rows, cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

int rgbmp_peer_alloc(size_t bytes, void** ptr, unsigned char handle[RGBMP_IPC_HANDLE_BYTES], int device) {
  static_assert(sizeof(cudaIpcMemHandle_t) == RGBMP_IPC_HANDLE_BYTES, "IPC handle size");
  if (!ptr || !handle || bytes == 0) return fail(RGBMP_EINVAL, "rgbmp_peer_alloc: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_peer_alloc: bad device");
  void* p = nullptr;
  RGBMP_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return cuda_fail(e, "cudaIpcGetMemHandle"); }
  memcpy(handle, &h, sizeof(h));
  *ptr = p;
  return 0;
}

int rgbmp_peer_free(void* ptr, int device) {
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_peer_free: bad device");
  if (ptr) RGBMP_CUDA(cudaFree(ptr));
  return 0;
}

int rgbmp_peer_open(const unsigned char handle[RGBMP_IPC_HANDLE_BYTES], void** ptr, int device) {
  if (!handle || !ptr) return fail(RGBMP_EINVAL, "rgbmp_peer_open: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_peer_open: bad device");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  RGBMP_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}

int rgbmp_peer_close(void* ptr, int device) {
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_peer_close: bad device");
  if (ptr) RGBMP_CUDA(cudaIpcCloseMemHandle(ptr));
  return 0;
}

int rgbmp_l2_persist(int device, size_t bytes, size_t* granted) {
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_l2_persist: bad device");
  int maxb = 0;
  RGBMP_CUDA(cudaDeviceGetAttribute(&maxb, cudaDevAttrMaxPersistingL2CacheSize, device));
  if (bytes > (size_t)maxb) bytes = (size_t)maxb;
  RGBMP_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes));
  size_t got = 0;
  RGBMP_CUDA(cudaDeviceGetLimit(&got, cudaLimitPersistingL2CacheSize));
  if (granted) *granted = got;
  return 0;
}

int rgbmp_row_scale(const void* X, int64_t ldx, const float* scale, int divide, void* Y, int64_t ldy, int64_t n_rows,
                    int F, int dtype, int device, void* stream) {
  if (!X || !scale || !Y || n_rows < 0 || F <= 0 || ldx < F || ldy < F) return fail(RGBMP_EINVAL, "rgbmp_row_scale: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_row_scale: bad device");
  if (n_rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == RGBMP_BF16)
    row_scale_kernel<__nv_bfloat16><<<kSMs * 8, 256, 0, st>>>((const __nv_bfloat16*)X, ldx, scale, divide, (__nv_bfloat16*)Y, ldy, n_rows, F);
  else
    row_scale_kernel<float><<<kSMs * 8, 256, 0, st>>>((const float*)X, ldx, scale, divide, (float*)Y, ldy, n_rows, F);
  RGBMP_LAUNCH_CHECK("row_scale_kernel");
  return 0;
}

int rgbmp_stage_rows(const float* X, int64_t ldx, const int32_t* src_map, const float* scale, float* Z0, float* U0, int64_t ld,
                     int64_t n_rows, int F, int device, void* stream) {
  if (!X || !scale || !U0 || n_rows < 0 || F <= 0 || ldx < F || ld < F) return fail(RGBMP_EINVAL, "rgbmp_stage_rows: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_stage_rows: bad device");
  if (n_rows == 0) return 0;
  stage_rows_kernel<<<kSMs * 8, 256, 0, (cudaStream_t)stream>>>(X, ldx, src_map, scale, Z0, U0, ld, n_rows, F);
  RGBMP_LAUNCH_CHECK("stage_rows_kernel");
  return 0;
}

int rgbmp_appnp_host(const rgbmp_graph_t* g, const float* dinv, const float* z0_host, float* out_host, int F, int K,
                     float alpha, float* dev_z0, float* dev_ping, float* dev_pong, float* dev_out, int64_t ld, void* ws,
                     size_t ws_bytes, int device, void* stream) {
  return rgbmp_appnp_host_mapped(g, nullptr, dinv, z0_host, out_host, F, K, alpha, dev_z0, dev_ping, dev_pong, dev_out, ld, ws,
                                 ws_bytes, device, stream);
}

int rgbmp_appnp_host_mapped(const rgbmp_graph_t* g, const int32_t* row_map, const float* dinv, const float* z0_host,
                            float* out_host, int F, int K, float alpha, float* dev_z0, float* dev_ping, float* dev_pong,
                            float* dev_out, int64_t ld, void* ws, size_t ws_bytes, int device, void* stream) {
  int rc = check_graph(g, "rgbmp_appnp_host", GRAPH_TAGS_OK | GRAPH_SQUARE);
  if (rc) return rc;
  if (!dinv || !z0_host || !out_host || !dev_z0 || !dev_ping || !dev_pong || !dev_out || F <= 0 || K < 1 || ld < F)
    return fail(RGBMP_EINVAL, "rgbmp_appnp_host: bad argument");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_appnp_host: bad device");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t N = g->n_rows;
  // One contiguous H2D at full PCIe rate into dev_out (used as the packed [N,F] staging area; a
  // pitched 2-D copy of 188-byte rows runs ~15x slower), then one kernel re-pitches to ld and
  // writes both z0 and u0 = D^-1/2 z0 (in the graph's node order when it is renamed).
  float* stage = dev_out;
  RGBMP_CUDA(cudaMemcpyAsync(stage, z0_host, (size_t)N * F * sizeof(float), cudaMemcpyHostToDevice, st));
  stage_rows_kernel<<<kSMs * 8, 256, 0, st>>>(stage, F, row_map, dinv, dev_z0, dev_pong, ld, N, F);
  RGBMP_LAUNCH_CHECK("stage_rows_kernel");
  rgbmp_epilogue_t e = {};
  e.row_scale = dinv;
  e.a = 1.0f - alpha;
  e.b = alpha;
  e.T = dev_z0;
  e.ldt = ld;
  e.out2_scale = dinv;
  e.row_map = row_map;
  // hop 1 reads u0 from pong and writes ping; the last hop writes the unscaled result to dev_out
  rc = rgbmp_khop(g, nullptr, dev_pong, ld, dev_ping, dev_pong, ld, dev_out, ld, nullptr, 0, 0, F, RGBMP_F32, K, &e, 0, ws,
                  ws_bytes, device, stream);
  if (rc) return rc;
  // pack [N, ld] -> [N, F] (ping is free once the last hop has run) and copy out contiguously
  float* packed = dev_ping;
  pack_rows_kernel<<<kSMs * 8, 256, 0, st>>>(dev_out, ld, packed, N, F);
  RGBMP_LAUNCH_CHECK("pack_rows_kernel");
  RGBMP_CUDA(cudaMemcpyAsync(out_host, packed, (size_t)N * F * sizeof(float), cudaMemcpyDeviceToHost, st));
  RGBMP_CUDA(cudaStreamSynchronize(st));
  return 0;
}

}  // extern "C"
