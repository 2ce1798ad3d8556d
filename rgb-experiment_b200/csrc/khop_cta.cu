// K-hop propagation of a SMALL graph in ONE launch of ONE thread-block cluster (sm_100a).
//
// On a Cora-sized graph (2.7 k nodes, 13 k edges, 7 classes) a hop moves ~0.5 MB; the K-launch path spends 15-18 us per
// hop on it -- three launches (short rows, long-row items, combine) whose cost is launch latency and the chain of
// dependent L2 loads that starts every row, not bytes (profiles/r02_small_graph_latency.txt).  APPNP K=10,
// Correct&Smooth's 50+50 hops and the PTA label propagation on the reference's own CPU-sized datasets
// (BASELINE configs[0]; itexperiments.py:520-526, appnp_stack.py:22, pta.py:79-84) are exactly this case.
//
// Here ONE cluster of C = 16 (8 where 16 cannot be placed) CTAs x 512 threads runs all K hops; the hops are separated
// by the hardware cluster barrier (barrier.cluster, release / acquire: a few hundred cycles) instead of kernel
// boundaries.  The iterate stays in the caller's ping / pong buffers, i.e. in L2.  A group of G lanes owns a row (lane l
// its l-th 16-byte vector) and walks the slots  g, g + C*512/G, ...  of the degree-sorted schedule; a row's epilogue
// operands are requested one row ahead; rows longer than 32 edges -- a hop's critical path -- are taken by a whole warp
// each (32/G edge slots, 4 gathers in flight per lane, fixed-order shuffle reduction).
// Two earlier cuts, measured on B200 and dropped (profiles/r02_small_graph_latency.txt):
//   * everything in ONE CTA's shared memory: issue-bound on its single SM, 12 us per hop -- no better than the launches;
//   * the iterate dealt over the cluster's DISTRIBUTED shared memory and gathered with ld.shared::cluster: no faster than
//     L2 (8 us per hop at F=7, 46 at F=64 -- remote shared-memory loads are served lane by lane);
//   * a hop barrier built from one remote mbarrier arrive per CTA (one release fence per CTA instead of one per thread)
//     in place of barrier.cluster: within noise of it (56 vs 54 us for APPNP K=10).
// Edges of a row accumulate sequentially in stable CSR order exactly as in spmm_rows_kernel (bit-identical for rows
// neither path splits); the epilogue is rgbmp_epilogue_t's, applied by the same ep_apply.
#include <stdlib.h>
#include "epilogue.cuh"

namespace rgbmp {

// 512 threads per CTA: 1,024 (64 registers, spills) measured 5-10 % slower, 256 40 % slower (profiles/r02_small_graph_latency.txt)
#ifndef RGBMP_KC_THREADS
#define RGBMP_KC_THREADS 512
#endif
constexpr int KC_THREADS = RGBMP_KC_THREADS;       // A/B: tools/build_variant.py kc1024 -DRGBMP_KC_THREADS=1024 --only khop_cta.cu
constexpr int KC_IDS = 32;            // column ids cached per lane group (rows up to this length)
constexpr int KC_LONG_CAP = 1024;     // rows a warp takes instead of a lane group, listed in shared memory
constexpr double KC_MAX_GATHER_BYTES = 8e6;        // per hop: beyond this 148 SMs beat 16
constexpr int64_t KC_MAX_ROWS = 200000;
// Wider rows leave a warp too few edge slots (32/G) for its long rows: measured on the Cora-shaped graph, F=64 (G=16): 22 us
// per hop here against 18 for the K launches, F=7 (G=2): 5.8 against 17.3 (profiles/r02_small_graph_latency.txt).
constexpr int KC_MAX_LD = 16;

struct KhopCtaParams {
  const int64_t* rowptr;
  const int32_t* col;
  const float* val;
  const int32_t* row_order;
  int n, F, ld, K;
  int lgC;
  int cache_rows, cache_ids;   // the first row of every group / warp (and its column ids) is kept in shared memory
  const float* X0;
  int64_t ldx0;
  float* ping;
  float* pong;
  int64_t ldp;
  float* out;
  int64_t ldo;
  float* hops;
  int64_t ld_hops, hop_stride;
  rgbmp_epilogue_t ep;
};

struct KcRow {          // one row of the schedule: edge range + epilogue operands (nothing here depends on the iterate)
  int row;
  int k0, len;
  float rs, s2;
  float4 t;
  bool reset;
};

__device__ __forceinline__ float4 f4_zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ uint32_t kc_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// the iterate is written by other CTAs of the cluster between two barriers: read it from L2 (ld.global.cg)
__device__ __forceinline__ float4 kc_ld(const float* in, int64_t ldin, int c, int f) {
  return __ldcg(reinterpret_cast<const float4*>(in + (int64_t)c * ldin + f));
}
__device__ __forceinline__ void kc_st(float* o, int64_t ldo, int row, int f, float4 v) {
  if (o) __stcg(reinterpret_cast<float4*>(o + (int64_t)row * ldo + f), v);
}
__device__ __forceinline__ void kc_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

__device__ __forceinline__ void kc_operands(const KhopCtaParams& p, int row, int f, bool vact, KcRow& r) {
  const rgbmp_epilogue_t& ep = p.ep;
  if (ep.row_scale) r.rs = __ldg(ep.row_scale + row);
  if (ep.out2_scale) r.s2 = __ldg(ep.out2_scale + row);
  if (ep.T && vact) r.t = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ep.T) + (int64_t)row * ep.ldt + f));
  if (ep.reset_when != 0) r.reset = ep.reset_mask[row] != 0;
}

__device__ __forceinline__ void kc_fetch(const KhopCtaParams& p, int slot, int f, bool vact, KcRow& r) {
  r.row = -1;
  r.k0 = r.len = 0;
  r.rs = r.s2 = 1.f;
  r.t = f4_zero();
  r.reset = false;
  if (slot >= p.n) return;
  const int row = p.row_order ? __ldg(p.row_order + slot) : slot;
  r.row = row;
  const int64_t a = __ldg(p.rowptr + row);
  r.k0 = (int)a;
  r.len = (int)(__ldg(p.rowptr + row + 1) - a);
  kc_operands(p, row, f, vact, r);
}

// epilogue of rgbmp_epilogue_t (include/rgbmp.h) for the 4 features [f, f+4) of one row; returns what the next hop gathers
__device__ __forceinline__ float4 kc_epilogue(const KhopCtaParams& p, const KcRow& r, int f, float4 s, float* y, int64_t ldy) {
  const rgbmp_epilogue_t& ep = p.ep;
  float v[4] = {s.x, s.y, s.z, s.w};
  const float t[4] = {r.t.x, r.t.y, r.t.z, r.t.w};
  float rv[4] = {0.f, 0.f, 0.f, 0.f};
  if (r.reset) {
#pragma unroll
    for (int i = 0; i < 4; ++i) rv[i] = (f + i < p.F) ? ep.reset_val[(int64_t)r.row * ep.ld_reset + f + i] : 0.f;
  }
  ep_apply<4>(ep, v, r.rs, r.reset, rv, t);
  if (y) {
    float* q = y + (int64_t)r.row * ldy + f;
    if ((ldy & 3) == 0 && ((reinterpret_cast<uintptr_t>(y) & 15) == 0)) {
      *reinterpret_cast<float4*>(q) = make_float4(v[0], v[1], v[2], v[3]);      // padded rows: the pad is written too
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (f + i < p.F) q[i] = v[i];
    }
  }
  if (ep.out2_scale) {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = __fmul_rn(r.s2, v[i]);
  }
  return make_float4(v[0], v[1], v[2], v[3]);
}

template <bool HASW>
__device__ __forceinline__ void kc_acc(float4& a, const float4 x, float w) {
  if constexpr (HASW) {
    a.x = __fmaf_rn(w, x.x, a.x); a.y = __fmaf_rn(w, x.y, a.y); a.z = __fmaf_rn(w, x.z, a.z); a.w = __fmaf_rn(w, x.w, a.w);
  } else {
    a.x = __fadd_rn(a.x, x.x); a.y = __fadd_rn(a.y, x.y); a.z = __fadd_rn(a.z, x.z); a.w = __fadd_rn(a.w, x.w);
  }
}

// ids (and weights) of up to 4 edges ids[0], ids[stride], ...; slots whose offset reaches `left` hold id 0 / weight 0 and
// are never accumulated.  `ids` points into global memory or into the CTA's cached copy (generic loads).
template <bool HASW>
__device__ __forceinline__ void kc_batch(const int32_t* ids, const float* wts, int stride, int left, int (&c)[4], float (&w)[4]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    c[u] = 0;
    w[u] = 0.f;
    if (u * stride < left) {
      c[u] = ids[u * stride];
      if constexpr (HASW) w[u] = __ldg(wts + u * stride);
    }
  }
}

constexpr int KC_LIDS = 256;          // cached column ids of a warp's first long row

template <int G, bool HASW>
__global__ void __launch_bounds__(KC_THREADS, 1) khop_cluster_kernel(const KhopCtaParams p) {
  __shared__ int32_t long_list[KC_LONG_CAP];
  __shared__ int warp_tot[KC_THREADS / 32];
  __shared__ int n_long_s;
  const int n = p.n, ld = p.ld;
  const int C = 1 << p.lgC;
  const int rank = (int)kc_ctarank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NG = KC_THREADS / G;
  const int gl = tid % G, grp = tid / G;
  const int f = gl * 4;
  const bool vact = f < ld;

  // Rows above a length threshold go to a whole warp (32/G edge slots x 4 gathers in flight: up to 128/G edges per L2
  // round trip) instead of a lane group (4 edges per round trip): the longest chain of dependent round trips IS the hop
  // (ncu: 25 of 26 resident warps wait at the barrier for it).  The threshold is the smallest of 8, 16, ..., 256 that
  // leaves at most KC_LONG_CAP such rows.  Every CTA builds the same ascending list, so that the cluster's warps can
  // share it out by position: thread t scans a contiguous run of rows, block-wide exclusive scan, ordered write.
  __shared__ int over[6];                                 // rows longer than 8 << i
  if (tid < 6) over[tid] = 0;
  __syncthreads();
  const int run = (n + KC_THREADS - 1) / KC_THREADS;
  const int r_lo = min(n, tid * run), r_hi = min(n, r_lo + run);
  {
    int cnt[6] = {0, 0, 0, 0, 0, 0};
    for (int r = r_lo; r < r_hi; ++r) {
      const int len = (int)(p.rowptr[r + 1] - p.rowptr[r]);
#pragma unroll
      for (int i = 0; i < 6; ++i) cnt[i] += len > (8 << i);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i)
      if (cnt[i]) atomicAdd(&over[i], cnt[i]);
  }
  __syncthreads();
  int long_thr = 8 << 5;
#pragma unroll
  for (int i = 5; i >= 0; --i)
    if (over[i] <= KC_LONG_CAP) long_thr = 8 << i;
  int mine = 0;
  for (int r = r_lo; r < r_hi; ++r) mine += (int)(p.rowptr[r + 1] - p.rowptr[r]) > long_thr;
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  int base = 0;
  for (int w = 0; w < warp; ++w) base += warp_tot[w];
  if (tid == KC_THREADS - 1) n_long_s = base + incl;
  int at = base + incl - mine;
  for (int r = r_lo; r < r_hi; ++r) {
    if ((int)(p.rowptr[r + 1] - p.rowptr[r]) > long_thr) {
      if (at < KC_LONG_CAP) long_list[at] = r;
      ++at;
    }
  }
  __syncthreads();
  const int n_long = n_long_s;
  const bool split_long = n_long > 0 && n_long <= KC_LONG_CAP;   // otherwise every row is walked by its group

  const int gslot0 = grp * C + rank;                      // consecutive slots (similar degrees) go to different CTAs
  const int gstride = NG * C;
  // Every group walks the SAME rows in every hop, and the cluster barrier flushes L1: without a copy in shared memory
  // each hop pays the schedule -> rowptr -> column id chain of dependent L2 round trips again (3 of the 4 per row).
  extern __shared__ __align__(16) unsigned char kc_dyn[];
  int4* sm_row = reinterpret_cast<int4*>(kc_dyn);                               // [NG]  {row, k0, len, reset}
  float4* sm_T = reinterpret_cast<float4*>(sm_row + NG);                        // [1024] teleport vector of my lane
  int4* sl_row = reinterpret_cast<int4*>(sm_T + KC_THREADS);                    // [32]  first long row of each warp
  float4* sl_T = reinterpret_cast<float4*>(sl_row + KC_THREADS / 32);           // [1024]
  float2* sm_sc = reinterpret_cast<float2*>(sl_T + KC_THREADS);                 // [NG]  {row_scale, out2_scale}
  float2* sl_sc = sm_sc + NG;                                                   // [32]
  int32_t* sm_ids = reinterpret_cast<int32_t*>(sl_sc + KC_THREADS / 32);        // [NG][KC_IDS]
  int32_t* sl_ids = sm_ids + NG * KC_IDS;                                       // [32][KC_LIDS]
  const int li0 = warp * C + rank;                        // my warp's first long row
  if (p.cache_rows) {
    KcRow r;
    kc_fetch(p, gslot0, f, vact, r);
    if (gl == 0) {
      sm_row[grp] = make_int4(r.row, r.k0, r.len, r.reset ? 1 : 0);
      sm_sc[grp] = make_float2(r.rs, r.s2);
    }
    sm_T[tid] = r.t;
    if (p.cache_ids && r.row >= 0 && r.len <= KC_IDS)
      for (int j = gl; j < r.len; j += G) sm_ids[grp * KC_IDS + j] = __ldg(p.col + r.k0 + j);
    if (split_long && li0 < n_long) {
      const int lg = lane % G, fl = lg * 4;
      const int row = long_list[li0];
      KcRow q;
      q.row = row;
      q.k0 = (int)__ldg(p.rowptr + row);
      q.len = (int)(__ldg(p.rowptr + row + 1) - __ldg(p.rowptr + row));
      q.rs = q.s2 = 1.f;
      q.t = f4_zero();
      q.reset = false;
      kc_operands(p, row, fl, fl < ld, q);
      if (lane == 0) {
        sl_row[warp] = make_int4(q.row, q.k0, q.len, q.reset ? 1 : 0);
        sl_sc[warp] = make_float2(q.rs, q.s2);
      }
      sl_T[tid] = q.t;
      if (p.cache_ids && q.len <= KC_LIDS)
        for (int j = lane; j < q.len; j += 32) sl_ids[warp * KC_LIDS + j] = __ldg(p.col + q.k0 + j);
    }
    __syncthreads();
  }
  const float* in = p.X0;
  int64_t ldin = p.ldx0;
  for (int k = 0; k < p.K; ++k) {
    const bool last = (k == p.K - 1);
    float* y = nullptr;
    int64_t ldy = 0;
    if (p.hops) { y = p.hops + (int64_t)k * p.hop_stride; ldy = p.ld_hops; }
    if (last && !p.hops) { y = p.out; ldy = p.ldo; }
    float* nxt = last ? nullptr : ((k & 1) ? p.pong : p.ping);      // what the next hop gathers (pre-scaled when folded)
    // ---- long rows first: a warp each, 32/G edge slots x 4 gathers in flight, fixed-order reduction ----
    if (split_long) {
      constexpr int S = 32 / G;
      const int s = lane / G, lg = lane % G, fl = lg * 4;
      const bool va = fl < ld;
      for (int i = li0; i < n_long; i += (KC_THREADS / 32) * C) {
        KcRow r;
        const int32_t* ids;
        if (p.cache_rows && i == li0) {
          const int4 m = sl_row[warp];
          const float2 sc = sl_sc[warp];
          r.row = m.x; r.k0 = m.y; r.len = m.z; r.reset = m.w != 0;
          r.rs = sc.x; r.s2 = sc.y;
          r.t = sl_T[tid];
          ids = (p.cache_ids && r.len <= KC_LIDS) ? sl_ids + warp * KC_LIDS : p.col + r.k0;
        } else {
          r.row = long_list[i];
          r.k0 = (int)__ldg(p.rowptr + r.row);
          r.len = (int)(__ldg(p.rowptr + r.row + 1) - __ldg(p.rowptr + r.row));
          r.rs = r.s2 = 1.f;
          r.t = f4_zero();
          r.reset = false;
          if (s == 0) kc_operands(p, r.row, fl, va, r);   // travel while the row is summed
          ids = p.col + r.k0;
        }
        const int row = r.row, k0 = r.k0, len = r.len;
        float4 acc = f4_zero();
        if (va) {
          for (int j = s; j < len; j += 4 * S) {
            int c[4];
            float w[4];
            kc_batch<HASW>(ids + j, p.val + k0 + j, S, len - j, c, w);
            float4 x[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) x[u] = kc_ld(in, ldin, c[u], fl);     // id 0: a valid row
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (u * S < len - j) kc_acc<HASW>(acc, x[u], HASW ? w[u] : 1.f);
          }
        }
#pragma unroll
        for (int o = G; o < 32; o <<= 1) {
          acc.x = __fadd_rn(acc.x, __shfl_xor_sync(0xffffffffu, acc.x, o));
          acc.y = __fadd_rn(acc.y, __shfl_xor_sync(0xffffffffu, acc.y, o));
          acc.z = __fadd_rn(acc.z, __shfl_xor_sync(0xffffffffu, acc.z, o));
          acc.w = __fadd_rn(acc.w, __shfl_xor_sync(0xffffffffu, acc.w, o));
        }
        if (s == 0 && va) kc_st(nxt, p.ldp, row, fl, kc_epilogue(p, r, fl, acc, y, ldy));
      }
    }
    // ---- rows walked by their lane group ----
    KcRow nx;
    if (p.cache_rows) {
      const int4 m = sm_row[grp];
      const float2 sc = sm_sc[grp];
      nx.row = m.x; nx.k0 = m.y; nx.len = m.z; nx.reset = m.w != 0;
      nx.rs = sc.x; nx.s2 = sc.y;
      nx.t = sm_T[tid];
    } else {
      kc_fetch(p, gslot0, f, vact, nx);
    }
    for (int slot = gslot0; slot < n; slot += gstride) {
      const KcRow r = nx;
      kc_fetch(p, slot + gstride, f, vact, nx);           // the next row's operands travel while this row is summed
      if (split_long && r.len > long_thr) continue;
      if (vact) {
        const int32_t* ids = (p.cache_rows && p.cache_ids && slot == gslot0 && r.len <= KC_IDS) ? sm_ids + grp * KC_IDS : p.col + r.k0;
        const float* wts = p.val + r.k0;
        float4 acc = f4_zero();
        int cn[4];
        float wn[4];
        kc_batch<HASW>(ids, wts, 1, r.len, cn, wn);
        for (int j = 0; j < r.len; j += 4) {
          int c[4];
          float w[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) { c[u] = cn[u]; w[u] = wn[u]; }
          const int left = r.len - j;
          kc_batch<HASW>(ids + j + 4, wts + j + 4, 1, left - 4, cn, wn);               // next batch's ids before this batch's rows
          float4 x[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) x[u] = kc_ld(in, ldin, c[u], f);
#pragma unroll
          for (int u = 0; u < 4; ++u)
            if (u < left) kc_acc<HASW>(acc, x[u], HASW ? w[u] : 1.f);
        }
        kc_st(nxt, p.ldp, r.row, f, kc_epilogue(p, r, f, acc, y, ldy));
      }
    }
    if (!last || (p.hops && p.out)) kc_cluster_sync();    // every row of the new iterate is visible to the whole cluster
    in = nxt;
    ldin = p.ldp;
  }
  // final iterate also requested in `out` next to the per-hop outputs: the un-scaled copy went to hops[K-1]
  if (p.hops && p.out) {
    const float* lastp = p.hops + (int64_t)(p.K - 1) * p.hop_stride;
    for (int t = rank * KC_THREADS + tid; t < n * p.F; t += KC_THREADS * C) {
      const int r = t / p.F, c = t - r * p.F;
      p.out[(int64_t)r * p.ldo + c] = __ldcg(lastp + (int64_t)r * p.ld_hops + c);
    }
  }
}

static int kc_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RGBMP_KHOP_CTA");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v;
}
static int g_kc_override = -1;
static long long g_kc_calls = 0;      // calls taken by this path (tests / tools check that it ran)
static int g_kc_lgC[64];              // per device: log2 of the largest cluster this kernel was placed with (0 = unknown)

template <typename Kern>
static int kc_launch_one(Kern kern, const KhopCtaParams& p0, int G, cudaStream_t st, int device) {
  RGBMP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  // shared-memory copy of every group's / warp's first row: descriptors + teleport vectors always, column ids when they fit
  const size_t NG = KC_THREADS / G;
  const size_t base_bytes = NG * 16 + KC_THREADS * 16 + (KC_THREADS / 32) * 16 + KC_THREADS * 16 + NG * 8 + (KC_THREADS / 32) * 8;
  const size_t ids_bytes = (NG * KC_IDS + (KC_THREADS / 32) * KC_LIDS) * sizeof(int32_t);
  size_t smem = base_bytes + ids_bytes;
  RGBMP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  for (int lgC = (device >= 0 && device < 64 && g_kc_lgC[device] > 0) ? g_kc_lgC[device] : 4; lgC >= 3; --lgC) {
    KhopCtaParams p = p0;
    const int C = 1 << lgC;
    p.lgC = lgC;
    p.cache_rows = 1;
    p.cache_ids = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(C);
    cfg.blockDim = dim3(KC_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, p);
    if (e == cudaSuccess) {
      if (device >= 0 && device < 64) g_kc_lgC[device] = lgC;
      return 0;
    }
    cudaGetLastError();                                  // a 16-CTA cluster may not be placeable: try 8
    if (lgC == 3) return cuda_fail(e, "khop_cluster_kernel");
  }
  return fail(RGBMP_EINVAL, "khop_cluster: unreachable");
}

template <int G>
static int kc_launch(const KhopCtaParams& p, cudaStream_t st, int device) {
  return p.val ? kc_launch_one(khop_cluster_kernel<G, true>, p, G, st, device)
               : kc_launch_one(khop_cluster_kernel<G, false>, p, G, st, device);
}

// *handled = 1 when the call was taken (return value = its status), 0 = not eligible: the caller runs the K-launch path.
// ep passed check_epilogue with EP_KHOP.  Eligible: fp32, 16-byte aligned padded rows everywhere, at most
// KC_MAX_GATHER_BYTES gathered per hop and KC_MAX_ROWS rows, rows of at most 4 vectors (KC_MAX_LD), K >= 2, no row map,
// no hot tags.
int khop_cta_try(const rgbmp_graph_t* g, const float* val, const void* X0, int64_t ldx0, void* ping, void* pong, int64_t ldp,
                 void* out, int64_t ldo, void* hops, int64_t ld_hops, int64_t hop_stride, int F, int dtype, int K,
                 const rgbmp_epilogue_t& ep, cudaStream_t st, int device, int* handled) {
  *handled = 0;
  const int on = g_kc_override >= 0 ? g_kc_override : kc_enabled();
  if (!on || dtype != RGBMP_F32 || g->col_tagged || g->n_rows < 1 || g->n_rows > KC_MAX_ROWS || g->nnz >= (1ll << 30)) return 0;
  if (ep.row_map) return 0;
  const int ld = (int)align_up((size_t)F, 4);
  if (ld > KC_MAX_LD || K < 2) return 0;
  if ((double)g->nnz * ld * 4.0 > KC_MAX_GATHER_BYTES) return 0;
  auto rows_ok = [&](const void* q, int64_t l) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0 && (l & 3) == 0 && l >= ld; };
  if (!rows_ok(X0, ldx0)) return 0;
  if (ep.T && !rows_ok(ep.T, ep.ldt)) return 0;
  if (K > 1 && (!ping || !pong || !rows_ok(ping, ldp) || !rows_ok(pong, ldp))) return 0;
  KhopCtaParams p;
  p.rowptr = g->rowptr;
  p.col = g->col;
  p.val = val;
  p.row_order = g->row_order;
  p.n = (int)g->n_rows;
  p.F = F;
  p.ld = ld;
  p.K = K;
  p.lgC = 0;
  p.X0 = (const float*)X0;
  p.ldx0 = ldx0;
  p.ping = (float*)ping;
  p.pong = (float*)pong;
  p.ldp = ldp;
  p.out = (float*)out;
  p.ldo = ldo;
  p.hops = (float*)hops;
  p.ld_hops = ld_hops;
  p.hop_stride = hop_stride;
  p.ep = ep;
  const int nvec = ld / 4;
  const int rc = nvec <= 1 ? kc_launch<1>(p, st, device) : (nvec <= 2 ? kc_launch<2>(p, st, device) : kc_launch<4>(p, st, device));
  if (rc != 0) {               // no 8-CTA cluster can be placed on this device / partition: leave the path off for good
    g_kc_override = 0;
    return 0;                  // not handled: the caller runs the K-launch path
  }
  *handled = 1;
  ++g_kc_calls;
  return 0;
}

}  // namespace rgbmp

extern "C" int rgbmp_set_khop_cta(int on) {
  const int old = rgbmp::g_kc_override >= 0 ? rgbmp::g_kc_override : rgbmp::kc_enabled();
  if (on == 0 || on == 1) rgbmp::g_kc_override = on;
  return old;
}
extern "C" long long rgbmp_khop_cta_calls(void) { return rgbmp::g_kc_calls; }
