// Fused edge-score attention + aggregate over CSR, forward and backward (sm_100a).
//
// ONE kernel family for the layers of the reference whose per-edge weight is a function of the two endpoints
// (SURVEY.md 8a rows a4, a5, a9), selected by the template parameter SC:
//   SC_GAT  GATConv (gat.py:18-21, A10):       e = leaky_relu(a_src[j] + a_dst[i]);                 softmax over i's in-edges
//   SC_MX   SuperGATConv MX (supergat.py:15-21, A12): e = leaky_relu((a_l[j] + a_r[i]) * sigmoid(<x_i, x_j>)); softmax
//   SC_SD   SuperGATConv SD (A12):             e = leaky_relu(logit_scale * <x_i, x_j>), logit_scale = 1/sqrt(C); softmax
//   SC_FA   FAConv (fagcn.py:15,31, A13):      w = tanh(a_l[j] + a_r[i]) * dinv[j] * dinv[i];        no softmax, H = 1
// out[i] = sum_j weight_ij * mask_ij * X[j].  No edge-sized tensor is ever written: the forward is one pass with
// an online softmax, the backward recomputes the weights from per-node statistics (A10 identities).
//
// Gather / segment-reduce: L2/HBM-bound by bytes and, for L2-resident X, issue-bound -- so the work per edge is
// kept in as few instructions as possible:
//   * a group of G lanes owns a row, a lane owns 8 consecutive channels (two float4) that never straddle a head:
//     the score work (exp, sigmoid, tanh) is shared by 8 channels, the per-head dot products of MX and of the
//     backward need log2(C/8) shuffles (none for C = 8);
//   * heads are independent, so wide layers (H*C > 128) are tiled over blockIdx.y in groups of HT heads;
//   * logits live in the log2 domain (a_src/a_dst pre-multiplied by log2 e; leaky_relu and the product with
//     sigmoid > 0 commute with a positive scale), exp is a bare ex2.approx;
//   * SpMM's row-split schedule (csr_work.cuh): degree/locality row schedule, one coalesced load of G column ids per
//     batch broadcast through shared memory, rows longer than `chunk` split into CTA work items whose partial
//     (max, sum, acc) states are merged in item order; software-pipelined full batches (forward).
// DETERMINISTIC, no atomics anywhere.  The gradient of the per-TARGET score term (da_dst / da_r) is a sum over a
// target's in-edges while the backward walks the transpose CSR; instead of atomics it uses linearity:
//   GAT:  da_dst[i] = sum_j alpha_ij l'_ij (mask_ij <dout_i, x_j> - S_i) = <dout_i, P_i> - S_i q_i
//         with P_i = sum_j alpha_ij l'_ij mask_ij x_j and q_i = sum_j alpha_ij l'_ij -- a SECOND aggregate the
//         training-mode forward accumulates next to out_i (l' = leaky_relu' in {1, slope}, known per edge);
//   FA:   da_r[i] = <dout_i, Q_i>,  Q_i = sum_j (1 - tanh^2) dinv_j dinv_i mask_ij x_j, likewise;
//   MX:   the logit <x_i, x_j> sends gradient to BOTH endpoints' features, so its backward runs one pass per
//         orientation anyway (forward CSR: dX_i += dlogit x_j, da_r; transpose CSR: dX_j += alpha dout_i + dlogit x_i, da_l).
//   SD:   MX without the score scalars and the sigmoid gate: the same two passes, no da_l / da_r.
#include <math.h>
#include <stdlib.h>
#include <type_traits>
#include "csr_work.cuh"
#include "philox.cuh"

namespace rgbmp {

constexpr unsigned FULLMASK = 0xffffffffu;
constexpr int ATT_THREADS = 256;
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;
constexpr int U = 2;       // edges per step
enum { SC_GAT = RGBMP_ATT_GAT, SC_MX = RGBMP_ATT_MX, SC_FA = RGBMP_ATT_FA, SC_SD = RGBMP_ATT_SD };

__device__ __forceinline__ float leaky_relu(float x, float slope) { return x > 0.f ? x : x * slope; }
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// sigmoid of a NATURAL-domain argument
__device__ __forceinline__ float sigmoidf(float x) { return rcp(1.0f + ex2(-x * LOG2E)); }
// packed fp32x2 FMA of sm_100 (one issue slot per two channels)
__device__ __forceinline__ void fma4(float4& a, float w, const float4& x) {
  unsigned long long lo, hi, wl;
  const float2 ww = make_float2(w, w);
  wl = reinterpret_cast<const unsigned long long&>(ww);
  float2 a0 = make_float2(a.x, a.y), a1 = make_float2(a.z, a.w), x0 = make_float2(x.x, x.y), x1 = make_float2(x.z, x.w);
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(lo) : "l"(wl), "l"(reinterpret_cast<unsigned long long&>(x0)), "l"(reinterpret_cast<unsigned long long&>(a0)));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(hi) : "l"(wl), "l"(reinterpret_cast<unsigned long long&>(x1)), "l"(reinterpret_cast<unsigned long long&>(a1)));
  const float2 r0 = reinterpret_cast<float2&>(lo), r1 = reinterpret_cast<float2&>(hi);
  a = make_float4(r0.x, r0.y, r1.x, r1.y);
}
__device__ __forceinline__ void scale4(float4& a, float w) { a.x *= w; a.y *= w; a.z *= w; a.w *= w; }
__device__ __forceinline__ float dot4(const float4& a, const float4& b) {
  return fmaf(a.x, b.x, fmaf(a.y, b.y, fmaf(a.z, b.z, a.w * b.w)));
}
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }

struct AttParams {
  CsrWork w;                          // the graph in the orientation of this pass
  // geometry: H heads of C channels, HT heads per blockIdx.y tile, LPH lanes per head
  int H, HT, C, LPH;
  float slope;
  // gathered (neighbour) operands
  const float* Xn;  int64_t ldn;      // feature row gathered per edge (fwd / bwd-F: x_j ; bwd-T: dout_i)
  const float* Xn2; int64_t ldn2;     // second gathered row (MX bwd-T: x_i)
  const float* sn;                    // [*,H] per-neighbour scalar (fwd / bwd-F: a_src scaled)
  const float4* stats;                // [n_dst,H] per-target statistics (bwd-T: gathered; bwd-F: own row)
  const float* dinv;                  // FA: deg^-1/2, indexed by both endpoints
  // own-row operands
  const float* Xo;  int64_t ldo_;     // own features (MX fwd / bwd-F: x_i ; bwd-T: x_j)
  const float* Do;  int64_t lddo;     // own dout (MX bwd-F)
  const float* so;                    // [*,H] own scalar (fwd: a_dst scaled ; bwd-T: a_src unscaled)
  // attention dropout: keep-mask / (1-p) in forward-CSR order [nnz,H]; tpos maps transpose entries to it
  const float* drop;
  const int32_t* tpos;
  // fused attention dropout (the DR instantiations): multiplier of entry k = dropout_mult(seed, eid[k], head),
  // eid = edge id of every entry of THIS pass's CSR (forward CSR or transpose CSR), read as a stream
  const int64_t* seed;
  const int32_t* eid;
  uint32_t thresh;
  float dscale;
  // outputs
  float* out;  int64_t ldo;           // fwd: out ; bwd: dX of the own row
  float* out2; int64_t ldo2;          // fwd TRAIN: second aggregate (P / Q)
  float* rowmax; float* rowsum; float* rowq;   // fwd: [n_rows,H]
  float* ds;                          // bwd: gradient of the own row's score scalar [n_rows,H]
  const float* acc_in; int64_t ld_acc;         // bwd-T: partial dX added in the epilogue (MX pass F result)
  // long-row scratch
  float* part_m; float* part_s; float* part_q; float* part_acc; float* part_acc2;
  int64_t ldp;
  // SD: natural-domain scale of the logit <x_i, x_j> (1/sqrt(C) of the UNPADDED head width); last, so that the
  // parameter offsets of the other variants do not move
  float logit_scale;
};

// ---------------------------------------------------------------------------------------------
// lane geometry
// ---------------------------------------------------------------------------------------------
struct Lane {
  int f;        // first channel (absolute, within the H*C row) of this lane's 8
  int h;        // absolute head of this lane (0 when H == 1)
  int nact;     // number of existing float4 vectors of this lane (0, 1 or 2)
  bool lead;    // first lane of its head (writes the per-head scalars)
};

__device__ __forceinline__ Lane lane_of(const AttParams& p, int gl) {
  Lane L;
  const int tile = blockIdx.y;
  int width, base;            // channels of this tile, first channel of this tile
  if (p.H == 1) { width = (p.C + 3) & ~3; base = 0; }
  else {
    const int h0 = tile * p.HT;
    const int ht = min(p.HT, p.H - h0);
    width = ht * p.C;
    base = h0 * p.C;
  }
  const int fl = gl * 8;
  L.nact = (fl < width ? 1 : 0) + (fl + 4 < width ? 1 : 0);
  L.f = base + (L.nact ? fl : 0);
  L.h = (p.H == 1) ? 0 : L.f / p.C;
  L.lead = L.nact > 0 && (p.H == 1 ? gl == 0 : (L.f % p.C) == 0);
  return L;
}

// the key is built once per thread from the device-resident seed; the hash runs per (entry, head)
template <bool DR>
__device__ __forceinline__ PhiloxKey drop_key(const AttParams& p) {
  if constexpr (DR) return philox_key((uint64_t)__ldg(p.seed));
  else return PhiloxKey{0u, 0u};
}
__device__ __forceinline__ float drop_mult(const AttParams& p, PhiloxKey key, int64_t k, int h) {
  return dropout_mult(key, (uint32_t)__ldg(p.eid + k), (uint32_t)h, p.thresh, p.dscale);
}

// sum over the LPH lanes of a head (all lanes of the warp execute)
__device__ __forceinline__ float head_sum(float v, int LPH) {
  for (int o = LPH >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(FULLMASK, v, o);
  return v;
}

// SD's raw score in the log2 domain; forward and both backward passes round it the same way
__device__ __forceinline__ float sd_raw(const AttParams& p, float logit) { return logit * (p.logit_scale * LOG2E); }

__device__ __forceinline__ void load_own(const float* X, int64_t ld, int64_t row, const Lane& L, float4 (&x)[2]) {
  x[0] = L.nact > 0 ? __ldg(reinterpret_cast<const float4*>(X + row * ld + L.f)) : zero4();
  x[1] = L.nact > 1 ? __ldg(reinterpret_cast<const float4*>(X + row * ld + L.f + 4)) : zero4();
}

// =============================================================================================
// forward
// =============================================================================================
struct FwdState {
  float m, s, q;            // running max (log2 domain), running sum, running sum of alpha*l'
  float4 acc[2], acc2[2];
};

template <int SC, bool TRAIN, int UU, bool DR>
__device__ __forceinline__ void fwd_consume(const AttParams& p, const float4 (&x)[UU][2], const float (&sn)[UU], const float (&dn)[UU],
                                            int nvalid, int64_t kbase, const Lane& L, float so, float d_own,
                                            const float4 (&xi)[2], PhiloxKey key, FwdState& st) {
  if constexpr (SC == SC_FA) {
#pragma unroll
    for (int u = 0; u < UU; ++u) {
      if (u < nvalid) {
        const float t = tanhf(sn[u] + so);
        float wgt = dn[u] * d_own;
        if constexpr (DR) wgt *= drop_mult(p, key, kbase + u, 0);
        else if (p.drop) wgt *= __ldg(p.drop + (kbase + u));
        const float w = t * wgt;
        fma4(st.acc[0], w, x[u][0]);
        fma4(st.acc[1], w, x[u][1]);
        if constexpr (TRAIN) {
          const float w2 = (1.0f - t * t) * wgt;
          fma4(st.acc2[0], w2, x[u][0]);
          fma4(st.acc2[1], w2, x[u][1]);
        }
      }
    }
  } else {
    float e[UU];
    float mb = -INFINITY;
#pragma unroll
    for (int u = 0; u < UU; ++u) {
      float raw;
      if constexpr (SC == SC_SD) {
        raw = sd_raw(p, head_sum(dot4(xi[0], x[u][0]) + dot4(xi[1], x[u][1]), p.LPH));
      } else {
        raw = sn[u] + so;                                   // log2 domain (both terms pre-scaled)
        if constexpr (SC == SC_MX) {
          const float dot = head_sum(dot4(xi[0], x[u][0]) + dot4(xi[1], x[u][1]), p.LPH);
          raw *= sigmoidf(dot);
        }
      }
      e[u] = leaky_relu(raw, p.slope);
      if (u < nvalid) mb = fmaxf(mb, e[u]);
    }
    if (mb > st.m) {                                        // rare after the first batches of a row
      const float sc = ex2(st.m - mb);                      // m = -inf on the first batch: ex2(-inf) = 0
      st.s *= sc;
      scale4(st.acc[0], sc);
      scale4(st.acc[1], sc);
      if constexpr (TRAIN) {
        st.q *= sc;
        scale4(st.acc2[0], sc);
        scale4(st.acc2[1], sc);
      }
      st.m = mb;
    }
#pragma unroll
    for (int u = 0; u < UU; ++u) {
      if (u < nvalid) {
        const float pe = ex2(e[u] - st.m);
        st.s += pe;
        float mu;
        if constexpr (DR) mu = drop_mult(p, key, kbase + u, L.h);
        else mu = p.drop ? __ldg(p.drop + (kbase + u) * p.H + L.h) : 1.0f;
        const float w = pe * mu;
        fma4(st.acc[0], w, x[u][0]);
        fma4(st.acc[1], w, x[u][1]);
        if constexpr (TRAIN) {
          const float pl = e[u] > 0.f ? pe : pe * p.slope;  // alpha * leaky_relu'
          st.q += pl;
          const float w2 = pl * mu;
          fma4(st.acc2[0], w2, x[u][0]);
          fma4(st.acc2[1], w2, x[u][1]);
        }
      }
    }
  }
}

// UU edges per step; PIPE: software-pipelined full batches (the gathers of step j+UU fly while step j is consumed)
template <int SC, bool TRAIN, int G, int UU, bool PIPE, bool DR>
__device__ __forceinline__ void fwd_range(const AttParams& p, int64_t k0, int64_t k1, int gl, const Lane& L, float so,
                                          float d_own, const float4 (&xi)[2], PhiloxKey key, int32_t* sm_ids, FwdState& st) {
  const int len = (k1 > k0) ? (int)(k1 - k0) : 0;
  const int maxlen = __reduce_max_sync(FULLMASK, len);
  if (maxlen == 0) return;
  const int32_t* __restrict__ col = p.w.col + k0;
  const char* xb0 = reinterpret_cast<const char*>(p.Xn + L.f);
  const char* xb1 = reinterpret_cast<const char*>(p.Xn + L.f + 4);
  const bool a0 = L.nact > 0, a1 = L.nact > 1;             // lanes beyond the row issue no feature load
  const uint32_t row_bytes = (uint32_t)(p.ldn * 4);
  const char* snb = reinterpret_cast<const char*>(p.sn + L.h);
  const uint32_t sn_bytes = (uint32_t)(p.H * 4);
  auto gather = [&](uint32_t c, float4 (&xx)[2], float& aa, float& dd) {
    xx[0] = a0 ? __ldg(reinterpret_cast<const float4*>(xb0 + (size_t)c * row_bytes)) : zero4();
    xx[1] = a1 ? __ldg(reinterpret_cast<const float4*>(xb1 + (size_t)c * row_bytes)) : zero4();
    if constexpr (SC == SC_SD) aa = 0.f;                    // SD has no per-neighbour scalar
    else aa = __ldg(reinterpret_cast<const float*>(snb + (size_t)c * sn_bytes));
    if constexpr (SC == SC_FA) dd = __ldg(p.dinv + c);
    else dd = 0.f;
  };
  const int lane = threadIdx.x & 31;
  int32_t* wids = sm_ids + (threadIdx.x & ~31);            // this warp's 32 slots
  const int32_t* gids = wids + (lane - gl);                // this group's G slots
  int32_t cn = (gl < len) ? __ldcs(col + gl) : 0;          // lanes past the row hold id 0: a valid row
  for (int off = 0; off < maxlen; off += G) {
    int nb = len - off;
    nb = nb < 0 ? 0 : (nb > G ? G : nb);
    __syncwarp();
    wids[lane] = cn;
    __syncwarp();
    cn = 0;
    if (off + G + gl < len) cn = __ldcs(col + off + G + gl);
    if (G >= 2 * UU && __all_sync(FULLMASK, nb == G)) {
      if constexpr (PIPE) {
        float4 x[UU][2];
        float as[UU], dn[UU];
        {
          uint32_t c[UU];
          lds_ids<UU>(gids, c);
#pragma unroll
          for (int u = 0; u < UU; ++u) gather(c[u], x[u], as[u], dn[u]);
        }
#pragma unroll 1
        for (int j = 0; j < G; j += UU) {
          float4 xn[UU][2];
          float asn[UU], dnn[UU];
          const int jn = (j + UU < G) ? j + UU : j;          // last step re-requests itself (L1 hit, unused)
          uint32_t c[UU];
          lds_ids<UU>(gids + jn, c);
#pragma unroll
          for (int u = 0; u < UU; ++u) gather(c[u], xn[u], asn[u], dnn[u]);
          fwd_consume<SC, TRAIN, UU, DR>(p, x, as, dn, UU, k0 + off + j, L, so, d_own, xi, key, st);
#pragma unroll
          for (int u = 0; u < UU; ++u) {
            as[u] = asn[u];
            dn[u] = dnn[u];
            x[u][0] = xn[u][0];
            x[u][1] = xn[u][1];
          }
        }
      } else {
#pragma unroll 1
        for (int j = 0; j < G; j += UU) {
          float4 x[UU][2];
          float as[UU], dn[UU];
          uint32_t c[UU];
          lds_ids<UU>(gids + j, c);
#pragma unroll
          for (int u = 0; u < UU; ++u) gather(c[u], x[u], as[u], dn[u]);
          fwd_consume<SC, TRAIN, UU, DR>(p, x, as, dn, UU, k0 + off + j, L, so, d_own, xi, key, st);
        }
      }
    } else {
      const int nbmax = __reduce_max_sync(FULLMASK, nb);
#pragma unroll 1
      for (int j = 0; j < nbmax; j += UU) {
        float4 x[UU][2];
        float as[UU], dn[UU];
        uint32_t c[UU];
        lds_ids<UU>(gids + (j & (G - 1)), c);
#pragma unroll
        for (int u = 0; u < UU; ++u) gather(c[u], x[u], as[u], dn[u]);
        int nv = nb - j;
        nv = nv < 0 ? 0 : (nv > UU ? UU : nv);
        fwd_consume<SC, TRAIN, UU, DR>(p, x, as, dn, nv, k0 + off + j, L, so, d_own, xi, key, st);
      }
    }
  }
}

// RGBMP_ATT_OCC (compile-time A/B of the resident-CTA targets, tools/build_variant.py; profiles/r02_att_occupancy.txt):
// 0 = round-2 first cut; 1 (default) = one more CTA per SM for the backward kernels (GAT fwd+bwd 6.59 -> 6.20 ms,
// SuperGAT-MX 14.6 -> 12.2 on the Reddit-shaped layer; 12-20 bytes of spill) and for the MX eval forward (3.32 -> 3.09);
// 2 = 4 CTAs/SM for every forward variant too (the training forms spill 100-200 bytes: 2-layer GAT epoch 24.7 -> 26.1).
#ifndef RGBMP_ATT_OCC
#define RGBMP_ATT_OCC 1
#endif
template <int SC, bool TRAIN>
constexpr int fwd_minb() { return RGBMP_ATT_OCC >= 2 ? 4 : (RGBMP_ATT_OCC == 1 ? (TRAIN ? 3 : 4) : ((TRAIN || SC == SC_MX) ? 3 : 4)); }

__device__ __forceinline__ void fwd_init(FwdState& st) {
  st.m = -INFINITY;
  st.s = st.q = 0.f;
  st.acc[0] = st.acc[1] = st.acc2[0] = st.acc2[1] = zero4();
}

template <int SC, bool TRAIN, int G, int UU, bool PIPE, bool DR>
__global__ void __launch_bounds__(ATT_THREADS, fwd_minb<SC, TRAIN>()) att_fwd_rows_kernel(const AttParams p) {
  __shared__ __align__(16) int32_t sm_ids[ATT_THREADS];
  const int gl = threadIdx.x % G;
  int64_t row, k0, k1;
  const bool live = short_row<G, ATT_THREADS>(p.w, row, k0, k1);
  const Lane L = lane_of(p, gl);
  float so = 0.f, d_own = 0.f;
  float4 xi[2] = {zero4(), zero4()};
  if (live) {
    if constexpr (SC != SC_SD) so = __ldg(p.so + row * p.H + L.h);
    if constexpr (SC == SC_FA) d_own = __ldg(p.dinv + row);
    if constexpr (SC == SC_MX || SC == SC_SD) load_own(p.Xo, p.ldo_, row, L, xi);
  }
  FwdState st;
  fwd_init(st);
  fwd_range<SC, TRAIN, G, UU, PIPE, DR>(p, k0, k1, gl, L, so, d_own, xi, drop_key<DR>(p), sm_ids, st);
  if (!live || L.nact == 0) return;
  float inv = 1.0f;
  if constexpr (SC != SC_FA) inv = (k1 > k0) ? 1.0f / (st.s + 1e-16f) : 0.f;
#pragma unroll
  for (int v = 0; v < 2; ++v) {
    if (v < L.nact) {
      scale4(st.acc[v], inv);
      __stcs(reinterpret_cast<float4*>(p.out + row * p.ldo + L.f + 4 * v), st.acc[v]);
      if constexpr (TRAIN) {
        scale4(st.acc2[v], inv);
        __stcs(reinterpret_cast<float4*>(p.out2 + row * p.ldo2 + L.f + 4 * v), st.acc2[v]);
      }
    }
  }
  if constexpr (SC != SC_FA) {
    if (L.lead) {
      p.rowsum[row * p.H + L.h] = st.s;
      p.rowmax[row * p.H + L.h] = (k1 > k0) ? st.m * LN2 : 0.f;
      if constexpr (TRAIN) p.rowq[row * p.H + L.h] = st.q * inv;
    }
  }
}

// long rows: one CTA per (work item, head tile); the CTA's Q groups take contiguous sub-ranges, their states
// are merged through shared memory in group order
template <int SC, bool TRAIN, int G, int UU, bool PIPE, bool DR>
__global__ void __launch_bounds__(ATT_THREADS, fwd_minb<SC, TRAIN>()) att_fwd_long_kernel(const AttParams p) {
  constexpr int Q = ATT_THREADS / G;
  constexpr int W = G * 8;
  __shared__ __align__(16) int32_t sm_ids[ATT_THREADS];
  __shared__ float sm_acc[Q * W];
  __shared__ float sm_acc2[TRAIN ? Q * W : 1];
  __shared__ float sm_m[Q][G], sm_s[Q][G], sm_q[Q][G];      // heads per tile <= lanes per group
  const int gl = threadIdx.x % G, q = threadIdx.x / G;
  int64_t row, k0, k1;
  long_item<G, ATT_THREADS>(p.w, row, k0, k1);
  const Lane L = lane_of(p, gl);
  const float so = (SC == SC_SD) ? 0.f : __ldg(p.so + row * p.H + L.h);
  float d_own = 0.f;
  float4 xi[2] = {zero4(), zero4()};
  if constexpr (SC == SC_FA) d_own = __ldg(p.dinv + row);
  if constexpr (SC == SC_MX || SC == SC_SD) load_own(p.Xo, p.ldo_, row, L, xi);
  FwdState st;
  fwd_init(st);
  fwd_range<SC, TRAIN, G, UU, PIPE, DR>(p, k0, k1, gl, L, so, d_own, xi, drop_key<DR>(p), sm_ids, st);
#pragma unroll
  for (int v = 0; v < 2; ++v) {
    const bool act = v < L.nact;
    float* d = sm_acc + q * W + gl * 8 + 4 * v;
    d[0] = act ? st.acc[v].x : 0.f; d[1] = act ? st.acc[v].y : 0.f; d[2] = act ? st.acc[v].z : 0.f; d[3] = act ? st.acc[v].w : 0.f;
    if constexpr (TRAIN) {
      float* d2 = sm_acc2 + q * W + gl * 8 + 4 * v;
      d2[0] = act ? st.acc2[v].x : 0.f; d2[1] = act ? st.acc2[v].y : 0.f; d2[2] = act ? st.acc2[v].z : 0.f; d2[3] = act ? st.acc2[v].w : 0.f;
    }
  }
  const int hl = (p.H == 1) ? 0 : L.h - blockIdx.y * p.HT;  // head index inside the tile
  if (L.lead) {
    sm_m[q][hl] = st.m;
    sm_s[q][hl] = st.s;
    sm_q[q][hl] = st.q;
  }
  __syncthreads();
  const int64_t item = blockIdx.x;
  const int h0 = (p.H == 1) ? 0 : blockIdx.y * p.HT;
  const int ht = (p.H == 1) ? 1 : min(p.HT, p.H - h0);
  const int width = (p.H == 1) ? p.C : ht * p.C;
  const int base = h0 * p.C;
  for (int t = threadIdx.x; t < width; t += ATT_THREADS) {
    const int hh = (p.H == 1) ? 0 : t / p.C;
    float a = 0.f, a2 = 0.f;
    if constexpr (SC == SC_FA) {
      for (int qq = 0; qq < Q; ++qq) {
        a += sm_acc[qq * W + t];
        if constexpr (TRAIN) a2 += sm_acc2[qq * W + t];
      }
    } else {
      float M = -INFINITY;
      for (int qq = 0; qq < Q; ++qq) M = fmaxf(M, sm_m[qq][hh]);
      for (int qq = 0; qq < Q; ++qq) {
        const float mq = sm_m[qq][hh];
        if (mq > -INFINITY) {
          const float sc = ex2(mq - M);
          a = fmaf(sm_acc[qq * W + t], sc, a);
          if constexpr (TRAIN) a2 = fmaf(sm_acc2[qq * W + t], sc, a2);
        }
      }
    }
    p.part_acc[item * p.ldp + base + t] = a;
    if constexpr (TRAIN) p.part_acc2[item * p.ldp + base + t] = a2;
  }
  if constexpr (SC != SC_FA) {
    if (threadIdx.x < ht) {
      const int hh = threadIdx.x;
      float M = -INFINITY;
      for (int qq = 0; qq < Q; ++qq) M = fmaxf(M, sm_m[qq][hh]);
      float s = 0.f, qv = 0.f;
      for (int qq = 0; qq < Q; ++qq) {
        const float mq = sm_m[qq][hh];
        if (mq > -INFINITY) {
          const float sc = ex2(mq - M);
          s = fmaf(sm_s[qq][hh], sc, s);
          qv = fmaf(sm_q[qq][hh], sc, qv);
        }
      }
      p.part_m[item * p.H + h0 + hh] = M;
      p.part_s[item * p.H + h0 + hh] = s;
      p.part_q[item * p.H + h0 + hh] = qv;
    }
  }
}

// one thread per (long row, channel): merge the items in order, normalise, record the statistics
template <int SC, bool TRAIN>
__global__ void __launch_bounds__(256) att_fwd_combine_kernel(const AttParams p) {
  const int HC = p.H * p.C;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t slot = t / HC;
  const int f = (int)(t - slot * HC);
  if (slot >= p.w.n_long) return;
  const int64_t row = p.w.long_rows[slot];
  const int h = (p.H == 1) ? 0 : f / p.C;
  const int32_t i0 = p.w.long_item_ptr[slot], i1 = p.w.long_item_ptr[slot + 1];
  float acc = 0.f, acc2 = 0.f, s = 0.f, qv = 0.f, M = -INFINITY, inv = 1.0f;
  if constexpr (SC == SC_FA) {
    for (int32_t it = i0; it < i1; ++it) {
      acc += p.part_acc[(int64_t)it * p.ldp + f];
      if constexpr (TRAIN) acc2 += p.part_acc2[(int64_t)it * p.ldp + f];
    }
  } else {
    for (int32_t it = i0; it < i1; ++it) M = fmaxf(M, p.part_m[(int64_t)it * p.H + h]);
    for (int32_t it = i0; it < i1; ++it) {
      const float mq = p.part_m[(int64_t)it * p.H + h];
      if (mq > -INFINITY) {
        const float sc = ex2(mq - M);
        s = fmaf(p.part_s[(int64_t)it * p.H + h], sc, s);
        acc = fmaf(p.part_acc[(int64_t)it * p.ldp + f], sc, acc);
        if constexpr (TRAIN) {
          qv = fmaf(p.part_q[(int64_t)it * p.H + h], sc, qv);
          acc2 = fmaf(p.part_acc2[(int64_t)it * p.ldp + f], sc, acc2);
        }
      }
    }
    inv = 1.0f / (s + 1e-16f);
  }
  p.out[row * p.ldo + f] = acc * inv;
  if constexpr (TRAIN) p.out2[row * p.ldo2 + f] = acc2 * inv;
  if constexpr (SC != SC_FA) {
    if (p.H == 1 ? (f == 0) : (f % p.C == 0)) {
      p.rowsum[row * p.H + h] = s;
      p.rowmax[row * p.H + h] = M * LN2;
      if constexpr (TRAIN) p.rowq[row * p.H + h] = qv * inv;
    }
  }
}

// out[e*H + h] = dropout multiplier of edge e, head h (edge order): the mask of the unfused paths and of the tests
__global__ void __launch_bounds__(256) att_dropout_mask_kernel(const int64_t* __restrict__ seed, int64_t n, int H,
                                                              uint32_t thresh, float scale, float* __restrict__ out) {
  const PhiloxKey key = philox_key((uint64_t)__ldg(seed));
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = t / H;
    out[t] = dropout_mult(key, (uint32_t)e, (uint32_t)(t - e * H), thresh, scale);
  }
}

// scaled copies of the score terms: out[i] = in[i] * log2(e)
__global__ void __launch_bounds__(256) att_scale_kernel(const float* __restrict__ in, int64_t n, float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i] * LOG2E;
}

// =============================================================================================
// backward
//   alpha_ij = exp(e_ij - max_i) / (sum_i + 1e-16),  dalpha_ij = mask_ij <dout_i, x_j>,  S_i = <dout_i, out_i>
//   de_ij = alpha_ij (dalpha_ij - S_i),  draw_ij = de_ij * leaky_relu'(raw_ij)
//   GAT: raw = a_src[j] + a_dst[i]:               da_src[j] += draw ; da_dst[i] = <dout_i, P_i> - S_i q_i
//   MX:  raw = u * s, u = a_l[j] + a_r[i], s = sigmoid(<x_i, x_j>):
//        da_l[j] += draw*s ; da_r[i] += draw*s ; dlogit = draw*u*s(1-s) ; dX_j += dlogit x_i ; dX_i += dlogit x_j
//   SD:  raw = logit_scale * <x_i, x_j>:           dlogit = draw*logit_scale ; dX_j += dlogit x_i ; dX_i += dlogit x_j
//   all: dX_j += alpha_ij mask_ij dout_i
//   FA:  w = tanh(u) dinv_j dinv_i: dX_j += w mask dout_i ; da_l[j] += <dout_i, x_j> dinv_j dinv_i mask (1 - tanh^2) ;
//        da_r[i] = <dout_i, Q_i>
// =============================================================================================
// per-(target, head) statistics + the node-level gradient of the target-side score term
template <int SC>
__global__ void __launch_bounds__(256)
att_bwd_prep_kernel(const float* __restrict__ dout, int64_t ldd, const float* __restrict__ out, int64_t ldo,
                    const float* __restrict__ out2, int64_t ldo2, const float* __restrict__ a_own,
                    const float* __restrict__ rowmax, const float* __restrict__ rowsum, const float* __restrict__ rowq,
                    const float* __restrict__ dinv, int64_t n, int H, int C, float4* __restrict__ stats,
                    float* __restrict__ da_own) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * H) return;
  const int64_t i = t / H;
  const int h = (int)(t - i * H);
  const float* a = dout + i * ldd + h * C;
  if constexpr (SC == SC_FA) {
    const float* b2 = out2 + i * ldo2 + h * C;
    float s2 = 0.f;
    for (int c = 0; c < C; ++c) s2 = fmaf(a[c], b2[c], s2);
    stats[t] = make_float4(a_own[t], dinv[i], 0.f, 0.f);
    da_own[t] = s2;
  } else {
    const float* b = out + i * ldo + h * C;
    float s = 0.f;
    for (int c = 0; c < C; ++c) s = fmaf(a[c], b[c], s);
    const float so = (SC == SC_SD) ? 0.f : a_own[t] * LOG2E;     // SD has no target-side scalar
    stats[t] = make_float4(so, rowmax[t] * LOG2E, 1.0f / (rowsum[t] + 1e-16f), s);
    if constexpr (SC == SC_GAT) {
      const float* b2 = out2 + i * ldo2 + h * C;
      float s2 = 0.f;
      for (int c = 0; c < C; ++c) s2 = fmaf(a[c], b2[c], s2);
      da_own[t] = s2 - s * rowq[t];
    }
  }
}

// ---- transpose pass: rows = sources j, neighbours = targets i -----------------------------------------------
template <int SC, int G, bool DR>
__device__ __forceinline__ void bwdT_range(const AttParams& p, int64_t k0, int64_t k1, int gl, const Lane& L, float so2,
                                           float d_own, const float4 (&xj)[2], PhiloxKey key, int32_t* sm_ids, float4 (&acc)[2],
                                           float& das) {
  constexpr int UB = (SC == SC_FA && G >= 8) ? 4 : 2;     // edges per step: 4 only where it measured faster (FAConv: 11.8 -> 11.05 ms fwd+bwd;
                                                          // GAT 6.6 -> 6.8, MX does not fit the registers)
  const int len = (k1 > k0) ? (int)(k1 - k0) : 0;
  const int maxlen = __reduce_max_sync(FULLMASK, len);
  if (maxlen == 0) return;
  const int32_t* __restrict__ col = p.w.col + k0;
  const char* db0 = reinterpret_cast<const char*>(p.Xn + L.f);
  const char* db1 = reinterpret_cast<const char*>(p.Xn + L.f + 4);
  const uint32_t d_bytes = (uint32_t)(p.ldn * 4);
  constexpr bool LOGIT = SC == SC_MX || SC == SC_SD;       // the score reads <x_i, x_j>: x_i is gathered too
  const char* xb0 = LOGIT ? reinterpret_cast<const char*>(p.Xn2 + L.f) : nullptr;
  const char* xb1 = LOGIT ? reinterpret_cast<const char*>(p.Xn2 + L.f + 4) : nullptr;
  const uint32_t x_bytes = (uint32_t)(p.ldn2 * 4);
  const char* stb = reinterpret_cast<const char*>(p.stats + L.h);
  const uint32_t st_bytes = (uint32_t)(p.H * 16);
  const bool a0 = L.nact > 0, a1 = L.nact > 1;
  const int lane = threadIdx.x & 31;
  int32_t* wids = sm_ids + (threadIdx.x & ~31);
  const int32_t* gids = wids + (lane - gl);
  int32_t cn = (gl < len) ? __ldcs(col + gl) : 0;
  for (int off = 0; off < maxlen; off += G) {
    int nb = len - off;
    nb = nb < 0 ? 0 : (nb > G ? G : nb);
    __syncwarp();
    wids[lane] = cn;
    __syncwarp();
    cn = 0;
    if (off + G + gl < len) cn = __ldcs(col + off + G + gl);
    const int nbmax = __reduce_max_sync(FULLMASK, nb);
#pragma unroll 1
    for (int j = 0; j < nbmax; j += UB) {
      float4 d[UB][2], x2[UB][2], st[UB];
      uint32_t cc[UB];
      lds_ids<UB>(gids + (j & (G - 1)), cc);
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        const uint32_t ci = cc[u];
        d[u][0] = a0 ? __ldg(reinterpret_cast<const float4*>(db0 + (size_t)ci * d_bytes)) : zero4();
        d[u][1] = a1 ? __ldg(reinterpret_cast<const float4*>(db1 + (size_t)ci * d_bytes)) : zero4();
        if constexpr (LOGIT) {
          x2[u][0] = a0 ? __ldg(reinterpret_cast<const float4*>(xb0 + (size_t)ci * x_bytes)) : zero4();
          x2[u][1] = a1 ? __ldg(reinterpret_cast<const float4*>(xb1 + (size_t)ci * x_bytes)) : zero4();
        }
        st[u] = __ldg(reinterpret_cast<const float4*>(stb + (size_t)ci * st_bytes));
      }
#pragma unroll
      for (int u = 0; u < UB; ++u) {
        // per-head dot products: lane-local, then reduced over the LPH lanes of the head (whole warp executes)
        const float dot = head_sum(dot4(d[u][0], xj[0]) + dot4(d[u][1], xj[1]), p.LPH);     // <dout_i, x_j>
        float sg = 1.0f, lg = 0.f;
        if constexpr (SC == SC_MX) sg = sigmoidf(head_sum(dot4(x2[u][0], xj[0]) + dot4(x2[u][1], xj[1]), p.LPH));
        if constexpr (SC == SC_SD) lg = head_sum(dot4(x2[u][0], xj[0]) + dot4(x2[u][1], xj[1]), p.LPH);  // <x_i, x_j>
        if (j + u < nb) {
          float mu = 1.0f;
          if constexpr (DR) mu = drop_mult(p, key, k0 + off + j + u, L.h);
          else if (p.drop) mu = __ldg(p.drop + (int64_t)__ldg(p.tpos + k0 + off + j + u) * p.H + L.h);
          if constexpr (SC == SC_FA) {
            const float t = tanhf(so2 + st[u].x);
            const float wgt = d_own * st[u].y * mu;
            const float w = t * wgt;
            fma4(acc[0], w, d[u][0]);
            fma4(acc[1], w, d[u][1]);
            das = fmaf(dot * wgt, 1.0f - t * t, das);
          } else {
            const float uu = so2 + st[u].x;                  // log2 domain
            const float raw = (SC == SC_SD) ? sd_raw(p, lg) : uu * sg;
            const float alpha = ex2(leaky_relu(raw, p.slope) - st[u].y) * st[u].z;
            const float w = alpha * mu;
            fma4(acc[0], w, d[u][0]);
            fma4(acc[1], w, d[u][1]);
            const float draw = alpha * (mu * dot - st[u].w) * (raw > 0.f ? 1.0f : p.slope);
            if constexpr (SC == SC_MX) {
              const float dlog = draw * (uu * LN2) * sg * (1.0f - sg);
              fma4(acc[0], dlog, x2[u][0]);
              fma4(acc[1], dlog, x2[u][1]);
              das = fmaf(draw, sg, das);
            } else if constexpr (SC == SC_SD) {
              const float dlog = draw * p.logit_scale;
              fma4(acc[0], dlog, x2[u][0]);
              fma4(acc[1], dlog, x2[u][1]);
            } else {
              das += draw;
            }
          }
        }
      }
    }
  }
}

template <int SC>
constexpr int bwdT_minb() {
  return RGBMP_ATT_OCC >= 1 ? (SC == SC_MX ? 3 : (SC == SC_GAT ? 4 : 3)) : (SC == SC_MX ? 2 : 3);
}

template <int SC, int G, bool DR>
__global__ void __launch_bounds__(ATT_THREADS, bwdT_minb<SC>()) att_bwdT_rows_kernel(const AttParams p) {
  __shared__ __align__(16) int32_t sm_ids[ATT_THREADS];
  const int gl = threadIdx.x % G;
  int64_t row, k0, k1;
  const bool live = short_row<G, ATT_THREADS>(p.w, row, k0, k1);
  const Lane L = lane_of(p, gl);
  float so2 = 0.f, d_own = 0.f;
  float4 xj[2] = {zero4(), zero4()}, acc[2] = {zero4(), zero4()};
  if (live) {
    if constexpr (SC != SC_SD) so2 = __ldg(p.so + row * p.H + L.h) * (SC == SC_FA ? 1.0f : LOG2E);
    if constexpr (SC == SC_FA) d_own = __ldg(p.dinv + row);
    load_own(p.Xo, p.ldo_, row, L, xj);
  }
  float das = 0.f;
  bwdT_range<SC, G, DR>(p, k0, k1, gl, L, so2, d_own, xj, drop_key<DR>(p), sm_ids, acc, das);
  if (!live || L.nact == 0) return;
#pragma unroll
  for (int v = 0; v < 2; ++v) {
    if (v < L.nact) {
      if (p.acc_in) {
        const float4 a = __ldcs(reinterpret_cast<const float4*>(p.acc_in + row * p.ld_acc + L.f + 4 * v));
        acc[v].x += a.x; acc[v].y += a.y; acc[v].z += a.z; acc[v].w += a.w;
      }
      __stcs(reinterpret_cast<float4*>(p.out + row * p.ldo + L.f + 4 * v), acc[v]);
    }
  }
  if (L.lead) p.ds[row * p.H + L.h] = das;
}

// long rows of a backward pass: plain sums (no running max), merged through shared memory in group order
template <int G>
__device__ __forceinline__ void bwd_long_merge(const AttParams& p, int gl, int q, const Lane& L, const float4 (&acc)[2], float das,
                                               float* sm_acc, float (*sm_s)[G]) {
  constexpr int Q = ATT_THREADS / G;
  constexpr int W = G * 8;
#pragma unroll
  for (int v = 0; v < 2; ++v) {
    const bool act = v < L.nact;
    float* d = sm_acc + q * W + gl * 8 + 4 * v;
    d[0] = act ? acc[v].x : 0.f; d[1] = act ? acc[v].y : 0.f; d[2] = act ? acc[v].z : 0.f; d[3] = act ? acc[v].w : 0.f;
  }
  const int hl = (p.H == 1) ? 0 : L.h - blockIdx.y * p.HT;
  if (L.lead) sm_s[q][hl] = das;
  __syncthreads();
  const int64_t item = blockIdx.x;
  const int h0 = (p.H == 1) ? 0 : blockIdx.y * p.HT;
  const int ht = (p.H == 1) ? 1 : min(p.HT, p.H - h0);
  const int width = (p.H == 1) ? p.C : ht * p.C;
  for (int t = threadIdx.x; t < width; t += ATT_THREADS) {
    float v = 0.f;
    for (int qq = 0; qq < Q; ++qq) v += sm_acc[qq * W + t];
    p.part_acc[item * p.ldp + h0 * p.C + t] = v;
  }
  if (threadIdx.x < ht) {
    float v = 0.f;
    for (int qq = 0; qq < Q; ++qq) v += sm_s[qq][threadIdx.x];
    p.part_s[item * p.H + h0 + threadIdx.x] = v;
  }
}

template <int SC, int G, bool DR>
__global__ void __launch_bounds__(ATT_THREADS, bwdT_minb<SC>()) att_bwdT_long_kernel(const AttParams p) {
  constexpr int Q = ATT_THREADS / G;
  __shared__ __align__(16) int32_t sm_ids[ATT_THREADS];
  __shared__ float sm_acc[Q * G * 8];
  __shared__ float sm_s[Q][G];
  const int gl = threadIdx.x % G, q = threadIdx.x / G;
  int64_t row, k0, k1;
  long_item<G, ATT_THREADS>(p.w, row, k0, k1);
  const Lane L = lane_of(p, gl);
  const float so2 = (SC == SC_SD) ? 0.f : __ldg(p.so + row * p.H + L.h) * (SC == SC_FA ? 1.0f : LOG2E);
  float d_own = 0.f;
  if constexpr (SC == SC_FA) d_own = __ldg(p.dinv + row);
  float4 xj[2], acc[2] = {zero4(), zero4()};
  load_own(p.Xo, p.ldo_, row, L, xj);
  float das = 0.f;
  bwdT_range<SC, G, DR>(p, k0, k1, gl, L, so2, d_own, xj, drop_key<DR>(p), sm_ids, acc, das);
  bwd_long_merge<G>(p, gl, q, L, acc, das, sm_acc, sm_s);
}

__global__ void __launch_bounds__(256) att_bwd_combine_kernel(const AttParams p) {
  const int HC = p.H * p.C;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t slot = t / HC;
  const int f = (int)(t - slot * HC);
  if (slot >= p.w.n_long) return;
  const int64_t row = p.w.long_rows[slot];
  const int h = (p.H == 1) ? 0 : f / p.C;
  float acc = 0.f, s = 0.f;
  for (int32_t it = p.w.long_item_ptr[slot]; it < p.w.long_item_ptr[slot + 1]; ++it) {
    acc += p.part_acc[(int64_t)it * p.ldp + f];
    s += p.part_s[(int64_t)it * p.H + h];
  }
  if (p.acc_in) acc += p.acc_in[row * p.ld_acc + f];
  p.out[row * p.ldo + f] = acc;
  if (p.H == 1 ? (f == 0) : (f % p.C == 0)) p.ds[row * p.H + h] = s;
}

// ---- MX / SD forward-orientation pass: rows = targets i, neighbours = sources j ----------------------------
//   dXf_i = sum_j dlogit_ij x_j ;  MX: da_r[i] = sum_j draw_ij * s_ij
template <int SC, int G, bool DR>
__device__ __forceinline__ void bwdF_range(const AttParams& p, int64_t k0, int64_t k1, int gl, const Lane& L, const float4 st_own,
                                           const float4 (&xi)[2], const float4 (&di)[2], PhiloxKey key, int32_t* sm_ids,
                                           float4 (&acc)[2], float& dar) {
  const int len = (k1 > k0) ? (int)(k1 - k0) : 0;
  const int maxlen = __reduce_max_sync(FULLMASK, len);
  if (maxlen == 0) return;
  const int32_t* __restrict__ col = p.w.col + k0;
  const char* xb0 = reinterpret_cast<const char*>(p.Xn + L.f);
  const char* xb1 = reinterpret_cast<const char*>(p.Xn + L.f + 4);
  const uint32_t row_bytes = (uint32_t)(p.ldn * 4);
  const char* snb = reinterpret_cast<const char*>(p.sn + L.h);
  const uint32_t sn_bytes = (uint32_t)(p.H * 4);
  const bool a0 = L.nact > 0, a1 = L.nact > 1;
  const int lane = threadIdx.x & 31;
  int32_t* wids = sm_ids + (threadIdx.x & ~31);
  const int32_t* gids = wids + (lane - gl);
  int32_t cn = (gl < len) ? __ldcs(col + gl) : 0;
  for (int off = 0; off < maxlen; off += G) {
    int nb = len - off;
    nb = nb < 0 ? 0 : (nb > G ? G : nb);
    __syncwarp();
    wids[lane] = cn;
    __syncwarp();
    cn = 0;
    if (off + G + gl < len) cn = __ldcs(col + off + G + gl);
    const int nbmax = __reduce_max_sync(FULLMASK, nb);
#pragma unroll 1
    for (int j = 0; j < nbmax; j += U) {
      float4 x[U][2];
      float as[U];
      uint32_t cc[U];
      lds_ids<U>(gids + (j & (G - 1)), cc);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const uint32_t cj = cc[u];
        x[u][0] = a0 ? __ldg(reinterpret_cast<const float4*>(xb0 + (size_t)cj * row_bytes)) : zero4();
        x[u][1] = a1 ? __ldg(reinterpret_cast<const float4*>(xb1 + (size_t)cj * row_bytes)) : zero4();
        if constexpr (SC == SC_MX) as[u] = __ldg(reinterpret_cast<const float*>(snb + (size_t)cj * sn_bytes));
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float dot = head_sum(dot4(di[0], x[u][0]) + dot4(di[1], x[u][1]), p.LPH);              // <dout_i, x_j>
        const float lg = head_sum(dot4(xi[0], x[u][0]) + dot4(xi[1], x[u][1]), p.LPH);              // <x_i, x_j>
        const float sg = (SC == SC_MX) ? sigmoidf(lg) : 0.f;
        if (j + u < nb) {
          float mu;
          if constexpr (DR) mu = drop_mult(p, key, k0 + off + j + u, L.h);
          else mu = p.drop ? __ldg(p.drop + (k0 + off + j + u) * p.H + L.h) : 1.0f;
          if constexpr (SC == SC_SD) {
            const float raw = sd_raw(p, lg);
            const float alpha = ex2(leaky_relu(raw, p.slope) - st_own.y) * st_own.z;
            const float draw = alpha * (mu * dot - st_own.w) * (raw > 0.f ? 1.0f : p.slope);
            const float dlog = draw * p.logit_scale;
            fma4(acc[0], dlog, x[u][0]);
            fma4(acc[1], dlog, x[u][1]);
          } else {
            const float uu = as[u] + st_own.x;
            const float raw = uu * sg;
            const float alpha = ex2(leaky_relu(raw, p.slope) - st_own.y) * st_own.z;
            const float draw = alpha * (mu * dot - st_own.w) * (raw > 0.f ? 1.0f : p.slope);
            const float dlog = draw * (uu * LN2) * sg * (1.0f - sg);
            fma4(acc[0], dlog, x[u][0]);
            fma4(acc[1], dlog, x[u][1]);
            dar = fmaf(draw, sg, dar);
          }
        }
      }
    }
  }
}

template <int SC, int G, bool DR>
__global__ void __launch_bounds__(ATT_THREADS, RGBMP_ATT_OCC >= 1 ? 3 : 2) att_bwdF_rows_kernel(const AttParams p) {
  __shared__ __align__(16) int32_t sm_ids[ATT_THREADS];
  const int gl = threadIdx.x % G;
  int64_t row, k0, k1;
  const bool live = short_row<G, ATT_THREADS>(p.w, row, k0, k1);
  const Lane L = lane_of(p, gl);
  float4 xi[2] = {zero4(), zero4()}, di[2] = {zero4(), zero4()}, acc[2] = {zero4(), zero4()};
  float4 st_own = zero4();
  if (live) {
    load_own(p.Xo, p.ldo_, row, L, xi);
    load_own(p.Do, p.lddo, row, L, di);
    st_own = __ldg(p.stats + row * p.H + L.h);
  }
  float dar = 0.f;
  bwdF_range<SC, G, DR>(p, k0, k1, gl, L, st_own, xi, di, drop_key<DR>(p), sm_ids, acc, dar);
  if (!live || L.nact == 0) return;
#pragma unroll
  for (int v = 0; v < 2; ++v)
    if (v < L.nact) __stcs(reinterpret_cast<float4*>(p.out + row * p.ldo + L.f + 4 * v), acc[v]);
  if (L.lead) p.ds[row * p.H + L.h] = dar;
}

template <int SC, int G, bool DR>
__global__ void __launch_bounds__(ATT_THREADS, RGBMP_ATT_OCC >= 1 ? 3 : 2) att_bwdF_long_kernel(const AttParams p) {
  constexpr int Q = ATT_THREADS / G;
  __shared__ __align__(16) int32_t sm_ids[ATT_THREADS];
  __shared__ float sm_acc[Q * G * 8];
  __shared__ float sm_s[Q][G];
  const int gl = threadIdx.x % G, q = threadIdx.x / G;
  int64_t row, k0, k1;
  long_item<G, ATT_THREADS>(p.w, row, k0, k1);
  const Lane L = lane_of(p, gl);
  float4 xi[2], di[2], acc[2] = {zero4(), zero4()};
  load_own(p.Xo, p.ldo_, row, L, xi);
  load_own(p.Do, p.lddo, row, L, di);
  const float4 st_own = __ldg(p.stats + row * p.H + L.h);
  float dar = 0.f;
  bwdF_range<SC, G, DR>(p, k0, k1, gl, L, st_own, xi, di, drop_key<DR>(p), sm_ids, acc, dar);
  bwd_long_merge<G>(p, gl, q, L, acc, dar, sm_acc, sm_s);
}

// =============================================================================================
// host side
// =============================================================================================
struct Shape { int G, HT, LPH, tiles; };

// heads per tile: as many as fit 128 channels; G = pow2 lanes covering the tile with 8 channels per lane
static bool att_shape(int H, int C, Shape* s) {
  if (H <= 0 || C <= 0 || C > 128) return false;
  int HT, width;
  if (H == 1) { HT = 1; width = C; }
  else {
    if (C < 8 || (C & (C - 1)) != 0) return false;          // pow2 >= 8: a lane's 8 channels stay inside one head
    HT = 128 / C;
    if (HT > H) HT = H;
    width = HT * C;
  }
  const int lanes = (int)ceil_div(width, 8);
  int g = 4;
  while (g < lanes) g <<= 1;
  s->G = g;
  s->HT = HT;
  s->LPH = (H == 1) ? g : C / 8;
  s->tiles = (int)ceil_div(H, HT);
  return g <= 16;
}

// scratch of the long-row split: part_m | part_s | part_q [n_items,H] and part_acc | part_acc2 [n_items, ldp]
static size_t split_bytes(int64_t n_items, int H, int HC) {
  if (n_items <= 0) return 0;
  return 5 * 256 + align_up((size_t)n_items * H * 4, 256) * 3 + align_up((size_t)n_items * align_up((size_t)HC, 4) * 4, 256) * 2;
}

static bool carve_split(AttParams& p, Carver& cv, int HC, int64_t n_items) {
  p.part_m = p.part_s = p.part_q = p.part_acc = p.part_acc2 = nullptr;
  p.ldp = (int64_t)align_up((size_t)HC, 4);
  if (n_items <= 0) return true;
  p.part_m = cv.take<float>((size_t)n_items * p.H);
  p.part_s = cv.take<float>((size_t)n_items * p.H);
  p.part_q = cv.take<float>((size_t)n_items * p.H);
  p.part_acc = cv.take<float>((size_t)n_items * p.ldp);
  p.part_acc2 = cv.take<float>((size_t)n_items * p.ldp);
  return cv.ok();
}

// Calls f(G) for the lanes per row att_shape chose, G as a std::integral_constant
template <class F>
static int with_group(int G, F&& f) {
  switch (G) {
    case 4: return f(std::integral_constant<int, 4>());
    case 8: return f(std::integral_constant<int, 8>());
    default: return f(std::integral_constant<int, 16>());
  }
}

// forward loop variant: 0 = 2 edges per step, software-pipelined (round 1's shape); 1 = 4 edges per step, plain;
// 2 = 2 edges per step, plain (default).  Measured on the Reddit-shaped 8x8 layer with the ids staged in shared
// memory (profiles/r02_att_variants.txt): 3.27 / 2.77 / 2.50 ms -- the explicit pipeline now only costs registers
// and issue slots.  RGBMP_ATT_FWD selects a variant for experiments.
static int att_fwd_variant() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("RGBMP_ATT_FWD");
    v = e ? atoi(e) : 2;
    if (v < 0 || v > 2) v = 2;
  }
  return v;
}

template <int SC, bool TRAIN, int UU, bool PIPE, bool DR>
static int launch_fwd_v(const AttParams& p, const Shape& s, cudaStream_t st) {
  return with_group(s.G, [&](auto g) {
    constexpr int G = decltype(g)::value;
    return launch_phases(
        p.w, ATT_THREADS / G, s.tiles, p.H * p.C, "att_fwd kernels",
        [&](dim3 grid) { att_fwd_rows_kernel<SC, TRAIN, G, UU, PIPE, DR><<<grid, ATT_THREADS, 0, st>>>(p); },
        [&](dim3 grid) { att_fwd_long_kernel<SC, TRAIN, G, UU, PIPE, DR><<<grid, ATT_THREADS, 0, st>>>(p); },
        [&](unsigned blocks) { att_fwd_combine_kernel<SC, TRAIN><<<blocks, 256, 0, st>>>(p); });
  });
}

// the fused-dropout and the SD forwards exist in the default loop variant only (SD spills in the other two)
template <int SC, bool TRAIN, bool DR>
static int launch_fwd(const AttParams& p, const Shape& s, cudaStream_t st) {
  if constexpr (DR || SC == SC_SD) {
    return launch_fwd_v<SC, TRAIN, 2, false, DR>(p, s, st);
  } else {
    switch (att_fwd_variant()) {
      case 1: return launch_fwd_v<SC, TRAIN, 4, false, false>(p, s, st);
      case 0: return launch_fwd_v<SC, TRAIN, 2, true, false>(p, s, st);
      default: return launch_fwd_v<SC, TRAIN, 2, false, false>(p, s, st);
    }
  }
}

template <int SC, bool DR>
static int launch_bwdT(const AttParams& p, const Shape& s, cudaStream_t st) {
  return with_group(s.G, [&](auto g) {
    constexpr int G = decltype(g)::value;
    return launch_phases(
        p.w, ATT_THREADS / G, s.tiles, p.H * p.C, "att_bwdT kernels",
        [&](dim3 grid) { att_bwdT_rows_kernel<SC, G, DR><<<grid, ATT_THREADS, 0, st>>>(p); },
        [&](dim3 grid) { att_bwdT_long_kernel<SC, G, DR><<<grid, ATT_THREADS, 0, st>>>(p); },
        [&](unsigned blocks) { att_bwd_combine_kernel<<<blocks, 256, 0, st>>>(p); });
  });
}

template <int SC, bool DR>
static int launch_bwdF(const AttParams& p, const Shape& s, cudaStream_t st) {
  return with_group(s.G, [&](auto g) {
    constexpr int G = decltype(g)::value;
    return launch_phases(
        p.w, ATT_THREADS / G, s.tiles, p.H * p.C, "att_bwdF kernels",
        [&](dim3 grid) { att_bwdF_rows_kernel<SC, G, DR><<<grid, ATT_THREADS, 0, st>>>(p); },
        [&](dim3 grid) { att_bwdF_long_kernel<SC, G, DR><<<grid, ATT_THREADS, 0, st>>>(p); },
        [&](unsigned blocks) { att_bwd_combine_kernel<<<blocks, 256, 0, st>>>(p); });
  });
}

// the scores and shapes the kernels take; FA is single-head
static bool att_ok(int score, int H, int C, Shape* s) {
  return score >= RGBMP_ATT_GAT && score <= RGBMP_ATT_SD && (score != RGBMP_ATT_FA || H == 1) && att_shape(H, C, s);
}

// Calls f(SC, DR) -- the score as a std::integral_constant, "fused dropout" as a std::bool_constant -- for a score
// att_ok admitted: the one place run-time arguments become kernel template arguments.  f guards with if constexpr
// what a score has no kernels for (MX / SD: a training-mode forward; GAT / FA: the backward's pass F).
template <class F>
static int with_kernel(int score, bool dr, F&& f) {
  const auto run = [&](auto sc) { return dr ? f(sc, std::true_type()) : f(sc, std::false_type()); };
  switch (score) {
    case RGBMP_ATT_GAT: return run(std::integral_constant<int, SC_GAT>());
    case RGBMP_ATT_MX: return run(std::integral_constant<int, SC_MX>());
    case RGBMP_ATT_FA: return run(std::integral_constant<int, SC_FA>());
    default: return run(std::integral_constant<int, SC_SD>());
  }
}

}  // namespace rgbmp

using namespace rgbmp;

extern "C" {

int rgbmp_att_supported(int score, int H, int C) {
  Shape s;
  return att_ok(score, H, C, &s) ? 1 : 0;
}

size_t rgbmp_att_forward_workspace_bytes(const rgbmp_graph_t* g, int H, int C) {
  if (!g || H <= 0 || C <= 0) return 256;
  return 1024 + align_up((size_t)g->n_cols * H * 4, 256) + align_up((size_t)g->n_rows * H * 4, 256) +
         split_bytes(g->n_items, H, H * C);
}

static void set_dropout(AttParams& p, const rgbmp_dropout_t* d, const int32_t* eid) {
  p.seed = d->seed;
  p.eid = eid;
  p.thresh = d->thresh;
  p.dscale = d->scale;
}

int rgbmp_att_forward(const rgbmp_graph_t* g, int score, const float* X, int64_t ldx, const float* a_nbr,
                      const float* a_own, const float* dinv, int H, int C, float slope, float logit_scale,
                      const float* drop, const rgbmp_dropout_t* d, float* out, int64_t ldo, float* rowmax,
                      float* rowsum, float* out2, int64_t ldo2, float* rowq, void* ws, size_t ws_bytes, int device,
                      void* stream) {
  const char* fn = "rgbmp_att_forward";
  const bool sd = score == RGBMP_ATT_SD;                   // X holds the features of both endpoints
  int rc = check_graph(g, fn, sd ? GRAPH_SQUARE : 0);
  if (rc) return rc;
  Shape s;
  if (!att_ok(score, H, C, &s))
    return fail(RGBMP_ERANGE, "%s: unsupported score %d / H %d / C %d (H == 1 with C <= 128, or C in {8..128} a power of two)",
                fn, score, H, C);
  if (sd && !isfinite(logit_scale)) return fail(RGBMP_EINVAL, "%s: SD needs a finite logit_scale", fn);
  if (drop && d) return fail(RGBMP_EINVAL, "%s: at most one of drop / d", fn);
  if (!X || (!sd && (!a_nbr || !a_own)) || !out || !ws) return fail(RGBMP_EINVAL, "%s: null pointer", fn);
  if (d && (!d->seed || (g->nnz > 0 && !d->eid))) return fail(RGBMP_EINVAL, "%s: dropout needs seed and eid", fn);
  const bool softmax = score != RGBMP_ATT_FA;
  if (softmax && (!rowmax || !rowsum)) return fail(RGBMP_EINVAL, "%s: rowmax / rowsum required", fn);
  if (!softmax && !dinv) return fail(RGBMP_EINVAL, "%s: FA needs dinv", fn);
  const bool train = out2 != nullptr;
  if (train && (score == RGBMP_ATT_MX || sd)) return fail(RGBMP_EINVAL, "%s: MX / SD have no second aggregate", fn);
  if (train && score == RGBMP_ATT_GAT && !rowq) return fail(RGBMP_EINVAL, "%s: rowq required with out2", fn);
  const int HC = H * C;
  const int64_t need_ld = (int64_t)align_up((size_t)HC, 4);
  if (!al16(X, ldx) || !al16(out, ldo) || ldx < need_ld || ldo < need_ld || (train && (!al16(out2, ldo2) || ldo2 < need_ld)))
    return fail(RGBMP_EALIGN, "%s: X/out/out2 need 16-byte aligned rows with ld >= roundup(H*C,4)", fn);
  if (ws_bytes < rgbmp_att_forward_workspace_bytes(g, H, C))
    return fail(RGBMP_EWORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes, rgbmp_att_forward_workspace_bytes(g, H, C));
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "%s: bad device", fn);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = g->n_rows;
  if (n == 0) return 0;
  AttParams p = {};
  p.w = csr_work(g);
  p.H = H; p.HT = s.HT; p.C = C; p.LPH = s.LPH; p.slope = slope; p.logit_scale = logit_scale;
  Carver cv(ws, ws_bytes);
  float* an2 = cv.take<float>((size_t)g->n_cols * H);
  float* ao2 = cv.take<float>((size_t)n * H);
  if (!carve_split(p, cv, HC, p.w.n_items) || !cv.ok()) return fail(RGBMP_EWORKSPACE, "%s: workspace carve", fn);
  p.Xn = X; p.ldn = ldx; p.Xo = X; p.ldo_ = ldx; p.dinv = dinv; p.drop = drop;
  if (d) set_dropout(p, d, d->eid);
  p.out = out; p.ldo = ldo; p.out2 = out2; p.ldo2 = ldo2; p.rowmax = rowmax; p.rowsum = rowsum; p.rowq = rowq;
  if (score == RGBMP_ATT_FA) {
    p.sn = a_nbr; p.so = a_own;
  } else if (!sd) {                                        // log2-domain copies of the score terms
    att_scale_kernel<<<(unsigned)ceil_div(g->n_cols * H, 256), 256, 0, st>>>(a_nbr, g->n_cols * H, an2);
    att_scale_kernel<<<(unsigned)ceil_div(n * H, 256), 256, 0, st>>>(a_own, n * H, ao2);
    RGBMP_LAUNCH_CHECK("att_scale_kernel");
    p.sn = an2; p.so = ao2;
  }
  return with_kernel(score, d != nullptr, [&](auto sc, auto dr) {
    constexpr int SC = decltype(sc)::value;
    constexpr bool DR = decltype(dr)::value;
    if constexpr (SC == SC_MX || SC == SC_SD) return launch_fwd<SC, false, DR>(p, s, st);
    else return train ? launch_fwd<SC, true, DR>(p, s, st) : launch_fwd<SC, false, DR>(p, s, st);
  });
}

size_t rgbmp_att_backward_workspace_bytes(const rgbmp_graph_t* g, const rgbmp_graph_t* gT, int H, int C) {
  if (!g || !gT || H <= 0 || C <= 0) return 256;
  const int64_t items = g->n_items > gT->n_items ? g->n_items : gT->n_items;
  return 2048 + align_up((size_t)g->n_rows * H * sizeof(float4), 256) + align_up((size_t)g->n_cols * H * 4, 256) +
         split_bytes(items, H, H * C);
}

int rgbmp_att_backward(const rgbmp_graph_t* g, const rgbmp_graph_t* gT, int score, const float* X, int64_t ldx,
                       const float* a_nbr, const float* a_own, const float* dinv, int H, int C, float slope,
                       float logit_scale, const float* drop, const int32_t* tpos, const rgbmp_dropout_t* d,
                       const float* rowmax, const float* rowsum, const float* rowq, const float* out, int64_t ldo,
                       const float* out2, int64_t ldo2, const float* dout, int64_t ldd, float* dX, int64_t lddx,
                       float* dXf, int64_t lddxf, float* da_nbr, float* da_own, void* ws, size_t ws_bytes, int device,
                       void* stream) {
  const char* fn = "rgbmp_att_backward";
  const bool sd = score == RGBMP_ATT_SD;
  int rc = check_graph(g, fn, sd ? GRAPH_SQUARE : 0);
  if (rc) return rc;
  rc = check_graph(gT, fn);
  if (rc) return rc;
  Shape s;
  if (!att_ok(score, H, C, &s)) return fail(RGBMP_ERANGE, "%s: unsupported score %d / H %d / C %d", fn, score, H, C);
  if (sd && (gT->n_rows != g->n_cols || gT->n_cols != g->n_rows || gT->nnz != g->nnz || !isfinite(logit_scale)))
    return fail(RGBMP_EINVAL, "%s: SD needs the transpose of g and a finite logit_scale", fn);
  if (drop && d) return fail(RGBMP_EINVAL, "%s: at most one of drop / d", fn);
  if (!X || !dout || !dX || (!sd && (!a_nbr || !a_own || !da_nbr || !da_own)) || !ws || (drop && !tpos))
    return fail(RGBMP_EINVAL, "%s: null pointer", fn);
  const bool logit = score == RGBMP_ATT_MX || sd;             // one pass per orientation
  if (d && (!d->seed || (gT->nnz > 0 && !d->eid_t) || (logit && g->nnz > 0 && !d->eid)))
    return fail(RGBMP_EINVAL, "%s: dropout needs seed, eid_t (and eid for MX / SD)", fn);
  const bool softmax = score != RGBMP_ATT_FA;
  if (softmax && (!rowmax || !rowsum || !out)) return fail(RGBMP_EINVAL, "%s: forward statistics required", fn);
  if (!logit && !out2) return fail(RGBMP_EINVAL, "%s: the training-mode forward's second aggregate is required", fn);
  if (score == RGBMP_ATT_GAT && !rowq) return fail(RGBMP_EINVAL, "%s: rowq required", fn);
  if (logit && !dXf) return fail(RGBMP_EINVAL, "%s: MX / SD need the dXf scratch [n, ld]", fn);
  if (!softmax && !dinv) return fail(RGBMP_EINVAL, "%s: FA needs dinv", fn);
  if (!al16(X, ldx) || !al16(dout, ldd) || !al16(dX, lddx) || (dXf && !al16(dXf, lddxf)))
    return fail(RGBMP_EALIGN, "%s: X/dout/dX need 16-byte aligned rows", fn);
  if (ws_bytes < rgbmp_att_backward_workspace_bytes(g, gT, H, C))
    return fail(RGBMP_EWORKSPACE, "%s: workspace %zu < %zu", fn, ws_bytes, rgbmp_att_backward_workspace_bytes(g, gT, H, C));
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "%s: bad device", fn);
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_dst = g->n_rows, n_src = gT->n_rows;
  if (n_dst == 0 || n_src == 0) return 0;
  const int HC = H * C;
  Carver cv(ws, ws_bytes);
  float4* stats = cv.take<float4>((size_t)n_dst * H);
  float* an2 = cv.take<float>((size_t)g->n_cols * H);
  AttParams pt = {};
  pt.w = csr_work(gT);
  pt.H = H; pt.HT = s.HT; pt.C = C; pt.LPH = s.LPH; pt.slope = slope; pt.logit_scale = logit_scale;
  if (!carve_split(pt, cv, HC, g->n_items > gT->n_items ? g->n_items : gT->n_items) || !cv.ok())
    return fail(RGBMP_EWORKSPACE, "%s: workspace carve", fn);
  const unsigned prep_grid = (unsigned)ceil_div(n_dst * H, 256);
  return with_kernel(score, d != nullptr, [&](auto sc, auto dr) {
    constexpr int SC = decltype(sc)::value;
    constexpr bool DR = decltype(dr)::value;
    att_bwd_prep_kernel<SC><<<prep_grid, 256, 0, st>>>(dout, ldd, out, ldo, out2, ldo2, a_own, rowmax, rowsum, rowq, dinv,
                                                       n_dst, H, C, stats, da_own);
    RGBMP_LAUNCH_CHECK("att_bwd_prep_kernel");
    if constexpr (SC == SC_MX || SC == SC_SD) {
      // pass F on the forward CSR: dXf_i = sum_j dlogit_ij x_j, da_r[i]
      AttParams pf = pt;
      pf.w = csr_work(g);
      if constexpr (SC == SC_MX) {
        att_scale_kernel<<<(unsigned)ceil_div(g->n_cols * H, 256), 256, 0, st>>>(a_nbr, g->n_cols * H, an2);
        RGBMP_LAUNCH_CHECK("att_scale_kernel");
        pf.sn = an2;
      }
      pf.Xn = X; pf.ldn = ldx; pf.stats = stats; pf.Xo = X; pf.ldo_ = ldx; pf.Do = dout; pf.lddo = ldd;
      // SD has no score scalars, but the passes (att_bwd_combine_kernel among them) write a per-row ds: the zeros
      // land in the slot of the scaled a_nbr copy, n_cols * H floats, which covers the rows of both orientations
      // because SD admits square graphs only
      pf.drop = drop; pf.out = dXf; pf.ldo = lddxf; pf.ds = SC == SC_SD ? an2 : da_own;
      if (d) set_dropout(pf, d, d->eid);
      const int rc = launch_bwdF<SC, DR>(pf, s, st);
      if (rc) return rc;
      pt.acc_in = dXf; pt.ld_acc = lddxf;
      pt.Xn2 = X; pt.ldn2 = ldx;
    }
    // pass T on the transpose CSR: dX_j, da_src[j]
    pt.Xn = dout; pt.ldn = ldd; pt.stats = stats; pt.Xo = X; pt.ldo_ = ldx;
    if constexpr (SC != SC_SD) { pt.dinv = dinv; pt.so = a_nbr; }
    pt.drop = drop; pt.tpos = tpos; pt.out = dX; pt.ldo = lddx; pt.ds = SC == SC_SD ? an2 : da_nbr;
    if (d) set_dropout(pt, d, d->eid_t);
    return launch_bwdT<SC, DR>(pt, s, st);
  });
}

int rgbmp_dropout_mask(const rgbmp_dropout_t* d, int64_t nnz, int H, float* out, int device, void* stream) {
  if (!d || !d->seed || nnz < 0 || H <= 0 || (nnz > 0 && !out))
    return fail(RGBMP_EINVAL, "rgbmp_dropout_mask: bad arguments");
  if (nnz > INT32_MAX) return fail(RGBMP_ERANGE, "rgbmp_dropout_mask: edge ids are 32-bit");
  DeviceGuard dg(device);
  if (!dg.ok) return fail(RGBMP_EINVAL, "rgbmp_dropout_mask: bad device");
  const int64_t n = nnz * H;
  if (n == 0) return 0;
  const int64_t blocks = ceil_div(n, 256);
  att_dropout_mask_kernel<<<(unsigned)(blocks < 148 * 64 ? blocks : 148 * 64), 256, 0, (cudaStream_t)stream>>>(
      d->seed, n, H, d->thresh, d->scale, out);
  RGBMP_LAUNCH_CHECK("att_dropout_mask_kernel");
  return 0;
}

}  // extern "C"
