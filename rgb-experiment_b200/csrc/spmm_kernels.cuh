// CSR SpMM kernels with fused epilogue (sm_100a) -- templates shared by the per-dtype
// instantiation units spmm_inst_*.cu.
//
// HBM-bound gather/segment-reduce (0.25-0.5 flop/B): no tensor cores.  Layout of the work:
//   * a GROUP of G lanes owns one output row; lane l of the group owns V 16-byte vectors of the
//     row (vector index l + v*G), so every gathered feature row is read with fully coalesced
//     16-byte loads and accumulated in registers with no cross-lane traffic;
//   * U edges are kept in flight per group (U*V independent 16-byte loads per lane) and the next
//     U column indices are prefetched while the current features are consumed;
//   * edges of a row are accumulated sequentially in CSR (= stable edge) order: unweighted sums are plain
//     IEEE adds and reproduce PyG-CPU scatter_add_ bit for bit; weighted sums use one fused multiply-add per
//     element (one rounding instead of two) and are held to the 1e-5 bar only;
//   * rows longer than `chunk` edges are split into CTA-sized work items (spmm_long_kernel) whose
//     partial sums are combined in a fixed order (spmm_combine_kernel) -- deterministic, no atomics;
//   * the epilogue (row scale, teleport, clamp, reset rows, pre-scaled second output) is applied
//     in registers before the single store of the row.
#pragma once
#include "csr_work.cuh"
#include "epilogue.cuh"

namespace rgbmp {

struct SpmmParams {
  CsrWork w;
  const float* val;
  float* partial;  // [n_items, ldpart]
  int64_t ldpart;
  // features
  const void* X;
  int64_t ldx;
  void* Y;
  int64_t ldy;
  int F;
  // cache policy: 1 = column ids, weights, teleport rows and outputs are touched once per launch ->
  // streaming (evict-first) loads/stores, so that L2 keeps the gathered feature rows instead
  int stream;
  // hinted = 1 (hot-tagged graph, or a policy set in the tune word): each gathered row carries an L2 eviction priority
  // (0 normal, 1 evict-first, 2 evict-last), pol_hot for column ids tagged hot (bit 31 set by rgbmp_col_tag), pol_cold
  // for the rest.  hinted = 0: one plain load per vector, no tag mask, no policy descriptor.
  int hinted;
  int pol_hot, pol_cold;
  // fused all-gather: 1 = the short-row kernel stages each finished row in shared memory and pushes it to every peer with
  // one bulk asynchronous copy (cp.async.bulk, TMA) instead of 16-byte st.global per lane
  int push_bulk;
  // epilogue
  rgbmp_epilogue_t ep;
};

template <typename S>
__device__ __forceinline__ S ld_stream(const S* q, int stream) {
  return stream ? __ldcs(q) : __ldg(q);
}

// ------------------------------------------------------------------------------------------
// vector load / store helpers.  EPV = elements per 16-byte vector (4 fp32, 8 bf16) or 1 (scalar).
// ------------------------------------------------------------------------------------------
template <typename T, int EPV>
struct Raw;
template <>
struct Raw<float, 4> {
  float4 r;
  __device__ __forceinline__ void load(const float* p) { r = __ldg(reinterpret_cast<const float4*>(p)); }
  __device__ __forceinline__ void zero() { r = make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ void unpack(float (&f)[4]) const { f[0] = r.x; f[1] = r.y; f[2] = r.z; f[3] = r.w; }
  __device__ __forceinline__ float2 pair(int i) const { return i == 0 ? make_float2(r.x, r.y) : make_float2(r.z, r.w); }
  static __device__ __forceinline__ void store(float* p, const float (&f)[4], int stream = 0) {
    const float4 v = make_float4(f[0], f[1], f[2], f[3]);
    if (stream) __stcs(reinterpret_cast<float4*>(p), v);
    else *reinterpret_cast<float4*>(p) = v;
  }
  __device__ __forceinline__ void load_stream(const float* p) { r = __ldcs(reinterpret_cast<const float4*>(p)); }
  __device__ __forceinline__ void load_hint(const float* p, uint64_t pol) {
    asm("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
        : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p), "l"(pol));
  }
};
template <>
struct Raw<float, 1> {
  float r;
  __device__ __forceinline__ void load(const float* p) { r = __ldg(p); }
  __device__ __forceinline__ void zero() { r = 0.f; }
  __device__ __forceinline__ void unpack(float (&f)[1]) const { f[0] = r; }
  __device__ __forceinline__ float2 pair(int) const { return make_float2(r, 0.f); }
  static __device__ __forceinline__ void store(float* p, const float (&f)[1], int = 0) { *p = f[0]; }
  __device__ __forceinline__ void load_stream(const float* p) { r = __ldcs(p); }
  __device__ __forceinline__ void load_hint(const float* p, uint64_t pol) {
    asm("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
  }
};
template <>
struct Raw<__nv_bfloat16, 8> {
  uint4 r;
  __device__ __forceinline__ void load(const __nv_bfloat16* p) { r = __ldg(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ void zero() { r = make_uint4(0, 0, 0, 0); }
  __device__ __forceinline__ void unpack(float (&f)[8]) const {
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    }
  }
  __device__ __forceinline__ float2 pair(int i) const {
    const uint32_t w = i == 0 ? r.x : (i == 1 ? r.y : (i == 2 ? r.z : r.w));
    return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u));
  }
  __device__ __forceinline__ void load_stream(const __nv_bfloat16* p) { r = __ldcs(reinterpret_cast<const uint4*>(p)); }
  __device__ __forceinline__ void load_hint(const __nv_bfloat16* p, uint64_t pol) {
    asm("ld.global.nc.L2::cache_hint.v4.u32 {%0, %1, %2, %3}, [%4], %5;"
        : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8], int stream = 0) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 h = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&h);
    }
    const uint4 v = make_uint4(w[0], w[1], w[2], w[3]);
    if (stream) __stcs(reinterpret_cast<uint4*>(p), v);
    else *reinterpret_cast<uint4*>(p) = v;
  }
};
template <>
struct Raw<__nv_bfloat16, 1> {
  __nv_bfloat16 r;
  __device__ __forceinline__ void load(const __nv_bfloat16* p) { r = *p; }
  __device__ __forceinline__ void zero() { r = __float2bfloat16(0.f); }
  __device__ __forceinline__ void unpack(float (&f)[1]) const { f[0] = __bfloat162float(r); }
  __device__ __forceinline__ float2 pair(int) const { return make_float2(__bfloat162float(r), 0.f); }
  __device__ __forceinline__ void load_stream(const __nv_bfloat16* p) { r = *p; }
  __device__ __forceinline__ void load_hint(const __nv_bfloat16* p, uint64_t) { r = *p; }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[1], int = 0) { *p = __float2bfloat16(f[0]); }
};

__device__ __forceinline__ float to_f(float x) { return x; }
__device__ __forceinline__ float to_f(__nv_bfloat16 x) { return __bfloat162float(x); }

// ------------------------------------------------------------------------------------------
// accumulate edges [k0, k1) of one row into acc (sequential, stable order).
//
// Lean inner loop (v2, after the v1 ncu profile showed 43 instructions per 16-byte gather):
//   * the G lanes of the group load G consecutive column ids (and weights) with ONE coalesced load
//     per lane and broadcast them with warp shuffles -- 1 LDG per lane per G edges instead of 2 per edge;
//   * the next batch of ids is prefetched while the current one is consumed;
//   * feature address = lane base + uint32(col) * row_bytes in one IMAD.WIDE.U32;
//   * multiply and add are the packed fp32x2 instructions of sm_100 (FMUL2 / FADD2): half the FP
//     issue slots, still one IEEE rounding per operation (bit-identical to scalar mul + add);
//   * full batches of U edges run unpredicated, only the last partial batch is masked.
// ------------------------------------------------------------------------------------------
// packed fp32x2 math of sm_100 (FFMA2 / FADD2): one instruction per two floats.  Weighted sums use
// a fused multiply-add (one rounding; ptxas contracts mul.rn + add.rn on f32x2 anyway), unweighted
// sums are plain IEEE adds in stable edge order and therefore bit-identical to PyG-CPU scatter_add_.
__device__ __forceinline__ float2 fma2_rn(float2 a, float2 b, float2 c) {
  unsigned long long r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(r)
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)),
        "l"(reinterpret_cast<unsigned long long&>(c)));
  return reinterpret_cast<float2&>(r);
}
__device__ __forceinline__ float2 add2_rn(float2 a, float2 b) {
  unsigned long long r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return reinterpret_cast<float2&>(r);
}

template <typename T, int EPV, bool HASW>
__device__ __forceinline__ void accum_vec(float2 (&acc)[(EPV + 1) / 2], const Raw<T, EPV>& raw, float w) {
  if constexpr (EPV == 1) {
    const float f = raw.pair(0).x;
    acc[0].x = HASW ? __fmaf_rn(w, f, acc[0].x) : __fadd_rn(acc[0].x, f);
  } else {
#pragma unroll
    for (int i = 0; i < EPV / 2; ++i)
      acc[i] = HASW ? fma2_rn(make_float2(w, w), raw.pair(i), acc[i]) : add2_rn(acc[i], raw.pair(i));
  }
}

// address of a gathered row for this lane: base + col * row_bytes in ONE IMAD.WIDE.U32
__device__ __forceinline__ const char* row_addr(const char* base, uint32_t c, uint32_t row_bytes) {
  unsigned long long r;
  asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(r) : "r"(c), "r"(row_bytes), "l"((unsigned long long)base));
  return reinterpret_cast<const char*>(r);
}

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ uint64_t make_policy(int kind) {
  uint64_t pol;
  if (kind == 2) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  else if (kind == 1) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  else asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

// gather one 16-byte vector of feature row `ctag` (act = false: no load, zeros; the tail batches pass it -- without the
// zero fill the predicated load's destination would stay live through the full-batch loop: +6 registers, spills).  Every lane
// loads: a lane beyond F has its base on the row's LAST vector (lane_bases), so there is no predicate, branch or zero fill
// in the full-batch loop.  Where another lane of the same instruction reads that vector anyway (every tile whose v-th
// slice holds at least one vector of the row -- all shapes choose_shape() picks for rows of at most 64 vectors) this
// costs no extra line or L1 wavefront.  A slice wholly beyond F (G32 V2: the last tile of a row wider than 64 vectors
// with at most 32 vectors left, e.g. F = 602 fp32, tile 3; or V2 tune words on narrow rows) issues one extra load of an
// already-requested line per edge, which the parent predicated off.
// (Round 1's dummy load of vector 0 did cost a second line per gathered row; profiles/r02_spmm_l1_wavefronts.txt.)
// HINTED: bit 31 of the id selects the policy.  The L2 policy travels in a memory DESCRIPTOR, which is warp-uniform on
// sm_100 (ptxas moves a per-lane policy through R2UR, i.e. silently applies one lane's choice to the whole warp), so
// the choice is expressed as two predicated loads with kernel-uniform policies.  Without HINTED: one plain load, no
// tag mask, no policy descriptor.
template <typename T, int EPV, bool HINTED>
__device__ __forceinline__ void gather_vec(Raw<T, EPV>& raw, const char* base, uint32_t ctag, uint32_t row_bytes,
                                           uint64_t pol_hot, uint64_t pol_cold, bool act) {
  const T* q = reinterpret_cast<const T*>(row_addr(base, HINTED ? ctag & 0x7fffffffu : ctag, row_bytes));
  if (!act) raw.zero();
  else if (!HINTED) raw.load(q);
  else if (ctag & 0x80000000u) raw.load_hint(q, pol_hot);
  else raw.load_hint(q, pol_cold);
}

// Column ids (and weights) of a batch reach the lanes of a group through SHARED MEMORY: each lane loads one id
// with a coalesced streaming load, the warp stores its 32 ids to its own 128-byte slot, and every lane then reads
// the UE ids of a step with ONE broadcast LDS (8 lanes of a group read the same address, the 4 groups of a warp
// 4 different ones: one wavefront).  The round-1 kernel broadcast each id with a warp shuffle; on sm_100 a SHFL
// occupies the LSU data pipe for 4 wavefronts, and with the gathers L2-resident that pipe is the limiter
// (l1tex__data_pipe_lsu_wavefronts 74 % busy, 37 % of it shuffles; profiles/r02_spmm_l1_wavefronts.txt).
struct IdStage {
  int32_t* ids;     // this warp's 32 ids   (shared memory)
  float* wts;       // this warp's 32 weights
};

template <int N>
__device__ __forceinline__ void lds_wts(const float* p, float (&w)[N]) {
  if constexpr (N == 8) {
    const float4 v = *reinterpret_cast<const float4*>(p), x = *reinterpret_cast<const float4*>(p + 4);
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w; w[4] = x.x; w[5] = x.y; w[6] = x.z; w[7] = x.w;
  } else if constexpr (N == 4) {
    const float4 v = *reinterpret_cast<const float4*>(p);
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
  } else if constexpr (N == 2) {
    const float2 v = *reinterpret_cast<const float2*>(p);
    w[0] = v.x; w[1] = v.y;
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) w[i] = p[i];
  }
}

// The loop is WARP-uniform: every lane of the warp runs the same number of batches (the maximum
// over the warp's groups; with the degree-sorted row schedule the groups of a warp have equal
// lengths, so nothing is wasted), which lets full batches run without a single predicate.
// xb[v]: this lane's base pointer for its v-th vector (a lane beyond F: the row's last vector, see gather_vec).
// PIPE: software-pipelined main loop -- the features of step j+1 are requested BEFORE the math of
// step j and consumed in the next loop iteration, so UE*V loads per lane are always in flight
// whatever order ptxas picks inside one iteration (without it, ptxas 12.9 sinks each LDG next to
// its FFMA2 and serialises the gathers).
template <typename T, int EPV, int G, int V, int U, bool HASW, bool PIPE, bool HINTED>
__device__ __forceinline__ void accumulate_edges(const SpmmParams& p, int64_t k0, int64_t k1, const char* const (&xb)[V],
                                                 const bool (&active)[V], int gl, const IdStage& sm,
                                                 float2 (&acc)[V][(EPV + 1) / 2]) {
  constexpr int UE = (U < G) ? U : G;   // edges per inner step (a batch holds G ids)
  constexpr bool LANE_BRANCH = HASW && EPV == 8;   // weighted bf16: lanes beyond F skip their load (see accumulate_range)
  bool act[V];
#pragma unroll
  for (int v = 0; v < V; ++v) act[v] = LANE_BRANCH ? active[v] : true;
  const uint32_t row_bytes = (uint32_t)(p.ldx * (int64_t)sizeof(T));
  uint64_t pol_hot = 0, pol_cold = 0;
  if constexpr (HINTED) {
    pol_hot = make_policy(p.pol_hot);
    pol_cold = make_policy(p.pol_cold);
  }
  const int32_t* __restrict__ col = p.w.col + k0;
  const float* __restrict__ val = HASW ? p.val + k0 : nullptr;
  const int len = (k1 > k0) ? (int)(k1 - k0) : 0;          // <= chunk / long sub-range, fits int
  const int maxlen = __reduce_max_sync(FULL, len);
  if (maxlen == 0) return;
  const int lane = threadIdx.x & 31;
  const int32_t* gid_ = sm.ids + (lane - gl);              // this group's G slots
  const float* gwt_ = sm.wts + (lane - gl);
  int32_t cn = (gl < len) ? ld_stream(col + gl, p.stream) : 0;   // lanes past the row hold id 0: a valid row
  float wn = 0.f;
  if constexpr (HASW) wn = (gl < len) ? ld_stream(val + gl, p.stream) : 0.f;
  for (int off = 0; off < maxlen; off += G) {
    int nb = len - off;
    nb = nb < 0 ? 0 : (nb > G ? G : nb);
    __syncwarp();                                   // everybody has read the previous batch
    sm.ids[lane] = cn;
    if constexpr (HASW) sm.wts[lane] = wn;
    __syncwarp();
    cn = 0;
    wn = 0.f;
    if (off + G + gl < len) {                       // prefetch the next batch of ids / weights
      cn = ld_stream(col + off + G + gl, p.stream);
      if constexpr (HASW) wn = ld_stream(val + off + G + gl, p.stream);
    }
    if (__all_sync(FULL, nb == G)) {                // every group has a full batch: no predicates
      if constexpr (PIPE && (G / UE) >= 2) {
        Raw<T, EPV> cur[UE][V];
        {
          uint32_t c[UE];
          lds_ids<UE>(gid_, c);
#pragma unroll
          for (int u = 0; u < UE; ++u)
#pragma unroll
            for (int v = 0; v < V; ++v) gather_vec<T, EPV, HINTED>(cur[u][v], xb[v], c[u], row_bytes, pol_hot, pol_cold, act[v]);
        }
#pragma unroll 1
        for (int j = 0; j < G; j += UE) {
          Raw<T, EPV> nxt[UE][V];
          const int jn = (j + UE < G) ? j + UE : j;   // last step re-requests itself (L1 hit, result unused)
          uint32_t c[UE];
          lds_ids<UE>(gid_ + jn, c);
#pragma unroll
          for (int u = 0; u < UE; ++u)
#pragma unroll
            for (int v = 0; v < V; ++v) gather_vec<T, EPV, HINTED>(nxt[u][v], xb[v], c[u], row_bytes, pol_hot, pol_cold, act[v]);
          float w[UE];
          if constexpr (HASW) lds_wts<UE>(gwt_ + j, w);
#pragma unroll
          for (int u = 0; u < UE; ++u) {
#pragma unroll
            for (int v = 0; v < V; ++v) accum_vec<T, EPV, HASW>(acc[v], cur[u][v], HASW ? w[u] : 1.0f);
          }
#pragma unroll
          for (int u = 0; u < UE; ++u)
#pragma unroll
            for (int v = 0; v < V; ++v) cur[u][v] = nxt[u][v];
        }
      } else {
#pragma unroll 1
        for (int j = 0; j < G; j += UE) {
          Raw<T, EPV> raw[UE][V];
          uint32_t c[UE];
          lds_ids<UE>(gid_ + j, c);
#pragma unroll
          for (int u = 0; u < UE; ++u)
#pragma unroll
            for (int v = 0; v < V; ++v) gather_vec<T, EPV, HINTED>(raw[u][v], xb[v], c[u], row_bytes, pol_hot, pol_cold, act[v]);
          float w[UE];
          if constexpr (HASW) lds_wts<UE>(gwt_ + j, w);
#pragma unroll
          for (int u = 0; u < UE; ++u) {
#pragma unroll
            for (int v = 0; v < V; ++v) accum_vec<T, EPV, HASW>(acc[v], raw[u][v], HASW ? w[u] : 1.0f);
          }
        }
      }
    } else {                                        // tail batches: per-group predicates
      const int nbmax = __reduce_max_sync(FULL, nb);
#pragma unroll 1
      for (int j = 0; j < nbmax; j += UE) {
        Raw<T, EPV> raw[UE][V];
        uint32_t c[UE];
        lds_ids<UE>(gid_ + j, c);
#pragma unroll
        for (int u = 0; u < UE; ++u) {
#pragma unroll
          for (int v = 0; v < V; ++v)   // an edge past the group's row loads nothing (zeros) and is not added
            gather_vec<T, EPV, HINTED>(raw[u][v], xb[v], c[u], row_bytes, pol_hot, pol_cold, act[v] && (j + u < nb));
        }
        float w[UE];
        if constexpr (HASW) lds_wts<UE>(gwt_ + j, w);
#pragma unroll
        for (int u = 0; u < UE; ++u) {
          if (j + u < nb) {
#pragma unroll
            for (int v = 0; v < V; ++v) accum_vec<T, EPV, HASW>(acc[v], raw[u][v], HASW ? w[u] : 1.0f);
          }
        }
      }
    }
  }
}

// hinted is kernel-uniform: one branch per launch, both edge loops inlined into the same kernel.  Weighted bf16 sums
// keep the previous loop (the hinted form, which also serves untagged graphs, with a per-lane branch): two loops in one
// kernel cost them 12 registers, and at 5 CTAs/SM (20-byte spill) or at 4 CTAs/SM the weighted bf16 hop of the
// papers100M-shaped block ran 7 % / 5 % slower (profiles/r04_spmm_untagged_gather.txt, section 6).
template <typename T, int EPV, int G, int V, int U, bool HASW, bool PIPE>
__device__ __forceinline__ void accumulate_range(const SpmmParams& p, int64_t k0, int64_t k1, const char* const (&xb)[V],
                                                 const bool (&active)[V], int gl, const IdStage& sm,
                                                 float2 (&acc)[V][(EPV + 1) / 2]) {
  if (HASW && EPV == 8) accumulate_edges<T, EPV, G, V, U, HASW, PIPE, true>(p, k0, k1, xb, active, gl, sm, acc);
  else if (p.hinted) accumulate_edges<T, EPV, G, V, U, HASW, PIPE, true>(p, k0, k1, xb, active, gl, sm, acc);
  else accumulate_edges<T, EPV, G, V, U, HASW, PIPE, false>(p, k0, k1, xb, active, gl, sm, acc);
}

// epilogue for EPV consecutive features [f, f+EPV) of row `row`
// push = false: the caller pushes the row to the peers itself (bulk copy of the staged row); s returns what is pushed
template <typename T, int EPV>
__device__ __forceinline__ void epilogue_store(const SpmmParams& p, int64_t row, int f, float (&s)[EPV], bool push = true) {
  const rgbmp_epilogue_t& ep = p.ep;
  const float rs = ep.row_scale ? __ldg(ep.row_scale + row) : 1.0f;
  const bool reset = (ep.reset_when != 0) && ep.reset_mask[row];
  float rv[EPV];
  if (reset) {
#pragma unroll
    for (int i = 0; i < EPV; ++i) rv[i] = (f + i < p.F) ? ep.reset_val[row * ep.ld_reset + f + i] : 0.f;
  }
  if (ep.acc_in) {
    Raw<T, EPV> ar;
    float a[EPV];
    ar.load_stream(reinterpret_cast<const T*>(ep.acc_in) + row * ep.ld_acc + f);
    ar.unpack(a);
#pragma unroll
    for (int i = 0; i < EPV; ++i) s[i] = __fadd_rn(a[i], s[i]);
  }
  float t[EPV];
  if (ep.T) {
    Raw<T, EPV> tr;
    if (p.stream) tr.load_stream(reinterpret_cast<const T*>(ep.T) + row * ep.ldt + f);
    else tr.load(reinterpret_cast<const T*>(ep.T) + row * ep.ldt + f);
    tr.unpack(t);
  }
  ep_apply<EPV>(ep, s, rs, reset, rv, t);
  if (p.Y) {
    const int64_t yrow = ep.row_map ? (int64_t)__ldg(ep.row_map + row) : row;
    Raw<T, EPV>::store(reinterpret_cast<T*>(p.Y) + yrow * p.ldy + f, s, p.stream);
  }
  if (ep.out2_scale) {                     // pre-scaled copy (folded D^-1/2): what the NEXT hop gathers
    const float s2 = __ldg(ep.out2_scale + row);
#pragma unroll
    for (int i = 0; i < EPV; ++i) s[i] = __fmul_rn(s2, s[i]);
    if (ep.Y2) Raw<T, EPV>::store(reinterpret_cast<T*>(ep.Y2) + row * ep.ldy2 + f, s, p.stream);
  }
  if (push)
    for (int q = 0; q < ep.n_peers; ++q)   // fused all-gather: push the finished row to every peer over NVLink
      Raw<T, EPV>::store(reinterpret_cast<T*>(ep.peer_out[q]) + (ep.peer_row0 + row) * ep.ld_peer + f, s, 0);
}

constexpr int SPMM_THREADS = 256;
// Min CTAs per SM a variant is compiled for (register cap = 65536 / (256 * minb)).  ptxas is generous
// with registers once the epilogue grew (86-93 for the main products variant -> 2 CTAs/SM, 4.16 ms instead
// of 2.95 ms per hop); capping the variants whose in-flight gather data needs <= 32 registers at 64
// costs no spills and restores 4 CTAs/SM.  Variants with more data in flight get proportionally more; the leanest
// (one vector, 4 edges) fit 5 CTAs/SM in 48 registers without spills (6 CTAs / 40 registers spill 16 bytes and gain
// nothing more: 2.77 vs 2.74 ms on the products-shaped hop).  With unpredicated gathers (round 4) one vector and 8
// edges needs 62 registers: 4 CTAs/SM, no spills (capped at 48 for 5 CTAs/SM it spills 224 bytes).
template <int EPV, int V, int U, bool PIPE>
constexpr int spmm_minb() {
  constexpr int raw = ((EPV > 1) ? 4 : 1) * V * U * (PIPE ? 2 : 1);   // registers holding gathered vectors
  constexpr int need = raw + V * EPV;                                  // + fp32 accumulators
  return need <= 24 ? 5 : (need <= 40 ? 4 : (need <= 56 ? 3 : (need <= 72 ? 2 : 1)));
}

// per-lane vector bases: lane l of the group owns vectors l, l+G, ... of the feature tile.  A vector beyond F
// (active[v] = false) is gathered from the row's last vector and its sum never stored.
template <typename T, int EPV, int G, int V>
__device__ __forceinline__ void lane_bases(const SpmmParams& p, int f0, const char* (&xb)[V], bool (&active)[V]) {
  const int last = (p.F - 1) / EPV * EPV;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int f = f0 + v * G * EPV;
    active[v] = f < p.F;
    xb[v] = reinterpret_cast<const char*>(p.X) + (size_t)(active[v] ? f : last) * sizeof(T);
  }
}

// short rows: one group of G lanes per row.  blockIdx.y = feature tile of G*V*EPV elements.
// Rows are taken in `row_order` (degree-sorted inside windows, built once per graph) so that the
// groups sharing a warp run rows of equal length -- no idle issue slots from divergent trip counts.
template <typename T, int EPV, int G, int V, int U, bool HASW, bool PIPE>
__global__ void __launch_bounds__(SPMM_THREADS, spmm_minb<EPV, V, U, PIPE>()) spmm_rows_kernel(const SpmmParams p) {
  const int gl = threadIdx.x % G;
  int64_t row, k0, k1;
  short_row<G, SPMM_THREADS>(p.w, row, k0, k1);
  const int f0 = blockIdx.y * (G * V * EPV) + gl * EPV;
  const char* xb[V];
  bool active[V];
  float2 acc[V][(EPV + 1) / 2];
  lane_bases<T, EPV, G, V>(p, f0, xb, active);
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int i = 0; i < (EPV + 1) / 2; ++i) acc[v][i] = make_float2(0.f, 0.f);
  __shared__ __align__(16) int32_t sm_ids[SPMM_THREADS];
  __shared__ __align__(16) float sm_wts[HASW ? SPMM_THREADS : 4];
  const IdStage stage = {sm_ids + (threadIdx.x & ~31), sm_wts + (HASW ? (threadIdx.x & ~31) : 0)};
  accumulate_range<T, EPV, G, V, U, HASW, PIPE>(p, k0, k1, xb, active, gl, stage, acc);
  if (row < 0 || (p.ep.skip_empty && k1 == k0)) return;
  // Fused all-gather, bulk form: the group's lanes lay the finished (pre-scaled) row out in shared memory and ONE lane hands
  // it to the TMA engine once per peer (cp.async.bulk shared -> global over NVLink): full-line writes issued off the LSU
  // path.  Optional (rgbmp_set_push_bulk): measured no faster than 16-byte st.global per lane at 2 and 4 GPUs.
  extern __shared__ __align__(16) unsigned char sm_push[];          // [SPMM_THREADS * V] 16-byte vectors when pushing in bulk
  const bool bulk = (EPV > 1) && p.push_bulk && p.ep.n_peers > 0;
  T* my_stage = reinterpret_cast<T*>(sm_push) + (size_t)(threadIdx.x / G) * (G * V * EPV);
#pragma unroll
  for (int v = 0; v < V; ++v) {
    if (active[v]) {
      float s[EPV];
#pragma unroll
      for (int i = 0; i < EPV; ++i) s[i] = (i & 1) ? acc[v][i / 2].y : acc[v][i / 2].x;
      epilogue_store<T, EPV>(p, row, f0 + v * G * EPV, s, !bulk);
      if (bulk) Raw<T, EPV>::store(my_stage + (v * G + gl) * EPV, s, 0);
    }
  }
  if (bulk) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // my generic-proxy writes, before the async proxy reads them
    const int lane = threadIdx.x & 31;
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane - gl));
    __syncwarp(gmask);
    if (gl == 0) {
      const int ftile = blockIdx.y * (G * V * EPV);
      const int nv = min(G * V, (p.F - ftile + EPV - 1) / EPV);        // vectors of this tile that exist
      const uint32_t src = (uint32_t)__cvta_generic_to_shared(my_stage);
      const uint32_t bytes = (uint32_t)nv * 16u;
      for (int q = 0; q < p.ep.n_peers; ++q) {
        T* dst = reinterpret_cast<T*>(p.ep.peer_out[q]) + (p.ep.peer_row0 + row) * p.ep.ld_peer + ftile;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the staged row may go once it has been read
    }
  }
}

// long rows: one CTA per work item (<= long_chunk edges of one row); the CTA's groups take
// contiguous sub-ranges, partial sums are reduced through shared memory in a fixed order.
template <typename T, int EPV, int G, int V, int U, bool HASW, bool PIPE>
__global__ void __launch_bounds__(SPMM_THREADS, spmm_minb<EPV, V, U, PIPE>()) spmm_long_kernel(const SpmmParams p) {
  constexpr int Q = SPMM_THREADS / G;      // groups per CTA
  constexpr int W = G * V * EPV;           // feature tile width
  extern __shared__ float sm[];            // [Q][W]
  const int gl = threadIdx.x % G, q = threadIdx.x / G;
  const int64_t item = blockIdx.x;
  int64_t row, k0, k1;
  long_item<G, SPMM_THREADS>(p.w, row, k0, k1);
  const int ftile = blockIdx.y * W;
  const int f0 = ftile + gl * EPV;
  const char* xb[V];
  bool active[V];
  float2 acc[V][(EPV + 1) / 2];
  lane_bases<T, EPV, G, V>(p, f0, xb, active);
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int i = 0; i < (EPV + 1) / 2; ++i) acc[v][i] = make_float2(0.f, 0.f);
  __shared__ __align__(16) int32_t sm_ids[SPMM_THREADS];
  __shared__ __align__(16) float sm_wts[HASW ? SPMM_THREADS : 4];
  const IdStage stage = {sm_ids + (threadIdx.x & ~31), sm_wts + (HASW ? (threadIdx.x & ~31) : 0)};
  accumulate_range<T, EPV, G, V, U, HASW, PIPE>(p, k0, k1, xb, active, gl, stage, acc);
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int i = 0; i < EPV; ++i)
      sm[q * W + (gl + v * G) * EPV + i] = active[v] ? ((i & 1) ? acc[v][i / 2].y : acc[v][i / 2].x) : 0.f;
  __syncthreads();
  for (int t = threadIdx.x; t < W; t += SPMM_THREADS) {
    float s = 0.f;
    for (int qq = 0; qq < Q; ++qq) s = __fadd_rn(s, sm[qq * W + t]);
    if (ftile + t < p.ldpart) p.partial[item * p.ldpart + ftile + t] = s;
  }
}

// combine the items of each long row in order and apply the epilogue (one thread per element)
template <typename T>
__global__ void __launch_bounds__(256) spmm_combine_kernel(const SpmmParams p) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t slot = t / p.F;
  const int f = (int)(t - slot * p.F);
  if (slot >= p.w.n_long) return;
  const int64_t row = p.w.long_rows[slot];
  float s[1] = {0.f};
  for (int32_t it = p.w.long_item_ptr[slot]; it < p.w.long_item_ptr[slot + 1]; ++it)
    s[0] = __fadd_rn(s[0], p.partial[(int64_t)it * p.ldpart + f]);
  epilogue_store<T, 1>(p, row, f, s);
}

template <typename T>
__global__ void __launch_bounds__(256)
row_scale_kernel(const T* __restrict__ X, int64_t ldx, const float* __restrict__ scale, int divide, T* __restrict__ Y,
                 int64_t ldy, int64_t n_rows, int F) {
  const int64_t total = n_rows * F;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    const int64_t r = t / F;
    const int f = (int)(t - r * F);
    const float xv = to_f(X[r * ldx + f]);
    float o[1] = {divide ? __fdiv_rn(xv, scale[r]) : __fmul_rn(scale[r], xv)};
    Raw<T, 1>::store(Y + r * ldy + f, o);
  }
}

// ------------------------------------------------------------------------------------------
// launch dispatch
// ------------------------------------------------------------------------------------------
template <typename T, int EPV, int G, int V, int U, bool HASW, bool PIPE>
int launch_cfg(const SpmmParams& p, cudaStream_t st) {
  constexpr int W = G * V * EPV;
  const size_t push_smem = (EPV > 1 && p.push_bulk && p.ep.n_peers > 0) ? (size_t)SPMM_THREADS * V * 16 : 0;
  return launch_phases(
      p.w, SPMM_THREADS / G, (unsigned)ceil_div(p.F, W), p.F, "spmm kernels",
      [&](dim3 grid) { spmm_rows_kernel<T, EPV, G, V, U, HASW, PIPE><<<grid, SPMM_THREADS, push_smem, st>>>(p); },
      [&](dim3 grid) {
        spmm_long_kernel<T, EPV, G, V, U, HASW, PIPE><<<grid, SPMM_THREADS, (SPMM_THREADS / G) * W * sizeof(float), st>>>(p);
      },
      [&](unsigned blocks) { spmm_combine_kernel<T><<<blocks, 256, 0, st>>>(p); });
}

template <typename T, int EPV, int G, int V, int U, bool PIPE>
int dispatch_w(const SpmmParams& p, cudaStream_t st) {
  return p.val ? launch_cfg<T, EPV, G, V, U, true, PIPE>(p, st) : launch_cfg<T, EPV, G, V, U, false, PIPE>(p, st);
}

// U field of the tune word: 2 / 4 = edges per step; +16 = software-pipelined main loop
// (V >= 3 and U = 8 never won a sweep on B200 and are no longer instantiated)
template <typename T, int EPV, int G, int V>
int dispatch_u(const SpmmParams& p, int U, cudaStream_t st) {
  switch (U) {
    case 2: return dispatch_w<T, EPV, G, V, 2, false>(p, st);
    case 8: return dispatch_w<T, EPV, G, V, 8, false>(p, st);
    case 18: return dispatch_w<T, EPV, G, V, 2, true>(p, st);
    case 20: return dispatch_w<T, EPV, G, V, 4, true>(p, st);
    default: return dispatch_w<T, EPV, G, V, 4, false>(p, st);
  }
}

template <typename T, int EPV, int G>
int dispatch_v(const SpmmParams& p, int V, int U, cudaStream_t st) {
  switch (V) {
    case 1: return dispatch_u<T, EPV, G, 1>(p, U, st);
    default: return dispatch_u<T, EPV, G, 2>(p, U, st);
  }
}

template <typename T, int EPV>
int dispatch_g(const SpmmParams& p, int G, int V, int U, cudaStream_t st) {
  switch (G) {
    case 1: return dispatch_v<T, EPV, 1>(p, V, U, st);
    case 2: return dispatch_v<T, EPV, 2>(p, V, U, st);
    case 4: return dispatch_v<T, EPV, 4>(p, V, U, st);
    case 8: return dispatch_v<T, EPV, 8>(p, V, U, st);
    case 16: return dispatch_v<T, EPV, 16>(p, V, U, st);
    default: return dispatch_v<T, EPV, 32>(p, V, U, st);
  }
}

// per-dtype instantiation units
int spmm_dispatch_f32v(const SpmmParams& p, int G, int V, int U, cudaStream_t st);
int spmm_dispatch_f32s(const SpmmParams& p, int G, int V, int U, cudaStream_t st);
int spmm_dispatch_bf16(const SpmmParams& p, int G, int V, int U, cudaStream_t st);

}  // namespace rgbmp
