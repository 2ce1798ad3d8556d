// The fused epilogue rgbmp_epilogue_t as the library reads it: the rules rgbmp_spmm and rgbmp_khop check it against, and
// the arithmetic the SpMM and the one-cluster K-hop kernels apply to a finished row sum.  Each kernel loads the operands
// (row scale, teleport row, reset row) its own way; the order of operations lives here only, so both give the same bits.
#pragma once
#include "common.cuh"

namespace rgbmp {

enum : unsigned {
  // rgbmp_khop: the driver owns each hop's stores (Y2 carries the next hop's input) and every hop rewrites every row,
  // so Y2, acc_in, skip_empty and peers have no meaning there
  EP_KHOP = 1,
  EP_HOPS = 2,  // rgbmp_khop with `hops`: every hop's output is kept, in the graph's own naming
};

// The epilogue rules of include/rgbmp.h; runs before any device is selected.  *out = the checked copy of *ep, or the
// identity epilogue {a = 1} when ep is NULL.  has_y: the call stores to Y.
inline int check_epilogue(const rgbmp_epilogue_t* ep, int F, bool has_y, const char* fn, unsigned rules,
                          rgbmp_epilogue_t* out) {
  rgbmp_epilogue_t e = {};
  e.a = 1.0f;
  if (ep) e = *ep;
  if (e.reset_when < 0 || e.reset_when > 2) return fail(RGBMP_EINVAL, "%s: bad reset_when %d", fn, e.reset_when);
  if (e.reset_when != 0 && (!e.reset_mask || !e.reset_val || e.ld_reset < F))
    return fail(RGBMP_EINVAL, "%s: reset rows need reset_mask, reset_val and ld_reset >= F", fn);
  if (e.T && e.ldt < F) return fail(RGBMP_EINVAL, "%s: T needs ldt >= F", fn);
  if (e.Y2 && (!e.out2_scale || e.ldy2 < F)) return fail(RGBMP_EINVAL, "%s: Y2 needs out2_scale and ldy2 >= F", fn);
  if (e.acc_in && e.ld_acc < F) return fail(RGBMP_EINVAL, "%s: acc_in needs ld_acc >= F", fn);
  if (e.n_peers < 0 || e.n_peers > RGBMP_MAX_PEERS) return fail(RGBMP_EINVAL, "%s: bad n_peers %d", fn, e.n_peers);
  for (int q = 0; q < e.n_peers; ++q) {
    if (!e.peer_out[q]) return fail(RGBMP_EINVAL, "%s: null peer buffer %d", fn, q);
    if ((((uintptr_t)e.peer_out[q]) & 15) != 0) return fail(RGBMP_EALIGN, "%s: peer buffer %d not 16-byte aligned", fn, q);
  }
  if (e.n_peers > 0 && e.ld_peer < F) return fail(RGBMP_EINVAL, "%s: peers need ld_peer >= F", fn);
  if (e.row_map && (e.n_peers > 0 || e.acc_in || e.reset_when != 0))
    return fail(RGBMP_EINVAL, "%s: row_map does not combine with peers, acc_in or reset rows", fn);
  if (!has_y && !e.Y2 && e.n_peers == 0) return fail(RGBMP_EINVAL, "%s: no output", fn);
  if ((rules & EP_KHOP) && (e.Y2 || e.acc_in || e.skip_empty || e.n_peers > 0))
    return fail(RGBMP_EINVAL, "%s: Y2, acc_in, skip_empty and peers are not K-hop epilogue fields", fn);
  if ((rules & EP_HOPS) && e.row_map) return fail(RGBMP_EINVAL, "%s: row_map does not combine with hops", fn);
  *out = e;
  return 0;
}

// Row scale or divide, reset-before, a * v + b * T, clamp, reset-after, for the N features s[] of one row.
// rs = row_scale[row] (read only with ep.row_scale), reset = this row is a reset row (only with ep.reset_when != 0),
// rv = its reset values (read only when reset), t = its teleport values (read only with ep.T).
template <int N>
__device__ __forceinline__ void ep_apply(const rgbmp_epilogue_t& ep, float (&s)[N], float rs, bool reset,
                                         const float (&rv)[N], const float (&t)[N]) {
#pragma unroll
  for (int i = 0; i < N; ++i) {
    float v = ep.row_scale ? (ep.row_div ? __fdiv_rn(s[i], rs) : __fmul_rn(rs, s[i])) : s[i];
    if (reset && ep.reset_when == 1) v = rv[i];
    v = __fmul_rn(ep.a, v);
    if (ep.T) v = __fadd_rn(v, __fmul_rn(ep.b, t[i]));
    if (ep.clamp) v = fminf(fmaxf(v, ep.lo), ep.hi);
    if (reset && ep.reset_when == 2) v = rv[i];
    s[i] = v;
  }
}

}  // namespace rgbmp
