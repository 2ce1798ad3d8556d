// Counter-based attention dropout: the keep rule shared by the fused attention kernels (csrc/att.cu), the mask
// kernel of the unfused paths (rgbmp_dropout_mask) and, compiled as host code, the test that checks it against the
// numpy restatement (oracle/philox.py).  Also the draws of SuperGAT's edge and negative sampling (below).
//
// For edge e (its id in the edited edge list) and head h:
//   u    = Philox4x32-10(counter = (e, h, 0, 0), key = (seed & 0xffffffff, seed >> 32)).word0
//   drop iff u < thresh,  thresh = floor(p * 2^32) computed on the host (p == 1: thresh = 2^32 - 1 and scale = 0)
//   mask = drop ? 0 : scale,  scale = float32(1 / (1 - p))
// Philox4x32-10 is Salmon et al., "Parallel random numbers: as easy as 1, 2, 3" (SC'11), as in Random123.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define RGBMP_HD __host__ __device__ __forceinline__
#else
#define RGBMP_HD inline
#endif

namespace rgbmp {

constexpr uint32_t PHILOX_M0 = 0xD2511F53u, PHILOX_M1 = 0xCD9E8D57u;
constexpr uint32_t PHILOX_W0 = 0x9E3779B9u, PHILOX_W1 = 0xBB67AE85u;

// The 64-bit seed split into the two key words, once per thread: the round keys k + r * W are then immediates
// added to these two registers.
struct PhiloxKey {
  uint32_t k0, k1;
};

RGBMP_HD PhiloxKey philox_key(uint64_t seed) {
  PhiloxKey k;
  k.k0 = (uint32_t)(seed & 0xffffffffu);
  k.k1 = (uint32_t)(seed >> 32);
  return k;
}

RGBMP_HD void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#if defined(__CUDA_ARCH__)
  hi = __umulhi(a, b);
  lo = a * b;
#else
  const uint64_t p = (uint64_t)a * (uint64_t)b;
  hi = (uint32_t)(p >> 32);
  lo = (uint32_t)p;
#endif
}

// All four output words of Philox4x32-10 (the known-answer test reads them).
RGBMP_HD void philox4x32_10(const uint32_t (&ctr)[4], PhiloxKey key, uint32_t (&out)[4]) {
  uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
  uint32_t k0 = key.k0, k1 = key.k1;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(PHILOX_M0, c0, hi0, lo0);
    philox_mulhilo(PHILOX_M1, c2, hi1, lo1);
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += PHILOX_W0;
    k1 += PHILOX_W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// word 0 for counter (e, h, 0, 0); the compiler drops the work that only feeds the other three words
RGBMP_HD uint32_t dropout_bits(PhiloxKey key, uint32_t e, uint32_t h) {
  const uint32_t ctr[4] = {e, h, 0u, 0u};
  uint32_t out[4];
  philox4x32_10(ctr, key, out);
  return out[0];
}

// the multiplier of edge e, head h: 0 (dropped) or scale (kept)
RGBMP_HD float dropout_mult(PhiloxKey key, uint32_t e, uint32_t h, uint32_t thresh, float scale) {
  return dropout_bits(key, e, h) < thresh ? 0.0f : scale;
}

// SuperGAT's self-supervised sampling (csrc/supergat_loss.cu).  Counter word 2 tells the streams apart: 0 attention
// dropout, 1 the positive keep rule, 2 the negative candidates.
//   positive edge e is dropped iff Philox(counter (e, 0, 1, 0)).word0 < thresh,  thresh = floor((1 - ratio) * 2^32)
//   negative candidate k of round r: (w0, w1, w2, w3) = Philox(counter (k, r, 2, 0)),
//     row = umulhi64(w1:w0, N), col = umulhi64(w3:w2, N)
// The 64-bit multiply-high maps a uniform 64-bit word onto [0, N) with a bias of at most N / 2^64 per value
// (< 2^-33 for N < 2^31): every id is hit by floor(2^64 / N) or that plus one of the 2^64 words.
RGBMP_HD uint32_t edge_sample_bits(PhiloxKey key, uint32_t e) {
  const uint32_t ctr[4] = {e, 0u, 1u, 0u};
  uint32_t out[4];
  philox4x32_10(ctr, key, out);
  return out[0];
}

// thresh is 64-bit so that ratio 0 (thresh = 2^32) drops every edge
RGBMP_HD bool edge_sample_keep(PhiloxKey key, uint32_t e, uint64_t thresh) {
  return thresh == 0 || (uint64_t)edge_sample_bits(key, e) >= thresh;
}

RGBMP_HD uint64_t umulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * (unsigned __int128)b) >> 64);
#endif
}

RGBMP_HD void neg_candidate(PhiloxKey key, uint32_t k, uint32_t round, uint64_t n, uint32_t& row, uint32_t& col) {
  const uint32_t ctr[4] = {k, round, 2u, 0u};
  uint32_t w[4];
  philox4x32_10(ctr, key, w);
  row = (uint32_t)umulhi64(((uint64_t)w[1] << 32) | w[0], n);
  col = (uint32_t)umulhi64(((uint64_t)w[3] << 32) | w[2], n);
}

}  // namespace rgbmp
