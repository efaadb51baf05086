// Counter-based RNG (Philox-4x32-10) + Dirichlet / uniform helpers for the self-play engine.
//
// Replaces the reference's global numpy RNG (lib/mcts.py:56 np.random.dirichlet, lib/utils.py:66,83
// np.random.choice).  Streams are addressed, not consumed: (seed, game uid, ply, descent, action)
// -> value, so any rank / launch order reproduces the same games.  The numpy bit-stream itself is
// not reproduced (it cannot be, it is MT19937 + legacy gamma); parity tests either inject the
// noise/uniforms or export the values generated here into the oracle.
#pragma once
#include <math.h>
#include <stdint.h>
#include "rules.cuh"

namespace caro {

struct Philox4 {
  uint32_t v[4];
};

CARO_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32); }

CARO_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  Philox4 o;
  o.v[0] = c0; o.v[1] = c1; o.v[2] = c2; o.v[3] = c3;
  return o;
}

// uniform in (0,1), 24 bits
CARO_HD float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }
// uniform in [0,1), 53 bits
CARO_HD double u01d(uint32_t hi, uint32_t lo) {
  const uint64_t x = (((uint64_t)hi << 32) | lo) >> 11;
  return (double)x * (1.0 / 9007199254740992.0);
}

// Stream tags
enum : uint32_t { kStreamDirichlet = 0x44495243u, kStreamChoice = 0x43484F49u, kStreamFirst = 0x46495253u,
                  kStreamResign = 0x52455347u, kStreamGumbel = 0x47554D42u };

// Gumbel(0, 1) draw of the Gumbel root search: g = -log(-log(u)) in double, u = k * 2^-53 from the top 53 bits k of the
// Philox word pair, with k = 0 replaced by 1/2 so that u lies in the open interval (0, 1) and g is always finite.
// Addressed by (seed, game uid, search index, ply, action).
CARO_HD double gumbel_draw(uint32_t seed_lo, uint32_t seed_hi, uint64_t uid, uint32_t search_index, uint32_t ply,
                           uint32_t action) {
  const Philox4 r = philox4x32_10((uint32_t)uid, (uint32_t)(uid >> 32), search_index, (ply << 8) | action,
                                  seed_lo ^ kStreamGumbel, seed_hi);
  const uint64_t k = ((((uint64_t)r.v[0]) << 32) | r.v[1]) >> 11;
  const double u = (k == 0 ? 0.5 : (double)k) * (1.0 / 9007199254740992.0);
  return -log(-log(u));
}

// Device code uses the fast-math intrinsics: the noise only has to be distributed correctly, and whatever is
// generated is what both the engine and (through noise_out) the oracle consume.
#if defined(__CUDA_ARCH__)
#define CARO_LOGF(x) __logf(x)
#define CARO_EXPF(x) __expf(x)
#define CARO_COSF(x) __cosf(x)
#else
#define CARO_LOGF(x) logf(x)
#define CARO_EXPF(x) expf(x)
#define CARO_COSF(x) cosf(x)
#endif

// Gamma(alpha, 1) for alpha < 1 via Marsaglia-Tsang on alpha+1 (with the x^4 squeeze) and the U^(1/alpha)
// boost.  `c0..c2` address the stream; the rejection loop walks c3.
CARO_HD float gamma_small(float alpha, uint32_t k0, uint32_t k1, uint32_t c0, uint32_t c1, uint32_t c2) {
  const float d = alpha + 1.0f - 1.0f / 3.0f;
  const float c = 1.0f / sqrtf(9.0f * d);
  const float inv_alpha = 1.0f / alpha;
  float g = d;  // fallback if the loop somehow exhausts
  for (uint32_t it = 0; it < 64u; ++it) {
    const Philox4 r = philox4x32_10(c0, c1, c2, it, k0, k1);
    // Box-Muller normal from r.v[0], r.v[1]
    const float u1 = u01(r.v[0]), u2 = u01(r.v[1]);
    const float x = sqrtf(-2.0f * CARO_LOGF(u1)) * CARO_COSF(6.283185307179586f * u2);
    float v = 1.0f + c * x;
    if (v <= 0.0f) continue;
    v = v * v * v;
    const float u = u01(r.v[2]);
    const float x2 = x * x;
    if (u < 1.0f - 0.0331f * x2 * x2 || CARO_LOGF(u) < 0.5f * x2 + d - d * v + d * CARO_LOGF(v)) {
      // boost: Gamma(alpha) = Gamma(alpha+1) * U^(1/alpha)
      g = d * v * CARO_EXPF(CARO_LOGF(u01(r.v[3])) * inv_alpha);
      break;
    }
  }
  return g;
}

}  // namespace caro
