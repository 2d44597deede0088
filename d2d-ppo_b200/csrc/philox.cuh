// The project's one random stream layout: Philox4x32-10 (Salmon et al., SC'11) and every way a kernel takes draws from
// it.  Each function names its counterpart in oracle/philox_np.py, the numpy restatement the parity tests compare with.
//   counter  (env_global_index, timestep, device | purpose << 16, block)          the generator's c0 .. c3
//   key      the 64-bit seed, as the round keys k + r * W (PhiloxKey)              _key
//   16-bit lane c of a call: word c / 2, high half when c is odd                  lanes16
//   32-bit word of device k: word k % 4 of the call whose device field is k / 4   word32
//   1-bit draw of device k (single-channel env): lane k % 8 of the call k / 8     lane16_shared
#pragma once
#include <stdint.h>

#include "../../include/d2d_b200.h"

namespace d2d {

constexpr uint32_t kPurposeSwitch = 0u, kPurposeArrival = 1u, kPurposePolicy = 2u;
constexpr uint32_t kEnvLevelDevice = 0xFFFFu;

// the round keys (k0 + r * W0, k1 + r * W1) of a 64-bit seed: carried by value in kernel arguments, so every key XOR
// reads a constant-bank operand
struct PhiloxKey {
  uint32_t rk0[10], rk1[10];
};

inline PhiloxKey philox_key(uint64_t seed) {   // _key
  PhiloxKey k;
  for (int r = 0; r < 10; ++r) {
    k.rk0[r] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
    k.rk1[r] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
  }
  return k;
}

// rounds R0 .. 9 of Philox4x32-10 on the state (c0, c1, c2, c3)
template <int R0>
__device__ __forceinline__ uint4 philox_rounds(const PhiloxKey& k, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
#pragma unroll
  for (int r = R0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k.rk0[r];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k.rk1[r];
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
  }
  return make_uint4(c0, c1, c2, c3);
}

// one call of the generator (the oracle's Philox4x32-10 function)
__device__ __forceinline__ uint4 philox(const PhiloxKey& k, uint32_t env, uint32_t t, uint32_t dev_purpose,
                                        uint32_t blk) {
  return philox_rounds<0>(k, env, t, dev_purpose, blk);
}

// A call split after its first two rounds, for callers that draw many counters (env, t, dp, blk) with the same env
// and blk.  With M0 = 0xD2511F53, M1 = 0xCD9E8D57 and hi / lo the halves of the 64-bit product, round 0 gives
//   c0 = hi(M1 dp) ^ t ^ rk0[0] =: A      c1 = lo(M1 dp)      c2 = hi(M0 env) ^ blk ^ rk1[0] =: X      c3 = lo(M0 env)
// and round 1 multiplies A and X:
//   c0 = hi(M1 X) ^ rk0[1] ^ lo(M1 dp)    c1 = lo(M1 X)       c2 = lo(M0 env) ^ rk1[1] ^ hi(M0 A)      c3 = lo(M0 A).
// So after two rounds the state is three words of (env, blk) (PhiloxEnvHead, once per thread) XOR three words of
// (t, dp) (PhiloxCallHead, warp-uniform; lo(M1 dp) is a constant for a compile-time dp), and a call continues at round 2.
// tests/test_philox_prefix.py restates the split in numpy.
struct PhiloxEnvHead {
  uint32_t e0, e1, e2;
};
struct PhiloxCallHead {
  uint32_t u0, u2, u3;
};

__device__ __forceinline__ PhiloxEnvHead philox_env_head(const PhiloxKey& k, uint32_t env, uint32_t blk) {
  const uint64_t p0 = (uint64_t)0xD2511F53u * env;
  const uint32_t x = (uint32_t)(p0 >> 32) ^ blk ^ k.rk1[0];
  const uint64_t p1 = (uint64_t)0xCD9E8D57u * x;
  return {(uint32_t)(p1 >> 32) ^ k.rk0[1], (uint32_t)p1, (uint32_t)p0 ^ k.rk1[1]};
}

__device__ __forceinline__ PhiloxCallHead philox_call_head(const PhiloxKey& k, uint32_t t, uint32_t dev_purpose) {
  const uint64_t p1 = (uint64_t)0xCD9E8D57u * dev_purpose;
  const uint32_t c0 = (uint32_t)(p1 >> 32) ^ t ^ k.rk0[0];
  const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
  return {(uint32_t)p1, (uint32_t)(p0 >> 32), (uint32_t)p0};
}

// philox(k, env, t, dp, blk) == philox(k, philox_env_head(k, env, blk), philox_call_head(k, t, dp))
__device__ __forceinline__ uint4 philox(const PhiloxKey& k, const PhiloxEnvHead& e, const PhiloxCallHead& u) {
  return philox_rounds<2>(k, e.e0 ^ u.u0, e.e1, e.e2 ^ u.u2, u.u3);
}

// ---- 16-bit lanes (lanes16, thr16) ----
// Bernoulli(thr / 65536) on a 16-bit lane is "lane < thr", thr in [0, 65536].  lanes_below takes it encoded once on the
// host: lt = lane_lt(thr) per lane, and `all` = the lanes whose thr is 65536.
inline uint32_t lane_lt(uint32_t thr) { return thr >= 65536u ? 0u : thr << 16; }

// bit c = (16-bit lane c of r < thr(c)) for c < NL <= 8, given lt(c) and `all` as above.  Lane 2j + 1 is the high half
// of word j, so it is below thr exactly when the word is below thr << 16; lane 2j is compared the same way after a
// shift.  One compare per lane.  A runtime lane count calls it once per 8-lane block (one call each).
template <int NL, typename LtFn>
__device__ __forceinline__ uint32_t lanes_below(const uint4& r, LtFn lt, uint32_t all) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
  uint32_t m = all;
#pragma unroll
  for (int c = 0; c < NL; ++c) {
    const uint32_t v = (c & 1) ? w[c >> 1] : (w[c >> 1] << 16);
    m |= (uint32_t)(v < lt(c)) << c;
  }
  return m;
}

// lanes16: bit c = (16-bit lane c < thr(c)) for c < n_lanes, lane c from block c / 8 of the counter (env, t, dp, .),
// lanes_below once per 8-lane block.  NL > 0 fixes the lane count at compile time (n_lanes unused).  The lanes of the
// last block at and above n_lanes are compared too: lt(c) must be readable there, and those bits are the caller's to
// mask.
template <int NL, typename LtFn>
__device__ __forceinline__ uint32_t lanes16_below(const PhiloxKey& k, uint32_t env, uint32_t t, uint32_t dp,
                                                  int n_lanes, LtFn lt, uint32_t all) {
  uint32_t m = 0;
#pragma unroll
  for (int blk = 0; blk < (NL ? (NL + 7) / 8 : D2D_MAX_CHANNELS / 8); ++blk)
    if (blk * 8 < (NL ? NL : n_lanes))
      m |= lanes_below<NL && NL < 8 ? NL : 8>(philox(k, env, t, dp, (uint32_t)blk),
                                               [&](int c) { return lt(8 * blk + c); }, all >> (8 * blk))
           << (8 * blk);
  return m;
}

// ---- calls shared between devices ----
// word32: device k's 32-bit word is word k % 4 of the call whose device field is word32_field(k) = k / 4.  A device
// loop that starts at a multiple of 4 draws the call at k % 4 == 0 and keeps it for the group.
__device__ __forceinline__ uint32_t word32_field(int k) { return (uint32_t)k >> 2; }
__device__ __forceinline__ uint32_t word32(const uint4& r, int k) {
  const int i = k & 3;
  return i == 0 ? r.x : (i == 1 ? r.y : (i == 2 ? r.z : r.w));
}

// lane16_shared: device k's 16-bit lane is lane lane16_shared_lane(k) = k % 8 of the call whose device field is
// lane16_shared_field(k) = k / 8 (one switch / policy bit per device of the single-channel env)
__device__ __forceinline__ uint32_t lane16_shared_field(int k) { return (uint32_t)k >> 3; }
__device__ __forceinline__ int lane16_shared_lane(int k) { return k & 7; }

// ---- arrival count of a 32-bit word (thr32, poisson_from_u32) ----
// Bernoulli: u < bern_thr (64-bit compare, thr in [0, 2^32]); Poisson: #{m : u >= cdf[m]} over the non-decreasing
// thresholds of the device's CDF row
__device__ __forceinline__ uint32_t arrival_count(uint32_t u, bool bernoulli, uint64_t bern_thr, const uint32_t* cdf) {
  if (bernoulli) return (uint64_t)u < bern_thr ? 1u : 0u;
  uint32_t n = 0;
#pragma unroll 1
  for (int m = 0; m < D2D_POISSON_KMAX; ++m) {
    if (u < cdf[m]) break;
    ++n;
  }
  return n;
}

}  // namespace d2d
