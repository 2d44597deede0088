// Shared device code of the env kernels: parameter blob, launch arguments, packet-buffer records, Philox draws,
// f32 row emission.  Included by env_kernels.cu and env_comb_step.cuh.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace d2d {


// ------------------------------------------------------------------------------------------------
// parameter blob (device global -> shared memory at block start)
// ------------------------------------------------------------------------------------------------
struct EnvParamsHdr {
  int32_t N, C, D, T, homog, kind, sum_dl, obs_rows, state_rows;
  int32_t off_cdf, off_sw, off_nbr_off, off_nbr_idx, total_bytes;
  int32_t self_nbr;   // single-channel env: every neighbourhood is the device itself (env.py:38-39 default)
  uint8_t deadline[D2D_MAX_AGENTS];
  uint8_t arrival_kind[D2D_MAX_AGENTS];
  uint16_t obs_off[D2D_MAX_AGENTS];
  uint16_t obs_dim[D2D_MAX_AGENTS];
  uint16_t sbuf_off[D2D_MAX_AGENTS];  // first row of device k's buffer inside `state`
  uint64_t bern_thr[D2D_MAX_AGENTS];
  float inv_count[D2D_MAX_AGENTS + 1];  // (float)(1.0 / count) -- channel_selection_env.py:137
};

struct StepArgs {
  uint32_t* buf;
  void* chan;
  uint32_t* disc;
  uint32_t* recv;
  uint32_t* stats;
  const uint8_t* params;
  int params_bytes;
  const void* actions;
  void* actions_out;
  float* obs;
  float* state;
  int32_t* reward;
  uint8_t* done;
  void* ack;
  const uint8_t* rp_arr;  // replay arrivals of this timestep, u8 [N][B]
  const void* rp_sw;      // replay switch draws of this timestep
  int B;
  uint32_t t;  // timestep being produced (0 = reset)
  uint32_t k0, k1;
  uint32_t rk0[10], rk1[10];  // Philox round keys (k + r * W), precomputed on the host: constant-bank operands
  uint32_t env_offset;
  uint64_t active;  // bit k: device k draws an arrival at timestep t
  int rng_mode;
  int act_mode;  // 0 = actions from memory, 1 = fused random-access policy
  uint32_t tp_thr;
  int done_flag;
  int reward_accum;  // 1: reward[b] += this step's reward (d2d_env_run_random_access), 0: overwrite
};

// the multi-step kernels (sc_run_kernel, sc_run_lanes_kernel, comb_run_kernel): n_inner steps of one episode per launch
struct RunArgs {
  const uint64_t* active;      // device copy of the per-timestep arrival masks, indexed by the episode timestep
  int t_plain;                 // episode timestep of the first step produced (a.t is its Philox counter)
  int n_inner;
  long long reward_stride;     // elements between the reward rows of consecutive steps (0 with reward_accum)
  long long obs_stride;        // elements between the observation blocks of consecutive steps (comb_run_kernel)
};

__device__ __forceinline__ const EnvParamsHdr* stage_params(const StepArgs& a, uint8_t* smem) {
  const uint32_t* src = reinterpret_cast<const uint32_t*>(a.params);
  uint32_t* dst = reinterpret_cast<uint32_t*>(smem);
  for (int i = threadIdx.x; i < a.params_bytes / 4; i += blockDim.x) dst[i] = src[i];
  __syncthreads();
  return reinterpret_cast<const EnvParamsHdr*>(smem);
}

// ------------------------------------------------------------------------------------------------
// packet-buffer records: W 32-bit words, byte d (little endian) = packets with d slots left
// ------------------------------------------------------------------------------------------------
template <int W>
struct Rec {
  uint32_t w[W];
};

template <int W>
__device__ __forceinline__ Rec<W> rec_load(const uint32_t* base, size_t idx) {
  Rec<W> r;
  if constexpr (W == 2) {
    const uint2 v = reinterpret_cast<const uint2*>(base)[idx];
    r.w[0] = v.x, r.w[1] = v.y;
  } else {
#pragma unroll
    for (int q = 0; q < W / 4; ++q) {
      const uint4 v = reinterpret_cast<const uint4*>(base)[idx * (W / 4) + q];
      r.w[4 * q] = v.x, r.w[4 * q + 1] = v.y, r.w[4 * q + 2] = v.z, r.w[4 * q + 3] = v.w;
    }
  }
  return r;
}

template <int W>
__device__ __forceinline__ void rec_store(uint32_t* base, size_t idx, const Rec<W>& r) {
  if constexpr (W == 2) {
    reinterpret_cast<uint2*>(base)[idx] = make_uint2(r.w[0], r.w[1]);
  } else {
#pragma unroll
    for (int q = 0; q < W / 4; ++q)
      reinterpret_cast<uint4*>(base)[idx * (W / 4) + q] =
          make_uint4(r.w[4 * q], r.w[4 * q + 1], r.w[4 * q + 2], r.w[4 * q + 3]);
  }
}

template <int W>
__device__ __forceinline__ bool rec_any(const Rec<W>& r) {
  uint32_t o = 0;
#pragma unroll
  for (int j = 0; j < W; ++j) o |= r.w[j];
  return o != 0;
}

// remove one packet from the earliest non-empty slot (combinatorial_env.py:169-170)
template <int W>
__device__ __forceinline__ void rec_pop_earliest(Rec<W>& r, bool enable) {
  bool done = !enable;
#pragma unroll
  for (int j = 0; j < W; ++j) {
    const uint32_t w = r.w[j];
    const bool hit = !done && w != 0;
    const int pos = (__ffs((int)w) - 1) & 24;  // bit offset of the lowest non-zero byte
    r.w[j] = hit ? w - (1u << pos) : w;
    done |= hit;
  }
}

// age by one slot (combinatorial_env.py:120-124); returns the expired count (old slot 0)
template <int W>
__device__ __forceinline__ uint32_t rec_age(Rec<W>& r) {
  const uint32_t expired = r.w[0] & 0xFFu;
#pragma unroll
  for (int j = 0; j + 1 < W; ++j) r.w[j] = __funnelshift_r(r.w[j], r.w[j + 1], 8);
  r.w[W - 1] >>= 8;
  return expired;
}

template <int W>
__device__ __forceinline__ void rec_set_byte(Rec<W>& r, int idx, uint32_t val) {
  // mask arithmetic on every word (not an indexed write): keeps the record in registers for a runtime idx
  const int s = (idx & 3) * 8;
  const uint32_t m = 0xFFu << s, v = val << s;
#pragma unroll
  for (int j = 0; j < W; ++j) {
    const uint32_t mj = (idx >> 2) == j ? m : 0u;
    r.w[j] = (r.w[j] & ~mj) | (v & mj);
  }
}

template <int W>
__device__ __forceinline__ uint32_t rec_sum(const Rec<W>& r) {
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < W; ++j) s += __vsadu4(r.w[j], 0u);
  return s;
}

// write the first `n` slots of a record as f32 rows p[0], p[B], p[2B], ...
template <int W>
__device__ __forceinline__ void rec_emit(const Rec<W>& r, int n, float* p, size_t B) {
#pragma unroll
  for (int d = 0; d < 4 * W; ++d) {
    if (d < n) {
      *p = (float)((r.w[d >> 2] >> (8 * (d & 3))) & 0xFFu);
      p += B;
    }
  }
}

// Arrival uniforms: one Philox call serves FOUR devices (counter device field = k / 4, device k takes word k % 4), so a
// step draws ceil(N / 4) arrival calls per env instead of N.
__device__ __forceinline__ uint32_t pick_word(const uint4& r, int i) {
  return i == 0 ? r.x : (i == 1 ? r.y : (i == 2 ? r.z : r.w));
}

__device__ __forceinline__ uint32_t arrival_from_u(const EnvParamsHdr* P, const uint32_t* cdf, int k, uint32_t u) {
  if (P->arrival_kind[k] == D2D_ARRIVAL_BERNOULLI) return (uint64_t)u < P->bern_thr[k] ? 1u : 0u;
  const uint32_t* c = cdf + k * D2D_POISSON_KMAX;
  uint32_t n = 0;
#pragma unroll 1
  for (int m = 0; m < D2D_POISSON_KMAX; ++m) {
    if (u < c[m]) break;  // thresholds are non-decreasing
    ++n;
  }
  return n;
}

// the four arrival words of device group k / 4, fetched once and reused while the device loop stays in the group
struct ArrivalWords {
  uint4 r;
  int group = -1;
  __device__ __forceinline__ uint32_t get(const StepArgs& a, uint32_t env, int k) {
    if ((k >> 2) != group) {
      group = k >> 2;
      r = philox4x32_10(env, a.t, (uint32_t)group | (kPurposeArrival << 16), 0u, a.k0, a.k1);
    }
    return pick_word(r, k & 3);
  }
};

// arrival of device k at timestep a.t (only called when the device is active)
__device__ __forceinline__ uint32_t draw_arrival(const StepArgs& a, const EnvParamsHdr* P, const uint32_t* cdf, int k,
                                                 int b, ArrivalWords& words) {
  if (a.rng_mode == D2D_RNG_REPLAY) return a.rp_arr[(size_t)k * a.B + b];
  return arrival_from_u(P, cdf, k, words.get(a, a.env_offset + (uint32_t)b, k));
}

// 16-bit lanes shared by EIGHT devices (single-channel env: one switch / policy bit per device): counter device field
// = k / 8, device k takes lane k % 8
struct LaneWords {
  uint4 r;
  int group = -1;
  __device__ __forceinline__ uint32_t get(const StepArgs& a, uint32_t env, int k, uint32_t purpose) {
    if ((k >> 3) != group) {
      group = k >> 3;
      r = philox4x32_10(env, a.t, (uint32_t)group | (purpose << 16), 0u, a.k0, a.k1);
    }
    const uint32_t w = pick_word(r, (k & 7) >> 1);
    return (k & 1) ? (w >> 16) : (w & 0xFFFFu);
  }
};

// Philox with the host-precomputed round keys of StepArgs (one constant-bank operand per XOR).
__device__ __forceinline__ uint4 philox_rk(const StepArgs& a, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ a.rk0[r];
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ a.rk1[r];
    c1 = (uint32_t)p1;
    c3 = (uint32_t)p0;
    c0 = n0;
    c2 = n2;
  }
  return make_uint4(c0, c1, c2, c3);
}

// bit c = (16-bit lane c < thr(c)) for c < C at Philox timestep t;  CFIX > 0 makes the lane count a compile-time constant
template <int CFIX, typename ThrFn>
__device__ __forceinline__ uint32_t lane_mask_rk(const StepArgs& a, uint32_t env, uint32_t t, uint32_t dev_purpose,
                                                 int C, ThrFn thr) {
  uint32_t m = 0;
  const int nl = CFIX ? CFIX : C;
#pragma unroll
  for (int blk = 0; blk < (CFIX ? (CFIX + 7) / 8 : 4); ++blk) {
    if (blk * 8 < nl) {
      const uint4 r = philox_rk(a, env, t, dev_purpose, (uint32_t)blk);
      const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        const int c = blk * 8 + l;
        if (c < nl) {
          const uint32_t u = (l & 1) ? (w[l >> 1] >> 16) : (w[l >> 1] & 0xFFFFu);
          m |= (uint32_t)(u < thr(c)) << c;
        }
      }
    }
  }
  return m;
}

// p += stride floats, as ONE 64-bit multiply-add on the (otherwise idle) FMA pipe
__device__ __forceinline__ float* next_row(float* p, uint32_t stride) {
  uint64_t q = reinterpret_cast<uint64_t>(p);
  asm("mad.wide.u32 %0, %1, 4, %0;" : "+l"(q) : "r"(stride));
  return reinterpret_cast<float*>(q);
}

__device__ __forceinline__ void st_f32(float* p, float v) {   // keeps the store in the global window (STG, not ST)
  asm volatile("st.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// byte `byte` of w as f32 without the quarter-rate I2F: splice it under the exponent of 2^23, subtract 2^23
template <int BYTE>
__device__ __forceinline__ float byte_f32(uint32_t w) {
  return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7650u | BYTE)) - 8388608.0f;
}

template <int W, int NB>
__device__ __forceinline__ float* emit_slots_fixed(const Rec<W>& r, float* p, uint32_t B) {
#pragma unroll
  for (int d = 0; d < NB; ++d) {
    const uint32_t w = r.w[d >> 2];
    st_f32(p, (d & 3) == 0 ? byte_f32<0>(w) : (d & 3) == 1 ? byte_f32<1>(w) : (d & 3) == 2 ? byte_f32<2>(w) : byte_f32<3>(w));
    p = next_row(p, B);
  }
  return p;
}

// first n slots of a record as f32 rows; the common deadlines (7, 14) get predicate-free code
template <int W>
__device__ __forceinline__ float* emit_slots(const Rec<W>& r, int n, float* p, uint32_t B) {
  if (n == 7) return emit_slots_fixed<W, 7>(r, p, B);
  if constexpr (W >= 4)
    if (n == 14) return emit_slots_fixed<W, 14>(r, p, B);
#pragma unroll
  for (int d = 0; d < 4 * W; ++d) {
    if (d < n) {
      const uint32_t w = r.w[d >> 2];
      st_f32(p, (d & 3) == 0 ? byte_f32<0>(w) : (d & 3) == 1 ? byte_f32<1>(w) : (d & 3) == 2 ? byte_f32<2>(w) : byte_f32<3>(w));
      p = next_row(p, B);
    }
  }
  return p;
}

template <int CFIX>
__device__ __forceinline__ float* emit_bits(uint32_t m, int C, float* p, uint32_t B) {
#pragma unroll
  for (int c = 0; c < (CFIX ? CFIX : D2D_MAX_CHANNELS); ++c) {
    if (CFIX || c < C) {
      st_f32(p, (m & (1u << c)) ? 1.0f : 0.0f);
      p = next_row(p, B);
    }
  }
  return p;
}

template <int CFIX>
__device__ __forceinline__ float* emit_ack(uint32_t acked, uint32_t nacked, int C, float* p, uint32_t B) {
#pragma unroll
  for (int c = 0; c < (CFIX ? CFIX : D2D_MAX_CHANNELS); ++c) {
    if (CFIX || c < C) {
      st_f32(p, (acked & (1u << c)) ? 1.0f : ((nacked & (1u << c)) ? -1.0f : 0.0f));
      p = next_row(p, B);
    }
  }
  return p;
}

}  // namespace d2d
