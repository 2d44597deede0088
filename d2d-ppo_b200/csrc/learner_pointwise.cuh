// Row-wise (pointwise) kernels of the learner: GRU gates, distribution heads, PPO loss derivatives,
// lambda-return / discounted-return scans, normalisation, Adam.  One thread per (agent, time, env) row.
#pragma once
#include "learner_kernels.cuh"

namespace d2d {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// ------------------------------------------------------------------------------------------------
// GRU cell, torch gate order (r, z, n):  r = s(gi_r + gh_r), z = s(gi_z + gh_z), n = tanh(gi_n + r * gh_n),
// h' = (1 - z) n + z h        (nn.GRU; reference d2d_ppo.py:30,52)
// ------------------------------------------------------------------------------------------------
struct GateArgs {
  View gi;      // [.. 3H ..] input projections of the observation at time t - back (view.t_off = -back + halo)
  View gh;      // [.. 3H ..] hidden projections of this step (forward) / d(gh) (backward out)
  View h_prev;  // [.. H ..]  (forward in; backward in)
  View h_out;   // [.. H ..]  forward: h'; backward: d(h_prev) out
  View acts;    // [.. 4H ..] stored r, z, n, gh_n (forward out if store; backward in)
  View dh;      // backward in: d(h')
  View dgi;     // backward: accumulated into (same time shift as gi)
  int H, B, t0, t1;
  int back;       // this step looks `back` observations into the past
  int padded;     // 1: observations before the episode start are zero INPUTS that still run (training windows)
                  // 0: those steps do not exist (rollout windows): h' = h
  int first;      // 1: h_prev is the zero initial state (not read)
  int store;      // forward: write acts
  int t_episode0; // absolute time index of the episode's first observation in units of this call's t (usually 0)
};

__global__ void gru_gate_fwd_kernel(const GateArgs a) {
  const int g = blockIdx.y, H = a.H;
  const long long per_t = (long long)H * a.B;
  const long long n = (long long)(a.t1 - a.t0) * per_t;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int t = a.t0 + (int)(i / per_t);
    const int u = (int)((i % per_t) / a.B), b = (int)(i % a.B);
    const long long uB = (long long)u * a.B, HB = per_t;
    const float hp = a.first ? 0.f : view_ptr(a.h_prev, g, t, a.B, b)[uB];
    float* ho = view_ptr(a.h_out, g, t, a.B, b) + uB;
    const bool exists = a.padded || (t - a.back >= a.t_episode0);
    if (!exists) {
      *ho = hp;
      continue;
    }
    const float* gi = view_ptr(a.gi, g, t, a.B, b) + uB;
    const float* gh = view_ptr(a.gh, g, t, a.B, b) + uB;
    const float ghn = gh[2 * HB];
    const float r = sigmoidf_(gi[0] + gh[0]);
    const float z = sigmoidf_(gi[HB] + gh[HB]);
    const float nn = tanhf(gi[2 * HB] + r * ghn);
    *ho = (1.0f - z) * nn + z * hp;
    if (a.store) {
      float* ac = view_ptr(a.acts, g, t, a.B, b) + uB;
      ac[0] = r, ac[HB] = z, ac[2 * HB] = nn, ac[3 * HB] = ghn;
    }
  }
}

// backward of one (always existing: training windows are padded) GRU step
__global__ void gru_gate_bwd_kernel(const GateArgs a) {
  const int g = blockIdx.y, H = a.H;
  const long long per_t = (long long)H * a.B;
  const long long n = (long long)(a.t1 - a.t0) * per_t;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int t = a.t0 + (int)(i / per_t);
    const int u = (int)((i % per_t) / a.B), b = (int)(i % a.B);
    const long long uB = (long long)u * a.B, HB = per_t;
    const float* ac = view_ptr(a.acts, g, t, a.B, b) + uB;
    const float r = ac[0], z = ac[HB], nn = ac[2 * HB], ghn = ac[3 * HB];
    const float hp = a.first ? 0.f : view_ptr(a.h_prev, g, t, a.B, b)[uB];
    const float dh = view_ptr(a.dh, g, t, a.B, b)[uB];
    const float dn = dh * (1.0f - z) * (1.0f - nn * nn);   // through tanh
    const float dz = dh * (hp - nn) * z * (1.0f - z);      // through sigmoid
    const float dr = dn * ghn * r * (1.0f - r);
    float* dgh = view_ptr(a.gh, g, t, a.B, b) + uB;
    dgh[0] = dr, dgh[HB] = dz, dgh[2 * HB] = dn * r;
    float* dgi = view_ptr(a.dgi, g, t, a.B, b) + uB;       // several windows share an observation: accumulate
    dgi[0] += dr, dgi[HB] += dz, dgi[2 * HB] += dn;
    view_ptr(a.h_out, g, t, a.B, b)[uB] = dh * z;          // direct path; dense_kernel adds d(gh) W_hh on top
  }
}

// ------------------------------------------------------------------------------------------------
// policy head: probabilities -> actions / log-prob / entropy, and the PPO surrogate derivative
// torch.distributions numerics (Bernoulli / Categorical built from `probs`), reference d2d_ppo.py:159-196
// ------------------------------------------------------------------------------------------------
enum { kOutSoftmax = 0, kOutSigmoid = 1, kOutIdentity = 2 };
enum { kDistBernoulli = 0, kDistCategorical = 1 };
enum { kActSample = 0, kActGreedy = 1, kActGiven = 2 };
constexpr int kMaxOut = 32;
constexpr float kProbEps = 1.1920928955078125e-07f;  // torch.finfo(float32).eps

// what select_action needs besides the probabilities (also embedded in the GRU window kernel's arguments, which
// selects the action in its epilogue: gru_tc.cuh)
struct DistArgs {
  int A, B, n_agents;
  int out_kind, dist_kind, act_mode;
  // actions: Bernoulli -> channel bitmask (mask_bytes per element), Categorical -> u8 index;  layout [t][N][B]
  void* actions;
  int mask_bytes;
  long long act_t_stride;   // elements between time blocks (N * B)
  int act_t_off;
  float* logp;              // [t][N][B] (same strides as actions)
  float* entropy;           // may be null
  uint32_t k0, k1, env_offset;
  int t_abs_off;            // Philox timestep = t + t_abs_off
};

struct HeadArgs : DistArgs {
  View logits;           // [.. A ..] pre-activation outputs of the last Linear
  View probs;            // optional out [.. A ..] (p == nullptr: not written)
  int t0, t1;
  // ---- loss / backward (ppo_dlogits_kernel) ----
  const float* logp_old;    // [t][N][B]
  const float* weight;      // per-row weight (advantage or HAPPO M): [t][N][B] if weight_per_agent else [t][B]
  int weight_per_agent;
  const int* cycle;         // HAPPO order (device, [N]) or null
  float* ratio_out;         // optional [t][N][B]
  View dlogits;             // out
  float inv_rows;           // 1 / R_total
  float cliprange, beta;
  double* loss_sums;        // [N][2]: sum over rows of min(surr1, surr2), sum of entropy
};

__device__ __forceinline__ void head_probs(const DistArgs& a, const float* lg, long long sB, float* p) {
  if (a.out_kind == kOutSigmoid) {
    for (int j = 0; j < a.A; ++j) p[j] = sigmoidf_(lg[j * sB]);
  } else if (a.out_kind == kOutSoftmax) {
    float m = -INFINITY;
    for (int j = 0; j < a.A; ++j) m = fmaxf(m, lg[j * sB]);
    float s = 0.f;
    for (int j = 0; j < a.A; ++j) {
      p[j] = expf(lg[j * sB] - m);
      s += p[j];
    }
    for (int j = 0; j < a.A; ++j) p[j] = p[j] / s;
  } else {
    for (int j = 0; j < a.A; ++j) p[j] = lg[j * sB];
  }
}

__device__ __forceinline__ float clamp_prob(float p) { return fminf(fmaxf(p, kProbEps), 1.0f - kProbEps); }
// ATen binary_cross_entropy_with_logits: (1 - y) x - log_sigmoid(x), log_sigmoid(x) = min(x, 0) - log1p(exp(-|x|))
__device__ __forceinline__ float bce_logits(float x, float y) {
  return (1.0f - y) * x - (fminf(x, 0.f) - log1pf(expf(-fabsf(x))));
}

__device__ __forceinline__ uint32_t load_action(const DistArgs& a, long long idx) {
  if (a.dist_kind == kDistCategorical || a.mask_bytes == 1) return reinterpret_cast<const uint8_t*>(a.actions)[idx];
  if (a.mask_bytes == 2) return reinterpret_cast<const uint16_t*>(a.actions)[idx];
  return reinterpret_cast<const uint32_t*>(a.actions)[idx];
}
__device__ __forceinline__ void store_action(const DistArgs& a, long long idx, uint32_t v) {
  if (a.dist_kind == kDistCategorical || a.mask_bytes == 1) reinterpret_cast<uint8_t*>(a.actions)[idx] = (uint8_t)v;
  else if (a.mask_bytes == 2) reinterpret_cast<uint16_t*>(a.actions)[idx] = (uint16_t)v;
  else reinterpret_cast<uint32_t*>(a.actions)[idx] = v;
}

// log-prob and entropy of action `act` under probs p (registers)
__device__ __forceinline__ void dist_logp_entropy(const DistArgs& a, const float* p, uint32_t act, float& logp,
                                                  float& ent) {
  if (a.dist_kind == kDistBernoulli) {
    float sl = 0.f, se = 0.f;
    for (int j = 0; j < a.A; ++j) {
      const float pc = clamp_prob(p[j]);
      const float l = logf(pc) - log1pf(-pc);
      sl += -bce_logits(l, (float)((act >> j) & 1u));
      se += bce_logits(l, p[j]);
    }
    logp = sl / (float)a.A;   // .mean(-1) over channels, d2d_ppo.py:168-169
    ent = se / (float)a.A;
  } else {
    float s = 0.f;
    for (int j = 0; j < a.A; ++j) s += p[j];
    float e = 0.f;
    logp = 0.f;
    for (int j = 0; j < a.A; ++j) {
      const float pn = p[j] / s;
      const float l = logf(clamp_prob(pn));
      if ((uint32_t)j == act) logp = l;
      e += l * pn;
    }
    ent = -e;
  }
}

// select_action / evaluate of one (agent g, time t, env b) row from its probabilities p (registers): act_mode
// sample / greedy / given -> action, log-prob, entropy (reference d2d_ppo.py:159-196)
__device__ __forceinline__ void policy_select(const DistArgs& a, int g, int t, int b, const float* p) {
  const long long idx = (long long)(t + a.act_t_off) * a.act_t_stride + (long long)g * a.B + b;
  uint32_t act = 0;
  if (a.act_mode == kActGiven) {
    act = load_action(a, idx);
  } else {
    if (a.dist_kind == kDistBernoulli) {
      if (a.act_mode == kActGreedy) {
        for (int j = 0; j < a.A; ++j) act |= (uint32_t)(p[j] > 0.5f) << j;      // d2d_ppo.py:166
      } else {
        for (int blk = 0; blk * 4 < a.A; ++blk) {
          const uint4 r = philox4x32_10(a.env_offset + (uint32_t)b, (uint32_t)(t + a.t_abs_off),
                                        (uint32_t)g | (kPurposePolicy << 16), (uint32_t)blk, a.k0, a.k1);
          const uint32_t u[4] = {r.x, r.y, r.z, r.w};
          for (int l = 0; l < 4 && blk * 4 + l < a.A; ++l) {
            const int j = blk * 4 + l;
            const double thr = (double)p[j] * 4294967296.0;          // P(u32 < thr) = p at 2^-32 resolution
            act |= (uint32_t)((double)u[l] < thr) << j;
          }
        }
      }
    } else {
      if (a.act_mode == kActGreedy) {
        float best = p[0];
        for (int j = 1; j < a.A; ++j)
          if (p[j] > best) best = p[j], act = (uint32_t)j;            // argmax, first maximum (d2d_ppo.py:176)
      } else {
        const uint4 r = philox4x32_10(a.env_offset + (uint32_t)b, (uint32_t)(t + a.t_abs_off),
                                      (uint32_t)g | (kPurposePolicy << 16), 0u, a.k0, a.k1);
        double s = 0.0;
        for (int j = 0; j < a.A; ++j) s += (double)p[j];
        const double uu = ((double)r.x + 0.5) * (1.0 / 4294967296.0) * s;
        double c = 0.0;
        act = (uint32_t)(a.A - 1);
        for (int j = 0; j < a.A; ++j) {
          c += (double)p[j];
          if (uu < c) {
            act = (uint32_t)j;
            break;
          }
        }
      }
    }
    store_action(a, idx, act);
  }
  float logp, ent;
  dist_logp_entropy(a, p, act, logp, ent);
  if (a.logp) a.logp[idx] = logp;
  if (a.entropy) a.entropy[idx] = ent;
}

__global__ void policy_head_kernel(const HeadArgs a) {
  const int g = blockIdx.y;
  const long long n = (long long)(a.t1 - a.t0) * a.B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int t = a.t0 + (int)(i / a.B), b = (int)(i % a.B);
    const float* lg = view_ptr(a.logits, g, t, a.B, b);
    float p[kMaxOut];
    head_probs(a, lg, a.B, p);
    if (a.probs.p) {
      float* q = view_ptr(a.probs, g, t, a.B, b);
      for (int j = 0; j < a.A; ++j) q[(long long)j * a.B] = p[j];
    }
    policy_select(a, g, t, b, p);
  }
}

// d(loss)/d(logits) of  loss = -mean_rows(min(ratio w, clip(ratio) w)) - beta mean_rows(entropy)
// (reference d2d_ppo.py:201-207, ippo.py:196-202).  One thread per (time, env) handles ALL agents so that the
// HAPPO weight M_j = adv * prod_{i before j in cycle} ratio_i (d2d_ppo.py:427-436) is a running product.
// part == nullptr: the loss sums are added to a.loss_sums with fp64 atomics (order not fixed).  Deterministic mode:
// warp w of the grid adds its sums to part[g][w][2] (zeroed by the caller, one writer per slot) and
// sum_partials_kernel reduces them in a fixed order.
template <bool PART>
__device__ __forceinline__ void ppo_dlogits_body(const HeadArgs& a, double* part) {
  const long long n = (long long)(a.t1 - a.t0) * a.B;
  const long long n_round = (n + blockDim.x - 1) / blockDim.x * blockDim.x;   // whole warps stay in the loop
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_round;
       i += (long long)gridDim.x * blockDim.x) {
    const bool live = i < n;
    const long long ii = live ? i : 0;
    const int t = a.t0 + (int)(ii / a.B), b = (int)(ii % a.B);
    float chain = 1.0f;
    for (int ord = 0; ord < a.n_agents; ++ord) {
      const int g = a.cycle ? a.cycle[ord] : ord;
      const float* lg = view_ptr(a.logits, g, t, a.B, b);
      float p[kMaxOut];
      head_probs(a, lg, a.B, p);
      const long long idx = (long long)(t + a.act_t_off) * a.act_t_stride + (long long)g * a.B + b;
      const uint32_t act = load_action(a, idx);
      float logp, ent;
      dist_logp_entropy(a, p, act, logp, ent);
      const float ratio = expf(logp - a.logp_old[idx]);
      float w = a.weight_per_agent ? a.weight[idx]
                                   : a.weight[(long long)(t + a.act_t_off) * a.B + b];
      if (a.cycle) {
        w *= chain;          // M for this agent (detached)
        chain *= ratio;      // M <- ratio * M with the PRE-update ratio
      }
      if (a.ratio_out && live) a.ratio_out[idx] = ratio;
      const float lo = 1.0f - a.cliprange, hi = 1.0f + a.cliprange;
      const float surr1 = ratio * w, surr2 = fminf(fmaxf(ratio, lo), hi) * w;
      // torch.min splits the gradient on ties (ratio inside the clip range: surr1 == surr2, both paths carry w)
      const float dratio = (ratio >= lo && ratio <= hi) ? w : (surr1 < surr2 ? w : 0.f);
      const float dlogp = -a.inv_rows * dratio * ratio;
      const float dent = -a.inv_rows * a.beta;
      double s0 = live ? (double)fminf(surr1, surr2) : 0.0, s1 = live ? (double)ent : 0.0;
      for (int o = 16; o > 0; o >>= 1) {
        s0 += __shfl_down_sync(0xFFFFFFFFu, s0, o);
        s1 += __shfl_down_sync(0xFFFFFFFFu, s1, o);
      }
      if ((threadIdx.x & 31) == 0) {
        if constexpr (PART) {
          const int n_warps = gridDim.x * (blockDim.x >> 5);
          double* q = part + 2 * ((long long)g * n_warps + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5));
          q[0] += s0, q[1] += s1;
        } else {
          atomicAdd(&a.loss_sums[2 * g], s0);
          atomicAdd(&a.loss_sums[2 * g + 1], s1);
        }
      }
      if (!live) continue;
      // ---- d/dp, then through the output activation ----
      float dp[kMaxOut];
      if (a.dist_kind == kDistBernoulli) {
        for (int j = 0; j < a.A; ++j) {
          const float pc = clamp_prob(p[j]);
          const float l = logf(pc) - log1pf(-pc);
          const float dl_dp = (p[j] >= kProbEps && p[j] <= 1.0f - kProbEps) ? 1.0f / (pc * (1.0f - pc)) : 0.f;
          const float y = (float)((act >> j) & 1u);
          // logp_j = -bce(l, y): d/dl = y - sigmoid(l) = y - pc;  ent_j = bce(l, p): d/dp = -l + (pc - p) dl/dp
          dp[j] = (dlogp * (y - pc) * dl_dp + dent * (-l + (pc - p[j]) * dl_dp)) / (float)a.A;
        }
      } else {
        float s = 0.f;
        for (int j = 0; j < a.A; ++j) s += p[j];
        float dpn[kMaxOut];
        float dot = 0.f;
        for (int j = 0; j < a.A; ++j) {
          const float pn = p[j] / s;
          const float pc = clamp_prob(pn);
          const float in = (pn >= kProbEps && pn <= 1.0f - kProbEps) ? 1.0f : 0.f;
          const float l = logf(pc);
          // logp = l[act]; ent = -sum l pn
          dpn[j] = ((uint32_t)j == act ? dlogp * in / pc : 0.f) + dent * (-(l + in * pn / pc));
          dot += dpn[j] * pn;
        }
        for (int j = 0; j < a.A; ++j) dp[j] = (dpn[j] - dot) / s;   // through pn = p / sum(p)
      }
      float* dl = view_ptr(a.dlogits, g, t, a.B, b);
      if (a.out_kind == kOutSigmoid) {
        for (int j = 0; j < a.A; ++j) dl[(long long)j * a.B] = dp[j] * p[j] * (1.0f - p[j]);
      } else if (a.out_kind == kOutSoftmax) {
        float dot = 0.f;
        for (int j = 0; j < a.A; ++j) dot += dp[j] * p[j];
        for (int j = 0; j < a.A; ++j) dl[(long long)j * a.B] = p[j] * (dp[j] - dot);
      } else {
        for (int j = 0; j < a.A; ++j) dl[(long long)j * a.B] = dp[j];
      }
    }
  }
}
__global__ void ppo_dlogits_kernel(const HeadArgs a) { ppo_dlogits_body<false>(a, nullptr); }
__global__ void ppo_dlogits_part_kernel(const HeadArgs a, double* part) { ppo_dlogits_body<true>(a, part); }

// critic: d(mse)/d(value) = 2 (v - target) / R ; loss sum accumulated in fp64
struct MseArgs {
  View value;        // [.. 1 ..]
  View dvalue;       // out
  const float* target;   // [t][N][B] if per_agent else [t][B]
  int per_agent;
  long long tgt_t_stride;
  int tgt_t_off;
  int B, t0, t1;
  float inv_rows;
  double* loss_sum;  // [N]
  float* value_out;  // optional [t][N][B] copy
  long long out_t_stride;
};

// part != nullptr (deterministic mode): warp w of agent g's blocks stores its sum to part[g][w] instead of the atomic
template <bool PART>
__device__ __forceinline__ void mse_dvalue_body(const MseArgs& a, double* part) {
  const int g = blockIdx.y;
  const long long n = (long long)(a.t1 - a.t0) * a.B;
  double local = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int t = a.t0 + (int)(i / a.B), b = (int)(i % a.B);
    const float v = *view_ptr(a.value, g, t, a.B, b);
    const long long ti = (long long)(t + a.tgt_t_off) * a.tgt_t_stride;
    const float y = a.per_agent ? a.target[ti + (long long)g * a.B + b] : a.target[ti + b];
    const float d = v - y;
    *view_ptr(a.dvalue, g, t, a.B, b) = 2.0f * d * a.inv_rows;
    local += (double)d * (double)d;
    if (a.value_out) a.value_out[(long long)(t + a.tgt_t_off) * a.out_t_stride + (long long)g * a.B + b] = v;
  }
  for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xFFFFFFFFu, local, o);
  if ((threadIdx.x & 31) == 0) {
    if constexpr (PART) part[(long long)g * gridDim.x * (blockDim.x >> 5) + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5)] = local;
    else atomicAdd(&a.loss_sum[g], local);
  }
}
__global__ void mse_dvalue_kernel(const MseArgs a) { mse_dvalue_body<false>(a, nullptr); }
__global__ void mse_dvalue_part_kernel(const MseArgs a, double* part) { mse_dvalue_body<true>(a, part); }

// ------------------------------------------------------------------------------------------------
// lambda-returns (compute_gae, d2d_ppo.py:100-110) and discounted returns (discount_rewards, :112-124)
// One thread per (agent column, env): reverse scan over the T steps of that env's episode, in float64 as
// the reference (numpy) does.  Rows of the reference are episode-major, so only the LAST env's final step
// keeps the `r - v` quirk of :102; every other episode end gives out = r exactly (done zeroes the bootstrap).
// ------------------------------------------------------------------------------------------------
struct ScanArgs {
  const int32_t* reward_i;   // [T][B] integer reward shared by the columns (number of successes / ack)
  const float* value;        // [T][N][B]  (N = n_cols)
  double* adv_raw;           // [T][N][B] out (unnormalised lambda-return), may be null
  double* ret_raw;           // [T][N][B] out (unnormalised discounted return), may be null
  double* stats;             // [N][4]: sum adv, sumsq adv, sum ret(f32-cast), sumsq ret(f32-cast)
  int T, B, n_cols;
  double gamma, lam;
  int last_env_is_global_last;  // this shard holds the globally last env (multi-GPU)
  // two-pass mode (kScanStats then kScanEmit): nothing but the normalised fp32 results ever reaches HBM
  int want_adv, want_ret;
  float* adv_out;            // [T][N][B] normalised lambda-returns (fp64 maths, numpy semantics)
  float* ret_out;            // [T][N][B] normalised discounted returns (cast to fp32 first, torch semantics)
  const double *adv_mean, *adv_std, *ret_mean, *ret_std;   // [N]
  const int *adv_norm, *ret_norm;                          // [N] normalise flags
};

enum { kScanRaw = 0, kScanStats = 1, kScanEmit = 2 };
// or-ed into kScanRaw / kScanStats (deterministic mode): warp w of column g's blocks stores its four sums to
// a.stats[g][w][4] (a scratch of n_cols x gridDim.x x 4 warps) for sum_partials_kernel instead of the atomics
constexpr int kScanPartials = 4;

// One thread per (column, env) walks the episode backwards in float64 as numpy does.  The chain is serial and short of
// arithmetic, so the kernel lives on memory-level parallelism and on a lean instruction stream:
//  * the U rows of the NEXT batch are requested before the current batch is reduced (two register buffers), and the
//    rewards stay as loaded (int32 / fp32 bits) until they are reduced -- converting at load time waits for the load;
//  * running row pointers with register strides instead of 64-bit index arithmetic per access (address arithmetic was
//    40 % of the 141 thread-instructions per element of the first version: ncu opcode mix, profiles/r02_*);
//  * the episode-end row (t = T - 1) is peeled, the main loop runs whole batches without predicates.
// Normalisation multiplies by the float64 reciprocal of the std (one division per thread instead of one per element;
// the result differs from numpy's quotient by at most one float64 ulp BEFORE the cast to fp32).
template <int MODE_BITS>
__global__ void __launch_bounds__(128, 7) returns_scan_kernel(const ScanArgs a) {
  constexpr int MODE = MODE_BITS & 3;
  const int g = blockIdx.y;
  const bool do_adv = MODE == kScanRaw ? a.adv_raw != nullptr : (MODE == kScanStats ? a.want_adv : a.adv_out != nullptr);
  const bool do_ret = MODE == kScanRaw ? a.ret_raw != nullptr : (MODE == kScanStats ? a.want_ret : a.ret_out != nullptr);
  double s_adv = 0, q_adv = 0, s_ret = 0, q_ret = 0;
  // "do not normalise" is the identity map (x - 0) * 1, exact in both precisions: no select per element
  double am = 0.0, a_inv = 1.0;
  float rmf = 0.f, rsf = 1.f, r_inv = 1.f;
  if (MODE == kScanEmit) {
    if (do_adv && a.adv_norm[g] != 0) am = a.adv_mean[g], a_inv = 1.0 / a.adv_std[g];
    if (do_ret && a.ret_norm[g] != 0) rmf = (float)a.ret_mean[g], rsf = (float)a.ret_std[g], r_inv = 1.0f / rsf;
  }
  constexpr int U = 6;   // time steps per register buffer: 72 registers = 7 blocks per SM (U = 8 spills there), which
                         // turns the 3,072 blocks of the c3 rollout into 2.97 waves instead of 3.46 (0.366 -> 0.357 ms)
  const ptrdiff_t B = a.B, step = (ptrdiff_t)a.n_cols * a.B;
  const double gamma = a.gamma, gl = a.gamma * a.lam;
  const int T = a.T;
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += gridDim.x * blockDim.x) {
    // running pointers, all starting at the LAST row (t = T - 1) of this (column, env) and walked towards t = 0:
    // lr / lv feed the loads (one batch ahead), oa / orr the stores
    const int32_t* lr = a.reward_i + (ptrdiff_t)(T - 1) * B + b;
    const ptrdiff_t col = ((ptrdiff_t)(T - 1) * a.n_cols + g) * B + b;
    const float* lv = do_adv ? a.value + col : nullptr;
    float* oa = (MODE == kScanEmit && do_adv) ? a.adv_out + col : nullptr;
    float* orr = (MODE == kScanEmit && do_ret) ? a.ret_out + col : nullptr;
    double* wa = (MODE == kScanRaw && do_adv) ? a.adv_raw + col : nullptr;
    double* wr = (MODE == kScanRaw && do_ret) ? a.ret_raw + col : nullptr;
    double gae = 0.0, run = 0.0, v_next = 0.0;
    auto emit = [&](double out_a, double run_v) {   // writes the row the output pointers stand on, then moves them up
      if (do_adv) {
        if (MODE == kScanRaw) *wa = out_a, wa -= step;
        if (MODE == kScanEmit) __stcs(oa, (float)((out_a - am) * a_inv)), oa -= step;
        if (MODE != kScanEmit) s_adv += out_a, q_adv += out_a * out_a;
      }
      if (do_ret) {
        if (MODE == kScanRaw) *wr = run_v, wr -= step;
        const float xf = (float)run_v;               // the reference casts to fp32 before normalising (:119)
        if (MODE == kScanEmit) {
          // (xf - mean) / std in fp32, as torch: quotient by Markstein's correction of x * rn(1 / std) (correctly
          // rounded except for divisors with an all-ones mantissa), 3 FMA-pipe instructions instead of a division
          const float x = xf - rmf, q = x * r_inv;
          __stcs(orr, fmaf(fmaf(-q, rsf, x), r_inv, q)), orr -= step;
        }
        const double rf = (double)xf;
        if (MODE != kScanEmit) s_ret += rf, q_ret += rf * rf;
      }
    };
    auto row = [&](int raw, float vf) {              // a row that is not the episode end
      const double r = (double)raw, v = (double)vf;
      double out = 0.0;
      if (do_adv) {
        const double delta = r + gamma * v_next - v;
        gae = delta + gl * gae;
        out = gae + v;
        v_next = v;
      }
      if (do_ret) run = r + run * gamma;
      emit(out, run);
    };
    {   // t = T - 1 (done): delta = r - v, gae = delta, out = gae + v = r; the globally last row keeps r - v (:102)
      const double r = (double)__ldg(lr), v = do_adv ? (double)__ldg(lv) : 0.0;
      lr -= B;
      if (do_adv) lv -= step;
      const bool quirk = a.last_env_is_global_last && b == a.B - 1;
      gae = quirk ? 0.0 : r - v;
      v_next = v;
      run = r;
      emit(quirk ? r - v : gae + v, run);
    }
    // rows T - 2 .. 0: whole batches of U, double buffered; the rewards stay int32 until they are reduced
    int rA[U], rB[U];
    float vA[U], vB[U];
    auto load = [&](int (&rr)[U], float (&vv)[U]) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        rr[u] = __ldg(lr), lr -= B;
        vv[u] = 0.f;
        if (do_adv) vv[u] = __ldg(lv), lv -= step;
      }
    };
    auto reduce = [&](const int (&rr)[U], const float (&vv)[U]) {
#pragma unroll
      for (int u = 0; u < U; ++u) row(rr[u], vv[u]);
    };
    const int n_batches = (T - 1) / U;
    if (n_batches > 0) load(rA, vA);
    for (int i = 0; i < n_batches; i += 2) {
      if (i + 1 < n_batches) load(rB, vB);           // next batch in flight while this one is reduced
      reduce(rA, vA);
      if (i + 1 >= n_batches) break;
      if (i + 2 < n_batches) load(rA, vA);
      reduce(rB, vB);
    }
    for (int k = n_batches * U + 1; k < T; ++k) {    // the (T - 1) % U rows nearest to t = 0
      const int raw = __ldg(lr);
      lr -= B;
      float vf = 0.f;
      if (do_adv) vf = __ldg(lv), lv -= step;
      row(raw, vf);
    }
  }
  if (MODE == kScanEmit) return;
  double vals[4] = {s_adv, q_adv, s_ret, q_ret};
  for (int k = 0; k < 4; ++k) {
    double v = vals[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    if constexpr ((MODE_BITS & kScanPartials) != 0) {
      const long long w = (long long)g * gridDim.x * (blockDim.x >> 5) + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
      if ((threadIdx.x & 31) == 0) a.stats[4 * w + k] = v;
    } else {
      if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(&a.stats[4 * g + k], v);
    }
  }
}

// out[grp][k] += sum over p = 0 .. n_parts - 1 of part[grp][p][k], in a fixed order: block = (grp, k), thread i sums
// p = i, i + 256, ... in turn, then a fixed tree over the 256 threads.  The deterministic mode's replacement of the
// fp64 atomics of the loss, returns-statistics and gradient-norm sums.
__global__ void __launch_bounds__(256) sum_partials_kernel(const double* __restrict__ part, int n_parts, int n_vals,
                                                           double* __restrict__ out) {
  __shared__ double sh[256];
  const int grp = blockIdx.x / n_vals, k = blockIdx.x % n_vals;
  const double* p = part + (long long)grp * n_parts * n_vals + k;
  double s = 0.0;
  for (int i = threadIdx.x; i < n_parts; i += 256) s += p[(long long)i * n_vals];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] += sh[0];
}

// d(gi) of the observations [c0 - halo, c1) of a chunk from the L d(gi) slices the SLICES BPTT kernels stored
// (gru_bptt_tc.cuh, gru_bwd_tc.cuh): slice s holds, at the local time l of window t = c0 + l, the d(gi) that window
// step s gives observation t - (L - 1 - s).  Hence, with halo = L - 1 and o the local time of the observation,
//   dgi[o] = sum_{s = 0 .. L - 1, 0 <= o - s < n_win} slice_s[o - s]
// summed in increasing s: the same terms as the atomic accumulation, in a fixed order.  Every element is written.
//   slices [L][n_win_cap][per_t] floats;  dgi [n_win + L - 1][per_t];  per_t = 3H N B (a multiple of 4)
__global__ void dgi_slice_sum_kernel(const float4* __restrict__ slices, float4* __restrict__ dgi, int L, int n_win,
                                     long long slice_t, long long per_t4) {
  const long long n = (long long)(n_win + L - 1) * per_t4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int o = (int)(i / per_t4);
    const long long e = i % per_t4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < L; ++s) {
      const int l = o - s;
      if (l < 0 || l >= n_win) continue;
      const float4 v = __ldcs(slices + (long long)s * slice_t + (long long)l * per_t4 + e);
      acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
    }
    dgi[i] = acc;
  }
}

// mean / std / normalise-flag of the lambda-returns (numpy population std, d2d_ppo.py:108-109) and of the returns (torch
// unbiased std, :121-123) from the all-reduced [n_cols][4] sums; one block.  The reference normalises only if EVERY
// column has a positive std; the one-pass (sum, sum of squares) form leaves rounding noise of the order
// 1e-16 n mean^2 where numpy / torch give exactly 0, hence the gate is relative to the column's mean square.
// out: [6][n_cols] doubles = adv mean, adv std, ret mean, ret std, then (as int32 pairs) the two flag vectors.
__global__ void norm_stats_kernel(const double* __restrict__ stats, int n_cols, double rows, double* adv_mean,
                                  double* adv_std, int* adv_norm, double* ret_mean, double* ret_std, int* ret_norm) {
  const int c = threadIdx.x;
  bool ok_a = true, ok_r = true;
  double ma = 0, sa = 0, mr = 0, sr = 0;
  if (c < n_cols) {
    ma = stats[4 * c] / rows;
    const double va = (stats[4 * c + 1] - rows * ma * ma) / rows;                 // ddof = 0
    sa = sqrt(fmax(va, 0.0));
    ok_a = va > 1e-9 * (stats[4 * c + 1] / rows);
    mr = stats[4 * c + 2] / rows;
    const double vr = (stats[4 * c + 3] - rows * mr * mr) / (rows - 1.0);         // ddof = 1
    sr = sqrt(fmax(vr, 0.0));
    ok_r = vr > 1e-9 * (stats[4 * c + 3] / rows);
  }
  const int all_a = __syncthreads_and(ok_a), all_r = __syncthreads_and(ok_r);
  if (c < n_cols) {
    adv_mean[c] = ma, adv_std[c] = sa, adv_norm[c] = all_a;
    ret_mean[c] = mr, ret_std[c] = sr, ret_norm[c] = all_r;
  }
}

// out = (raw - mean) / std  per column (or a plain cast when do_norm[g] == 0), written as fp32
struct NormArgs {
  const double* raw;   // [T][N][B]
  float* out;          // [T][N][B]
  const double* mean;  // [N]
  const double* std;   // [N]
  const int* do_norm;  // [N]
  int fp32_math;       // 1: torch semantics of discount_rewards (cast first, normalise in fp32)
  long long per_t;     // N * B
  int B;
  long long n;         // T * N * B
};

__global__ void normalize_kernel(const NormArgs a) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.n; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)((i % a.per_t) / a.B);
    if (a.fp32_math) {   // the same Markstein quotient as returns_scan_kernel<kScanEmit> (bit-identical results)
      const float xf = (float)a.raw[i];
      const float sd = (float)a.std[g], inv = 1.0f / sd, x = xf - (float)a.mean[g], q = x * inv;
      a.out[i] = a.do_norm[g] ? fmaf(fmaf(-q, sd, x), inv, q) : xf;
    } else {   // reciprocal multiply, exactly as returns_scan_kernel<kScanEmit> does (bit-identical results)
      const double x = a.raw[i];
      a.out[i] = (float)(a.do_norm[g] ? (x - a.mean[g]) * (1.0 / a.std[g]) : x);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// optimiser: per-agent gradient norm (clip_grad_norm_, d2d_ppo.py:211,445) and torch.optim.Adam defaults
// ------------------------------------------------------------------------------------------------
// deterministic mode: one 512-thread block per agent; thread i sums elements i, i + 512, ... in turn, then a fixed tree;
// out[agent] is stored (no zeroing needed)
__global__ void __launch_bounds__(512) grad_sqnorm_tree_kernel(const float* __restrict__ g, long long per_agent,
                                                               double* __restrict__ out) {
  __shared__ double sh[512];
  const float* p = g + blockIdx.x * per_agent;
  double s = 0.0;
  for (long long i = threadIdx.x; i < per_agent; i += 512) {
    const double v = p[i];
    s += v * v;
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = 256; w > 0; w >>= 1) {
    if (threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

__global__ void grad_sqnorm_kernel(const float* __restrict__ g, long long per_agent, double* __restrict__ out) {
  const int a = blockIdx.y;
  double s = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < per_agent;
       i += (long long)gridDim.x * blockDim.x) {
    const double v = g[a * per_agent + i];
    s += v * v;
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xFFFFFFFFu, s, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(&out[a], s);
}

struct AdamArgs {
  float* p;
  float* m;
  float* v;
  const float* g;
  const double* sqnorm;   // [N] or null (no clipping)
  long long per_agent;
  float lr, beta1, beta2, eps, max_norm;
  float bc1, bc2;         // 1 - beta^t
};

__global__ void adam_kernel(const AdamArgs a) {
  const int ag = blockIdx.y;
  float coef = 1.0f;
  if (a.sqnorm) {
    const float total = (float)sqrt(a.sqnorm[ag]);
    coef = fminf(a.max_norm / (total + 1e-6f), 1.0f);
  }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.per_agent;
       i += (long long)gridDim.x * blockDim.x) {
    const long long j = ag * a.per_agent + i;
    const float g = a.g[j] * coef;
    const float m = a.beta1 * a.m[j] + (1.0f - a.beta1) * g;
    const float v = a.beta2 * a.v[j] + (1.0f - a.beta2) * g * g;
    a.m[j] = m, a.v[j] = v;
    const float denom = sqrtf(v) / sqrtf(a.bc2) + a.eps;
    a.p[j] = a.p[j] - (a.lr / a.bc1) * (m / denom);
  }
}

// inputs_bf16_exact guard: elements of x whose low 16 mantissa bits are not all zero (grid.y = time block)
__global__ void check_bf16_exact_kernel(const float* x, long long count, long long t_stride,
                                        unsigned long long* n_inexact) {
  const float* p = x + (long long)blockIdx.y * t_stride;
  unsigned int bad = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x)
    bad += (__float_as_uint(p[i]) & 0xFFFFu) != 0u;
  bad = __reduce_add_sync(0xFFFFFFFFu, bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(n_inexact, (unsigned long long)bad);
}

// max |x| over a buffer, as the bit pattern of a non-negative float (atomicMax on uint32); *out zeroed by the caller
__global__ void absmax_kernel(const float* __restrict__ x, long long n, unsigned int* out) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(x[i]));
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out, __float_as_uint(m));
}

}  // namespace d2d
