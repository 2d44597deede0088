// Lockstep step/reset of the three channel-access environments for B envs x N devices on one B200.
//
// Replaces (file:line under /root/reference):
//   envs/combinatorial_env.py:61-114 reset, :127-242 step     -> comb_reset_kernel / comb_step_kernel
//   envs/env.py:51-101 reset, :118-217 step                   -> sc_reset_kernel / sc_step_kernel
//   envs/channel_selection_env.py:49-98 reset, :116-214 step  -> sel_reset_kernel / sel_step_kernel
//   algorithms/baselines.py:181-183 CombinatorialRandomAccess.act (fused, act_mode = 1)
//
// Design (sm_100a, HBM-bound integer/byte work -- no tensor cores on purpose):
//   * one THREAD per env, devices looped in-thread.  Per-channel collision / success resolution is then pure
//     bitmask arithmetic in registers (once / twice accumulators over the devices' channel masks): no
//     shuffles, no idle lanes for N = 6, and every per-device parameter (deadline, switch thresholds,
//     arrival law) is warp-uniform, so there is no divergence on heterogeneous devices.
//   * env-minor structure of arrays: record k of env b lives at X[k][b]; a warp of 32 consecutive envs
//     issues one fully coalesced 128..512-byte request per row.  Packet buffers are one 8/16/32-byte record
//     per (device, env) (byte d = packets with d slots to the deadline), moved with one vector load/store.
//   * observations are emitted as f32 rows obs[row][b]: each warp store writes one full 128-byte line.
//   * grid-stride persistent launch sized in whole waves of the SM count; per-env parameters are staged
//     once per block in shared memory and read by broadcast.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "env_common.cuh"

namespace d2d {

template <int W>
int launch_comb_step(const StepArgs& a, int N, int C, int mask_bytes, cudaStream_t s);  // env_comb_w{2,4,8}.cu
template <int W>
int launch_comb_run(const StepArgs& a, const RunArgs& ra, int C, cudaStream_t s);         // env_comb_w{2,4}.cu

// ================================================================================================
// CombinatorialEnv reset (the step kernel lives in env_comb_step.cuh)
// ================================================================================================
template <int W, typename MaskT>
__global__ void __launch_bounds__(256) comb_reset_kernel(const StepArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const int N = P->N, C = P->C;
  const size_t B = (size_t)a.B;
  MaskT* chan = reinterpret_cast<MaskT*>(a.chan);
  const uint32_t cmask = C >= 32 ? 0xFFFFFFFFu : ((1u << C) - 1u);
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += gridDim.x * blockDim.x) {
    ArrivalWords arr_words;
    for (int k = 0; k < N; ++k) {
      const size_t idx = (size_t)k * B + b;
      Rec<W> r;
#pragma unroll
      for (int j = 0; j < W; ++j) r.w[j] = 0;
      uint32_t arrived = 0;
      const int dl = P->deadline[k];
      if ((a.active >> k) & 1ull) {
        arrived = draw_arrival(a, P, cdf, k, b, arr_words);
        rec_set_byte<W>(r, dl - 1, arrived);
      }
      rec_store<W>(a.buf, idx, r);
      chan[idx] = (MaskT)cmask;          // combinatorial_env.py:88
      a.disc[idx] = 0;                   // :91
      a.recv[idx] = arrived;             // :92
      if (a.obs) {                       // :102-109 -- channel and ack/nack slots are ones at reset
        float* o = a.obs + (size_t)P->obs_off[k] * B + b;
        const int nb = P->homog ? P->D : dl;
        rec_emit<W>(r, nb, o, B);
        o += (size_t)nb * B;
        for (int c = 0; c < 2 * C; ++c) o[(size_t)c * B] = 1.0f;
      }
      if (a.state) rec_emit<W>(r, dl, a.state + (size_t)P->sbuf_off[k] * B + b, B);
    }
    if (a.state) {                       // :110-112
      float* s = a.state + (size_t)P->sum_dl * B + b;
      for (int c = 0; c < (N + 1) * C; ++c) s[(size_t)c * B] = 1.0f;
    }
  }
}

// ================================================================================================
// D2DEnv (single channel)
// ================================================================================================
// NK > 0: register-resident fast path for N <= NK devices (records and channel bits are loaded once, kept in
// registers across the passes and stored once; the device loops are unrolled).  NK = 0: any N, records re-read
// from L1 in the second pass.  With the default self-only neighbourhoods (env.py:38-39) the observation of device k
// is emitted in the second pass from registers; other neighbourhoods take the gather pass at the end.
template <int W, int NK>
__global__ void __launch_bounds__(256, NK ? 5 : 4) sc_step_kernel(const StepArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const uint32_t* swthr = reinterpret_cast<const uint32_t*>(smem + P->off_sw);
  const int32_t* nbr_off = reinterpret_cast<const int32_t*>(smem + P->off_nbr_off);
  const uint8_t* nbr_idx = smem + P->off_nbr_idx;
  const int N = P->N;
  const size_t B = (size_t)a.B;
  const uint32_t Bu = (uint32_t)a.B;
  uint8_t* chan = reinterpret_cast<uint8_t*>(a.chan);
  const uint8_t* act = reinterpret_cast<const uint8_t*>(a.actions);
  uint8_t* act_out = reinterpret_cast<uint8_t*>(a.actions_out);
  const uint8_t* rp_sw = reinterpret_cast<const uint8_t*>(a.rp_sw);
  const bool self_obs = a.obs != nullptr && P->self_nbr != 0;
  constexpr int KR = NK ? NK : 1;

  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += gridDim.x * blockDim.x) {
    ArrivalWords arr_words;
    const uint32_t env = a.env_offset + (uint32_t)b;
    LaneWords pol_lanes, sw_lanes;   // one Philox call per eight devices for the 1-bit policy / switch draws
    Rec<W> rec[KR];
    uint32_t chv[KR], wantv[KR];
    // ---- pass 1 (env.py:125-127): attempts and the lone transmitter's channel ----
    uint64_t att = 0, good = 0;
    if constexpr (NK > 0) {
#pragma unroll
      for (int k = 0; k < NK; ++k) {           // every load of the env is issued before the first use
        const size_t idx = (size_t)min(k, N - 1) * B + b;
        rec[k] = rec_load<W>(a.buf, idx);
        chv[k] = chan[idx];
        wantv[k] = a.act_mode == 0 ? act[idx] : 0u;
      }
#pragma unroll
      for (int k = 0; k < NK; ++k) {
        if (k < N) {
          uint32_t want = wantv[k] != 0;
          if (a.act_mode != 0) {
            want = pol_lanes.get(a, env, k, kPurposePolicy) < a.tp_thr;
            if (act_out) act_out[(size_t)k * B + b] = (uint8_t)want;
          }
          const uint64_t at = (want && rec_any<W>(rec[k])) ? 1ull : 0ull;
          att |= at << k;
          good |= (at & (uint64_t)(chv[k] & 1u)) << k;
        }
      }
    } else {
      for (int k = 0; k < N; ++k) {
        const size_t idx = (size_t)k * B + b;
        const Rec<W> r = rec_load<W>(a.buf, idx);
        uint32_t want;
        if (a.act_mode == 0) {
          want = act[idx] != 0;
        } else {
          want = pol_lanes.get(a, env, k, kPurposePolicy) < a.tp_thr;
          if (act_out) act_out[idx] = (uint8_t)want;
        }
        const uint64_t at = (want && rec_any<W>(r)) ? 1ull : 0ull;
        att |= at << k;
        good |= (at & (uint64_t)(chan[idx] & 1u)) << k;
      }
    }
    const int n_att = __popcll(att);
    // env.py:130-152: exactly one attempt is decoded iff its channel is good (binomial(1, state) is deterministic)
    const bool lone = n_att == 1;
    const bool decoded = lone && good != 0;
    const int ack = n_att > 1 ? -1 : (decoded ? 1 : 0);
    const float ackf = (float)ack;
    // Counters are read-modified-written only when they change.  Fast path: every counter this env may touch is
    // requested here in ONE batch (one exposed DRAM latency instead of one per dependent update further down).
    uint32_t discv[KR], recvv[KR], st0 = 0, st1 = 0;
    if constexpr (NK > 0) {
      if (lone && !decoded) st0 = a.stats[b];
      if (n_att > 1) st1 = a.stats[B + b];
#pragma unroll
      for (int k = 0; k < NK; ++k) {
        discv[k] = recvv[k] = 0;
        if (k < N) {
          const size_t idx = (size_t)k * B + b;
          if (rec[k].w[0] & 0xFFu) discv[k] = a.disc[idx];    // slot 0 occupied: it may expire this step
          if ((a.active >> k) & 1ull) recvv[k] = a.recv[idx];
        }
      }
      if (lone && !decoded) a.stats[b] = st0 + 1;     // channel_errors (:147)
      if (n_att > 1) a.stats[B + b] = st1 + 1;        // n_collisions   (:150)
    } else {
      if (lone && !decoded) a.stats[b] += 1;
      if (n_att > 1) a.stats[B + b] += 1;
    }

    // ---- pass 2: serve, age, switch, arrive (+ state row, + observation when the neighbourhood is the device) ----
    auto second = [&](int k, Rec<W> r, uint32_t ch_old, uint32_t disc_v, uint32_t recv_v) {
      const size_t idx = (size_t)k * B + b;
      rec_pop_earliest<W>(r, decoded && ((att >> k) & 1ull));   // :137-144
      const uint32_t expired = rec_age<W>(r);                   // :157
      if (expired) a.disc[idx] = (NK > 0 ? disc_v : a.disc[idx]) + expired;   // :158
      uint32_t sw;                                              // :107-109
      if (a.rng_mode == D2D_RNG_REPLAY) {
        sw = rp_sw[idx] & 1u;
      } else {
        sw = sw_lanes.get(a, env, k, kPurposeSwitch) < swthr[k];
      }
      const uint32_t ch_new = (ch_old ^ sw) & 1u;
      chan[idx] = (uint8_t)ch_new;
      const int dl = P->deadline[k];
      if ((a.active >> k) & 1ull) {                             // :162-180
        const uint32_t arrived = draw_arrival(a, P, cdf, k, b, arr_words);
        rec_set_byte<W>(r, dl - 1, arrived);
        if (arrived) a.recv[idx] = (NK > 0 ? recv_v : a.recv[idx]) + arrived;
      }
      rec_store<W>(a.buf, idx, r);
      const float chf = ch_new ? 1.0f : 0.0f;
      if (a.state) {                                            // :189-190
        emit_slots<W>(r, dl, a.state + (size_t)P->sbuf_off[k] * B + b, Bu);
        st_f32(a.state + ((size_t)P->sum_dl + k) * B + b, chf);
      }
      if (self_obs) {                                           // :183-187 with neighbourhoods[k] = [k]
        float* o = emit_slots<W>(r, dl, a.obs + (size_t)P->obs_off[k] * B + b, Bu);
        st_f32(o, chf);                                         // post-switch channel
        st_f32(next_row(o, Bu), ackf);
      }
    };
    if constexpr (NK > 0) {
#pragma unroll
      for (int k = 0; k < NK; ++k)
        if (k < N) second(k, rec[k], chv[k], discv[k], recvv[k]);
    } else {
      for (int k = 0; k < N; ++k) {
        const size_t idx = (size_t)k * B + b;
        second(k, rec_load<W>(a.buf, idx), chan[idx], 0u, 0u);
      }
    }
    if (a.state) st_f32(a.state + ((size_t)P->sum_dl + N) * B + b, ackf);
    // ---- pass 3: general neighbourhood observations (env.py:183-187), channel is the post-switch state ----
    if (a.obs && !self_obs) {
      for (int k = 0; k < N; ++k) {
        float* o = a.obs + (size_t)P->obs_off[k] * B + b;
        for (int j = nbr_off[k]; j < nbr_off[k + 1]; ++j) {
          const int i = nbr_idx[j];
          const Rec<W> r = rec_load<W>(a.buf, (size_t)i * B + b);
          rec_emit<W>(r, P->deadline[i], o, B);
          o += (size_t)P->deadline[i] * B;
        }
        for (int j = nbr_off[k]; j < nbr_off[k + 1]; ++j, o += B) *o = (float)chan[(size_t)nbr_idx[j] * B + b];
        *o = ackf;
      }
    }
    a.reward[b] = (a.reward_accum ? a.reward[b] : 0) + ack;     // :191 rewards = zeros(N) + ack
    if (a.done) a.done[b] = (uint8_t)a.done_flag;
  }
}

// n_inner consecutive random-access steps of ONE episode in one launch (d2d_env_run_random_access without per-step
// outputs): the env's records, channel bits and counters are loaded once, live in registers for every step and are
// stored once; each step is the three Philox calls of sc_step_kernel (policy lanes, switch lanes, arrival words: one
// call each serves all N <= 4 devices) plus the serve / age / switch / arrive logic.  A thread only ever touches its own
// env, so no step needs a grid-wide barrier.  The per-step kernel at the named c2 size (4,096 envs) is launch-latency
// bound (8.2 us a step for ~0.5 MB of state); this one is bound by the dependent-issue chain of a single warp.
// Same Philox counters and the same update order as sc_step_kernel: trajectories are bit-identical.
// (RunArgs: env_common.cuh)
template <int W, int NK>
__global__ void __launch_bounds__(256) sc_run_kernel(const StepArgs a, const RunArgs ra) {
  extern __shared__ __align__(16) uint8_t smem[];
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const uint32_t* swthr = reinterpret_cast<const uint32_t*>(smem + P->off_sw);
  const int N = P->N;
  const size_t B = (size_t)a.B;
  uint8_t* chan = reinterpret_cast<uint8_t*>(a.chan);
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= a.B) return;
  const uint32_t env = a.env_offset + (uint32_t)b;
  Rec<W> rec[NK];
  uint32_t chv[NK], discv[NK], recvv[NK], thr_sw[NK];
  int dl[NK];
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    const int kk = min(k, N - 1);
    const size_t idx = (size_t)kk * B + b;
    rec[k] = rec_load<W>(a.buf, idx);
    chv[k] = chan[idx] & 1u, discv[k] = a.disc[idx], recvv[k] = a.recv[idx];
    thr_sw[k] = swthr[kk], dl[k] = P->deadline[kk];
  }
  uint32_t st0 = a.stats[b], st1 = a.stats[B + b];
  int32_t rew = a.reward_accum ? a.reward[b] : 0;
  auto lane16 = [](const uint4& r, int k) {
    const uint32_t w = pick_word(r, k >> 1);
    return (k & 1) ? (w >> 16) : (w & 0xFFFFu);
  };
#pragma unroll 1
  for (int i = 0; i < ra.n_inner; ++i) {
    const uint32_t t = a.t + (uint32_t)i;
    const uint64_t active = ra.active[ra.t_plain + i];
    // the three draws are independent of the state: their Philox rounds interleave
    const uint4 pol = philox_rk(a, env, t, kPurposePolicy << 16, 0u);
    const uint4 sw4 = philox_rk(a, env, t, kPurposeSwitch << 16, 0u);
    uint4 ar4 = make_uint4(0u, 0u, 0u, 0u);
    if (active) ar4 = philox_rk(a, env, t, kPurposeArrival << 16, 0u);
    uint32_t att = 0, good = 0;                                 // env.py:125-127
#pragma unroll
    for (int k = 0; k < NK; ++k) {
      if (k < N) {
        const uint32_t at = (lane16(pol, k) < a.tp_thr && rec_any<W>(rec[k])) ? 1u : 0u;
        att |= at << k;
        good |= (at & chv[k]) << k;
      }
    }
    const int n_att = __popc(att);                              // :130-152
    const bool lone = n_att == 1;
    const bool decoded = lone && good != 0;
    const int ack = n_att > 1 ? -1 : (decoded ? 1 : 0);
    st0 += (lone && !decoded) ? 1u : 0u;
    st1 += n_att > 1 ? 1u : 0u;
#pragma unroll
    for (int k = 0; k < NK; ++k) {
      if (k < N) {
        rec_pop_earliest<W>(rec[k], decoded && ((att >> k) & 1u));   // :137-144
        discv[k] += rec_age<W>(rec[k]);                              // :157-158
        chv[k] ^= lane16(sw4, k) < thr_sw[k] ? 1u : 0u;              // :107-109
        if ((active >> k) & 1ull) {                                  // :162-180
          const uint32_t arrived = arrival_from_u(P, cdf, k, pick_word(ar4, k));
          rec_set_byte<W>(rec[k], dl[k] - 1, arrived);
          recvv[k] += arrived;
        }
      }
    }
    if (a.reward_accum) rew += ack;                             // :191
    else a.reward[(size_t)i * ra.reward_stride + b] = ack;
  }
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    if (k < N) {
      const size_t idx = (size_t)k * B + b;
      rec_store<W>(a.buf, idx, rec[k]);
      chan[idx] = (uint8_t)chv[k];
      a.disc[idx] = discv[k], a.recv[idx] = recvv[k];
    }
  }
  a.stats[b] = st0, a.stats[B + b] = st1;
  if (a.reward_accum) a.reward[b] = rew;
  if (a.done) a.done[b] = (uint8_t)a.done_flag;
}

// The same episode-in-one-launch loop with FOUR LANES PER ENV (lane = device) for small batches, where sc_run_kernel is
// bound by the dependent-issue chain of its few warps (4,096 envs = 128 warps on 148 SMs): every lane keeps ONE device's
// record and counters, lanes 0 / 1 / 2 of a quad compute the policy / switch / arrival Philox call (one call per lane
// and step instead of three per thread) and hand the words round with shuffles, the attempt bits meet in a ballot.
// Same Philox counters and update order: trajectories are bit-identical to sc_run_kernel / sc_step_kernel.
template <int W>
__global__ void __launch_bounds__(128) sc_run_lanes_kernel(const StepArgs a, const RunArgs ra) {
  extern __shared__ __align__(16) uint8_t smem[];
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const uint32_t* swthr = reinterpret_cast<const uint32_t*>(smem + P->off_sw);
  const int N = P->N;
  const size_t B = (size_t)a.B;
  uint8_t* chan = reinterpret_cast<uint8_t*>(a.chan);
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int k = gid & 3, lane = threadIdx.x & 31, quad0 = lane & ~3;
  int b = gid >> 2;
  const bool env_ok = b < a.B;                       // whole quads are in or out; out-of-range quads still shuffle
  if (!env_ok) b = a.B - 1;
  const bool live = env_ok && k < N;
  const int kk = min(k, N - 1);
  const size_t idx = (size_t)kk * B + b;
  const uint32_t env = a.env_offset + (uint32_t)b;
  Rec<W> rec = rec_load<W>(a.buf, idx);
  uint32_t chv = chan[idx] & 1u, discv = a.disc[idx], recvv = a.recv[idx];
  const uint32_t thr_sw = swthr[kk];
  const int dl = P->deadline[kk];
  uint32_t st0 = a.stats[b], st1 = a.stats[B + b];
  int32_t rew = a.reward_accum ? a.reward[b] : 0;
#pragma unroll 1
  for (int i = 0; i < ra.n_inner; ++i) {
    const uint32_t t = a.t + (uint32_t)i;
    const uint64_t active = ra.active[ra.t_plain + i];
    // lane 0: policy words, lane 1: switch words, lane 2: arrival words (only when a device is active this step)
    uint4 r = make_uint4(0u, 0u, 0u, 0u);
    if (k < 2 || (k == 2 && active)) r = philox_rk(a, env, t, (k == 0 ? kPurposePolicy : (k == 1 ? kPurposeSwitch : kPurposeArrival)) << 16, 0u);
    // 16-bit policy / switch lanes of device k live in word k >> 1 (x or y for k < 4); the arrival word is word k
    const uint32_t px = __shfl_sync(0xFFFFFFFFu, r.x, quad0), py = __shfl_sync(0xFFFFFFFFu, r.y, quad0);
    const uint32_t sx = __shfl_sync(0xFFFFFFFFu, r.x, quad0 + 1), sy = __shfl_sync(0xFFFFFFFFu, r.y, quad0 + 1);
    const uint32_t ax = __shfl_sync(0xFFFFFFFFu, r.x, quad0 + 2), ay = __shfl_sync(0xFFFFFFFFu, r.y, quad0 + 2);
    const uint32_t az = __shfl_sync(0xFFFFFFFFu, r.z, quad0 + 2), aw = __shfl_sync(0xFFFFFFFFu, r.w, quad0 + 2);
    const uint32_t pw = (k >> 1) ? py : px, sw = (k >> 1) ? sy : sx;
    const uint32_t pol16 = (k & 1) ? (pw >> 16) : (pw & 0xFFFFu);
    const uint32_t sw16 = (k & 1) ? (sw >> 16) : (sw & 0xFFFFu);
    const uint32_t arw = k == 0 ? ax : (k == 1 ? ay : (k == 2 ? az : aw));
    const bool at = live && pol16 < a.tp_thr && rec_any<W>(rec);          // env.py:125-127
    const uint32_t att = (__ballot_sync(0xFFFFFFFFu, at) >> quad0) & 0xFu;
    const uint32_t good = (__ballot_sync(0xFFFFFFFFu, at && chv) >> quad0) & 0xFu;
    const int n_att = __popc(att);                                        // :130-152
    const bool lone = n_att == 1;
    const bool decoded = lone && good != 0;
    const int ack = n_att > 1 ? -1 : (decoded ? 1 : 0);
    st0 += (lone && !decoded) ? 1u : 0u;
    st1 += n_att > 1 ? 1u : 0u;
    if (live) {
      rec_pop_earliest<W>(rec, decoded && at);                            // :137-144
      discv += rec_age<W>(rec);                                           // :157-158
      chv ^= sw16 < thr_sw ? 1u : 0u;                                     // :107-109
      if ((active >> k) & 1ull) {                                         // :162-180
        const uint32_t arrived = arrival_from_u(P, cdf, k, arw);
        rec_set_byte<W>(rec, dl - 1, arrived);
        recvv += arrived;
      }
    }
    if (a.reward_accum) rew += ack;                                       // :191
    else if (k == 0 && env_ok) a.reward[(size_t)i * ra.reward_stride + b] = ack;
  }
  if (live) {
    rec_store<W>(a.buf, idx, rec);
    chan[idx] = (uint8_t)chv;
    a.disc[idx] = discv, a.recv[idx] = recvv;
  }
  if (k == 0 && env_ok) {
    a.stats[b] = st0, a.stats[B + b] = st1;
    if (a.reward_accum) a.reward[b] = rew;
    if (a.done) a.done[b] = (uint8_t)a.done_flag;
  }
}

template <int W>
__global__ void __launch_bounds__(256) sc_reset_kernel(const StepArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const int32_t* nbr_off = reinterpret_cast<const int32_t*>(smem + P->off_nbr_off);
  const uint8_t* nbr_idx = smem + P->off_nbr_idx;
  const int N = P->N;
  const size_t B = (size_t)a.B;
  uint8_t* chan = reinterpret_cast<uint8_t*>(a.chan);
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += gridDim.x * blockDim.x) {
    ArrivalWords arr_words;
    for (int k = 0; k < N; ++k) {
      const size_t idx = (size_t)k * B + b;
      Rec<W> r;
#pragma unroll
      for (int j = 0; j < W; ++j) r.w[j] = 0;
      uint32_t arrived = 0;
      if ((a.active >> k) & 1ull) {
        arrived = draw_arrival(a, P, cdf, k, b, arr_words);
        rec_set_byte<W>(r, P->deadline[k] - 1, arrived);
      }
      rec_store<W>(a.buf, idx, r);
      chan[idx] = 1;                     // env.py:79
      a.disc[idx] = 0;
      a.recv[idx] = arrived;
      if (a.state) {
        rec_emit<W>(r, P->deadline[k], a.state + (size_t)P->sbuf_off[k] * B + b, B);
        a.state[((size_t)P->sum_dl + k) * B + b] = 1.0f;
      }
    }
    a.stats[b] = 0;
    a.stats[B + b] = 0;
    if (a.state) a.state[((size_t)P->sum_dl + N) * B + b] = 0.0f;   // last_feedback = 0 (env.py:87,99)
    if (a.obs) {                                                    // env.py:92-96
      for (int k = 0; k < N; ++k) {
        float* o = a.obs + (size_t)P->obs_off[k] * B + b;
        for (int j = nbr_off[k]; j < nbr_off[k + 1]; ++j) {
          const int i = nbr_idx[j];
          const Rec<W> r = rec_load<W>(a.buf, (size_t)i * B + b);
          rec_emit<W>(r, P->deadline[i], o, B);
          o += (size_t)P->deadline[i] * B;
        }
        for (int j = nbr_off[k]; j < nbr_off[k + 1]; ++j, o += B) *o = 1.0f;
        *o = 0.0f;
      }
    }
  }
}

// ================================================================================================
// ChannelSelectionEnv
// ================================================================================================
constexpr int kCountPlanes = 7;  // bit-sliced per-channel attempt counters, counts up to 127 >= N

template <int W>
__global__ void __launch_bounds__(256, 4) sel_step_kernel(const StepArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const uint32_t* swthr = reinterpret_cast<const uint32_t*>(smem + P->off_sw);
  const int N = P->N, C1 = P->C + 1;
  const size_t B = (size_t)a.B;
  const uint32_t Bu = (uint32_t)a.B;
  uint32_t* chan = reinterpret_cast<uint32_t*>(a.chan);
  const uint8_t* act = reinterpret_cast<const uint8_t*>(a.actions);
  uint8_t* act_out = reinterpret_cast<uint8_t*>(a.actions_out);
  const uint32_t* rp_sw = reinterpret_cast<const uint32_t*>(a.rp_sw);
  const uint32_t cmask = C1 >= 32 ? 0xFFFFFFFFu : ((1u << C1) - 1u);
  const int n_planes = 32 - __clz(N);     // a channel is picked by at most N devices: bits(N) counter planes suffice
  // act_mode 1: fused RandomAccess policy (algorithms/baselines.py:10-14): every device draws a channel id uniformly
  // from 0..C (0 = stay idle) -- floor(u32 (C + 1) / 2^32) of the Philox policy stream, one call per four devices --
  // and devices without a packet are set to 0.  The drawn ids are kept in a local array for the second pass.
  const bool fused_policy = a.act_mode != 0;

  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += gridDim.x * blockDim.x) {
    ArrivalWords arr_words;
    const uint32_t env = a.env_offset + (uint32_t)b;
    const uint32_t ch = chan[b];
    // ---- pass 1 (channel_selection_env.py:124-128): per-channel attempt counts, bit-sliced ----
    uint32_t plane[kCountPlanes];
#pragma unroll
    for (int j = 0; j < kCountPlanes; ++j) plane[j] = 0;
#pragma unroll 4
    uint8_t drawn[D2D_MAX_AGENTS];
    uint4 pol4 = make_uint4(0u, 0u, 0u, 0u);
    for (int k = 0; k < N; ++k) {
      const size_t idx = (size_t)k * B + b;
      const Rec<W> r = rec_load<W>(a.buf, idx);
      uint32_t sel;
      if (fused_policy) {
        if ((k & 3) == 0) pol4 = philox4x32_10(env, a.t, (uint32_t)(k >> 2) | (kPurposePolicy << 16), 0u, a.k0, a.k1);
        sel = rec_any<W>(r) ? __umulhi(pick_word(pol4, k & 3), (uint32_t)C1) : 0u;
        drawn[k] = (uint8_t)sel;
        if (act_out) act_out[idx] = (uint8_t)sel;
      } else {
        sel = act[idx];
      }
      uint32_t carry = (sel != 0 && rec_any<W>(r)) ? (1u << sel) : 0u;
#pragma unroll
      for (int j = 0; j < kCountPlanes; ++j) {
        if (j < n_planes) {
          const uint32_t s = plane[j] ^ carry;
          carry &= plane[j];
          plane[j] = s;
        }
      }
    }
    uint32_t selected = 0, multi = 0;
#pragma unroll
    for (int j = 0; j < kCountPlanes; ++j) {
      selected |= plane[j];
      if (j > 0) multi |= plane[j];
    }
    const uint32_t win = plane[0] & ~multi & ch;                 // :140-141 one attempt on a good channel
    if (selected) {                                              // counters move only when somebody transmitted
      const uint32_t s0 = a.stats[b], s1 = a.stats[B + b];
      a.stats[b] = s0 + __popc(selected & ch);                   // :132 selected_channel_qualities
      a.stats[B + b] = s1 + __popc(selected);                    // :133 number_selected_channel
    }

    // ---- pass 2: device k + 1's record and counters are fetched while device k is processed ----
    int n_success = 0;
    Rec<W> r_nx = rec_load<W>(a.buf, (size_t)b);                 // second touch of the record: L1 hit
    uint32_t sel_nx = fused_policy ? drawn[0] : act[b];
    uint32_t disc_nx = (r_nx.w[0] & 0xFFu) ? a.disc[b] : 0u;
    uint32_t recv_nx = (a.active & 1ull) ? a.recv[b] : 0u;
#pragma unroll 1
    for (int k = 0; k < N; ++k) {
      const size_t idx = (size_t)k * B + b;
      Rec<W> r = r_nx;
      const uint32_t sel = sel_nx, disc_v = disc_nx, recv_v = recv_nx;
      if (k + 1 < N) {
        const size_t nx = idx + B;
        r_nx = rec_load<W>(a.buf, nx);
        sel_nx = fused_policy ? drawn[k + 1] : act[nx];
        disc_nx = (r_nx.w[0] & 0xFFu) ? a.disc[nx] : 0u;
        if ((a.active >> (k + 1)) & 1ull) recv_nx = a.recv[nx];
      }
      const bool success = sel != 0 && rec_any<W>(r) && ((win >> sel) & 1u);   // :142
      n_success += success;
      rec_pop_earliest<W>(r, success);
      const uint32_t expired = rec_age<W>(r);
      if (expired) a.disc[idx] = disc_v + expired;
      const int dl = P->deadline[k];
      if ((a.active >> k) & 1ull) {
        const uint32_t arrived = draw_arrival(a, P, cdf, k, b, arr_words);
        rec_set_byte<W>(r, dl - 1, arrived);
        if (arrived) a.recv[idx] = recv_v + arrived;
      }
      rec_store<W>(a.buf, idx, r);
      if (a.obs) emit_slots<W>(r, dl, a.obs + (size_t)P->obs_off[k] * B + b, Bu);
      if (a.state) emit_slots<W>(r, dl, a.state + (size_t)P->sbuf_off[k] * B + b, Bu);
    }
    uint32_t sw;                                                 // :104-107 C+1 scalar draws
    if (a.rng_mode == D2D_RNG_REPLAY) {
      sw = rp_sw[b];
    } else {
      sw = philox_lane_mask(env, a.t, kEnvLevelDevice | (kPurposeSwitch << 16), C1, a.k0, a.k1,
                            [swthr](int c) { return swthr[c]; });
    }
    const uint32_t ch_new = (ch ^ sw) & cmask;
    chan[b] = ch_new;
    // ack/nack vector (:129-137): 0 unused, -1 bad channel, 1/count good channel -- computed once per channel into
    // registers, then streamed to every device's observation rows with a running row pointer
    float v[D2D_MAX_CHANNELS];
#pragma unroll
    for (int c = 0; c < D2D_MAX_CHANNELS; ++c) {
      int cnt = 0;
#pragma unroll
      for (int j = 0; j < kCountPlanes; ++j)
        if (j < n_planes) cnt |= (int)((plane[j] >> c) & 1u) << j;
      v[c] = cnt == 0 ? 0.0f : (((ch >> c) & 1u) ? P->inv_count[cnt] : -1.0f);
    }
    if (a.obs) {                                                 // :181-184
      for (int k = 0; k < N; ++k) {
        float* o = a.obs + ((size_t)P->obs_off[k] + P->deadline[k]) * B + b;
#pragma unroll
        for (int c = 0; c < D2D_MAX_CHANNELS; ++c) {
          if (c < C1) {
            st_f32(o, v[c]);
            o = next_row(o, Bu);
          }
        }
      }
    }
    if (a.ack) {
      float* q = reinterpret_cast<float*>(a.ack) + b;
#pragma unroll
      for (int c = 0; c < D2D_MAX_CHANNELS; ++c) {
        if (c < C1) {
          st_f32(q, v[c]);
          q = next_row(q, Bu);
        }
      }
    }
    if (a.state) {                                               // :186
      float* q = a.state + (size_t)P->sum_dl * B + b;
#pragma unroll
      for (int c = 0; c < D2D_MAX_CHANNELS; ++c) {
        if (c < C1) {
          st_f32(q, ((ch_new >> c) & 1u) ? 1.0f : 0.0f);
          q = next_row(q, Bu);
        }
      }
    }
    a.reward[b] = (a.reward_accum ? a.reward[b] : 0) + n_success;  // :188
    if (a.done) a.done[b] = (uint8_t)a.done_flag;
  }
}

template <int W>
__global__ void __launch_bounds__(256) sel_reset_kernel(const StepArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const int N = P->N, C1 = P->C + 1;
  const size_t B = (size_t)a.B;
  uint32_t* chan = reinterpret_cast<uint32_t*>(a.chan);
  const uint32_t cmask = C1 >= 32 ? 0xFFFFFFFFu : ((1u << C1) - 1u);
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < a.B; b += gridDim.x * blockDim.x) {
    ArrivalWords arr_words;
    for (int k = 0; k < N; ++k) {
      const size_t idx = (size_t)k * B + b;
      Rec<W> r;
#pragma unroll
      for (int j = 0; j < W; ++j) r.w[j] = 0;
      uint32_t arrived = 0;
      if ((a.active >> k) & 1ull) {
        arrived = draw_arrival(a, P, cdf, k, b, arr_words);
        rec_set_byte<W>(r, P->deadline[k] - 1, arrived);
      }
      rec_store<W>(a.buf, idx, r);
      a.disc[idx] = 0;
      a.recv[idx] = arrived;
      if (a.obs) {                        // channel_selection_env.py:90-94 (ack/nack slot is zeros)
        float* o = a.obs + (size_t)P->obs_off[k] * B + b;
        rec_emit<W>(r, P->deadline[k], o, B);
        o += (size_t)P->deadline[k] * B;
        for (int c = 0; c < C1; ++c) o[(size_t)c * B] = 0.0f;
      }
      if (a.state) rec_emit<W>(r, P->deadline[k], a.state + (size_t)P->sbuf_off[k] * B + b, B);
    }
    chan[b] = cmask;                      // :76
    a.stats[b] = 0;
    a.stats[B + b] = 0;
    if (a.state)
      for (int c = 0; c < C1; ++c) a.state[((size_t)P->sum_dl + c) * B + b] = 1.0f;
  }
}

// ------------------------------------------------------------------------------------------------
// small utilities
// ------------------------------------------------------------------------------------------------
// u8 [B][N][C] 0/1 -> bitmask [N][B]
template <typename MaskT>
__global__ void pack_actions_kernel(const uint8_t* __restrict__ src, MaskT* __restrict__ dst, int B, int N, int C) {
  const long long total = (long long)B * N;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i / B), b = (int)(i % B);
    const uint8_t* s = src + ((size_t)b * N + k) * C;
    uint32_t m = 0;
    for (int c = 0; c < C; ++c) m |= (uint32_t)(s[c] != 0) << c;
    dst[i] = (MaskT)m;
  }
}

// per-env URLLC score, Jain index, channel score (combinatorial_env.py:245-264), in float64 like numpy
__global__ void scores_kernel(const uint32_t* __restrict__ disc, const uint32_t* __restrict__ recv,
                              const uint32_t* __restrict__ stats, int kind, int B, int N, double* urllc,
                              double* jains, double* chscore) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    double sd = 0, sr = 0, s1 = 0, s2 = 0;
    for (int k = 0; k < N; ++k) {
      const double d = disc[(size_t)k * B + b], r = recv[(size_t)k * B + b];
      sd += d, sr += r;
      const double u = r > 0 ? 1.0 - d / r : 1.0;
      s1 += u, s2 += u * u;
    }
    if (urllc) urllc[b] = 1.0 - sd / sr;
    if (jains) jains[b] = s1 * s1 / N / s2;
    if (chscore) {
      double v = 1.0;
      if (kind == D2D_ENV_CHANNEL_SELECTION && stats[(size_t)B + b] != 0)
        v = (double)stats[b] / (double)stats[(size_t)B + b];
      chscore[b] = v;
    }
  }
}

}  // namespace d2d

// ================================================================================================
// C ABI
// ================================================================================================
using namespace d2d;

struct d2d_env {
  int kind, B, N, C, T, homog, rng_mode;
  uint64_t seed, env_offset;
  int D, W, CB;  // max deadline, words per record, bytes per channel mask element
  int t;
  long long episode = -1;   // index of the current episode (number of resets - 1): folded into the Philox counter
  bool is_reset;
  std::vector<int> deadlines, obs_off, obs_dim;
  std::vector<uint64_t> active;
  uint64_t* active_dev = nullptr;   // device copy of `active` (multi-step kernels index it by the episode timestep)
  int obs_rows, state_rows, sum_dl;
  uint32_t* buf = nullptr;
  void* chan = nullptr;
  uint32_t* disc = nullptr;
  uint32_t* recv = nullptr;
  uint32_t* stats = nullptr;
  uint8_t* params = nullptr;
  int params_bytes = 0;
  const uint8_t* rp_arr = nullptr;
  const void* rp_sw = nullptr;
  int rp_len = 0;
  struct HostPipe* pipe = nullptr;   // lazily created by d2d_env_step_host
  size_t chan_elems() const { return kind == D2D_ENV_CHANNEL_SELECTION ? (size_t)B : (size_t)N * B; }
};

// Staging of the host-buffer step (d2d_env_step_host): two calls in flight, copies on their own streams so the
// H2D of call k + 1 and the D2H of call k - 1 overlap the kernels of call k.
struct HostPipe {
  static constexpr int kSlots = 2;
  cudaStream_t h2d = nullptr, d2h = nullptr;
  uint8_t* stage[kSlots] = {nullptr, nullptr};    // device copy of the host actions, as the host laid them out
  uint8_t* hpacked[kSlots] = {nullptr, nullptr};  // pinned host buffers: the actions packed to bitmasks on the host
  // host packing pays only while the host packs faster than PCIe would move the unpacked bytes; the first calls are
  // timed and a host that is too slow (a loaded box: 37 GB/s measured instead of ~80) falls back for good
  int pack_samples = 0;
  double pack_ms_sum = 0.0;
  int host_pack_state = -1;                       // -1 not used yet, 1 active, 0 switched off after the timed calls
  void* masks[kSlots] = {nullptr, nullptr};       // device-layout actions [N][B] (packed from `stage` if needed)
  int32_t* reward[kSlots] = {nullptr, nullptr};
  uint8_t* done[kSlots] = {nullptr, nullptr};
  cudaEvent_t in_ready[kSlots], step_done[kSlots], out_done[kSlots];
  bool events = false;
  uint64_t calls = 0;
  size_t stage_bytes = 0;
};

// host_pack.cpp
namespace d2d {
void host_pack_actions(const uint8_t* src, void* dst, long long B, int N, int C, int mask_bytes);
bool host_pack_is_fast(int C, int mask_bytes);
int host_threads();
}  // namespace d2d
// fewer threads than this pack no faster than PCIe moves the unpacked bytes (measured: 16 threads 82 GB/s of action
// bytes, 8 threads about the 50 - 55 GB/s of the link)
constexpr int kHostPackMinThreads = 12;
constexpr int kHostPackSamples = 8;
constexpr int kRunLanesMaxEnvs = 32768;   // up to here the multi-step env kernel runs four lanes per env

static void pipe_free(HostPipe* p) {
  if (!p) return;
  if (p->h2d) cudaStreamSynchronize(p->h2d);
  if (p->d2h) cudaStreamSynchronize(p->d2h);
  for (int i = 0; i < HostPipe::kSlots; ++i) {
    cudaFree(p->stage[i]), cudaFree(p->masks[i]), cudaFree(p->reward[i]), cudaFree(p->done[i]);
    if (p->hpacked[i]) cudaFreeHost(p->hpacked[i]);
    if (p->events) cudaEventDestroy(p->in_ready[i]), cudaEventDestroy(p->step_done[i]), cudaEventDestroy(p->out_done[i]);
  }
  if (p->h2d) cudaStreamDestroy(p->h2d);
  if (p->d2h) cudaStreamDestroy(p->d2h);
  delete p;
}

static int env_free(d2d_env* e) {
  if (!e) return D2D_OK;
  pipe_free(e->pipe);
  cudaFree(e->buf), cudaFree(e->chan), cudaFree(e->disc), cudaFree(e->recv), cudaFree(e->stats), cudaFree(e->params);
  cudaFree(e->active_dev);
  delete e;
  return D2D_OK;
}

extern "C" int d2d_env_create(const d2d_env_config* cfg, d2d_env** out) {
  D2D_REQUIRE(cfg && out, "d2d_env_create: null argument");
  *out = nullptr;
  D2D_REQUIRE(cfg->kind >= 0 && cfg->kind <= 2, "d2d_env_create: unknown env kind %d", cfg->kind);
  D2D_REQUIRE(cfg->n_envs > 0, "d2d_env_create: n_envs must be positive");
  D2D_REQUIRE(cfg->n_agents > 0 && cfg->n_agents <= D2D_MAX_AGENTS, "d2d_env_create: n_agents %d not in 1..%d",
              cfg->n_agents, D2D_MAX_AGENTS);
  const int maxC = cfg->kind == D2D_ENV_CHANNEL_SELECTION ? D2D_MAX_CHANNELS - 1 : D2D_MAX_CHANNELS;
  D2D_REQUIRE(cfg->n_channels > 0 && cfg->n_channels <= maxC, "d2d_env_create: n_channels %d not in 1..%d",
              cfg->n_channels, maxC);
  D2D_REQUIRE(cfg->kind != D2D_ENV_SINGLE_CHANNEL || cfg->n_channels == 1,
              "d2d_env_create: the single-channel env has n_channels = 1");
  D2D_REQUIRE(cfg->episode_length > 0, "d2d_env_create: episode_length must be positive");
  D2D_REQUIRE(cfg->rng_mode == D2D_RNG_PHILOX || cfg->rng_mode == D2D_RNG_REPLAY, "d2d_env_create: bad rng_mode");
  D2D_REQUIRE(cfg->deadlines && cfg->arrival_kind && cfg->arrival_active && cfg->poisson_cdf && cfg->bernoulli_thr &&
                  cfg->switch_thr,
              "d2d_env_create: null table pointer");
  D2D_REQUIRE((uint64_t)cfg->n_envs + cfg->env_offset <= 0xFFFFFFFFull, "d2d_env_create: env index exceeds 32 bits");

  d2d_env* e = new (std::nothrow) d2d_env();
  D2D_REQUIRE(e, "d2d_env_create: out of host memory");
  e->kind = cfg->kind, e->B = cfg->n_envs, e->N = cfg->n_agents, e->C = cfg->n_channels, e->T = cfg->episode_length;
  e->homog = cfg->homogeneous_size != 0, e->rng_mode = cfg->rng_mode, e->seed = cfg->seed;
  e->env_offset = cfg->env_offset, e->t = 0, e->is_reset = false;
  const int N = e->N, C = e->C;
  e->D = 0, e->sum_dl = 0;
  for (int k = 0; k < N; ++k) {
    const int dl = cfg->deadlines[k];
    if (dl < 1 || dl > D2D_MAX_DEADLINE) {
      set_error("d2d_env_create: deadline[%d] = %d not in 1..%d", k, dl, D2D_MAX_DEADLINE);
      env_free(e);
      return D2D_ERR_INVALID;
    }
    e->deadlines.push_back(dl);
    e->D = std::max(e->D, dl);
    e->sum_dl += dl;
  }
  e->W = e->D <= 8 ? 2 : (e->D <= 16 ? 4 : 8);
  e->CB = C <= 8 ? 1 : (C <= 16 ? 2 : 4);
  if (e->kind == D2D_ENV_SINGLE_CHANNEL) e->CB = 1;
  if (e->kind == D2D_ENV_CHANNEL_SELECTION) e->CB = 4;
  e->active.assign(cfg->arrival_active, cfg->arrival_active + e->T + 1);

  // ---- parameter blob ----
  std::vector<int> nbr_off(N + 1, 0);
  std::vector<uint8_t> nbr_idx;
  if (e->kind == D2D_ENV_SINGLE_CHANNEL) {
    for (int k = 0; k < N; ++k) {
      if (cfg->nbr_offset && cfg->nbr_index) {
        for (int j = cfg->nbr_offset[k]; j < cfg->nbr_offset[k + 1]; ++j) {
          const int i = cfg->nbr_index[j];
          if (i < 0 || i >= N) {
            set_error("d2d_env_create: neighbour index %d out of range", i);
            env_free(e);
            return D2D_ERR_INVALID;
          }
          nbr_idx.push_back((uint8_t)i);
        }
      } else {
        nbr_idx.push_back((uint8_t)k);
      }
      nbr_off[k + 1] = (int)nbr_idx.size();
    }
  }
  const int n_sw = e->kind == D2D_ENV_COMBINATORIAL ? N * C : (e->kind == D2D_ENV_SINGLE_CHANNEL ? N : C + 1);
  auto align16 = [](int x) { return (x + 15) & ~15; };
  EnvParamsHdr h;
  memset(&h, 0, sizeof(h));
  h.N = N, h.C = C, h.D = e->D, h.T = e->T, h.homog = e->homog, h.kind = e->kind, h.sum_dl = e->sum_dl;
  h.self_nbr = 1;
  for (int k = 0; k < N && e->kind == D2D_ENV_SINGLE_CHANNEL; ++k)
    if (nbr_off[k + 1] - nbr_off[k] != 1 || nbr_idx[nbr_off[k]] != k) h.self_nbr = 0;
  h.off_cdf = align16((int)sizeof(EnvParamsHdr));
  h.off_sw = h.off_cdf + align16(N * D2D_POISSON_KMAX * 4);
  h.off_nbr_off = h.off_sw + align16(n_sw * 4);
  h.off_nbr_idx = h.off_nbr_off + align16((N + 1) * 4);
  h.total_bytes = h.off_nbr_idx + align16((int)nbr_idx.size() + 1);
  int row = 0, srow = 0;
  for (int k = 0; k < N; ++k) {
    int dim;
    if (e->kind == D2D_ENV_COMBINATORIAL) {
      dim = (e->homog ? e->D : e->deadlines[k]) + 2 * C;                 // combinatorial_env.py:47-53
    } else if (e->kind == D2D_ENV_SINGLE_CHANNEL) {
      dim = 1;                                                           // env.py:43-44
      for (int j = nbr_off[k]; j < nbr_off[k + 1]; ++j) dim += e->deadlines[nbr_idx[j]] + 1;
    } else {
      dim = e->deadlines[k] + C + 1;                                     // channel_selection_env.py:41-42
    }
    e->obs_off.push_back(row), e->obs_dim.push_back(dim);
    h.deadline[k] = (uint8_t)e->deadlines[k];
    h.arrival_kind[k] = (uint8_t)cfg->arrival_kind[k];
    h.obs_off[k] = (uint16_t)row, h.obs_dim[k] = (uint16_t)dim, h.sbuf_off[k] = (uint16_t)srow;
    h.bern_thr[k] = cfg->bernoulli_thr[k];
    row += dim, srow += e->deadlines[k];
  }
  for (int n = 1; n <= D2D_MAX_AGENTS; ++n) h.inv_count[n] = (float)(1.0 / (double)n);
  e->obs_rows = row;
  e->state_rows = e->kind == D2D_ENV_COMBINATORIAL ? e->sum_dl + C * (N + 1)       // combinatorial_env.py:57-58
                  : e->kind == D2D_ENV_SINGLE_CHANNEL ? e->sum_dl + N + 1          // env.py:47-48
                                                      : e->sum_dl + C + 1;         // channel_selection_env.py:45-46
  h.obs_rows = e->obs_rows, h.state_rows = e->state_rows;
  std::vector<uint8_t> blob(h.total_bytes, 0);
  memcpy(blob.data(), &h, sizeof(h));
  memcpy(blob.data() + h.off_cdf, cfg->poisson_cdf, (size_t)N * D2D_POISSON_KMAX * 4);
  memcpy(blob.data() + h.off_sw, cfg->switch_thr, (size_t)n_sw * 4);
  memcpy(blob.data() + h.off_nbr_off, nbr_off.data(), (size_t)(N + 1) * 4);
  if (!nbr_idx.empty()) memcpy(blob.data() + h.off_nbr_idx, nbr_idx.data(), nbr_idx.size());
  e->params_bytes = h.total_bytes;

  const size_t nb = (size_t)N * e->B;
  cudaError_t err = cudaSuccess;
  auto alloc = [&](void** p, size_t bytes) {
    if (err == cudaSuccess) err = cudaMalloc(p, bytes);
    if (err == cudaSuccess) err = cudaMemset(*p, 0, bytes);
  };
  alloc((void**)&e->buf, nb * e->W * 4);
  alloc(&e->chan, e->chan_elems() * e->CB);
  alloc((void**)&e->disc, nb * 4);
  alloc((void**)&e->recv, nb * 4);
  alloc((void**)&e->stats, (size_t)2 * e->B * 4);
  alloc((void**)&e->params, blob.size());
  if (err == cudaSuccess) err = cudaMemcpy(e->params, blob.data(), blob.size(), cudaMemcpyHostToDevice);
  alloc((void**)&e->active_dev, e->active.size() * 8);
  if (err == cudaSuccess)
    err = cudaMemcpy(e->active_dev, e->active.data(), e->active.size() * 8, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) {
    set_error("d2d_env_create: CUDA allocation failed: %s", cudaGetErrorString(err));
    env_free(e);
    return D2D_ERR_CUDA;
  }
  *out = e;
  return D2D_OK;
}

extern "C" int d2d_env_destroy(d2d_env* env) { return env_free(env); }
extern "C" int d2d_env_obs_rows(const d2d_env* e) { return e ? e->obs_rows : D2D_ERR_INVALID; }
extern "C" int d2d_env_obs_offset(const d2d_env* e, int k) {
  return (e && k >= 0 && k < e->N) ? e->obs_off[k] : D2D_ERR_INVALID;
}
extern "C" int d2d_env_obs_dim(const d2d_env* e, int k) {
  return (e && k >= 0 && k < e->N) ? e->obs_dim[k] : D2D_ERR_INVALID;
}
extern "C" int d2d_env_state_rows(const d2d_env* e) { return e ? e->state_rows : D2D_ERR_INVALID; }
extern "C" int d2d_env_timestep(const d2d_env* e) { return e ? e->t : D2D_ERR_INVALID; }
extern "C" int d2d_env_record_bytes(const d2d_env* e) { return e ? e->W * 4 : D2D_ERR_INVALID; }
extern "C" int d2d_env_mask_bytes(const d2d_env* e) { return e ? e->CB : D2D_ERR_INVALID; }
extern "C" int64_t d2d_env_episode(const d2d_env* e) { return e ? e->episode : D2D_ERR_INVALID; }
extern "C" int d2d_env_set_episode(d2d_env* e, int64_t next_episode) {
  D2D_REQUIRE(e && next_episode >= 0, "d2d_env_set_episode: null env or negative episode index");
  e->episode = next_episode - 1;   // the next reset() starts episode `next_episode`
  return D2D_OK;
}

extern "C" int d2d_env_set_replay(d2d_env* e, const uint8_t* arrivals, const void* switches, int t_len) {
  D2D_REQUIRE(e, "d2d_env_set_replay: null env");
  D2D_REQUIRE(e->rng_mode == D2D_RNG_REPLAY, "d2d_env_set_replay: env was not created with D2D_RNG_REPLAY");
  D2D_REQUIRE(arrivals && switches && t_len >= 1, "d2d_env_set_replay: null stream or empty length");
  e->rp_arr = arrivals, e->rp_sw = switches, e->rp_len = t_len;
  return D2D_OK;
}

static int fill_args(d2d_env* e, StepArgs& a, uint32_t t, const char* who) {
  memset(&a, 0, sizeof(a));
  a.buf = e->buf, a.chan = e->chan, a.disc = e->disc, a.recv = e->recv, a.stats = e->stats;
  a.params = e->params, a.params_bytes = e->params_bytes;
  // Philox streams: the counter's timestep field is t + episode * (T + 1), so that every episode of an env draws
  // fresh traffic (replayed streams, arrival phases and the done flag use the plain episode timestep)
  const uint32_t t_ctr = t + (uint32_t)((unsigned long long)std::max<long long>(e->episode, 0) * (unsigned)(e->T + 1));
  a.B = e->B, a.t = t_ctr, a.k0 = (uint32_t)(e->seed & 0xFFFFFFFFull), a.k1 = (uint32_t)(e->seed >> 32);
  for (int r = 0; r < 10; ++r) a.rk0[r] = a.k0 + (uint32_t)r * 0x9E3779B9u, a.rk1[r] = a.k1 + (uint32_t)r * 0xBB67AE85u;
  a.env_offset = (uint32_t)e->env_offset, a.active = e->active[t], a.rng_mode = e->rng_mode;
  a.done_flag = (int)t >= e->T;
  if (e->rng_mode == D2D_RNG_REPLAY) {
    D2D_REQUIRE(e->rp_arr && (int)t < e->rp_len, "%s: replay streams missing or shorter than timestep %u", who, t);
    const size_t nb = (size_t)e->N * e->B;
    a.rp_arr = e->rp_arr + (size_t)t * nb;
    a.rp_sw = reinterpret_cast<const uint8_t*>(e->rp_sw) + (size_t)t * e->chan_elems() * e->CB;
  }
  return D2D_OK;
}

// one_per_thread: ceil(B / 256) short blocks (the hardware block scheduler balances them better than a persistent
// grid-stride launch, whose ~3.5 envs per resident thread leave a 4-vs-3 iteration imbalance)
template <typename K>
static int launch_env(K kernel, const StepArgs& a, int params_bytes, void* stream, bool one_per_thread = false) {
  const int block = 256;
  kernel<<<grid_for(a.B, block, one_per_thread ? (1 << 20) : 8), block, params_bytes, as_stream(stream)>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_env_reset(d2d_env* e, float* obs, float* state, void* stream) {
  D2D_REQUIRE(e, "d2d_env_reset: null env");
  StepArgs a;
  e->episode += 1;
  int rc = fill_args(e, a, 0u, "d2d_env_reset");
  if (rc) {
    e->episode -= 1;
    return rc;
  }
  a.obs = obs, a.state = state;
  if (e->kind == D2D_ENV_COMBINATORIAL) {
#define D2D_RESET_CASE(WW, MT) rc = launch_env(comb_reset_kernel<WW, MT>, a, e->params_bytes, stream)
    if (e->W == 2 && e->CB == 1) D2D_RESET_CASE(2, uint8_t);
    else if (e->W == 2 && e->CB == 2) D2D_RESET_CASE(2, uint16_t);
    else if (e->W == 2) D2D_RESET_CASE(2, uint32_t);
    else if (e->W == 4 && e->CB == 1) D2D_RESET_CASE(4, uint8_t);
    else if (e->W == 4 && e->CB == 2) D2D_RESET_CASE(4, uint16_t);
    else if (e->W == 4) D2D_RESET_CASE(4, uint32_t);
    else if (e->CB == 1) D2D_RESET_CASE(8, uint8_t);
    else if (e->CB == 2) D2D_RESET_CASE(8, uint16_t);
    else D2D_RESET_CASE(8, uint32_t);
#undef D2D_RESET_CASE
  } else if (e->kind == D2D_ENV_SINGLE_CHANNEL) {
    rc = e->W == 2 ? launch_env(sc_reset_kernel<2>, a, e->params_bytes, stream)
         : e->W == 4 ? launch_env(sc_reset_kernel<4>, a, e->params_bytes, stream)
                     : launch_env(sc_reset_kernel<8>, a, e->params_bytes, stream);
  } else {
    rc = e->W == 2 ? launch_env(sel_reset_kernel<2>, a, e->params_bytes, stream)
         : e->W == 4 ? launch_env(sel_reset_kernel<4>, a, e->params_bytes, stream)
                     : launch_env(sel_reset_kernel<8>, a, e->params_bytes, stream);
  }
  if (rc) return rc;
  e->t = 0, e->is_reset = true;
  return D2D_OK;
}

static int env_step_impl(d2d_env* e, StepArgs& a, void* stream) {
  int rc;
  if (e->kind == D2D_ENV_COMBINATORIAL) {
    rc = e->W == 2 ? launch_comb_step<2>(a, e->N, e->C, e->CB, as_stream(stream))
         : e->W == 4 ? launch_comb_step<4>(a, e->N, e->C, e->CB, as_stream(stream))
                     : launch_comb_step<8>(a, e->N, e->C, e->CB, as_stream(stream));
  } else if (e->kind == D2D_ENV_SINGLE_CHANNEL) {
    if (e->N <= 4 && e->W == 2) rc = launch_env(sc_step_kernel<2, 4>, a, e->params_bytes, stream, true);
    else if (e->N <= 4 && e->W == 4) rc = launch_env(sc_step_kernel<4, 4>, a, e->params_bytes, stream, true);
    else
      rc = e->W == 2 ? launch_env(sc_step_kernel<2, 0>, a, e->params_bytes, stream, true)
           : e->W == 4 ? launch_env(sc_step_kernel<4, 0>, a, e->params_bytes, stream, true)
                       : launch_env(sc_step_kernel<8, 0>, a, e->params_bytes, stream, true);
  } else {
    rc = e->W == 2 ? launch_env(sel_step_kernel<2>, a, e->params_bytes, stream, true)
         : e->W == 4 ? launch_env(sel_step_kernel<4>, a, e->params_bytes, stream, true)
                     : launch_env(sel_step_kernel<8>, a, e->params_bytes, stream, true);
  }
  if (rc) return rc;
  e->t += 1;
  return D2D_OK;
}

extern "C" int d2d_env_step(d2d_env* e, const void* actions, float* obs, float* state, int32_t* reward,
                            uint8_t* done, void* ack, void* stream) {
  D2D_REQUIRE(e && actions && reward, "d2d_env_step: null env, actions or reward");
  if (!e->is_reset) {
    set_error("d2d_env_step: reset() has not been called");
    return D2D_ERR_STATE;
  }
  if (e->t >= e->T) {
    set_error("d2d_env_step: episode is over (timestep %d >= episode_length %d); call reset()", e->t, e->T);
    return D2D_ERR_STATE;
  }
  StepArgs a;
  int rc = fill_args(e, a, (uint32_t)(e->t + 1), "d2d_env_step");
  if (rc) return rc;
  a.actions = actions, a.obs = obs, a.state = state, a.reward = reward, a.done = done, a.ack = ack, a.act_mode = 0;
  return env_step_impl(e, a, stream);
}

extern "C" int d2d_env_step_random_access(d2d_env* e, double tp, void* actions_out, float* obs, float* state,
                                          int32_t* reward, uint8_t* done, void* ack, void* stream) {
  D2D_REQUIRE(e && reward, "d2d_env_step_random_access: null env or reward");
  D2D_REQUIRE(tp >= 0.0 && tp <= 1.0, "d2d_env_step_random_access: transmission_prob must be in [0, 1]");
  if (!e->is_reset) {
    set_error("d2d_env_step_random_access: reset() has not been called");
    return D2D_ERR_STATE;
  }
  if (e->t >= e->T) {
    set_error("d2d_env_step_random_access: episode is over (timestep %d >= %d); call reset()", e->t, e->T);
    return D2D_ERR_STATE;
  }
  StepArgs a;
  int rc = fill_args(e, a, (uint32_t)(e->t + 1), "d2d_env_step_random_access");
  if (rc) return rc;
  a.actions_out = actions_out, a.obs = obs, a.state = state, a.reward = reward, a.done = done, a.ack = ack;
  a.act_mode = 1;
  a.tp_thr = (uint32_t)std::min(65536.0, std::max(0.0, std::floor(tp * 65536.0 + 0.5)));
  return env_step_impl(e, a, stream);
}

// n_steps fused random-access steps enqueued back to back by the library: the inner loop of
// CombinatorialRandomAccess.run (algorithms/baselines.py:199-213) without a host round trip per step
extern "C" int d2d_env_run_random_access(d2d_env* e, double tp, int n_steps, int auto_reset, float* obs,
                                         int64_t obs_step_stride, float* state, int64_t state_step_stride,
                                         int32_t* reward, int64_t reward_step_stride, int reward_accumulate,
                                         uint8_t* done, void* stream, int* steps_done) {
  D2D_REQUIRE(e && reward && n_steps >= 0, "d2d_env_run_random_access: null env / reward or negative n_steps");
  D2D_REQUIRE(tp >= 0.0 && tp <= 1.0, "d2d_env_run_random_access: transmission_prob must be in [0, 1]");
  D2D_REQUIRE(!(reward_accumulate && reward_step_stride != 0),
              "d2d_env_run_random_access: reward_accumulate sums into ONE i32 [B] buffer (reward_step_stride 0)");
  if (steps_done) *steps_done = 0;
  if (!e->is_reset) {
    if (!auto_reset) {
      set_error("d2d_env_run_random_access: reset() has not been called");
      return D2D_ERR_STATE;
    }
  }
  const uint32_t tp_thr = (uint32_t)std::min(65536.0, std::max(0.0, std::floor(tp * 65536.0 + 0.5)));
  // the steps of one episode run inside ONE kernel with the env state in registers: the single-channel env with N <= 4
  // and no per-step observation rows (sc_run_kernel), the combinatorial env with N <= 8, C = 4 or 8 and the
  // one-thread-per-env mapping, observations at any stride or none (comb_run_kernel); never with state rows
  const bool philox = e->rng_mode == D2D_RNG_PHILOX && (e->W == 2 || e->W == 4) && !state &&
                      d2d_get_kernel_switch(D2D_SWITCH_ENV_MULTISTEP) == 1;
  const bool comb_multi = philox && e->kind == D2D_ENV_COMBINATORIAL && e->N <= 8 && (e->C == 4 || e->C == 8);
  const bool multi = comb_multi || (philox && e->kind == D2D_ENV_SINGLE_CHANNEL && e->N <= 4 && !obs);
  for (int i = 0; i < n_steps; ++i) {
    float* obs_i = obs ? obs + (size_t)i * obs_step_stride : nullptr;
    float* state_i = state ? state + (size_t)i * state_step_stride : nullptr;
    if (!e->is_reset || e->t >= e->T) {
      if (!auto_reset) break;               // episode over: the caller resets (as the reference's loop does)
      // the reset's observation goes to the slot of the step that follows and is overwritten by it
      int rc = d2d_env_reset(e, obs_i ? obs_i : nullptr, state_i, stream);
      if (rc) return rc;
    }
    if (multi) {
      const int n_inner = std::min(n_steps - i, e->T - e->t);
      StepArgs a;
      int rc = fill_args(e, a, (uint32_t)(e->t + 1), "d2d_env_run_random_access");
      if (rc) return rc;
      a.reward = reward + (size_t)i * reward_step_stride, a.done = done;
      a.act_mode = 1, a.tp_thr = tp_thr, a.reward_accum = reward_accumulate ? 1 : 0;
      a.done_flag = e->t + n_inner >= e->T;
      RunArgs ra;
      ra.active = e->active_dev, ra.t_plain = e->t + 1, ra.n_inner = n_inner, ra.reward_stride = reward_step_stride;
      ra.obs_stride = obs_step_stride;
      if (comb_multi) {
        a.obs = obs_i;
        rc = e->W == 2 ? launch_comb_run<2>(a, ra, e->C, as_stream(stream))
                       : launch_comb_run<4>(a, ra, e->C, as_stream(stream));
        if (rc) return rc;
      } else if (e->B <= kRunLanesMaxEnvs) {
        // small batches: four lanes per env (sc_run_lanes_kernel), 64-thread blocks = 16 envs spread over the SMs
        const int block = 64, grid = (int)(((long long)e->B * 4 + block - 1) / block);
        if (e->W == 2) sc_run_lanes_kernel<2><<<grid, block, e->params_bytes, as_stream(stream)>>>(a, ra);
        else sc_run_lanes_kernel<4><<<grid, block, e->params_bytes, as_stream(stream)>>>(a, ra);
        D2D_LAUNCHED();
      } else {
        // few envs: 64-thread blocks spread the warps over the SMs (each warp is one dependent-issue chain)
        const int block = e->B >= 148 * 256 ? 256 : 64, grid = (e->B + block - 1) / block;
        if (e->W == 2) sc_run_kernel<2, 4><<<grid, block, e->params_bytes, as_stream(stream)>>>(a, ra);
        else sc_run_kernel<4, 4><<<grid, block, e->params_bytes, as_stream(stream)>>>(a, ra);
        D2D_LAUNCHED();
      }
      e->t += n_inner;
      i += n_inner - 1;
      if (steps_done) *steps_done = i + 1;
      continue;
    }
    StepArgs a;
    int rc = fill_args(e, a, (uint32_t)(e->t + 1), "d2d_env_run_random_access");
    if (rc) return rc;
    a.obs = obs_i, a.state = state_i, a.reward = reward + (size_t)i * reward_step_stride, a.done = done;
    a.act_mode = 1, a.tp_thr = tp_thr, a.reward_accum = reward_accumulate ? 1 : 0;
    if ((rc = env_step_impl(e, a, stream))) return rc;
    if (steps_done) *steps_done = i + 1;
  }
  return D2D_OK;
}

extern "C" int d2d_pack_actions(const uint8_t* src, void* dst, int B, int N, int C, void* stream) {
  D2D_REQUIRE(src && dst && B > 0 && N > 0 && C > 0 && C <= D2D_MAX_CHANNELS, "d2d_pack_actions: bad argument");
  const int block = 256, grid = grid_for((long long)B * N, block);
  if (C <= 8) pack_actions_kernel<uint8_t><<<grid, block, 0, as_stream(stream)>>>(src, (uint8_t*)dst, B, N, C);
  else if (C <= 16) pack_actions_kernel<uint16_t><<<grid, block, 0, as_stream(stream)>>>(src, (uint16_t*)dst, B, N, C);
  else pack_actions_kernel<uint32_t><<<grid, block, 0, as_stream(stream)>>>(src, (uint32_t*)dst, B, N, C);
  D2D_LAUNCHED();
  return D2D_OK;
}

// ------------------------------------------------------------------------------------------------
// host-buffer step: the call a host-side caller of the reference's env.step(actions) makes
// ------------------------------------------------------------------------------------------------
static int pipe_create(d2d_env* e) {
  HostPipe* p = new (std::nothrow) HostPipe();
  D2D_REQUIRE(p, "d2d_env_step_host: out of host memory");
  e->pipe = p;
  const size_t nb = (size_t)e->N * e->B;
  p->stage_bytes = e->kind == D2D_ENV_COMBINATORIAL ? nb * e->C : nb;
  D2D_CUDA(cudaStreamCreateWithFlags(&p->h2d, cudaStreamNonBlocking));
  D2D_CUDA(cudaStreamCreateWithFlags(&p->d2h, cudaStreamNonBlocking));
  for (int i = 0; i < HostPipe::kSlots; ++i) {
    D2D_CUDA(cudaMalloc((void**)&p->stage[i], p->stage_bytes));
    D2D_CUDA(cudaMalloc(&p->masks[i], nb * (e->kind == D2D_ENV_COMBINATORIAL ? e->CB : 1)));
    D2D_CUDA(cudaMalloc((void**)&p->reward[i], (size_t)e->B * 4));
    D2D_CUDA(cudaMalloc((void**)&p->done[i], (size_t)e->B));
    D2D_CUDA(cudaEventCreateWithFlags(&p->in_ready[i], cudaEventDisableTiming));
    D2D_CUDA(cudaEventCreateWithFlags(&p->step_done[i], cudaEventDisableTiming));
    D2D_CUDA(cudaEventCreateWithFlags(&p->out_done[i], cudaEventDisableTiming));
  }
  p->events = true;
  return D2D_OK;
}

extern "C" int d2d_env_step_host(d2d_env* e, const void* actions_host, int layout, float* obs, float* state,
                                 int32_t* reward_host, uint8_t* done_host, void* ack, void* stream,
                                 uint64_t* ticket) {
  D2D_REQUIRE(e && actions_host && reward_host, "d2d_env_step_host: null env, actions or reward");
  D2D_REQUIRE(layout == D2D_ACT_HOST_REFERENCE || layout == D2D_ACT_HOST_DEVICE_LAYOUT,
              "d2d_env_step_host: unknown action layout %d", layout);
  if (!e->is_reset) {
    set_error("d2d_env_step_host: reset() has not been called");
    return D2D_ERR_STATE;
  }
  if (e->t >= e->T) {
    set_error("d2d_env_step_host: episode is over (timestep %d >= episode_length %d); call reset()", e->t, e->T);
    return D2D_ERR_STATE;
  }
  int rc;
  if (!e->pipe && (rc = pipe_create(e))) return rc;
  HostPipe* p = e->pipe;
  const int slot = (int)(p->calls % HostPipe::kSlots);
  const bool reused = p->calls >= HostPipe::kSlots;
  const size_t nb = (size_t)e->N * e->B;
  const bool comb = e->kind == D2D_ENV_COMBINATORIAL;
  D2D_REQUIRE(comb || layout == D2D_ACT_HOST_DEVICE_LAYOUT,
              "d2d_env_step_host: D2D_ACT_HOST_REFERENCE is defined for the combinatorial env only");
  bool need_pack = comb && layout == D2D_ACT_HOST_REFERENCE;
  cudaStream_t s = as_stream(stream);
  // 0. reference layout with enough host threads: pack u8 [B][N][C] to the [N][B] bitmasks ON THE HOST (host_pack.cpp),
  //    so that 1/C of the bytes cross PCIe.  The call blocks for the packing; the copy and the step stay asynchronous,
  //    so the host packs call k + 1 while the device runs call k.
  const void* src_host = actions_host;
  if (need_pack && d2d_get_kernel_switch(D2D_SWITCH_HOST_PACK) == 1 && d2d::host_threads() >= kHostPackMinThreads &&
      d2d::host_pack_is_fast(e->C, e->CB) && p->host_pack_state != 0) {
    if (!p->hpacked[slot]) D2D_CUDA(cudaHostAlloc((void**)&p->hpacked[slot], nb * e->CB, cudaHostAllocDefault));
    if (reused) D2D_CUDA(cudaEventSynchronize(p->in_ready[slot]));   // the copy of call k - 2 has left this buffer
    const auto t0 = std::chrono::steady_clock::now();
    d2d::host_pack_actions(reinterpret_cast<const uint8_t*>(actions_host), p->hpacked[slot], e->B, e->N, e->C, e->CB);
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    src_host = p->hpacked[slot];
    need_pack = false;
    p->host_pack_state = 1;
    // calls 2 .. 9 are timed (the first two fault the buffers in): slower on average than the unpacked bytes at
    // 40 GB/s of PCIe -> the following calls copy them as they are and pack on the device
    if (p->calls >= 2 && p->pack_samples < kHostPackSamples) {
      p->pack_ms_sum += ms;
      if (++p->pack_samples == kHostPackSamples &&
          p->pack_ms_sum / kHostPackSamples > (double)(nb * e->C) / 40.0e6)
        p->host_pack_state = 0;
    }
  }
  // 1. host -> device on the copy-in stream, once the step of call k - 2 has consumed this slot.  The copy is NOT
  //    ordered after the caller's stream (that would serialise it behind the previous call's step and lose the
  //    copy / compute overlap): actions_host must be complete on the host when the call is made (d2d_b200.h)
  if (reused) D2D_CUDA(cudaStreamWaitEvent(p->h2d, p->step_done[slot], 0));
  void* dst = need_pack ? (void*)p->stage[slot] : p->masks[slot];
  const size_t bytes = need_pack ? nb * e->C : nb * (comb ? e->CB : 1);
  D2D_CUDA(cudaMemcpyAsync(dst, src_host, bytes, cudaMemcpyHostToDevice, p->h2d));
  D2D_CUDA(cudaEventRecord(p->in_ready[slot], p->h2d));
  // 2. pack + step on the caller's stream
  D2D_CUDA(cudaStreamWaitEvent(s, p->in_ready[slot], 0));
  if (reused) D2D_CUDA(cudaStreamWaitEvent(s, p->out_done[slot], 0));
  if (need_pack && (rc = d2d_pack_actions(p->stage[slot], p->masks[slot], e->B, e->N, e->C, stream))) return rc;
  StepArgs a;
  if ((rc = fill_args(e, a, (uint32_t)(e->t + 1), "d2d_env_step_host"))) return rc;
  a.actions = p->masks[slot], a.obs = obs, a.state = state, a.reward = p->reward[slot], a.done = p->done[slot];
  a.ack = ack, a.act_mode = 0;
  if ((rc = env_step_impl(e, a, stream))) return rc;
  D2D_CUDA(cudaEventRecord(p->step_done[slot], s));
  // 3. device -> host on the copy-out stream
  D2D_CUDA(cudaStreamWaitEvent(p->d2h, p->step_done[slot], 0));
  D2D_CUDA(cudaMemcpyAsync(reward_host, p->reward[slot], (size_t)e->B * 4, cudaMemcpyDeviceToHost, p->d2h));
  if (done_host) D2D_CUDA(cudaMemcpyAsync(done_host, p->done[slot], (size_t)e->B, cudaMemcpyDeviceToHost, p->d2h));
  D2D_CUDA(cudaEventRecord(p->out_done[slot], p->d2h));
  if (ticket) *ticket = p->calls;
  p->calls += 1;
  return D2D_OK;
}

extern "C" int d2d_env_host_pack_state(const d2d_env* e) {
  return (e && e->pipe) ? e->pipe->host_pack_state : -1;
}

extern "C" int d2d_env_host_wait(d2d_env* e, uint64_t ticket) {
  D2D_REQUIRE(e && e->pipe, "d2d_env_host_wait: no host-buffer step has been issued on this env");
  HostPipe* p = e->pipe;
  D2D_REQUIRE(ticket < p->calls, "d2d_env_host_wait: ticket %llu has not been issued", (unsigned long long)ticket);
  // a slot's event is re-recorded by call ticket + kSlots, whose copy-out is stream-ordered after this one's:
  // waiting on the newest record of the slot therefore always covers `ticket`
  D2D_CUDA(cudaEventSynchronize(p->out_done[ticket % HostPipe::kSlots]));
  return D2D_OK;
}

extern "C" int d2d_env_export_state(const d2d_env* e, uint8_t* buffers, void* channel, uint32_t* discarded,
                                    uint32_t* received, uint32_t* stats, void* stream) {
  D2D_REQUIRE(e, "d2d_env_export_state: null env");
  const size_t nb = (size_t)e->N * e->B;
  cudaStream_t s = as_stream(stream);
  if (buffers) D2D_CUDA(cudaMemcpyAsync(buffers, e->buf, nb * e->W * 4, cudaMemcpyDeviceToDevice, s));
  if (channel) D2D_CUDA(cudaMemcpyAsync(channel, e->chan, e->chan_elems() * e->CB, cudaMemcpyDeviceToDevice, s));
  if (discarded) D2D_CUDA(cudaMemcpyAsync(discarded, e->disc, nb * 4, cudaMemcpyDeviceToDevice, s));
  if (received) D2D_CUDA(cudaMemcpyAsync(received, e->recv, nb * 4, cudaMemcpyDeviceToDevice, s));
  if (stats) D2D_CUDA(cudaMemcpyAsync(stats, e->stats, (size_t)2 * e->B * 4, cudaMemcpyDeviceToDevice, s));
  return D2D_OK;
}

extern "C" int d2d_env_import_state(d2d_env* e, const uint8_t* buffers, const void* channel,
                                    const uint32_t* discarded, const uint32_t* received, const uint32_t* stats,
                                    int timestep, void* stream) {
  D2D_REQUIRE(e, "d2d_env_import_state: null env");
  D2D_REQUIRE(timestep >= 0 && timestep <= e->T, "d2d_env_import_state: timestep out of range");
  const size_t nb = (size_t)e->N * e->B;
  cudaStream_t s = as_stream(stream);
  if (buffers) D2D_CUDA(cudaMemcpyAsync(e->buf, buffers, nb * e->W * 4, cudaMemcpyDeviceToDevice, s));
  if (channel) D2D_CUDA(cudaMemcpyAsync(e->chan, channel, e->chan_elems() * e->CB, cudaMemcpyDeviceToDevice, s));
  if (discarded) D2D_CUDA(cudaMemcpyAsync(e->disc, discarded, nb * 4, cudaMemcpyDeviceToDevice, s));
  if (received) D2D_CUDA(cudaMemcpyAsync(e->recv, received, nb * 4, cudaMemcpyDeviceToDevice, s));
  if (stats) D2D_CUDA(cudaMemcpyAsync(e->stats, stats, (size_t)2 * e->B * 4, cudaMemcpyDeviceToDevice, s));
  e->t = timestep, e->is_reset = true;
  return D2D_OK;
}

// EarliestDeadlineFirstScheduler.act (algorithms/baselines.py:55-76) for every env: the one device whose oldest packet
// is closest to its deadline transmits (ties: the first such device, as numpy's argmin); a uniformly drawn device when
// no buffer holds a packet.  use_channel: devices whose channel is bad are skipped (:91-94).  One thread per env.
__global__ void edf_policy_kernel(const uint32_t* __restrict__ buf, const uint8_t* __restrict__ chan, int N, int B,
                                  int W, int use_channel, uint8_t* __restrict__ actions, uint32_t k0, uint32_t k1,
                                  uint32_t env_offset, uint32_t t, uint32_t episode) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    int best = -1, best_d = 1 << 30;
    for (int i = 0; i < N; ++i) {
      if (use_channel && !(chan[(size_t)i * B + b] & 1)) continue;
      const uint32_t* rec = buf + ((size_t)i * B + b) * W;
      int d = -1;
      for (int w = 0; w < W && d < 0; ++w) {
        const uint32_t v = rec[w];
        if (v) d = 4 * w + ((__ffs(v) - 1) >> 3);        // first non-zero byte = packets with the fewest slots left
      }
      if (d >= 0 && d < best_d) best_d = d, best = i;
    }
    if (best < 0) {
      const uint4 r = philox4x32_10(env_offset + (uint32_t)b, t, kPurposePolicy << 16, episode, k0, k1);
      best = (int)(((unsigned long long)r.x * (unsigned long long)N) >> 32);
    }
    for (int i = 0; i < N; ++i) actions[(size_t)i * B + b] = (uint8_t)(i == best);
  }
}

extern "C" int d2d_env_policy_edf(const d2d_env* e, int use_channel, uint8_t* actions, void* stream) {
  D2D_REQUIRE(e && actions, "d2d_env_policy_edf: null argument");
  D2D_REQUIRE(e->kind == D2D_ENV_SINGLE_CHANNEL, "d2d_env_policy_edf: the scheduler grants the one shared channel of D2DEnv");
  D2D_REQUIRE(e->is_reset, "d2d_env_policy_edf: call reset first");
  edf_policy_kernel<<<grid_for(e->B, 128), 128, 0, as_stream(stream)>>>(
      e->buf, reinterpret_cast<const uint8_t*>(e->chan), e->N, e->B, e->W, use_channel != 0, actions,
      (uint32_t)(e->seed & 0xFFFFFFFFull), (uint32_t)(e->seed >> 32), (uint32_t)e->env_offset, (uint32_t)e->t,
      (uint32_t)e->episode);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_env_scores(const d2d_env* e, double* urllc, double* jains, double* channel_score, void* stream) {
  D2D_REQUIRE(e, "d2d_env_scores: null env");
  const int block = 256;
  scores_kernel<<<grid_for(e->B, block), block, 0, as_stream(stream)>>>(e->disc, e->recv, e->stats, e->kind, e->B,
                                                                         e->N, urllc, jains, channel_score);
  D2D_LAUNCHED();
  return D2D_OK;
}
