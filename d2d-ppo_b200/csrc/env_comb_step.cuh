// CombinatorialEnv.step (envs/combinatorial_env.py:127-242) for B lockstep envs: kernel + launcher template.
#pragma once
#include "env_common.cuh"

namespace d2d {

// W: words per buffer record; MaskT: channel-mask element; CFIX: compile-time channel count (0 = runtime);
// PACK: the N attempt masks fit one 64-bit register (N * 8 * sizeof(MaskT) <= 64), else a local array.
// MODE bit 0: replayed random streams (parity) instead of Philox; bit 1: fused random-access policy instead of
// actions from memory.  Compile-time so that the Philox kernel carries no predicated-off replay loads (they
// shared scoreboard slots with the prefetch loads and exposed a DRAM latency per device).
// G: device groups per env.  G = 1: one thread per env (the flagship shape: N = 6 devices, >= 1M envs).  G = 8: a block is
// 32 envs x 8 groups, warp g serves devices [g NG, (g + 1) NG) of the block's 32 envs (lanes stay consecutive envs, so
// every access is still a coalesced row) and the per-channel (once, twice, good) masks and the success count are
// combined across the 8 warps through shared memory.  For many devices per env (xp_n_agents.py sweep, N = 64) the
// one-thread-per-env mapping leaves 65,536 threads with 64-device serial loops: 20 % occupancy, 0.43 of HBM.
constexpr int kCombGroups = 8;
template <int W, typename MaskT, int CFIX, bool PACK, int MODE, int G = 1>
__global__ void __launch_bounds__(256, 4) comb_step_kernel(const StepArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  constexpr bool REPLAY = (MODE & 1) != 0, RA = (MODE & 2) != 0;
  const EnvParamsHdr* P = stage_params(a, smem);
  const uint32_t* cdf = reinterpret_cast<const uint32_t*>(smem + P->off_cdf);
  const uint32_t* swlt = reinterpret_cast<const uint32_t*>(smem + P->off_sw);
  const int N = P->N;
  const int C = CFIX ? CFIX : P->C;
  const size_t B = (size_t)a.B;
  const uint32_t Bu = (uint32_t)a.B;
  constexpr int MBITS = 8 * (int)sizeof(MaskT);
  MaskT* chan = reinterpret_cast<MaskT*>(a.chan);
  const MaskT* act = reinterpret_cast<const MaskT*>(a.actions);
  MaskT* act_out = reinterpret_cast<MaskT*>(a.actions_out);
  const MaskT* rp_sw = reinterpret_cast<const MaskT*>(a.rp_sw);
  const uint32_t cmask = C >= 32 ? 0xFFFFFFFFu : ((1u << C) - 1u);
  __shared__ uint32_t s_comb[G > 1 ? 4 : 1][G > 1 ? G : 1][32];   // once, twice, good_any, n_success per (group, lane)
  const int grp = G > 1 ? (int)(threadIdx.x >> 5) : 0;
  const int NG = G > 1 ? (((N + G - 1) / G + 3) & ~3) : N;         // devices per group, a multiple of 4 (Philox arrival
                                                                   // calls are shared by 4 consecutive devices)
  const int k_lo = G > 1 ? min(N, grp * NG) : 0, k_hi = G > 1 ? min(N, k_lo + NG) : N;
  const int b_first = G > 1 ? (int)(blockIdx.x * 32 + (threadIdx.x & 31)) : (int)(blockIdx.x * blockDim.x + threadIdx.x);
  const int b_step = G > 1 ? a.B : (int)(gridDim.x * blockDim.x);  // G > 1: one env per thread row, B % 32 == 0

  for (int b = b_first; b < a.B; b += b_step) {
    const uint32_t env = a.env_offset + (uint32_t)b;
    uint64_t att_pack = 0;
    MaskT att_arr[PACK ? 1 : D2D_MAX_AGENTS];

    // ---- pass 1: who transmits where (combinatorial_env.py:135-148) ----
    // Loads are issued CH devices at a time before any use, so one DRAM latency is exposed per chunk.
    constexpr int CH = W <= 4 ? 6 : 3;
    uint32_t once = 0, twice = 0, good_any = 0;
    uint64_t slot0 = 0;  // bit k: device k has a packet in slot 0 (it may expire this step)
    for (int k0 = k_lo; k0 < k_hi; k0 += CH) {
      Rec<W> rr[CH];
      uint32_t cc[CH], ww[CH];
#pragma unroll
      for (int j = 0; j < CH; ++j) {
        const int k = min(k0 + j, N - 1);
        const size_t idx = (size_t)k * B + b;
        rr[j] = rec_load<W>(a.buf, idx);
        cc[j] = chan[idx];
        if constexpr (!RA) ww[j] = act[idx];
        else ww[j] = 0u;
      }
#pragma unroll
      for (int j = 0; j < CH; ++j) {
        const int k = k0 + j;
        if (k < k_hi) {
          uint32_t want = ww[j] & cmask;
          if constexpr (RA) {
            want = lanes16_below<CFIX>(a.key, env, a.t, (uint32_t)k | (kPurposePolicy << 16), C,
                                       [&a](int) { return a.tp_lt; }, a.tp_all) & cmask;
            if (act_out) act_out[(size_t)k * B + b] = (MaskT)want;
          }
          const uint32_t at = rec_any<W>(rr[j]) ? want : 0u;
          twice |= once & at;
          once |= at;
          good_any |= at & cc[j];
          slot0 |= (uint64_t)((rr[j].w[0] & 0xFFu) != 0) << (k - k_lo);
          if constexpr (PACK) att_pack |= (uint64_t)at << ((k - k_lo) * MBITS);
          else att_arr[k - k_lo] = (MaskT)at;
        }
      }
    }
    if constexpr (G > 1) {   // combine the groups' masks: (o1, t1) + (o2, t2) = (o1 | o2, t1 | t2 | (o1 & o2))
      const int lane = threadIdx.x & 31;
      s_comb[0][grp][lane] = once, s_comb[1][grp][lane] = twice, s_comb[2][grp][lane] = good_any;
      __syncthreads();
      once = twice = good_any = 0;
#pragma unroll
      for (int q = 0; q < G; ++q) {
        const uint32_t o2 = s_comb[0][q][lane];
        twice |= s_comb[1][q][lane] | (once & o2);
        once |= o2;
        good_any |= s_comb[2][q][lane];
      }
    }
    // ack/nack per channel (combinatorial_env.py:155-157): +1 iff exactly one user and its channel is good
    const uint32_t acked = once & ~twice & good_any;
    const uint32_t nacked = once & ~acked;

    // ---- pass 2: serve, age, switch, arrive, observe; device k+1's state is fetched while k is processed ----
    int n_success = 0;
    uint4 arr4 = make_uint4(0u, 0u, 0u, 0u);
    const int k_first = G > 1 ? min(k_lo, N - 1) : 0;
    const size_t first = (size_t)k_first * B + b;
    Rec<W> r_nx = rec_load<W>(a.buf, first);       // second touch of the record: L1 hit
    uint32_t ch_nx = chan[first];
    uint32_t disc_nx = (slot0 & 1ull) ? a.disc[first] : 0u;
    uint32_t recv_nx = ((a.active >> k_first) & 1ull) ? a.recv[first] : 0u;
#pragma unroll 1
    for (int k = k_lo; k < k_hi; ++k) {
      const size_t idx = (size_t)k * B + b;
      Rec<W> r = r_nx;
      const uint32_t ch = ch_nx, disc_v = disc_nx, recv_v = recv_nx;
      if (k + 1 < k_hi) {
        const size_t nx = idx + B;
        r_nx = rec_load<W>(a.buf, nx);
        ch_nx = chan[nx];
        if ((slot0 >> (k + 1 - k_lo)) & 1ull) disc_nx = a.disc[nx];
        if ((a.active >> (k + 1)) & 1ull) recv_nx = a.recv[nx];
      }
      uint32_t at;
      if constexpr (PACK) at = (uint32_t)(att_pack >> ((k - k_lo) * MBITS)) & (uint32_t)(MaskT)~(MaskT)0;
      else at = att_arr[k - k_lo];
      const bool success = (at & ch & acked) != 0;                // :160-161
      n_success += success;
      rec_pop_earliest<W>(r, success);                            // :164-170
      const uint32_t expired = rec_age<W>(r);                     // :173
      if (expired) a.disc[idx] = disc_v + expired;                // :174
      uint32_t sw;                                                // :175, :116-118
      if constexpr (REPLAY) {
        sw = rp_sw[idx];
      } else {
        const uint32_t* lt = swlt + k * P->sw_row;
        sw = lanes16_below<CFIX>(a.key, env, a.t, (uint32_t)k | (kPurposeSwitch << 16), C,
                                 [lt](int c) { return lt[c]; }, P->sw_all[k]);
      }
      const uint32_t ch_new = (ch ^ sw) & cmask;
      chan[idx] = (MaskT)ch_new;
      const int dl = P->deadline[k];
      if constexpr (!REPLAY) arrival_call(a, env, k, arr4);   // k_lo is a multiple of 4
      if ((a.active >> k) & 1ull) {                               // :178-196
        const uint32_t arrived = REPLAY ? a.rp_arr[idx]
                                        : arrival_count(word32(arr4, k), P->arrival_kind[k] == D2D_ARRIVAL_BERNOULLI,
                                                        P->bern_thr[k], cdf + k * D2D_POISSON_KMAX);
        rec_set_byte<W>(r, dl - 1, arrived);
        if (arrived) a.recv[idx] = recv_v + arrived;
      }
      rec_store<W>(a.buf, idx, r);
      if (a.obs) {                                                // :199-206
        float* o = a.obs + (size_t)P->obs_off[k] * B + b;
        o = emit_slots<W>(r, P->homog ? P->D : dl, o, Bu);
        o = emit_bits<CFIX>(ch, C, o, Bu);                        // pre-switch copy (:145)
        emit_ack<CFIX>(acked, nacked, C, o, Bu);
      }
      if (a.state) {                                              // :207-209
        emit_slots<W>(r, dl, a.state + (size_t)P->sbuf_off[k] * B + b, Bu);
        emit_bits<CFIX>(ch_new, C, a.state + ((size_t)P->sum_dl + (size_t)k * C) * B + b, Bu);
      }
    }
    if constexpr (G > 1) {   // the env's success count: sum over the groups; group 0 writes the per-env outputs
      const int lane = threadIdx.x & 31;
      s_comb[3][grp][lane] = (uint32_t)n_success;
      __syncthreads();
      if (grp != 0) continue;
      n_success = 0;
#pragma unroll
      for (int q = 0; q < G; ++q) n_success += (int)s_comb[3][q][lane];
    }
    if (a.state) emit_ack<CFIX>(acked, nacked, C, a.state + ((size_t)P->sum_dl + (size_t)N * C) * B + b, Bu);
    if (a.ack) {
      int8_t* q = reinterpret_cast<int8_t*>(a.ack) + b;
      for (int c = 0; c < C; ++c) q[(size_t)c * B] = (int8_t)((int)((acked >> c) & 1u) - (int)((nacked >> c) & 1u));
    }
    a.reward[b] = (a.reward_accum ? a.reward[b] : 0) + n_success;  // :211
    if (a.done) a.done[b] = (uint8_t)a.done_flag;                 // :233-236
  }
}


// MODE from the call: replayed streams and / or the fused policy.  The CFIX > 0 fast paths are Philox-only
// (launch_comb_step), so they instantiate modes 0 and 2 alone.
template <int W, typename MaskT, int CFIX, bool PACK>
int launch_comb_mode(const StepArgs& a, int grid, int block, cudaStream_t s) {
  const int mode = (a.rng_mode == D2D_RNG_REPLAY ? 1 : 0) | (a.act_mode != 0 ? 2 : 0);
  if (mode == 0) comb_step_kernel<W, MaskT, CFIX, PACK, 0><<<grid, block, a.params_bytes, s>>>(a);
  else if (mode == 2) comb_step_kernel<W, MaskT, CFIX, PACK, 2><<<grid, block, a.params_bytes, s>>>(a);
  else if constexpr (CFIX == 0) {
    if (mode == 1) comb_step_kernel<W, MaskT, CFIX, PACK, 1><<<grid, block, a.params_bytes, s>>>(a);
    else comb_step_kernel<W, MaskT, CFIX, PACK, 3><<<grid, block, a.params_bytes, s>>>(a);
  }
  D2D_LAUNCHED();
  return D2D_OK;
}

// many devices per env: 32 envs x 8 device groups per block (Philox modes only)
template <int W, int CFIX>
int launch_comb_grouped(const StepArgs& a, cudaStream_t s) {
  const int g = a.B / 32;
  if (a.act_mode == 0) comb_step_kernel<W, uint8_t, CFIX, true, 0, kCombGroups><<<g, 256, a.params_bytes, s>>>(a);
  else comb_step_kernel<W, uint8_t, CFIX, true, 2, kCombGroups><<<g, 256, a.params_bytes, s>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

// n_inner consecutive fused random-access steps of ONE episode in one launch, one thread per env (the run form of
// comb_step_kernel<W, uint8_t, C, true, 2>, as sc_run_kernel is of sc_step_kernel).  The env's N <= 8 records,
// channel masks and disc / recv counters are loaded once, live in registers for every step and are stored once, so a
// step moves no state through HBM: what it writes is the observation rows and the reward.  With the observations of
// every step written to the same block (obs_stride 0, CombinatorialRandomAccess.run / bench.py) those rows of the
// resident envs can stay in L2 (2 blocks of 256 per SM: 75,776 envs x 720 B = 55 MB of the 126 MB; one block per SM
// measured slower, DESIGN.md section 3).  Same Philox counters and update order as comb_step_kernel: bit-identical.
// A step is bound by the instructions each warp issues, so the step body is straight-line code:
//  - NF: the device count as a constant (no per-device guards or dead slots); 0 = any N <= 8 at run time;
//  - DH: every device's observation carries DH slots (homogeneous sizes, D = DH), which fixes the rows of each device
//    at compile time; 0 = the slot count and rows come from the tables at run time;
//  - the env tables are kernel parameters (CombRunParams: constant-bank operands, no staging, no LDS);
//  - each Philox call starts at round 2 from the thread's and the call's two-round heads (philox.cuh);
//  - the ack / nack floats are formed once per step and stored for every device;
//  - observation rows are plain stores, which ptxas may schedule among the Philox rounds (emit_slots_run).
template <int W, int C, int NF, int DH>
__global__ void __launch_bounds__(256, 2) comb_run_kernel(const StepArgs a, const RunArgs ra,
                                                          const __grid_constant__ CombRunParams p) {
  constexpr int NK = NF ? NF : kRunMaxN;
  constexpr uint32_t cmask = (1u << C) - 1u;
  const int N = NF ? NF : p.N;
  const size_t B = (size_t)a.B;
  const int Bi = a.B;
  uint8_t* chan = reinterpret_cast<uint8_t*>(a.chan);
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= a.B) return;
  const uint32_t env = a.env_offset + (uint32_t)b;
  Rec<W> rec[NK];
  uint32_t chv[NK], discv[NK], recvv[NK];
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    const size_t idx = (size_t)(NF ? k : min(k, N - 1)) * B + b;
    rec[k] = rec_load<W>(a.buf, idx);
    chv[k] = chan[idx], discv[k] = a.disc[idx], recvv[k] = a.recv[idx];
  }
  int32_t rew = a.reward_accum ? a.reward[b] : 0;
  const PhiloxEnvHead eh = philox_env_head(a.key, env, 0u);   // C <= 8 and arrivals: block 0 only
#pragma unroll 1
  for (int i = 0; i < ra.n_inner; ++i) {
    const uint32_t t = a.t + (uint32_t)i;
    const uint64_t active = ra.active[ra.t_plain + i];
    // ---- who transmits where (combinatorial_env.py:135-148); the draws do not depend on the state ----
    uint32_t once = 0, twice = 0, good_any = 0;
    uint64_t att_pack = 0;
#pragma unroll
    for (int k = 0; k < NK; ++k) {
      if (NF || k < N) {
        const uint4 r = philox(a.key, eh, philox_call_head(a.key, t, (uint32_t)k | (kPurposePolicy << 16)));
        const uint32_t want = lanes_below<C>(r, [&a](int) { return a.tp_lt; }, a.tp_all);
        const uint32_t at = rec_any<W>(rec[k]) ? (want & cmask) : 0u;
        twice |= once & at;
        once |= at;
        good_any |= at & chv[k];
        att_pack |= (uint64_t)at << (k * 8);
      }
    }
    const uint32_t acked = once & ~twice & good_any;          // :155-157
    const uint32_t nacked = once & ~acked;
    float* obs_i = a.obs ? a.obs + (size_t)i * (size_t)ra.obs_stride + b : nullptr;
    float ackf[C];
    if (obs_i) {
#pragma unroll
      for (int c = 0; c < C; ++c) ackf[c] = ((acked >> c) & 1u) ? 1.0f : (((nacked >> c) & 1u) ? -1.0f : 0.0f);
    }
    // ---- serve, age, switch, arrive, observe (:160-206) ----
    int n_success = 0;
    uint4 arr4 = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int k = 0; k < NK; ++k) {
      if (NF || k < N) {
        Rec<W>& r = rec[k];
        const uint32_t at = (uint32_t)(att_pack >> (k * 8)) & 0xFFu;
        const uint32_t ch = chv[k];
        const bool success = (at & ch & acked) != 0;
        n_success += success;
        rec_pop_earliest<W>(r, success);
        discv[k] += rec_age<W>(r);
        const uint4 rs = philox(a.key, eh, philox_call_head(a.key, t, (uint32_t)k | (kPurposeSwitch << 16)));
        const uint32_t sw = lanes_below<C>(rs, [&p, k](int c) { return p.sw_lt[k][c]; }, p.sw_all[k]);
        chv[k] = (ch ^ sw) & cmask;
        const int dl = p.deadline[k];
        // arrival_call's draw, from the heads
        if ((k & 3) == 0 && ((active >> k) & 0xFull))
          arr4 = philox(a.key, eh, philox_call_head(a.key, t, word32_field(k) | (kPurposeArrival << 16)));
        if ((active >> k) & 1ull) {
          const uint32_t arrived =
              arrival_count(word32(arr4, k), p.arrival_kind[k] == D2D_ARRIVAL_BERNOULLI, p.bern_thr[k], p.cdf[k]);
          rec_set_byte<W>(r, dl - 1, arrived);
          recvv[k] += arrived;
        }
        if (obs_i) {
          float* o = obs_i + (size_t)(DH ? k * (DH + 2 * C) : (int)p.obs_off[k]) * B;
          o = emit_slots_run<W, DH>(r, DH ? DH : (p.homog_slots ? p.homog_slots : dl), o, Bi);
#pragma unroll
          for (int c = 0; c < C; ++c, o += Bi) *o = ((ch >> c) & 1u) ? 1.0f : 0.0f;   // pre-switch copy (:145)
#pragma unroll
          for (int c = 0; c < C; ++c, o += Bi) *o = ackf[c];
        }
      }
    }
    if (a.reward_accum) rew += n_success;                     // :211
    else a.reward[(size_t)i * ra.reward_stride + b] = n_success;
  }
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    if (NF || k < N) {
      const size_t idx = (size_t)k * B + b;
      rec_store<W>(a.buf, idx, rec[k]);
      chan[idx] = (uint8_t)chv[k];
      a.disc[idx] = discv[k], a.recv[idx] = recvv[k];
    }
  }
  if (a.reward_accum) a.reward[b] = rew;
  if (a.done) a.done[b] = (uint8_t)a.done_flag;
}

// d2d_env_run_random_access's episode-in-one-launch path for the combinatorial env; C must be 4 or 8, N <= 8.
// Exact-N kernels for N = 4, 6, 8 with homogeneous observations of the record's usual deadline (7 for 8-byte records,
// 14 for 16-byte ones: setup_8_channels and c1-c5); every other shape runs the general kernel.
template <int W>
int launch_comb_run(const StepArgs& a, const RunArgs& ra, const CombRunParams& p, int C, cudaStream_t s) {
  const int block = 256, grid = (a.B + block - 1) / block;
  constexpr int DH = W == 4 ? 14 : 7;
  const int nf = p.homog_slots == DH && (p.N == 4 || p.N == 6 || p.N == 8) ? p.N : 0;
#define D2D_RUN(CC)                                                                              \
  switch (nf) {                                                                                  \
    case 4: comb_run_kernel<W, CC, 4, DH><<<grid, block, 0, s>>>(a, ra, p); break;               \
    case 6: comb_run_kernel<W, CC, 6, DH><<<grid, block, 0, s>>>(a, ra, p); break;               \
    case 8: comb_run_kernel<W, CC, 8, DH><<<grid, block, 0, s>>>(a, ra, p); break;               \
    default: comb_run_kernel<W, CC, 0, 0><<<grid, block, 0, s>>>(a, ra, p); break;               \
  }
  if (C == 8) D2D_RUN(8) else D2D_RUN(4)
#undef D2D_RUN
  D2D_LAUNCHED();
  return D2D_OK;
}

// one translation unit per record width (env_comb_w2.cu / _w4.cu / _w8.cu) so that nvcc compiles them in parallel
template <int W>
int launch_comb_step(const StepArgs& a, int N, int C, int mask_bytes, cudaStream_t s) {
  // one env per thread, ceil(B / 256) blocks: with ~3.5 envs per resident thread a persistent grid-stride launch
  // leaves a 4-vs-3 iteration imbalance (13%); the hardware block scheduler balances 4096 short blocks better.
  const int block = 256, grid = grid_for(a.B, block, 1 << 20);
  const bool pack = N * 8 * mask_bytes <= 64;
  // grouped mapping: when one thread per env cannot fill the GPU (few envs, many devices each)
  const int ng = ((N + kCombGroups - 1) / kCombGroups + 3) & ~3;
  if (a.rng_mode != D2D_RNG_REPLAY && N >= 32 && a.B % 32 == 0 && a.B < 148 * 1024 && ng * 8 * mask_bytes <= 64) {
    if (C == 4) return launch_comb_grouped<W, 4>(a, s);
    if (C == 8) return launch_comb_grouped<W, 8>(a, s);
  }
#define D2D_CASE(MT, CF) return pack ? launch_comb_mode<W, MT, CF, true>(a, grid, block, s) \
                                     : launch_comb_mode<W, MT, CF, false>(a, grid, block, s)
  if (a.rng_mode != D2D_RNG_REPLAY) {   // Philox fast paths with a compile-time channel count
    if (C == 8) D2D_CASE(uint8_t, 8);
    if (C == 4) D2D_CASE(uint8_t, 4);
    if (C == 16) D2D_CASE(uint16_t, 16);
  }
  if (mask_bytes == 1) D2D_CASE(uint8_t, 0);
  if (mask_bytes == 2) D2D_CASE(uint16_t, 0);
  D2D_CASE(uint32_t, 0);
#undef D2D_CASE
}

}  // namespace d2d
