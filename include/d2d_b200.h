/*
 * d2d_b200.h -- C ABI of the B200-native D2D-PPO hot path (libd2d_b200.so).
 *
 * The reference (benrobaglia/D2D-PPO) is pure Python and defines no FFI; its
 * boundary for this path is the Python env/agent API.  Each entry point below
 * names the reference function (file:line under /root/reference) whose work it
 * replaces.  The Python classes in d2d-ppo_b200/ keep the reference signatures
 * and call these through ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - extern "C", plain C types; no torch / C++ types cross the boundary.
 *   - every function returns int: 0 = ok, negative = D2D_ERR_*; the message is
 *     in d2d_last_error() (thread-local).  Nothing throws.
 *   - all data pointers are DEVICE pointers borrowed for the duration of the
 *     call (PyTorch owns them) unless a parameter is documented as "host".
 *   - calls are asynchronous on the given cudaStream_t (passed as void*); no
 *     hidden synchronisation.
 *   - a handle is not thread-safe; distinct handles are independent.
 *
 * Device layout ("env-minor" structure of arrays): every per-(env, device)
 * quantity is stored as X[row][env] with the env index fastest, so that a warp
 * of 32 consecutive envs reads/writes 32 consecutive elements.  B = n_envs.
 */
#ifndef D2D_B200_H
#define D2D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D2D_ABI_VERSION 1

#define D2D_OK 0
#define D2D_ERR_INVALID (-1)   /* bad argument / unsupported shape */
#define D2D_ERR_CUDA (-2)      /* a CUDA runtime call failed */
#define D2D_ERR_STATE (-3)     /* call sequence error (e.g. step before reset) */

/* env kinds */
#define D2D_ENV_COMBINATORIAL 0      /* envs/combinatorial_env.py:4  CombinatorialEnv    */
#define D2D_ENV_SINGLE_CHANNEL 1     /* envs/env.py:4                D2DEnv              */
#define D2D_ENV_CHANNEL_SELECTION 2  /* envs/channel_selection_env.py:4 ChannelSelectionEnv */

/* random streams */
#define D2D_RNG_PHILOX 0  /* counter-based Philox4x32-10 keyed by (seed, env, t, device) */
#define D2D_RNG_REPLAY 1  /* pre-drawn arrival / switch streams (parity with the reference) */

/* arrival distributions (combinatorial_env.py:180 poisson, :185/:195 binomial) */
#define D2D_ARRIVAL_POISSON 0
#define D2D_ARRIVAL_BERNOULLI 1

#define D2D_MAX_AGENTS 64
#define D2D_MAX_CHANNELS 32
#define D2D_MAX_DEADLINE 32
#define D2D_POISSON_KMAX 16

const char* d2d_last_error(void);
int d2d_abi_version(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
uint64_t d2d_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Environments.  Replaces CombinatorialEnv / D2DEnv / ChannelSelectionEnv __init__/reset/step.
 * All pointers in the config are HOST pointers, copied by d2d_env_create.
 * ------------------------------------------------------------------------------------------ */
typedef struct d2d_env_config {
  int32_t kind;              /* D2D_ENV_*                                                   */
  int32_t n_envs;            /* B lockstep env instances on this GPU                        */
  int32_t n_agents;          /* N <= D2D_MAX_AGENTS                                         */
  int32_t n_channels;        /* C (1 for D2D_ENV_SINGLE_CHANNEL); C+1 <= 32 for selection   */
  int32_t episode_length;    /* T: done = (timestep >= T)   combinatorial_env.py:233        */
  int32_t homogeneous_size;  /* combinatorial_env.py:47-53: pad buffer obs to max deadline  */
  int32_t rng_mode;          /* D2D_RNG_*                                                   */
  int32_t reserved0;
  uint64_t seed;             /* Philox key                                                  */
  uint64_t env_offset;       /* global index of local env 0 (multi-GPU sharding)            */
  const int32_t* deadlines;        /* [N], each in 1..D2D_MAX_DEADLINE                      */
  const int32_t* arrival_kind;     /* [N] D2D_ARRIVAL_*                                     */
  const uint64_t* arrival_active;  /* [T+1] bit k: device k draws an arrival at timestep t
                                      (t = 0 is reset); encodes traffic_model / period / offsets */
  const uint32_t* poisson_cdf;     /* [N][D2D_POISSON_KMAX]: floor(CDF(m) 2^32), clamped    */
  const uint64_t* bernoulli_thr;   /* [N]: round(arrival_prob 2^32) in 0..2^32              */
  const uint32_t* switch_thr;      /* round(p 65536) in 0..65536; combinatorial [N][C],
                                      single-channel [N], selection [C+1]                   */
  const int32_t* nbr_offset;       /* single-channel only: CSR neighbourhoods, [N+1]; NULL = self */
  const int32_t* nbr_index;        /* single-channel only: [nbr_offset[N]]                  */
} d2d_env_config;

typedef struct d2d_env d2d_env;

int d2d_env_create(const d2d_env_config* cfg, d2d_env** out);
int d2d_env_destroy(d2d_env* env);

/* layout queries (rows of the env-minor obs / state matrices) */
int d2d_env_obs_rows(const d2d_env* env);               /* sum_k obs_dim[k]                 */
int d2d_env_obs_offset(const d2d_env* env, int agent);  /* first row of device k            */
int d2d_env_obs_dim(const d2d_env* env, int agent);     /* observation_space[k].shape[0]    */
int d2d_env_state_rows(const d2d_env* env);             /* state_space.shape[0]             */
int d2d_env_timestep(const d2d_env* env);

/* Episode index of the Philox streams.  The reference draws fresh traffic in every episode from numpy's global
 * generator (combinatorial_env.py:68,117,180); here every reset() starts episode e = (number of resets - 1) and the
 * Philox counter's timestep field is t + e * (episode_length + 1), so consecutive episodes of an env are
 * independent.  d2d_env_set_episode makes the NEXT reset() start episode `next_episode` (checkpoint / resume,
 * reproducing a given episode); d2d_env_episode returns the current one (-1 before the first reset). */
int64_t d2d_env_episode(const d2d_env* env);
int d2d_env_set_episode(d2d_env* env, int64_t next_episode);

/* Replay streams (device, borrowed until the next set_replay/destroy):
 *   arrivals  u8 [t_len][N][B]           value device k would draw at timestep t (0 = reset)
 *   switches  combinatorial: mask [t_len][N][B], element = 1/2/4 bytes for C <= 8/16/32, bit c = flip
 *             single-channel: u8 [t_len][N][B] (bit 0); selection: u32 [t_len][B] (bit c, c = 0..C)
 *   index 0 of `switches` is unused (reset draws no switch).                                  */
int d2d_env_set_replay(d2d_env* env, const uint8_t* arrivals, const void* switches, int t_len);

/* reset(): combinatorial_env.py:61-114, env.py:51-101, channel_selection_env.py:49-98.
 *   obs   f32 [obs_rows][B]   (required)
 *   state f32 [state_rows][B] (may be NULL)                                                   */
int d2d_env_reset(d2d_env* env, float* obs, float* state, void* stream);

/* step(actions): combinatorial_env.py:127-242, env.py:118-217, channel_selection_env.py:116-214.
 *   actions  combinatorial: channel bitmask [N][B] (1/2/4 bytes per element, bit c = transmit on c)
 *            single-channel: u8 [N][B] 0/1;  selection: u8 [N][B] channel id 0..C (0 = idle)
 *   obs      f32 [obs_rows][B]       next observations (may be NULL: not emitted)
 *   state    f32 [state_rows][B]     next global state (may be NULL)
 *   reward   i32 [B]   combinatorial/selection: number of successful devices; single-channel: ack
 *   done     u8  [B]   (may be NULL)
 *   ack      combinatorial: i8 [C][B]; single-channel: NULL; selection: f32 [C+1][B] (may be NULL)  */
int d2d_env_step(d2d_env* env, const void* actions, float* obs, float* state, int32_t* reward,
                 uint8_t* done, void* ack, void* stream);

/* step with the fused random-access policy: the actions come from the Philox policy stream inside the step kernel.
 *   combinatorial / single-channel: algorithms/baselines.py:181-183 (CombinatorialRandomAccess.act = Bernoulli(tp)
 *                     per (device, channel) resp. per device)
 *   selection:        algorithms/baselines.py:10-14 (RandomAccess.act: every device with a packet picks a channel id
 *                     uniformly from 0..C, 0 = stay idle); transmission_prob is ignored
 * actions_out (same layout as `actions`) may be NULL. */
int d2d_env_step_random_access(d2d_env* env, double transmission_prob, void* actions_out, float* obs,
                               float* state, int32_t* reward, uint8_t* done, void* ack, void* stream);

/* n_steps steps of d2d_env_step_random_access enqueued back to back by the library: the inner loop of
 * CombinatorialRandomAccess.run (algorithms/baselines.py:199-213) without one host call per step (at 8 ranks the
 * per-step Python -> C launch path, not the GPU, bounded short runs).
 *   auto_reset        1: an env that is not reset, or whose episode is over, is reset before the next step (the
 *                     reset's observation lands in that step's obs slot and is overwritten by the step);
 *                     0: the run stops at the end of the episode, as the reference's `while not done` loop
 *   obs / state       f32 [..][obs_rows][B] / [..][state_rows][B]: step i writes at + i * *_step_stride floats
 *                     (stride 0: every step overwrites the same block); NULL: not emitted
 *   reward            i32: step i writes reward + i * reward_step_stride ([B] each); with reward_accumulate = 1
 *                     (stride 0) every step ADDS its reward into the one [B] buffer (zero it first): the
 *                     per-episode reward sum of baselines.py:211
 *   done              u8 [B] of the last step (may be NULL);  *steps_done (may be NULL): steps actually run
 * With Philox streams and state == NULL the steps of an episode run in ONE launch with the env state in registers,
 * bit-identical to the per-step launches (D2D_SWITCH_ENV_MULTISTEP = 0 restores them): the single-channel env with
 * N <= 4 and obs == NULL (rewards only, RandomAccess.run; sc_run_kernel), and the combinatorial env with N <= 8 and
 * C = 4 or 8, observations at any stride or NULL (CombinatorialRandomAccess.run; comb_run_kernel).  Everything else
 * (replayed streams, state rows, C = 16, N > 8) runs one step kernel per step.  Resets stay launches of their own. */
int d2d_env_run_random_access(d2d_env* env, double transmission_prob, int n_steps, int auto_reset, float* obs,
                              int64_t obs_step_stride, float* state, int64_t state_step_stride, int32_t* reward,
                              int64_t reward_step_stride, int reward_accumulate, uint8_t* done, void* stream,
                              int* steps_done);

/* pack reference-layout actions u8 [B][N][C] (0/1) into the bitmask layout above */
int d2d_pack_actions(const uint8_t* actions_bnc, void* packed, int n_envs, int n_agents, int n_channels,
                     void* stream);

/* step(actions) with HOST buffers: what a host-side caller of the reference's env.step(actions)
 * (combinatorial_env.py:127) hands over and gets back, with the host<->device copies done by the library.
 *   actions_host  D2D_ACT_HOST_REFERENCE (combinatorial only): u8 [B][N][C] 0/1, the reference's (N, C) action
 *                 array of every env back to back;  D2D_ACT_HOST_DEVICE_LAYOUT: the `actions` layout of
 *                 d2d_env_step ([N][B] masks / flags / channel ids).  Pinned memory for asynchronous copies.
 *   reward_host   i32 [B] (required), done_host u8 [B] (may be NULL): pinned host memory
 *   obs / state / ack: DEVICE pointers as in d2d_env_step (may be NULL)
 * The call is asynchronous and pipelined: the H2D copy runs on the handle's copy-in stream, pack + step on
 * `stream`, the D2H copy on the copy-out stream, so consecutive calls overlap.  Up to two calls are in flight;
 * actions_host must be COMPLETE ON THE HOST when the call is made (the copy-in stream is deliberately not ordered
 * after `stream`: a caller that fills actions_host with asynchronous work must synchronise that work first) and
 * must stay untouched until the call's step ran (d2d_env_host_wait of the same ticket suffices).
 * *ticket (may be NULL) identifies the call; d2d_env_host_wait(env, ticket) blocks the host thread until
 * reward_host / done_host of that call are valid.
 * With D2D_ACT_HOST_REFERENCE, 8 channels, an AVX2 host and at least 12 host threads (d2d_get_host_threads) the library
 * packs the [B][N][C] bytes into the [N][B] channel bitmasks ON THE HOST (thread pool) and copies 1/8 of the bytes; the
 * call then blocks for the packing (actions_host may be reused as soon as it returns), the copy and the step stay
 * asynchronous. */
#define D2D_ACT_HOST_REFERENCE 0
#define D2D_ACT_HOST_DEVICE_LAYOUT 1
int d2d_env_step_host(d2d_env* env, const void* actions_host, int layout, float* obs, float* state,
                      int32_t* reward_host, uint8_t* done_host, void* ack, void* stream, uint64_t* ticket);
int d2d_env_host_wait(d2d_env* env, uint64_t ticket);
/* Host-side packing of this env's host-buffer steps: -1 not used (so far), 1 active, 0 switched off -- calls 2 .. 9 are
 * timed, and a host that packs slower than 40 GB/s of PCIe would move the unpacked bytes keeps the unpacked copy. */
int d2d_env_host_pack_state(const d2d_env* env);

/* Host-side helpers of the host-buffer step (csrc/host_pack.cpp, no CUDA involved).
 * d2d_set_host_threads(n): size of the library's host thread pool (0 = default: the CPUs of the process's affinity
 * mask, at most 16); d2d_pack_actions_host: d2d_pack_actions on HOST pointers (u8 [B][N][C] -> bitmasks [N][B]). */
int d2d_set_host_threads(int n);
int d2d_get_host_threads(void);
int d2d_pack_actions_host(const uint8_t* actions_bnc, void* packed, int n_envs, int n_agents, int n_channels);

/* Counters and raw state, env-minor: buffers u8 [N][Dmax][B]... exported as
 *   buffers  u8  [N][B][rec]   rec = d2d_env_record_bytes() (8/16/32), byte d = packets with d slots left
 *   channel  combinatorial: mask [N][B]; single-channel u8 [N][B]; selection u32 [B]
 *   discarded / received  u32 [N][B]     (combinatorial_env.py:91-92,174,181)
 *   stats    u32 [2][B]   single-channel: channel_errors, n_collisions (env.py:147,150);
 *                         selection: selected_channel_qualities, number_selected_channel (:132-133)
 * Any pointer may be NULL.  import is the inverse (used by tests to force a state). */
int d2d_env_record_bytes(const d2d_env* env);
int d2d_env_mask_bytes(const d2d_env* env);
int d2d_env_export_state(const d2d_env* env, uint8_t* buffers, void* channel, uint32_t* discarded,
                         uint32_t* received, uint32_t* stats, void* stream);
int d2d_env_import_state(d2d_env* env, const uint8_t* buffers, const void* channel, const uint32_t* discarded,
                         const uint32_t* received, const uint32_t* stats, int timestep, void* stream);

/* compute_urllc / compute_jains / compute_channel_score per env
 * (combinatorial_env.py:245-264): f64 [B] each, any may be NULL. */
int d2d_env_scores(const d2d_env* env, double* urllc, double* jains, double* channel_score, void* stream);

/* EarliestDeadlineFirstScheduler.act (algorithms/baselines.py:55-76) on the env's current buffers, all B envs: actions
 * u8 [N][B] one-hot over the devices -- the device whose oldest packet is closest to expiry (first one on ties), a
 * uniformly drawn device (Philox policy stream) when no buffer holds a packet.  use_channel = 1 skips devices whose
 * channel is bad (:91-94).  D2DEnv (D2D_ENV_SINGLE_CHANNEL) only: the scheduler grants its one shared channel. */
int d2d_env_policy_edf(const d2d_env* env, int use_channel, uint8_t* actions, void* stream);


/* ------------------------------------------------------------------------------------------
 * Learner: the per-agent actor / critic networks of algorithms/d2d_ppo.py and algorithms/ippo.py, evaluated
 * for all N agents in one launch.  All matrices are env-minor f32: M[time block][feature row][env].
 *
 * A "net set" is N independent networks of one architecture (the reference builds one PPO object per agent,
 * d2d_ppo.py:252-262, ippo.py:254-264); the D2DPPO central critic (d2d_ppo.py:265) is a net set with N = 1.
 * Parameters live in ONE caller-owned f32 buffer [N][param_stride]; inside an agent's block the tensors are
 * stored contiguously in the reference's state_dict order, row-major as torch stores them:
 *   GRU ("RNN", d2d_ppo.py:24-59):  lstm.weight_ih_l0 [3H, I], lstm.weight_hh_l0 [3H, H], lstm.bias_ih_l0 [3H],
 *                                   lstm.bias_hh_l0 [3H], layers.0.weight [H, H], layers.0.bias [H],
 *                                   layers.2.weight [O, H], layers.2.bias [O]
 *   GRU Q-network (irdqn.py:58-72, head_layers = 2): the same with layers.2 [H, H] and layers.4.weight [O, H],
 *                                   layers.4.bias [O]
 *   MLP ("Policy"/"Value", :62-98): linear1.weight [H, I], linear1.bias [H], linear2.weight [O, H], linear2.bias [O]
 * ------------------------------------------------------------------------------------------ */
#define D2D_NET_MLP 0
#define D2D_NET_GRU 1
#define D2D_OUT_SOFTMAX 0   /* Policy.forward, RNN with combinatorial=False (d2d_ppo.py:56,81) */
#define D2D_OUT_SIGMOID 1   /* RNN with combinatorial=True (d2d_ppo.py:58)                     */
#define D2D_OUT_IDENTITY 2  /* Value, RNN(use_activation=False) (ippo.py:46,146)               */
#define D2D_DIST_BERNOULLI 0    /* combinatorial=True: Bernoulli(probs), mean over channels    */
#define D2D_DIST_CATEGORICAL 1
#define D2D_ACT_SAMPLE 0   /* select_action(train=True)  */
#define D2D_ACT_GREEDY 1   /* select_action(train=False) */
#define D2D_ACT_GIVEN 2    /* evaluate(states, actions)  */

typedef struct d2d_net_config {
  int32_t arch;            /* D2D_NET_*                                                         */
  int32_t out_kind;        /* D2D_OUT_*                                                         */
  int32_t n_agents;        /* N networks                                                        */
  int32_t n_envs;          /* B                                                                 */
  int32_t hidden;          /* H, 1..128 (16 / 32 / 48 / 64: tcgen05 kernels; others: FP32 kernels)      */
  int32_t n_out;           /* O: action_space[k].n for policies, 1 for critics (<= 32)          */
  int32_t history_len;     /* L: GRU window (d2d_ppo.py:302); ignored for MLP                   */
  int32_t in_rows;         /* feature rows per time block of the input matrix                   */
  const int32_t* in_dim;   /* [N] host: input size of agent k                                   */
  const int32_t* in_off;   /* [N] host: first feature row of agent k inside a time block        */
  int64_t scratch_bytes;   /* activation scratch budget per call (0: 2 GiB)                     */
  int32_t inputs_bf16_exact; /* 1: every input value is exactly representable in bf16 (the integer-valued
                                observations of CombinatorialEnv / D2DEnv): allows the tcgen05 GRU-window
                                kernel, whose input projection uses a single bf16 plane for x            */
  int32_t head_layers;     /* hidden Linear+ReLU layers behind the GRU: 0 or 1 = the PPO nets (layers.0, layers.2);
                              2 = the Q-network of algorithms/irdqn.py:58-72 (layers.0, layers.2, layers.4; GRU only) */
} d2d_net_config;

typedef struct d2d_net d2d_net;
int d2d_net_create(const d2d_net_config* cfg, d2d_net** out);
int d2d_net_destroy(d2d_net* net);
int64_t d2d_net_param_stride(const d2d_net* net);       /* floats per agent block                        */
int d2d_net_num_tensors(const d2d_net* net);            /* 8 (GRU), 10 (GRU Q-network) or 4 (MLP)        */
/* state_dict tensor `index` of agent `agent`: offset inside the agent's block, rows, cols (cols = 1: vector) */
int d2d_net_tensor(const d2d_net* net, int agent, int index, int64_t* offset, int32_t* rows, int32_t* cols);

/* Forward of time blocks [t0, t1): net(x windows) -> PRE-activation outputs.
 *   x       f32 [x_lead + T][in_rows][B]; block x_lead + t holds time t; for GRU nets x_lead >= L - 1 and the
 *           blocks before time 0 are zero (the left zero padding of preprocess_input_for_rnn, d2d_ppo.py:385-398)
 *   padded  1: training windows (zero inputs before the episode start still run a GRU step)
 *           0: rollout windows (d2d_ppo.py:302: those steps do not exist)
 *   out     f32 [t1 - t0][N][O][B]                                                                           */
int d2d_net_forward(d2d_net* net, const float* params, const float* x, int x_lead, int t0, int t1, int padded,
                    float* out, void* stream);

/* Guard of the inputs_bf16_exact promise: counts the inputs of time blocks [t0, t1) (all agents' rows) that are NOT
 * exactly representable in bf16, into *n_inexact (device, u64).  The learners run it over every rollout they
 * collect and refuse to train on a non-zero count: a wrong flag would otherwise silently truncate the observations
 * to 8 significant bits in the tensor-core GRU window. */
int d2d_net_check_inputs(const d2d_net* net, const float* x, int x_lead, int t0, int t1,
                         unsigned long long* n_inexact, void* stream);

/* Kernel switches: A/B comparison and debugging (the library reads no environment variables).  All three are enabled
 * by default; any other id is rejected with D2D_ERR_INVALID.  Process-wide, not thread-safe: set before the first
 * launch. */
#define D2D_SWITCH_ALL_TC 5           /* 0: every GEMM, GRU window and BPTT of the learner runs on its FP32 CUDA-core
                                         kernel instead of the tensor cores */
#define D2D_SWITCH_ENV_MULTISTEP 9    /* 0: d2d_env_run_random_access launches one step kernel per step even where a
                                         register-resident multi-step kernel applies (Philox streams, no state rows:
                                         single-channel env with N <= 4 and no observations; combinatorial env with
                                         N <= 8 and C = 4 or 8) */
#define D2D_SWITCH_HOST_PACK 10       /* 0: d2d_env_step_host always copies the reference-layout actions as they are and
                                         packs them on the device (default: packed on the host when >= 12 host threads) */
int d2d_set_kernel_switch(int which, int enabled);
int d2d_get_kernel_switch(int which);

/* Rollout step (PPO.select_action's network call, d2d_ppo.py:302-303): forward of the single time block t on
 * the UNPADDED window.  The input projections of the previous L - 1 observations are kept in a ring inside the
 * handle, so each observation is projected once per episode instead of L times.  Call with t = 0, 1, 2, ... in
 * order within an episode; `params` must not change between the calls of one episode.  out f32 [1][N][O][B].   */
int d2d_net_rollout_step(d2d_net* net, const float* params, const float* x, int x_lead, int t, float* out,
                         void* stream);

/* PPO.select_action for all N agents at time t (d2d_ppo.py:159-181 called at :298-309): network forward on the
 * unpadded window, then the action (sampled from the Philox policy stream, greedy, or given) and its log-prob.
 * When the tensor-core GRU window kernel takes the net, window + head + selection + log-prob are ONE launch and the
 * outputs never leave the SM; otherwise d2d_net_rollout_step + d2d_policy_head.
 *   actions     [N][B] of time t (channel bitmask u8 / i16 / i32 for Bernoulli, u8 index for Categorical); read when
 *               act_mode = D2D_ACT_GIVEN, written otherwise;   logp f32 [N][B] of time t
 *   logits_out  f32 [1][N][O][B] or NULL (pre-activation outputs, for callers that want them)                    */
int d2d_net_rollout_act(d2d_net* net, const float* params, const float* x, int x_lead, int t, int dist_kind,
                        int act_mode, void* actions, float* logp, uint64_t seed, uint64_t env_offset, int t_abs0,
                        float* logits_out, void* stream);

/* Distribution head on pre-activation outputs (PPO.select_action / PPO.evaluate, d2d_ppo.py:159-196).
 *   logits   f32 [n_t][N][O][B]
 *   actions  Bernoulli: channel bitmask [n_t][N][B] (1/2/4 bytes for O <= 8/16/32); Categorical: u8 index.
 *            Written for D2D_ACT_SAMPLE / GREEDY, read for D2D_ACT_GIVEN.
 *   logp, entropy  f32 [n_t][N][B] (entropy may be NULL);  probs f32 [n_t][N][O][B] or NULL
 *   sampling uses Philox4x32-10 keyed (seed; env_offset + b, t_abs0 + t, agent, purpose = policy)            */
int d2d_policy_head(int n_agents, int n_envs, int n_out, int n_t, int out_kind, int dist_kind, int act_mode,
                    const float* logits, void* actions, float* logp, float* entropy, float* probs, uint64_t seed,
                    uint64_t env_offset, int t_abs0, void* stream);

/* PPO clipped-surrogate gradient of all N policies over time blocks [t0, t1)  (PPO.train_step, d2d_ppo.py:198-216,
 * ippo.py:194-206): forward on padded windows, loss, backward.
 *   actions, logp_old   [T][N][B] (indexed by absolute time)
 *   weight              f32 advantages [T][N][B] (weight_per_agent = 1, IPPO) or [T][B] (= 0, D2DPPO)
 *   cycle               int32 device [N] or NULL: HAPPO order; agent cycle[j] is weighted by
 *                       weight * prod_{i<j} ratio_{cycle[i]} (the sequential M chain of d2d_ppo.py:427-436)
 *   inv_rows            1 / (rows of the whole batch, over all ranks): the loss is a mean over rows
 *   grads               f32 [N][param_stride], ACCUMULATED into
 *   loss_sums           f64 device [N][2], ACCUMULATED: sum_rows min(surr1, surr2), sum_rows entropy
 *   ratio_out           f32 [T][N][B] or NULL                                                            */
int d2d_ppo_policy_grad(d2d_net* net, const float* params, const float* x, int x_lead, int t0, int t1,
                        int dist_kind, const void* actions, const float* logp_old, const float* weight,
                        int weight_per_agent, const int32_t* cycle, float inv_rows, float cliprange, float beta,
                        float* grads, double* loss_sums, float* ratio_out, void* stream);

/* Critic MSE gradient over time blocks [t0, t1) (ippo.py:208-215, d2d_ppo.py:440-446).
 *   target     f32 [T][N][B] (per_agent = 1) or [T][B] (= 0);  value_out f32 [T][N][B] or NULL
 *   loss_sum   f64 device [N], ACCUMULATED: sum_rows (v - target)^2                                      */
int d2d_value_grad(d2d_net* net, const float* params, const float* x, int x_lead, int t0, int t1, int padded,
                   const float* target, int per_agent, float inv_rows, float* grads, double* loss_sum,
                   float* value_out, void* stream);

/* torch.optim.Adam (betas 0.9 / 0.999, eps 1e-8) on [N][per_agent] buffers, step counter `step` (1-based).
 * max_norm > 0: clip_grad_norm_(max_norm) per agent first (d2d_ppo.py:211,445); sqnorm: f64 device [N] scratch. */
int d2d_adam_step(float* params, float* m, float* v, const float* grads, int n_agents, int64_t per_agent,
                  float lr, int step, float max_norm, double* sqnorm, void* stream);

/* compute_gae (d2d_ppo.py:100-110) and discount_rewards (:112-124) as reverse scans in float64.
 *   reward   i32 [T][B] (all agents of an env share the reward, combinatorial_env.py:211)
 *   value    f32 [T][n_cols][B] (NULL: no lambda-returns)
 *   adv_raw / ret_raw  f64 [T][n_cols][B] outputs (either may be NULL)
 *   stats    f64 device [n_cols][4], ACCUMULATED: sum / sum of squares of adv_raw, of (float)ret_raw
 *   last_shard  1 if this GPU holds the globally last env (its final row keeps the r - v quirk of :102)  */
int d2d_returns_scan(const int32_t* reward, const float* value, double* adv_raw, double* ret_raw, double* stats,
                     int T, int n_envs, int n_cols, double gamma, double lam, int last_shard, void* stream);
/* Normalisation statistics from the (all-reduced over ranks) [n_cols][4] sums of d2d_returns_stats and the global row
 * count: lambda-returns with numpy's population std (d2d_ppo.py:108-109), returns with torch's unbiased std
 * (:121-123); *_norm = 1 iff EVERY column has a positive std (the reference's `.all()` gate), tested relative to the
 * column's mean square (var > 1e-9 mean(x^2)) because the one-pass sums leave rounding noise where numpy / torch give
 * an exact 0.  All outputs are device arrays of n_cols elements; one tiny launch, no host round trip. */
int d2d_returns_norm_stats(const double* stats, int n_cols, double rows, double* adv_mean, double* adv_std,
                           int32_t* adv_norm, double* ret_mean, double* ret_std, int32_t* ret_norm, void* stream);

/* The same scans in two passes without fp64 intermediates in HBM (17 B per element instead of 45):
 * d2d_returns_stats accumulates `stats` only (want_adv / want_ret select the scans); after the caller has
 * reduced the statistics over ranks, d2d_returns_emit repeats the scans and writes the NORMALISED results
 *   adv_out f32 [T][n_cols][B] = (lambda-return - mean) / std in float64, numpy semantics (d2d_ppo.py:107-109)
 *   ret_out f32 [T][n_cols][B] = ((float)return - mean) / std in float32, torch semantics (d2d_ppo.py:119-123)
 * (either may be NULL; *_norm[col] == 0 skips the normalisation of that column, :108 / :122). */
int d2d_returns_stats(const int32_t* reward, const float* value, double* stats, int T, int n_envs, int n_cols,
                      double gamma, double lam, int last_shard, int want_adv, int want_ret, void* stream);
int d2d_returns_emit(const int32_t* reward, const float* value, float* adv_out, float* ret_out,
                     const double* adv_mean, const double* adv_std, const int32_t* adv_norm,
                     const double* ret_mean, const double* ret_std, const int32_t* ret_norm, int T, int n_envs,
                     int n_cols, double gamma, double lam, int last_shard, void* stream);
/* out[i] = (raw[i] - mean[col]) / std[col] as f32 (do_norm[col] == 0: plain cast); fp32_math = 1 reproduces
 * discount_rewards (cast to f32 first, normalise in f32).  mean/std f64 device [n_cols], do_norm i32 device. */
int d2d_normalize(const double* raw, float* out, const double* mean, const double* std, const int32_t* do_norm,
                  int fp32_math, int T, int n_envs, int n_cols, void* stream);

/* ------------------------------------------------------------------------------------------
 * Independent recurrent DQN (algorithms/irdqn.py), SURVEY.md section 8(f)4.  The Q-networks are net sets with
 * head_layers = 2 and D2D_OUT_IDENTITY; forward / rollout go through d2d_net_forward / d2d_net_rollout_step.
 * ------------------------------------------------------------------------------------------ */
#define D2D_QLOSS_HUBER 0   /* F.smooth_l1_loss (beta 1), irdqn.py:120 */
#define D2D_QLOSS_MSE 1     /* F.mse_loss                             */

/* torch.optim.Adam with a caller-chosen eps (irdqn.py:130 passes adam_epsilon); otherwise d2d_adam_step. */
int d2d_adam_step_eps(float* params, float* m, float* v, const float* grads, int n_agents, int64_t per_agent,
                      float lr, float eps, int step, float max_norm, double* sqnorm, void* stream);

/* DQN.act / DQN.predict for all N agents and B envs (irdqn.py:150-166, called at :244-253 and :323-328).
 *   q          f32 [N][O][B] Q-values of the current windows
 *   act_mode   D2D_ACT_SAMPLE: greedy iff training_ready and uniform >= epsilon, else a uniform draw from
 *              {0, .., n_random - 1} (the reference draws np.random.randint(0, 2): n_random = 2, whatever O is);
 *              D2D_ACT_GREEDY: argmax, first maximum (predict); D2D_ACT_GIVEN: action_idx is read, not written
 *   action_idx u8 [N][B];  action_mask: one-hot channel bitmask 1 << idx, [N][B] of mask_bytes (1/2/4) bytes each,
 *              the action_binary rows of irdqn.py:249-250 in the device action layout (may be NULL)
 *   draws: Philox4x32-10 keyed (seed; env_offset + b, t_abs, agent, purpose = policy)                        */
int d2d_q_select(int n_agents, int n_envs, int n_out, const float* q, int act_mode, float epsilon,
                 int training_ready, int n_random, uint8_t* action_idx, void* action_mask, int mask_bytes,
                 uint64_t seed, uint64_t env_offset, int t_abs, void* stream);

/* td_target = rewards + (1 - dones) * gamma * max_a Q_target(s')  (irdqn.py:136-139), fp32 in torch's op order.
 *   q_next f32 [N][O][B];  reward i32 [B] (all agents of an env share it);  done u8 [B];  target f32 [N][B]  */
int d2d_q_td_target(int n_agents, int n_envs, int n_out, const float* q_next, const int32_t* reward,
                    const uint8_t* done, float gamma, float* target, void* stream);

/* DQN.train_step up to the optimiser (irdqn.py:140-145) for all N agents over time blocks [t0, t1): forward on
 * padded windows, loss(Q[action], target) with reduction 'mean' over the rows, backward.
 *   actions u8 [T][N][B], target f32 [T][N][B] (absolute time);  inv_rows = 1 / rows of the whole batch
 *   grads f32 [N][param_stride] ACCUMULATED;  loss_sum f64 device [N] ACCUMULATED (sum over rows of the loss
 *   terms: the loss is loss_sum * inv_rows);  q_out f32 [T][N][B] or NULL: Q of the taken action             */
int d2d_q_grad(d2d_net* net, const float* params, const float* x, int x_lead, int t0, int t1,
               const uint8_t* actions, const float* target, int loss_kind, float inv_rows, float* grads,
               double* loss_sum, float* q_out, void* stream);

/* ReplayBuffer.sample_chunk (irdqn.py:24-42) on a device-resident ring.  Every env column b holds its own deque
 * of transitions, episode-major: the ring keeps the last n_ep_slots episodes as
 *   obs_ring f32 [n_ep_slots][T + 1][rows][B]  (state of transition t = block t, state_next = block t + 1)
 *   act_ring u8  [n_ep_slots][T][N][B],  rew_ring i32 [n_ep_slots][T][B]
 * and ep0 is the slot of the OLDEST stored episode (deque index 0).  Minibatch element j is the chunk of `chunk`
 * consecutive transitions start[j] .. start[j] + chunk - 1 (deque indices, may straddle an episode end as in the
 * reference) of env column env_col[j].  Outputs are env-minor minibatch matrices with B = mb:
 *   xs, xn f32 [chunk][rows][mb] (states / next states of the chunk);  act u8 [N][mb], rew i32 [mb], done u8 [mb]
 *   of the LAST transition of the chunk (irdqn.py:293-296).                                                  */
int d2d_replay_gather(const float* obs_ring, const uint8_t* act_ring, const int32_t* rew_ring,
                      const int32_t* start, const int32_t* env_col, int ep0, int n_ep_slots, int T, int chunk,
                      int rows, int n_agents, int n_envs, int mb, float* xs, float* xn, uint8_t* act, int32_t* rew,
                      uint8_t* done, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* D2D_B200_H */
