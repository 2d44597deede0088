// Host orchestration + C ABI of the learner (PPO / IPPO networks, losses, returns, optimiser).
//
// Replaces (file:line under /root/reference):
//   RNN / Policy / Value forward            algorithms/d2d_ppo.py:24-98, algorithms/ippo.py:14-90  -> d2d_net_forward
//   PPO.select_action / PPO.evaluate        d2d_ppo.py:159-196, ippo.py:154-191                    -> d2d_policy_head
//   PPO.train_step (policy part)            d2d_ppo.py:198-216, ippo.py:194-206                    -> d2d_ppo_policy_grad
//   critic MSE step                         d2d_ppo.py:440-446, ippo.py:208-215                    -> d2d_value_grad
//   compute_gae / discount_rewards          d2d_ppo.py:100-124                                     -> d2d_returns_scan
//   clip_grad_norm_ + Adam                  d2d_ppo.py:211-212,445-446                             -> d2d_adam_step
//   DQN.act / predict, train_step, replay   algorithms/irdqn.py:24-42,133-166                      -> d2d_q_select,
//                                                                    d2d_q_td_target, d2d_q_grad, d2d_replay_gather
//
// A net set evaluates N independent per-agent networks with grid.y = agent.  Time blocks are processed in
// chunks sized to the activation-scratch budget; the GRU window is unrolled step by step over the chunk with
// the input projection of every observation computed ONCE and shared by the up-to-L windows that contain it.
#include <algorithm>
#include <cstring>
#include <new>
#include <vector>

#include "gru_tc.cuh"
#include "gru_bwd_tc.cuh"
#include "gru_bptt_tc.cuh"
#include "wgrad_tc.cuh"
#include "dense_tc.cuh"
#include "head_fused.cuh"
#include "learner_pointwise.cuh"
#include "dqn_pointwise.cuh"

using namespace d2d;

struct d2d_net {
  int arch, out_kind, N, B, H, O, L, in_rows;
  int x_exact = 0;   // inputs are exactly representable in bf16 (integer observations): tensor-core GRU path allowed
  std::vector<int> in_dim, in_off;
  int max_in;
  long long stride;  // floats per agent block
  // per-agent tensor offsets inside the block
  std::vector<int> o_wih, o_whh, o_bih, o_bhh, o_w1, o_b1, o_w2, o_b2;
  int head2 = 0;              // 1: the Q-network head of algorithms/irdqn.py:63-69 (Linear-ReLU-Linear-ReLU-Linear)
  std::vector<int> o_w1b, o_b1b;   // its second hidden layer, layers.2 [H, H]; the output layer is then layers.4
  long long scratch_bytes;
  float* scratch = nullptr;
  long long scratch_cap = 0;  // floats
  float* gi_ring = nullptr;   // [L][N][3H][B] input projections of the last L observations (rollout)
  float* partial = nullptr;   // wgrad partial sums
  long long part_stride = 0;
  int n_strips = 0;
};

// ------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------
static View make_view(float* p, long long t_stride, int t_off, int N, int feat_per_agent, int B) {
  View v;
  memset(&v, 0, sizeof(v));
  v.p = p, v.t_stride = t_stride, v.t_off = t_off;
  for (int g = 0; g < N; ++g) v.f_off[g] = g * feat_per_agent;
  (void)B;
  return v;
}

// the observations: agent g's features are rows in_off[g] ... of each time block; time block t is x_lead blocks in
static View input_view(const d2d_net* n, const float* x, int x_lead) {
  View v;
  memset(&v, 0, sizeof(v));
  v.p = const_cast<float*>(x), v.t_stride = (long long)n->in_rows * n->B, v.t_off = x_lead;
  for (int g = 0; g < n->N; ++g) v.f_off[g] = n->in_off[g];
  return v;
}

// Kernel switches (d2d_set_kernel_switch in the C ABI): an A/B and debugging control set explicitly by the caller --
// the library reads no environment variables.  Not thread-safe; set before the first launch.
static int g_all_tc = 1, g_env_multistep = 1, g_host_pack = 1;
static int* switch_ptr(int which) {
  switch (which) {
    case D2D_SWITCH_ALL_TC: return &g_all_tc;
    case D2D_SWITCH_ENV_MULTISTEP: return &g_env_multistep;
    case D2D_SWITCH_HOST_PACK: return &g_host_pack;
    default: return nullptr;
  }
}
static bool tc_enabled() { return g_all_tc != 0; }

extern "C" int d2d_set_kernel_switch(int which, int enabled) {
  int* sw = switch_ptr(which);
  D2D_REQUIRE(sw, "d2d_set_kernel_switch: unknown switch %d", which);
  *sw = enabled ? 1 : 0;
  return D2D_OK;
}
extern "C" int d2d_get_kernel_switch(int which) {
  const int* sw = switch_ptr(which);
  return sw ? *sw : D2D_ERR_INVALID;
}

template <int RPT, int OPT>
static int launch_dense_tile(const d2d_net* n, const DenseArgs& a, int max_in, cudaStream_t s) {
  constexpr int ROWS = 32 * RPT;
  const size_t smem = ((size_t)std::max(max_in, 1) * 8 * OPT + 8 * OPT + 2 * kDenseKC * ROWS) * sizeof(float);
  static bool attr = false;
  if (!attr) {
    D2D_CUDA(cudaFuncSetAttribute(dense_tile_kernel<RPT, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  200 * 1024));
    attr = true;
  }
  const int tiles = (a.t1 - a.t0) * ((n->B + ROWS - 1) / ROWS);
  if (tiles <= 0) return D2D_OK;
  // persistent grid: exactly the number of blocks that are resident at once (registers + shared memory)
  int per_sm = 1;
  D2D_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dense_tile_kernel<RPT, OPT>, 256, smem));
  per_sm = std::max(per_sm, 1);
  const int gx = std::max(1, std::min(tiles, (148 * per_sm) / n->N));
  dense_tile_kernel<RPT, OPT><<<dim3(gx, n->N), 256, smem, s>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

static int launch_dense(const d2d_net* n, DenseArgs& a, int max_in, cudaStream_t s, int x_exact = 0) {
  a.B = n->B;
  // more than 192 outputs (3H of the hidden sizes above 64, e.g. the reference's iRDQN networks with H = 100): the
  // register-tiled kernel takes at most 192, so the output rows are split into equal slices that each go through it
  // (the generic kernel below is ~5x slower: profiles/r02_n_irdqn_launch_summary.txt)
  if (a.out_dim > 192 && n->B % 4 == 0 && (size_t)std::max(max_in, 1) * 8 * 24 * 4 <= 150 * 1024) {
    const int parts = (a.out_dim + 191) / 192;
    const int slice = ((a.out_dim + parts - 1) / parts + 7) / 8 * 8;
    for (int o0 = 0; o0 < a.out_dim; o0 += slice) {
      DenseArgs p = a;
      p.out_dim = std::min(slice, a.out_dim - o0);
      for (int g = 0; g < n->N; ++g) {
        p.w_off[g] = a.w_off[g] + (a.trans ? o0 : o0 * a.w_ld[g]);
        if (a.b_off[g] >= 0) p.b_off[g] = a.b_off[g] + o0;
        p.y.f_off[g] = a.y.f_off[g] + o0;
        if (a.aux.p) p.aux.f_off[g] = a.aux.f_off[g] + o0;
      }
      const int rc = launch_dense(n, p, max_in, s, x_exact);
      if (rc) return rc;
    }
    return D2D_OK;
  }
  // a reduction too long for the register-tiled kernel's resident weight tile (K = 3H of the hidden sizes above 64 in
  // d(h) += d(gh) W_hh): split along K into accumulating launches instead of falling to the generic kernel, which
  // re-stages the whole matrix per block (322 us for a 64-row minibatch: profiles/r02_n_irdqn_launch_summary.txt)
  if ((a.epilogue == kEpiAccum || a.epilogue == kEpiNone) && n->B % 4 == 0 && a.out_dim <= 192 && max_in > 160 &&
      (size_t)max_in * 8 * (a.out_dim > 64 ? 24 : (a.out_dim > 32 ? 8 : 4)) * 4 > 160 * 1024) {
    const int parts = (max_in + 159) / 160;
    const int slice = ((max_in + parts - 1) / parts + 3) / 4 * 4;
    for (int k0 = 0; k0 < max_in; k0 += slice) {
      DenseArgs p = a;
      if (k0 > 0) p.epilogue = kEpiAccum;
      for (int g = 0; g < n->N; ++g) {
        p.in_dim[g] = std::max(0, std::min(slice, a.in_dim[g] - k0));
        p.w_off[g] = a.w_off[g] + (a.trans ? k0 * a.w_ld[g] : k0);
        if (k0 > 0) p.b_off[g] = -1;
        p.x.f_off[g] = a.x.f_off[g] + k0;
      }
      const int rc = launch_dense(n, p, std::min(slice, max_in - k0), s, x_exact);
      if (rc) return rc;
    }
    return D2D_OK;
  }
  // tensor-core path (dense_tc.cuh) for single-chunk reductions (K <= 64); with K = 3H the three stage -> MMA round
  // trips per tile serialise inside a slot and the register-tiled FP32 kernel is faster (measured 212 vs 480 us)
  if (tc_enabled() && n->B >= 256 && a.out_dim <= 192 && max_in <= tcd::kKc &&
      tcd::smem_bytes(max_in, a.out_dim) <= 225 * 1024) {
    static bool attr = false;
    if (!attr) {
      D2D_CUDA(cudaFuncSetAttribute(dense_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024));
      attr = true;
    }
    const int pairs = (a.t1 - a.t0) * ((n->B + 255) / 256);
    if (pairs <= 0) return D2D_OK;
    const int gx = std::max(1, std::min(pairs, 148 / n->N));
    dense_tc_kernel<<<dim3(gx, n->N), tcd::kThreads, tcd::smem_bytes(max_in, a.out_dim), s>>>(a, x_exact);
    D2D_LAUNCHED();
    return D2D_OK;
  }
  const int tile_opt = a.out_dim > 64 ? 24 : (a.out_dim > 32 ? 8 : 4), tile_rows = a.out_dim > 64 ? 128 : 256;
  const size_t tile_smem = ((size_t)std::max(max_in, 1) * 8 * tile_opt + 8 * tile_opt + 2 * kDenseKC * tile_rows) * 4;
  if (n->B % 4 == 0 && a.out_dim <= 192 && tile_smem <= 200 * 1024) {   // register-tiled path (rows moved as float4)
    if (a.out_dim > 64) return launch_dense_tile<4, 24>(n, a, max_in, s);
    if (a.out_dim > 32) return launch_dense_tile<8, 8>(n, a, max_in, s);
    return launch_dense_tile<8, 4>(n, a, max_in, s);
  }
  const int OC = a.out_dim >= 64 ? 64 : 16;
  const int out_pad = (a.out_dim + OC - 1) / OC * OC;
  const size_t smem = ((size_t)max_in * out_pad + out_pad) * sizeof(float);
  const int tiles = (a.t1 - a.t0) * ((n->B + kRowsPerBlock - 1) / kRowsPerBlock);
  if (tiles <= 0) return D2D_OK;
  // persistent over row tiles: the weight matrix is staged in shared memory once per block
  const int gx = std::max(1, std::min(tiles, (148 * 4 + n->N - 1) / n->N));
  dim3 grid(gx, n->N);
  if (OC == 64) {
    static bool attr64 = false;
    if (!attr64) {
      D2D_CUDA(cudaFuncSetAttribute(dense_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr64 = true;
    }
    dense_kernel<64><<<grid, kRowsPerBlock, smem, s>>>(a);
  } else {
    static bool attr16 = false;
    if (!attr16) {
      D2D_CUDA(cudaFuncSetAttribute(dense_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr16 = true;
    }
    dense_kernel<16><<<grid, kRowsPerBlock, smem, s>>>(a);
  }
  D2D_LAUNCHED();
  return D2D_OK;
}

// weight tensor descriptor: offsets per agent, input dims per agent
struct Wt {
  const std::vector<int>* w_off;
  const std::vector<int>* b_off;   // may be null
  const std::vector<int>* in_dim;  // per agent rows' length of the stored matrix (K)
  int in_const;                    // used when in_dim == nullptr
  int out_dim;
};

static void fill_dense_w(const d2d_net* n, DenseArgs& a, const float* params, const Wt& w, int trans) {
  a.w = params, a.w_agent_stride = n->stride, a.trans = trans;
  for (int g = 0; g < n->N; ++g) {
    const int K = w.in_dim ? (*w.in_dim)[g] : w.in_const;
    a.w_off[g] = (*w.w_off)[g];
    a.b_off[g] = (w.b_off && !trans) ? (*w.b_off)[g] : -1;
    a.w_ld[g] = K;
    a.in_dim[g] = trans ? w.out_dim : K;
  }
  a.out_dim = trans ? (w.in_dim ? 0 : w.in_const) : w.out_dim;
}

template <int TO, int TK>
static void launch_wgrad_t(const WgradArgs& a, dim3 grid, cudaStream_t s) {
  const size_t smem = (size_t)(16 * TO + 16 * TK) * (kWgRows + 1) * sizeof(float);
  wgrad_kernel<TO, TK><<<grid, 256, smem, s>>>(a);
}

// row length of the gradient of `w` per agent (zero_in: the input was zero, only the bias gradient is taken)
static int wgrad_in_dims(const d2d_net* n, const Wt& w, bool zero_in, int* in_dim) {
  int maxK = 0;
  for (int g = 0; g < n->N; ++g) {
    in_dim[g] = zero_in ? 0 : (w.in_dim ? (*w.in_dim)[g] : w.in_const);
    maxK = std::max(maxK, in_dim[g]);
  }
  return maxK;
}

// dW (+ db) of `w` += the fixed-order sum of the `strips` per-CTA partial sums in n->partial
static int launch_wreduce(const d2d_net* n, const Wt& w, bool zero_in, int strips, float* grads, cudaStream_t s) {
  WreduceArgs r;
  memset(&r, 0, sizeof(r));
  r.partial = n->partial, r.part_stride = n->part_stride, r.n_strips = strips, r.grads = grads;
  r.g_agent_stride = n->stride, r.out_dim = w.out_dim, r.with_bias = w.b_off != nullptr;
  for (int g = 0; g < n->N; ++g) {
    r.w_off[g] = (*w.w_off)[g];
    r.b_off[g] = w.b_off ? (*w.b_off)[g] : 0;
  }
  const int total = w.out_dim * wgrad_in_dims(n, w, zero_in, r.in_dim) + w.out_dim;
  wreduce_kernel<<<dim3((total + 255) / 256, n->N), 256, 0, s>>>(r);
  D2D_LAUNCHED();
  return D2D_OK;
}

// dW (+ db) of `w` from dy [out_dim] and x [K]; accumulated into grads
static int launch_wgrad(d2d_net* n, const View& dy, const View& x, const Wt& w, bool zero_in, float* grads, int t0,
                        int t1, cudaStream_t s, bool x_is_input = false) {
  WgradArgs a;
  memset(&a, 0, sizeof(a));
  a.x_planes = (x_is_input && n->x_exact) ? 1 : 0;   // x = the observations, exact in bf16 by the caller's promise
  a.dy = dy, a.x = x, a.partial = n->partial, a.part_stride = n->part_stride;
  a.out_dim = w.out_dim, a.B = n->B, a.t0 = t0, a.t1 = t1, a.with_bias = w.b_off != nullptr;
  const int maxK = wgrad_in_dims(n, w, zero_in, a.in_dim);
  int strips = n->n_strips;
  const int O = w.out_dim;
  if (maxK > 128) {
    set_error("learner: weight-gradient reduction width %d exceeds the supported 128", maxK);
    return D2D_ERR_INVALID;
  }
  if (O > 192) {   // hidden sizes above 64: 3H output rows are handled as blocks of <= 192 rows
    for (int o0 = 0; o0 < O; o0 += 192) {
      Wt wb = w;
      wb.out_dim = std::min(192, O - o0);
      std::vector<int> woff(n->N), boff(n->N);
      View dyb = dy;
      for (int g = 0; g < n->N; ++g) {
        const int K = w.in_dim ? (*w.in_dim)[g] : w.in_const;   // row length of the stored matrix
        woff[g] = (*w.w_off)[g] + o0 * K;
        boff[g] = w.b_off ? (*w.b_off)[g] + o0 : 0;
        dyb.f_off[g] += o0;
      }
      wb.w_off = &woff;
      wb.b_off = w.b_off ? &boff : nullptr;
      const int rc = launch_wgrad(n, dyb, x, wb, zero_in, grads, t0, t1, s, x_is_input);
      if (rc) return rc;
    }
    return D2D_OK;
  }
  if (tc_enabled() && n->B % 8 == 0) {
    // tensor-core path (wgrad_tc.cuh): bf16 x 3 planes on tcgen05, accumulators in TMEM
    const size_t smem = tcw::smem_bytes(maxK);
    static bool attr = false;
    if (!attr) {
      D2D_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
      attr = true;
    }
    strips = std::max(1, std::min(n->n_strips, 296 / n->N));   // two CTAs per SM
    wgrad_tc_kernel<<<dim3(strips, n->N), tcw::kThreads, smem, s>>>(a);
  } else {
    dim3 grid(strips, n->N);
    const int to = O > 64 ? 12 : (O > 16 ? 4 : 1);
    const int tk = maxK > 64 ? 8 : (maxK > 32 ? 4 : 2);
#define WG(TO_, TK_) if (to == TO_ && tk == TK_) launch_wgrad_t<TO_, TK_>(a, grid, s)
    WG(12, 2); WG(12, 4); WG(12, 8); WG(4, 2); WG(4, 4); WG(4, 8); WG(1, 2); WG(1, 4); WG(1, 8);
#undef WG
  }
  D2D_LAUNCHED();
  return launch_wreduce(n, w, zero_in, strips, grads, s);
}

// fused hidden projection + gates (B % 4 == 0)
static int launch_gru_step(const d2d_net* n, GruStepArgs& a, const float* params, cudaStream_t s) {
  a.w = params, a.w_agent_stride = n->stride, a.H = n->H, a.B = n->B;
  for (int g = 0; g < n->N; ++g) a.whh_off[g] = n->o_whh[g], a.bhh_off[g] = n->o_bhh[g];
  constexpr int ROWS = 128, OUT_PAD = 192;
  const size_t smem = ((size_t)std::max(a.first ? 0 : n->H, 1) * OUT_PAD + OUT_PAD + 2 * kDenseKC * ROWS) * sizeof(float);
  static bool attr = false;
  if (!attr) {
    D2D_CUDA(cudaFuncSetAttribute(gru_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = true;
  }
  const int tiles = (a.t1 - a.t0) * ((n->B + ROWS - 1) / ROWS);
  if (tiles <= 0) return D2D_OK;
  int per_sm = 1;
  D2D_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, gru_step_kernel, 256, smem));
  const int gx = std::max(1, std::min(tiles, (148 * std::max(per_sm, 1)) / n->N));
  for (int u0 = 0; u0 < n->H; u0 += 64) {      // H > 64: every slice reads all of h_prev and writes its own units
    a.u0 = u0;
    gru_step_kernel<<<dim3(gx, n->N), 256, smem, s>>>(a);
    D2D_LAUNCHED();
  }
  return D2D_OK;
}

// Which kernels a call on the net runs.  It depends on the net's shape and D2D_SWITCH_ALL_TC only, and is evaluated
// per call (plan_chunk keeps it in Chunk::plan) because the switch may change between calls on the same net: the
// scratch layout and the launches all read this one decision.
enum class Bptt { kFp32, kRecompute, kStoredTc };
enum class Head { kDense, kKernel, kWindow };
struct Plan {
  bool window_tc;   // GRU forward on the tcgen05 window kernel (gru_tc.cuh); else input projection + FP32 step kernels
  Bptt bptt;        // kRecompute: gru_bptt_tc recomputes the gates, the forward keeps h only; kStoredTc: gru_bwd_tc
                    // reads the gates the forward stored; kFp32: gate kernels + FP32 GEMMs on the stored gates
  Head head;        // kWindow: fused behind the window kernel; kKernel: head_fused_kernel; kDense: dense kernels
};

static Plan make_plan(const d2d_net* n) {
  const bool gru = n->arch == D2D_NET_GRU, all_tc = tc_enabled(), h32_64 = n->H == 32 || n->H == 64;
  Plan p;
  // the window stages the inputs as one fp16 plane (integer observations, the caller's promise) with I <= 32
  p.window_tc = all_tc && gru && n->x_exact && n->max_in <= tc::kKx && (h32_64 || n->H == 16 || n->H == 48);
  p.bptt = !(all_tc && gru && h32_64) ? Bptt::kFp32 : (p.window_tc ? Bptt::kRecompute : Bptt::kStoredTc);
  const bool head_fused = gru && h32_64 && n->O <= 16 && !n->head2;
  p.head = !head_fused ? Head::kDense : (p.window_tc ? Head::kWindow : Head::kKernel);
  return p;
}

template <int H, int STORE, int OMAX>
static int launch_gru_tc_k(const d2d_net* n, const GruTcArgs& a, cudaStream_t s) {
  const size_t smem =
      OMAX > 0 ? ((tc::Smem<H>::bytes + 15) & ~(size_t)15) + tc::Smem<H>::head_bytes(OMAX) : tc::Smem<H>::bytes;
  static bool attr = false;
  if (!attr) {
    D2D_CUDA(cudaFuncSetAttribute(gru_window_tc_kernel<H, STORE, OMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    attr = true;
  }
  const int pairs = (a.t1 - a.t0) * ((n->B + 2 * tc::kM - 1) / (2 * tc::kM));
  if (pairs <= 0) return D2D_OK;
  const int gx = std::max(1, std::min(pairs, 148 / n->N));   // one CTA per SM (all of its shared memory and TMEM)
  gru_window_tc_kernel<H, STORE, OMAX><<<dim3(gx, n->N), tc::kThreads, smem, s>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

// Only the instantiations a plan reaches: H 32 / 64 train for the recomputing BPTT (STORE 2: h only) and may have the
// head fused (OMAX > 0); H 16 / 48 train for the FP32 gate backward (STORE 1: h and the gates), their head runs apart.
template <int H>
static int launch_gru_tc_h(const d2d_net* n, const GruTcArgs& a, cudaStream_t s, bool head) {
  constexpr int kStore = (H == 32 || H == 64) ? 2 : 1;
  if constexpr (H == 32 || H == 64) {
    if (head) {
      if (a.O <= 1) return a.store ? launch_gru_tc_k<H, kStore, 1>(n, a, s) : launch_gru_tc_k<H, 0, 1>(n, a, s);
      if (a.O <= 8) return a.store ? launch_gru_tc_k<H, kStore, 8>(n, a, s) : launch_gru_tc_k<H, 0, 8>(n, a, s);
      return a.store ? launch_gru_tc_k<H, kStore, 16>(n, a, s) : launch_gru_tc_k<H, 0, 16>(n, a, s);
    }
  }
  return a.store ? launch_gru_tc_k<H, kStore, 0>(n, a, s) : launch_gru_tc_k<H, 0, 0>(n, a, s);
}

// tensor-core fused GRU window (gru_tc.cuh): x windows -> last hidden state in h_out, no intermediate in HBM.
// hs != nullptr (training): h of every step goes to *hs instead, the L steps hs_step floats apart, and the gates to
// *acts (4 hs_step apart) unless acts->p is null.  out != nullptr: the network head is fused behind the window and
// *out receives the pre-activation outputs (out->p == nullptr: not written), *y1 relu(W1 h + b1) if given; sel turns
// the outputs into actions and log-probs.
static int launch_gru_tc(const d2d_net* n, const float* params, const View& x, const View& h_out, int t0, int t1,
                         int padded, cudaStream_t s, const View* hs, const View* acts, long long hs_step,
                         const View* out, const View* y1, const DistArgs* sel) {
  GruTcArgs a;
  memset(&a, 0, sizeof(a));
  a.x = x, a.h_out = h_out, a.w = params, a.w_agent_stride = n->stride;
  if (hs) a.store = 1, a.acts = *acts, a.hs = *hs, a.acts_step = 4 * hs_step, a.hs_step = hs_step;
  for (int g = 0; g < n->N; ++g) {
    a.wih_off[g] = n->o_wih[g], a.whh_off[g] = n->o_whh[g], a.bih_off[g] = n->o_bih[g], a.bhh_off[g] = n->o_bhh[g];
    a.in_dim[g] = n->in_dim[g];
    a.w1_off[g] = n->o_w1[g], a.b1_off[g] = n->o_b1[g], a.w2_off[g] = n->o_w2[g], a.b2_off[g] = n->o_b2[g];
  }
  a.L = n->L, a.B = n->B, a.t0 = t0, a.t1 = t1, a.padded = padded, a.O = n->O;
  if (out) a.out = *out;
  if (y1) a.y1 = *y1;
  if (sel) a.sel = *sel;
  switch (n->H) {
    case 16: return launch_gru_tc_h<16>(n, a, s, false);
    case 32: return launch_gru_tc_h<32>(n, a, s, out != nullptr);
    case 48: return launch_gru_tc_h<48>(n, a, s, false);
    default: return launch_gru_tc_h<64>(n, a, s, out != nullptr);
  }
}

// fused network head (head_fused.cuh): out = W2 relu(W1 h + b1) + b2; y1 == nullptr: first-layer outputs not kept
template <int H, int OMAX>
static void launch_head_fused_t(const HeadFusedArgs& a, int N, int tiles, cudaStream_t s) {
  const int gx = std::max(1, std::min(tiles, (148 * 2) / N));
  if (a.y1.p) head_fused_kernel<H, OMAX, true><<<dim3(gx, N), kHeadThreads, 0, s>>>(a);
  else head_fused_kernel<H, OMAX, false><<<dim3(gx, N), kHeadThreads, 0, s>>>(a);
}

static int launch_head_fused(const d2d_net* n, const float* params, const View& h, float* y1, const View& out, int t0,
                             int t1, cudaStream_t s) {
  HeadFusedArgs a;
  memset(&a, 0, sizeof(a));
  const long long NB = (long long)n->N * n->B;
  a.h = h, a.out = out, a.w = params, a.w_agent_stride = n->stride, a.O = n->O, a.B = n->B, a.t0 = t0, a.t1 = t1;
  if (y1) a.y1 = make_view(y1, n->H * NB, -t0, n->N, n->H, n->B);
  for (int g = 0; g < n->N; ++g)
    a.w1_off[g] = n->o_w1[g], a.b1_off[g] = n->o_b1[g], a.w2_off[g] = n->o_w2[g], a.b2_off[g] = n->o_b2[g];
  const int tiles = (t1 - t0) * ((n->B + 2 * kHeadThreads - 1) / (2 * kHeadThreads));
  if (tiles <= 0) return D2D_OK;
  const int om = n->O <= 1 ? 1 : (n->O <= 8 ? 8 : 16);
#define HF(H_, O_) if (n->H == H_ && om == O_) launch_head_fused_t<H_, O_>(a, n->N, tiles, s)
  HF(32, 1); HF(32, 8); HF(32, 16); HF(64, 1); HF(64, 8); HF(64, 16);
#undef HF
  D2D_LAUNCHED();
  return D2D_OK;
}

template <int H>
static int launch_gru_bptt_tc_h(const d2d_net* n, const GruBpttArgs& a, cudaStream_t s, int* strips) {
  static bool attr = false;
  if (!attr) {
    D2D_CUDA(cudaFuncSetAttribute(gru_bptt_tc_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)tcr::Smem<H>::bytes));
    attr = true;
  }
  const int tiles = (a.t1 - a.t0) * ((n->B + tc::kM - 1) / tc::kM);
  if (tiles <= 0) return D2D_OK;
  const int gx = std::max(1, std::min(std::min(tiles, 148 / n->N), n->n_strips));
  gru_bptt_tc_kernel<H><<<dim3(gx, n->N), tcr::kThreads, tcr::Smem<H>::bytes, s>>>(a);
  D2D_LAUNCHED();
  *strips = gx;
  return D2D_OK;
}

template <int H>
static int launch_gru_bwd_tc_h(const d2d_net* n, const GruBwdTcArgs& a, cudaStream_t s, int* strips) {
  static bool attr = false;
  if (!attr) {
    D2D_CUDA(cudaFuncSetAttribute(gru_bwd_tc_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)tcb::Smem<H>::bytes));
    attr = true;
  }
  const int tiles = (a.t1 - a.t0) * ((n->B + tc::kM - 1) / tc::kM);
  if (tiles <= 0) return D2D_OK;
  const int gx = std::max(1, std::min(std::min(tiles, 148 / n->N), n->n_strips));
  gru_bwd_tc_kernel<H><<<dim3(gx, n->N), tcb::kThreads, tcb::Smem<H>::bytes, s>>>(a);
  D2D_LAUNCHED();
  *strips = gx;
  return D2D_OK;
}

static int launch_gate(const GateArgs& a, int N, bool bwd, cudaStream_t s) {
  const long long n = (long long)(a.t1 - a.t0) * a.H * a.B;
  if (n <= 0) return D2D_OK;
  dim3 grid(grid_for(n, 256), N);
  if (bwd) gru_gate_bwd_kernel<<<grid, 256, 0, s>>>(a);
  else gru_gate_fwd_kernel<<<grid, 256, 0, s>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

// ------------------------------------------------------------------------------------------------
// scratch carving for one chunk of Tc time blocks
// ------------------------------------------------------------------------------------------------
struct Chunk {
  int Tc, halo;
  Plan plan;
  float *gi, *gh, *acts, *hs, *y1, *y2, *logits, *dl, *dy1, *dy2, *dh0, *dh1, *dgi;
};

static long long floats_per_t(const d2d_net* n, bool train, const Plan& plan) {
  const long long NB = (long long)n->N * n->B;
  const long long H = n->H, O = n->O, L = n->arch == D2D_NET_GRU ? n->L : 0;
  long long f = H + O;                                // y1, logits
  if (n->head2) f += train ? 2 * H : H;               // y2 (+ dy2)
  if (n->arch == D2D_NET_GRU) f += 3 * H + 3 * H;     // gi, gh
  // hs of every step; the 4H activations per step only for the BPTT kernels that do not recompute them
  if (n->arch == D2D_NET_GRU) f += train ? L * H + (plan.bptt == Bptt::kRecompute ? 0 : 4 * L * H) : 2 * H;
  if (train) f += O + H;                              // dl, dy1
  if (train && n->arch == D2D_NET_GRU) f += 2 * H + 3 * H;   // dh ping-pong, dgi
  return f * NB;
}

static int plan_chunk(d2d_net* n, bool train, int n_t, Chunk& c) {
  const long long NB = (long long)n->N * n->B;
  const int halo = n->arch == D2D_NET_GRU ? n->L - 1 : 0;
  c.plan = make_plan(n);
  const long long per_t = floats_per_t(n, train, c.plan);
  const long long halo_f = (long long)halo * 3 * n->H * NB * (train ? 2 : 1);
  long long budget = n->scratch_bytes / 4;
  int Tc = (int)std::max<long long>(1, std::min<long long>(n_t, (budget - halo_f) / per_t));
  const long long need = per_t * Tc + halo_f;
  if (need > n->scratch_cap) {
    if (n->scratch) cudaFree(n->scratch);
    n->scratch = nullptr, n->scratch_cap = 0;
    D2D_CUDA(cudaMalloc((void**)&n->scratch, (size_t)need * 4));
    n->scratch_cap = need;
  }
  c.Tc = Tc, c.halo = halo;
  float* p = n->scratch;
  auto take = [&](long long f) { float* q = p; p += f; return q; };
  const long long H = n->H, O = n->O, L = n->L;
  c.gi = c.gh = c.acts = c.hs = c.dl = c.dy1 = c.dh0 = c.dh1 = c.dgi = nullptr;
  if (n->arch == D2D_NET_GRU) {
    c.gi = take((long long)(Tc + halo) * 3 * H * NB);
    c.gh = take((long long)Tc * 3 * H * NB);
    if (train) {
      c.hs = take((long long)L * Tc * H * NB);
      if (c.plan.bptt != Bptt::kRecompute) c.acts = take((long long)L * Tc * 4 * H * NB);
    } else {
      c.hs = take((long long)2 * Tc * H * NB);
    }
  }
  c.y1 = take((long long)Tc * H * NB);
  c.y2 = c.dy2 = nullptr;
  if (n->head2) c.y2 = take((long long)Tc * H * NB);
  c.logits = take((long long)Tc * O * NB);
  if (train) {
    c.dl = take((long long)Tc * O * NB);
    c.dy1 = take((long long)Tc * H * NB);
    if (n->head2) c.dy2 = take((long long)Tc * H * NB);
    if (n->arch == D2D_NET_GRU) {
      c.dh0 = take((long long)Tc * H * NB);
      c.dh1 = take((long long)Tc * H * NB);
      c.dgi = take((long long)(Tc + halo) * 3 * H * NB);
    }
  }
  return D2D_OK;
}

// hidden state buffer of window step s for the chunk (training keeps all L of them)
static float* hs_ptr(const d2d_net* n, const Chunk& c, bool train, int s) {
  const long long per = (long long)c.Tc * n->H * n->N * n->B;
  return c.hs + per * (train ? s : (s & 1));
}

// network head on the CUDA-core dense kernels: y1 = relu(W1 last + b1) [, y2 = relu(W1b y1 + b1b)], out = W2 y + b2
static int head_dense(const d2d_net* n, const float* params, const View& last, const View& y1, float* y2p,
                      const View& lg, int t0, int t1, cudaStream_t s) {
  const int H = n->H, O = n->O;
  const long long NB = (long long)n->N * n->B;
  Wt w1{&n->o_w1, &n->o_b1, nullptr, H, H};
  Wt w2{&n->o_w2, &n->o_b2, nullptr, H, O};
  if (n->arch == D2D_NET_MLP) w1.in_dim = &n->in_dim;
  int rc;
  {
    DenseArgs a;
    memset(&a, 0, sizeof(a));
    fill_dense_w(n, a, params, w1, 0);
    a.x = last, a.y = y1, a.epilogue = kEpiRelu, a.t0 = t0, a.t1 = t1;
    if ((rc = launch_dense(n, a, n->arch == D2D_NET_MLP ? n->max_in : H, s))) return rc;
  }
  View top = y1;
  if (n->head2) {
    Wt w1b{&n->o_w1b, &n->o_b1b, nullptr, H, H};
    top = make_view(y2p, H * NB, -t0, n->N, H, n->B);
    DenseArgs a;
    memset(&a, 0, sizeof(a));
    fill_dense_w(n, a, params, w1b, 0);
    a.x = y1, a.y = top, a.epilogue = kEpiRelu, a.t0 = t0, a.t1 = t1;
    if ((rc = launch_dense(n, a, H, s))) return rc;
  }
  DenseArgs a;
  memset(&a, 0, sizeof(a));
  fill_dense_w(n, a, params, w2, 0);
  a.x = top, a.y = lg, a.epilogue = kEpiNone, a.t0 = t0, a.t1 = t1;
  return launch_dense(n, a, H, s);
}

// forward of chunk [c0, c1) (c1 - c0 <= Tc): fills c.logits (local time index t - c0)
static int forward_chunk(d2d_net* n, const float* params, const float* x, int x_lead, int c0, int c1, int padded,
                         bool train, const Chunk& c, cudaStream_t s) {
  const int N = n->N, B = n->B, H = n->H, O = n->O;
  const long long NB = (long long)N * B;
  const View xin = input_view(n, x, x_lead);
  const View y1 = make_view(c.y1, H * NB, -c0, N, H, B);
  const View lg = make_view(c.logits, O * NB, -c0, N, O, B);
  int rc;
  View last = xin;
  if (n->arch == D2D_NET_GRU) {
    const int L = n->L, halo = c.halo;
    if (c.plan.window_tc) {   // tcgen05 fused window (gru_tc.cuh); training windows are padded and keep every step's h
      const bool head = c.plan.head == Head::kWindow;   // window + head (+ y1 when training) in one launch
      const View hl = make_view(hs_ptr(n, c, train, L - 1), H * NB, -c0, N, H, B);
      const View hv = make_view(c.hs, H * NB, -c0, N, H, B);
      const View av = make_view(c.acts, 4 * H * NB, -c0, N, 4 * H, B);   // c.acts null: the BPTT recomputes the gates
      rc = launch_gru_tc(n, params, xin, hl, c0, c1, padded, s, train ? &hv : nullptr, train ? &av : nullptr,
                         (long long)c.Tc * H * NB, head ? &lg : nullptr, head && train ? &y1 : nullptr, nullptr);
      if (rc || head) return rc;
    } else {
      // input projections of every observation the chunk's windows touch: times [c0 - halo, c1)
      const View gi = make_view(c.gi, 3 * H * NB, -(c0 - halo), N, 3 * H, B);
      {
        DenseArgs a;
        memset(&a, 0, sizeof(a));
        Wt wih{&n->o_wih, &n->o_bih, &n->in_dim, 0, 3 * H};
        fill_dense_w(n, a, params, wih, 0);
        a.x = xin, a.y = gi, a.epilogue = kEpiNone, a.t0 = c0 - halo, a.t1 = c1;
        if ((rc = launch_dense(n, a, n->max_in, s, n->x_exact))) return rc;
      }
      const View gh = make_view(c.gh, 3 * H * NB, -c0, N, 3 * H, B);
      for (int st = 0; st < L; ++st) {
        const View hprev = make_view(hs_ptr(n, c, train, st - 1 < 0 ? 0 : st - 1), H * NB, -c0, N, H, B);
        const View hout = make_view(hs_ptr(n, c, train, st), H * NB, -c0, N, H, B);
        if (B % 4 == 0 && H <= 128) {   // fused hidden projection + gates (a register tile covers 64 units; H > 64: 2 launches)
          GruStepArgs fa;
          memset(&fa, 0, sizeof(fa));
          fa.h_prev = hprev, fa.h_out = hout, fa.gi = gi, fa.gi.t_off = gi.t_off - (L - 1 - st);
          if (train) fa.acts = make_view(c.acts + (long long)st * c.Tc * 4 * H * NB, 4 * H * NB, -c0, N, 4 * H, B);
          fa.t0 = c0, fa.t1 = c1, fa.back = L - 1 - st, fa.padded = padded, fa.first = st == 0, fa.store = train;
          if ((rc = launch_gru_step(n, fa, params, s))) return rc;
          continue;
        }
        {
          DenseArgs a;
          memset(&a, 0, sizeof(a));
          Wt whh{&n->o_whh, &n->o_bhh, nullptr, st == 0 ? 0 : H, 3 * H};   // step 0: h = 0, gh = b_hh
          fill_dense_w(n, a, params, whh, 0);
          for (int g = 0; g < N; ++g) a.w_ld[g] = H;
          a.x = hprev, a.y = gh, a.epilogue = kEpiNone, a.t0 = c0, a.t1 = c1;
          if ((rc = launch_dense(n, a, H, s))) return rc;
        }
        GateArgs ga;
        memset(&ga, 0, sizeof(ga));
        ga.gi = gi, ga.gi.t_off = gi.t_off - (L - 1 - st);
        ga.gh = gh, ga.h_prev = hprev, ga.h_out = hout;
        if (train) ga.acts = make_view(c.acts + (long long)st * c.Tc * 4 * H * NB, 4 * H * NB, -c0, N, 4 * H, B);
        ga.H = H, ga.B = B, ga.t0 = c0, ga.t1 = c1, ga.back = L - 1 - st, ga.padded = padded, ga.first = st == 0;
        ga.store = train, ga.t_episode0 = 0;
        if ((rc = launch_gate(ga, N, false, s))) return rc;
      }
    }
    last = make_view(hs_ptr(n, c, train, L - 1), H * NB, -c0, N, H, B);
  }
  if (c.plan.head == Head::kKernel) return launch_head_fused(n, params, last, train ? c.y1 : nullptr, lg, c0, c1, s);
  return head_dense(n, params, last, y1, c.y2, lg, c0, c1, s);
}

// backward of chunk [c0, c1) given c.dl = d(loss)/d(pre-activation outputs); accumulates into grads
static int backward_chunk(d2d_net* n, const float* params, const float* x, int x_lead, int c0, int c1,
                          const Chunk& c, float* grads, float inv_rows, cudaStream_t s) {
  const int N = n->N, B = n->B, H = n->H, O = n->O;
  const long long NB = (long long)N * B;
  const View xin = input_view(n, x, x_lead);
  const View y1 = make_view(c.y1, H * NB, -c0, N, H, B);
  const View dl = make_view(c.dl, O * NB, -c0, N, O, B);
  const View dy1 = make_view(c.dy1, H * NB, -c0, N, H, B);
  Wt w1{&n->o_w1, &n->o_b1, nullptr, H, H};
  Wt w2{&n->o_w2, &n->o_b2, nullptr, H, O};
  int rc;
  if (n->head2) {
    // Q-network head: dW2 = dl^T y2 ; dy2 = (dl W2) * relu'(y2) ; dW1b = dy2^T y1 ; dy1 = (dy2 W1b) * relu'(y1)
    const View y2 = make_view(c.y2, H * NB, -c0, N, H, B);
    const View dy2 = make_view(c.dy2, H * NB, -c0, N, H, B);
    Wt w1b{&n->o_w1b, &n->o_b1b, nullptr, H, H};
    if ((rc = launch_wgrad(n, dl, y2, w2, false, grads, c0, c1, s))) return rc;
    {
      DenseArgs a;
      memset(&a, 0, sizeof(a));
      fill_dense_w(n, a, params, w2, 1);
      a.out_dim = H;
      a.x = dl, a.y = dy2, a.aux = y2, a.epilogue = kEpiReluBwd, a.t0 = c0, a.t1 = c1;
      if ((rc = launch_dense(n, a, O, s))) return rc;
    }
    if ((rc = launch_wgrad(n, dy2, y1, w1b, false, grads, c0, c1, s))) return rc;
    DenseArgs a;
    memset(&a, 0, sizeof(a));
    fill_dense_w(n, a, params, w1b, 1);
    a.out_dim = H;
    a.x = dy2, a.y = dy1, a.aux = y1, a.epilogue = kEpiReluBwd, a.t0 = c0, a.t1 = c1;
    if ((rc = launch_dense(n, a, H, s))) return rc;
  } else {
    // head: dW2 = dl^T y1 ; dy1 = (dl W2) * relu'(y1)
    if ((rc = launch_wgrad(n, dl, y1, w2, false, grads, c0, c1, s))) return rc;
    DenseArgs a;
    memset(&a, 0, sizeof(a));
    fill_dense_w(n, a, params, w2, 1);
    a.out_dim = H;
    a.x = dl, a.y = dy1, a.aux = y1, a.epilogue = kEpiReluBwd, a.t0 = c0, a.t1 = c1;
    if ((rc = launch_dense(n, a, O, s))) return rc;
  }
  if (n->arch == D2D_NET_MLP) {
    w1.in_dim = &n->in_dim;
    return launch_wgrad(n, dy1, xin, w1, false, grads, c0, c1, s, true);
  }
  const int L = n->L, halo = c.halo;
  const View hlast = make_view(hs_ptr(n, c, true, L - 1), H * NB, -c0, N, H, B);
  if ((rc = launch_wgrad(n, dy1, hlast, w1, false, grads, c0, c1, s))) return rc;
  float* dh_cur = c.dh0;
  float* dh_nxt = c.dh1;
  {
    DenseArgs a;   // d(h_last) = dy1 W1
    memset(&a, 0, sizeof(a));
    fill_dense_w(n, a, params, w1, 1);
    a.out_dim = H;
    a.x = dy1, a.y = make_view(dh_cur, H * NB, -c0, N, H, B), a.epilogue = kEpiNone, a.t0 = c0, a.t1 = c1;
    if ((rc = launch_dense(n, a, H, s))) return rc;
  }
  D2D_CUDA(cudaMemsetAsync(c.dgi, 0, (size_t)(c.Tc + halo) * 3 * H * NB * 4, s));
  const View dgi = make_view(c.dgi, 3 * H * NB, -(c0 - halo), N, 3 * H, B);
  const View dgh = make_view(c.gh, 3 * H * NB, -c0, N, 3 * H, B);
  Wt whh{&n->o_whh, &n->o_bhh, nullptr, H, 3 * H};
  if (c.plan.bptt != Bptt::kFp32) {
    // one kernel walks the whole window backwards (d(h) in registers, d(gh) W_hh on tcgen05) and accumulates d(gi) per
    // observation and dW_hh / db_hh per CTA
    int strips = 0;
    if (c.plan.bptt == Bptt::kRecompute) {
      // gru_bptt_tc RECOMPUTES every step's gates from (x, h_prev) on the tensor cores: the forward kept only h
      GruBpttArgs ba;
      memset(&ba, 0, sizeof(ba));
      ba.x = xin;
      ba.hs = make_view(c.hs, H * NB, -c0, N, H, B);
      ba.dh = make_view(dh_cur, H * NB, -c0, N, H, B);
      ba.dgi = dgi;
      ba.w = params, ba.w_agent_stride = n->stride;
      for (int g = 0; g < N; ++g) {
        ba.wih_off[g] = n->o_wih[g], ba.whh_off[g] = n->o_whh[g], ba.bih_off[g] = n->o_bih[g], ba.bhh_off[g] = n->o_bhh[g];
        ba.in_dim[g] = n->in_dim[g];
      }
      ba.hs_step = (long long)c.Tc * H * NB;
      // d(gh) ~ 1 / rows (the loss is a mean): the kernel scales it into the fp16 range by a power of two taken from
      // the largest |dh| of the chunk
      {
        unsigned int* amax = reinterpret_cast<unsigned int*>(n->partial + (long long)n->N * n->n_strips * n->part_stride);
        D2D_CUDA(cudaMemsetAsync(amax, 0, 4, s));
        const long long cnt = (long long)(c1 - c0) * H * NB;
        absmax_kernel<<<grid_for(cnt, 256), 256, 0, s>>>(dh_cur, cnt, amax);
        D2D_LAUNCHED();
        ba.dh_absmax = reinterpret_cast<const float*>(amax);
      }
      (void)inv_rows;
      ba.L = L, ba.B = B, ba.t0 = c0, ba.t1 = c1;
      ba.partial = n->partial, ba.part_stride = n->part_stride;
      rc = n->H == 32 ? launch_gru_bptt_tc_h<32>(n, ba, s, &strips) : launch_gru_bptt_tc_h<64>(n, ba, s, &strips);
    } else {
      // gru_bwd_tc reads the gates the forward stored; it leaves d(gh) of step s in the first 3H features of that
      // step's activation block
      GruBwdTcArgs ba;
      memset(&ba, 0, sizeof(ba));
      ba.acts = make_view(c.acts, 4 * H * NB, -c0, N, 4 * H, B);
      ba.hs = make_view(c.hs, H * NB, -c0, N, H, B);
      ba.dh = make_view(dh_cur, H * NB, -c0, N, H, B);
      ba.dgi = dgi;
      ba.w = params, ba.w_agent_stride = n->stride;
      for (int g = 0; g < N; ++g) ba.whh_off[g] = n->o_whh[g];
      ba.acts_step = (long long)c.Tc * 4 * H * NB, ba.hs_step = (long long)c.Tc * H * NB;
      ba.L = L, ba.B = B, ba.t0 = c0, ba.t1 = c1;
      ba.partial = n->partial, ba.part_stride = n->part_stride;
      rc = n->H == 32 ? launch_gru_bwd_tc_h<32>(n, ba, s, &strips) : launch_gru_bwd_tc_h<64>(n, ba, s, &strips);
    }
    if (rc) return rc;
    if (strips > 0 && (rc = launch_wreduce(n, whh, false, strips, grads, s))) return rc;
  }
  for (int st = L - 1; st >= 0 && c.plan.bptt == Bptt::kFp32; --st) {
    const View hprev = make_view(hs_ptr(n, c, true, st - 1 < 0 ? 0 : st - 1), H * NB, -c0, N, H, B);
    GateArgs ga;
    memset(&ga, 0, sizeof(ga));
    ga.gh = dgh, ga.h_prev = hprev;
    ga.h_out = make_view(dh_nxt, H * NB, -c0, N, H, B);
    ga.dh = make_view(dh_cur, H * NB, -c0, N, H, B);
    ga.acts = make_view(c.acts + (long long)st * c.Tc * 4 * H * NB, 4 * H * NB, -c0, N, 4 * H, B);
    ga.dgi = dgi, ga.dgi.t_off = dgi.t_off - (L - 1 - st);
    ga.H = H, ga.B = B, ga.t0 = c0, ga.t1 = c1, ga.back = L - 1 - st, ga.padded = 1, ga.first = st == 0;
    if ((rc = launch_gate(ga, N, true, s))) return rc;
    // dW_hh += d(gh)^T h_{s-1}, db_hh += sum d(gh)   (h_{-1} = 0: bias only)
    if ((rc = launch_wgrad(n, dgh, hprev, whh, st == 0, grads, c0, c1, s))) return rc;
    if (st > 0) {
      DenseArgs a;   // d(h_{s-1}) += d(gh) W_hh
      memset(&a, 0, sizeof(a));
      fill_dense_w(n, a, params, whh, 1);
      a.out_dim = H;
      a.x = dgh, a.y = make_view(dh_nxt, H * NB, -c0, N, H, B), a.epilogue = kEpiAccum, a.t0 = c0, a.t1 = c1;
      if ((rc = launch_dense(n, a, 3 * H, s))) return rc;
    }
    std::swap(dh_cur, dh_nxt);
  }
  // dW_ih = d(gi)^T x over every observation the chunk touched (zero observations before t = 0 feed b_ih only)
  Wt wih{&n->o_wih, &n->o_bih, &n->in_dim, 0, 3 * H};
  return launch_wgrad(n, dgi, xin, wih, false, grads, c0 - halo, c1, s, true);
}

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" int d2d_net_create(const d2d_net_config* cfg, d2d_net** out) {
  D2D_REQUIRE(cfg && out, "d2d_net_create: null argument");
  *out = nullptr;
  D2D_REQUIRE(cfg->arch == D2D_NET_MLP || cfg->arch == D2D_NET_GRU, "d2d_net_create: unknown arch");
  D2D_REQUIRE(cfg->out_kind >= 0 && cfg->out_kind <= 2, "d2d_net_create: unknown out_kind");
  D2D_REQUIRE(cfg->n_agents >= 1 && cfg->n_agents <= D2D_MAX_AGENTS, "d2d_net_create: n_agents out of range");
  D2D_REQUIRE(cfg->n_envs >= 1, "d2d_net_create: n_envs must be positive");
  D2D_REQUIRE(cfg->hidden >= 1 && cfg->hidden <= 128, "d2d_net_create: hidden size %d not in 1..128 (this build)",
              cfg->hidden);
  D2D_REQUIRE(cfg->n_out >= 1 && cfg->n_out <= kMaxOut, "d2d_net_create: n_out not in 1..%d", kMaxOut);
  D2D_REQUIRE(cfg->arch == D2D_NET_MLP || (cfg->history_len >= 1 && cfg->history_len <= 64),
              "d2d_net_create: history_len out of range");
  D2D_REQUIRE(cfg->in_dim && cfg->in_off, "d2d_net_create: null in_dim / in_off");
  D2D_REQUIRE(cfg->head_layers >= 0 && cfg->head_layers <= 2 && (cfg->head_layers != 2 || cfg->arch == D2D_NET_GRU),
              "d2d_net_create: head_layers must be 0 / 1 (PPO nets) or 2 (GRU Q-network)");
  d2d_net* n = new (std::nothrow) d2d_net();
  D2D_REQUIRE(n, "d2d_net_create: out of host memory");
  n->arch = cfg->arch, n->out_kind = cfg->out_kind, n->N = cfg->n_agents, n->B = cfg->n_envs, n->H = cfg->hidden;
  n->O = cfg->n_out, n->L = cfg->arch == D2D_NET_GRU ? cfg->history_len : 1, n->in_rows = cfg->in_rows;
  n->scratch_bytes = cfg->scratch_bytes > 0 ? cfg->scratch_bytes : (2ll << 30);
  n->x_exact = cfg->inputs_bf16_exact != 0;
  n->head2 = cfg->head_layers == 2;
  n->max_in = 0, n->stride = 0;
  const int H = n->H, O = n->O;
  for (int g = 0; g < n->N; ++g) {
    const int I = cfg->in_dim[g];
    if (I < 1 || I > 128 || cfg->in_off[g] < 0 || cfg->in_off[g] + I > cfg->in_rows) {
      set_error("d2d_net_create: agent %d input rows [%d, %d) invalid (in_rows %d, max 128 inputs)", g,
                cfg->in_off[g], cfg->in_off[g] + I, cfg->in_rows);
      delete n;
      return D2D_ERR_INVALID;
    }
    n->in_dim.push_back(I), n->in_off.push_back(cfg->in_off[g]);
    n->max_in = std::max(n->max_in, I);
    int o = 0;
    if (n->arch == D2D_NET_GRU) {
      n->o_wih.push_back(o), o += 3 * H * I;
      n->o_whh.push_back(o), o += 3 * H * H;
      n->o_bih.push_back(o), o += 3 * H;
      n->o_bhh.push_back(o), o += 3 * H;
      n->o_w1.push_back(o), o += H * H;
    } else {
      n->o_w1.push_back(o), o += H * I;
    }
    n->o_b1.push_back(o), o += H;
    if (n->head2) {
      n->o_w1b.push_back(o), o += H * H;
      n->o_b1b.push_back(o), o += H;
    }
    n->o_w2.push_back(o), o += O * H;
    n->o_b2.push_back(o), o += O;
    n->stride = std::max<long long>(n->stride, o);
  }
  n->n_strips = 64;
  n->part_stride = (long long)std::max(3 * H, std::max(H, O)) * std::max(n->max_in, 3 * H) + 3 * H + 64;
  cudaError_t e = cudaMalloc((void**)&n->partial, (size_t)n->N * n->n_strips * n->part_stride * 4 + 64);   // + scalars
  if (e != cudaSuccess) {
    set_error("d2d_net_create: cudaMalloc failed: %s", cudaGetErrorString(e));
    delete n;
    return D2D_ERR_CUDA;
  }
  *out = n;
  return D2D_OK;
}

extern "C" int d2d_net_destroy(d2d_net* n) {
  if (!n) return D2D_OK;
  cudaFree(n->scratch), cudaFree(n->partial), cudaFree(n->gi_ring);
  delete n;
  return D2D_OK;
}
extern "C" int64_t d2d_net_param_stride(const d2d_net* n) { return n ? n->stride : D2D_ERR_INVALID; }
extern "C" int d2d_net_num_tensors(const d2d_net* n) {
  return n ? (n->arch == D2D_NET_GRU ? (n->head2 ? 10 : 8) : 4) : D2D_ERR_INVALID;
}
extern "C" int d2d_net_tensor(const d2d_net* n, int g, int index, int64_t* offset, int32_t* rows, int32_t* cols) {
  D2D_REQUIRE(n && offset && rows && cols && g >= 0 && g < n->N, "d2d_net_tensor: bad argument");
  const int H = n->H, O = n->O, I = n->in_dim[g];
  if (n->arch == D2D_NET_GRU && n->head2) {
    // irdqn.py:58-72 state_dict order: the four GRU tensors, layers.0, layers.2 (hidden), layers.4 (output)
    const int off[10] = {n->o_wih[g], n->o_whh[g], n->o_bih[g], n->o_bhh[g], n->o_w1[g],
                         n->o_b1[g],  n->o_w1b[g], n->o_b1b[g], n->o_w2[g],  n->o_b2[g]};
    const int r[10] = {3 * H, 3 * H, 3 * H, 3 * H, H, H, H, H, O, O};
    const int c[10] = {I, H, 1, 1, H, 1, H, 1, H, 1};
    D2D_REQUIRE(index >= 0 && index < 10, "d2d_net_tensor: index out of range");
    *offset = off[index], *rows = r[index], *cols = c[index];
  } else if (n->arch == D2D_NET_GRU) {
    // state_dict order: weight_ih, weight_hh, bias_ih, bias_hh, layers.0.weight, layers.0.bias, layers.2.weight, .bias
    const int off[8] = {n->o_wih[g], n->o_whh[g], n->o_bih[g], n->o_bhh[g], n->o_w1[g], n->o_b1[g], n->o_w2[g], n->o_b2[g]};
    const int r[8] = {3 * H, 3 * H, 3 * H, 3 * H, H, H, O, O};
    const int c[8] = {I, H, 1, 1, H, 1, H, 1};
    D2D_REQUIRE(index >= 0 && index < 8, "d2d_net_tensor: index out of range");
    *offset = off[index], *rows = r[index], *cols = c[index];
  } else {
    const int off[4] = {n->o_w1[g], n->o_b1[g], n->o_w2[g], n->o_b2[g]};
    const int r[4] = {H, H, O, O};
    const int c[4] = {I, 1, H, 1};
    D2D_REQUIRE(index >= 0 && index < 4, "d2d_net_tensor: index out of range");
    *offset = off[index], *rows = r[index], *cols = c[index];
  }
  return D2D_OK;
}

static int check_range(const d2d_net* n, int x_lead, int t0, int t1, const char* who) {
  D2D_REQUIRE(t0 >= 0 && t1 > t0, "%s: empty or negative time range [%d, %d)", who, t0, t1);
  D2D_REQUIRE(n->arch == D2D_NET_MLP || x_lead >= n->L - 1,
              "%s: GRU inputs need x_lead >= history_len - 1 zero blocks before time 0", who);
  D2D_REQUIRE(x_lead >= 0, "%s: negative x_lead", who);
  return D2D_OK;
}

extern "C" int d2d_net_forward(d2d_net* n, const float* params, const float* x, int x_lead, int t0, int t1,
                               int padded, float* out, void* stream) {
  D2D_REQUIRE(n && params && x && out, "d2d_net_forward: null argument");
  int rc = check_range(n, x_lead, t0, t1, "d2d_net_forward");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  Chunk c;
  if ((rc = plan_chunk(n, false, t1 - t0, c))) return rc;
  const long long per_t = (long long)n->N * n->O * n->B;
  for (int c0 = t0; c0 < t1; c0 += c.Tc) {
    const int c1 = std::min(t1, c0 + c.Tc);
    if ((rc = forward_chunk(n, params, x, x_lead, c0, c1, padded, false, c, s))) return rc;
    D2D_CUDA(cudaMemcpyAsync(out + (long long)(c0 - t0) * per_t, c.logits, (size_t)(c1 - c0) * per_t * 4,
                             cudaMemcpyDeviceToDevice, s));
  }
  return D2D_OK;
}

// Guard of the `inputs_bf16_exact` promise (d2d_net_config): the tensor-core GRU window stages the observations as ONE
// bf16 plane (the top 16 bits of the fp32 word), so an input with more than 8 significant bits would silently be
// truncated.  Counts such inputs over time blocks [t0, t1) of every agent's rows.
extern "C" int d2d_net_check_inputs(const d2d_net* n, const float* x, int x_lead, int t0, int t1,
                                    unsigned long long* n_inexact, void* stream) {
  D2D_REQUIRE(n && x && n_inexact && t1 > t0 && x_lead + t0 >= 0, "d2d_net_check_inputs: bad argument");
  cudaStream_t s = as_stream(stream);
  D2D_CUDA(cudaMemsetAsync(n_inexact, 0, sizeof(unsigned long long), s));
  for (int g = 0; g < n->N; ++g) {
    const long long count = (long long)n->in_dim[g] * n->B;
    const float* base = x + ((long long)(x_lead + t0) * n->in_rows + n->in_off[g]) * n->B;
    check_bf16_exact_kernel<<<dim3(grid_for(count, 256, 4096), t1 - t0), 256, 0, s>>>(base, count,
                                                                                       (long long)n->in_rows * n->B,
                                                                                       n_inexact);
    D2D_LAUNCHED();
  }
  return D2D_OK;
}

extern "C" int d2d_net_rollout_step(d2d_net* n, const float* params, const float* x, int x_lead, int t, float* out,
                                    void* stream) {
  D2D_REQUIRE(n && params && x && out, "d2d_net_rollout_step: null argument");
  if (n->arch == D2D_NET_MLP || n->B % 4 != 0 || n->H > 128)
    return d2d_net_forward(n, params, x, x_lead, t, t + 1, 0, out, stream);
  int rc = check_range(n, x_lead, t, t + 1, "d2d_net_rollout_step");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  const int N = n->N, B = n->B, H = n->H, O = n->O, L = n->L;
  const long long NB = (long long)N * B;
  Chunk c;
  if ((rc = plan_chunk(n, false, 1, c))) return rc;
  const View xin = input_view(n, x, x_lead);
  const View hl = make_view(hs_ptr(n, c, false, L - 1), H * NB, -t, N, H, B);
  const View lg = make_view(out, O * NB, -t, N, O, B);
  if (c.plan.window_tc) {   // the tensor-core window kernel re-reads the L observations (L x I floats per row): no ring
    const bool head = c.plan.head == Head::kWindow;   // window + head in ONE launch, outputs written in place
    rc = launch_gru_tc(n, params, xin, hl, t, t + 1, 0, s, nullptr, nullptr, 0, head ? &lg : nullptr, nullptr, nullptr);
    if (rc || head) return rc;
  } else {
    if (!n->gi_ring) D2D_CUDA(cudaMalloc((void**)&n->gi_ring, (size_t)L * 3 * H * NB * 4));
    {   // input projection of the NEW observation only; the previous L - 1 are still in the ring
      DenseArgs a;
      memset(&a, 0, sizeof(a));
      Wt wih{&n->o_wih, &n->o_bih, &n->in_dim, 0, 3 * H};
      fill_dense_w(n, a, params, wih, 0);
      a.x = xin, a.y = make_view(n->gi_ring, 3 * H * NB, (t % L) - t, N, 3 * H, B), a.epilogue = kEpiNone;
      a.t0 = t, a.t1 = t + 1;
      if ((rc = launch_dense(n, a, n->max_in, s))) return rc;
    }
    for (int st = 0; st < L; ++st) {
      const int back = L - 1 - st;
      if (t - back < 0 && st < L - 1) continue;   // the step does not exist and h stays zero: nothing to do
      GruStepArgs fa;
      memset(&fa, 0, sizeof(fa));
      const bool first = (t - back <= 0) || st == 0;   // first EXISTING step starts from h = 0
      fa.h_prev = make_view(hs_ptr(n, c, false, st - 1 < 0 ? 0 : st - 1), H * NB, -t, N, H, B);
      fa.h_out = make_view(hs_ptr(n, c, false, st), H * NB, -t, N, H, B);
      fa.gi = make_view(n->gi_ring, 3 * H * NB, -back, N, 3 * H, B);
      fa.t_mod_gi = L;
      fa.t0 = t, fa.t1 = t + 1, fa.back = back, fa.padded = 0, fa.first = first, fa.store = 0;
      if ((rc = launch_gru_step(n, fa, params, s))) return rc;
    }
  }
  if (c.plan.head == Head::kKernel) return launch_head_fused(n, params, hl, nullptr, lg, t, t + 1, s);
  return head_dense(n, params, hl, make_view(c.y1, H * NB, -t, N, H, B), c.y2, lg, t, t + 1, s);
}

static void fill_head(HeadArgs& h, int N, int B, int O, int out_kind, int dist_kind) {
  memset(&h, 0, sizeof(h));
  h.A = O, h.B = B, h.n_agents = N, h.out_kind = out_kind, h.dist_kind = dist_kind;
  h.mask_bytes = O <= 8 ? 1 : (O <= 16 ? 2 : 4);
  h.act_t_stride = (long long)N * B;
}

extern "C" int d2d_policy_head(int N, int B, int O, int n_t, int out_kind, int dist_kind, int act_mode,
                               const float* logits, void* actions, float* logp, float* entropy, float* probs,
                               uint64_t seed, uint64_t env_offset, int t_abs0, void* stream) {
  D2D_REQUIRE(logits && actions, "d2d_policy_head: null logits or actions");
  D2D_REQUIRE(N >= 1 && N <= D2D_MAX_AGENTS && B >= 1 && O >= 1 && O <= kMaxOut && n_t >= 1,
              "d2d_policy_head: bad shape");
  D2D_REQUIRE(act_mode >= 0 && act_mode <= 2 && (dist_kind == 0 || dist_kind == 1) && out_kind >= 0 && out_kind <= 2,
              "d2d_policy_head: bad mode");
  HeadArgs h;
  fill_head(h, N, B, O, out_kind, dist_kind);
  h.logits = make_view(const_cast<float*>(logits), (long long)N * O * B, 0, N, O, B);
  if (probs) h.probs = make_view(probs, (long long)N * O * B, 0, N, O, B);
  h.t0 = 0, h.t1 = n_t, h.act_mode = act_mode, h.actions = actions, h.logp = logp, h.entropy = entropy;
  h.k0 = (uint32_t)(seed & 0xFFFFFFFFull), h.k1 = (uint32_t)(seed >> 32), h.env_offset = (uint32_t)env_offset;
  h.t_abs_off = t_abs0;
  const long long rows = (long long)n_t * B;
  policy_head_kernel<<<dim3(grid_for(rows, 128), N), 128, 0, as_stream(stream)>>>(h);
  D2D_LAUNCHED();
  return D2D_OK;
}

// PPO.select_action for all agents at time t in as few launches as possible: GRU window + head + action selection +
// log-prob in ONE kernel when the tensor-core window kernel takes the net, else rollout_step + policy_head
extern "C" int d2d_net_rollout_act(d2d_net* n, const float* params, const float* x, int x_lead, int t, int dist_kind,
                                   int act_mode, void* actions, float* logp, uint64_t seed, uint64_t env_offset,
                                   int t_abs0, float* logits_out, void* stream) {
  D2D_REQUIRE(n && params && x && actions && logp, "d2d_net_rollout_act: null argument");
  D2D_REQUIRE(n->out_kind != D2D_OUT_IDENTITY, "d2d_net_rollout_act: net has no probability output");
  D2D_REQUIRE(act_mode >= 0 && act_mode <= 2 && (dist_kind == 0 || dist_kind == 1), "d2d_net_rollout_act: bad mode");
  int rc = check_range(n, x_lead, t, t + 1, "d2d_net_rollout_act");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  const int N = n->N, B = n->B, H = n->H, O = n->O;
  const long long NB = (long long)N * B;
  Chunk c;
  if ((rc = plan_chunk(n, false, 1, c))) return rc;
  if (c.plan.head == Head::kWindow && O > 1 && n->B % 4 == 0) {
    HeadArgs h;
    fill_head(h, N, B, O, n->out_kind, dist_kind);
    h.act_mode = act_mode, h.actions = actions, h.logp = logp, h.act_t_off = -t;
    h.k0 = (uint32_t)(seed & 0xFFFFFFFFull), h.k1 = (uint32_t)(seed >> 32), h.env_offset = (uint32_t)env_offset;
    h.t_abs_off = t_abs0 - t;
    const View hl = make_view(hs_ptr(n, c, false, n->L - 1), H * NB, -t, N, H, B);
    const View lgo = make_view(logits_out, O * NB, -t, N, O, B);   // p == nullptr: outputs are not written
    const DistArgs sel = h;
    return launch_gru_tc(n, params, input_view(n, x, x_lead), hl, t, t + 1, 0, s, nullptr, nullptr, 0, &lgo, nullptr,
                         &sel);
  }
  // generic path: outputs into the chunk scratch (or the caller's buffer), then the head kernel
  float* lg = logits_out ? logits_out : c.logits;
  if ((rc = d2d_net_rollout_step(n, params, x, x_lead, t, lg, stream))) return rc;
  return d2d_policy_head(N, B, O, 1, n->out_kind, dist_kind, act_mode, lg, actions, logp, nullptr, nullptr, seed,
                         env_offset, t_abs0, stream);
}

extern "C" int d2d_ppo_policy_grad(d2d_net* n, const float* params, const float* x, int x_lead, int t0, int t1,
                                   int dist_kind, const void* actions, const float* logp_old, const float* weight,
                                   int weight_per_agent, const int32_t* cycle, float inv_rows, float cliprange,
                                   float beta, float* grads, double* loss_sums, float* ratio_out, void* stream) {
  D2D_REQUIRE(n && params && x && actions && logp_old && weight && grads && loss_sums,
              "d2d_ppo_policy_grad: null argument");
  D2D_REQUIRE(n->out_kind != D2D_OUT_IDENTITY, "d2d_ppo_policy_grad: net has no probability output");
  int rc = check_range(n, x_lead, t0, t1, "d2d_ppo_policy_grad");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  Chunk c;
  if ((rc = plan_chunk(n, true, t1 - t0, c))) return rc;
  const long long NB = (long long)n->N * n->B;
  for (int c0 = t0; c0 < t1; c0 += c.Tc) {
    const int c1 = std::min(t1, c0 + c.Tc);
    if ((rc = forward_chunk(n, params, x, x_lead, c0, c1, 1, true, c, s))) return rc;
    HeadArgs h;
    fill_head(h, n->N, n->B, n->O, n->out_kind, dist_kind);
    h.logits = make_view(c.logits, n->O * NB, -c0, n->N, n->O, n->B);
    h.dlogits = make_view(c.dl, n->O * NB, -c0, n->N, n->O, n->B);
    h.t0 = c0, h.t1 = c1, h.actions = const_cast<void*>(actions), h.logp_old = logp_old, h.weight = weight;
    h.weight_per_agent = weight_per_agent, h.cycle = cycle, h.ratio_out = ratio_out, h.inv_rows = inv_rows;
    h.cliprange = cliprange, h.beta = beta, h.loss_sums = loss_sums;
    const long long rows = (long long)(c1 - c0) * n->B;
    ppo_dlogits_kernel<<<grid_for(rows, 128), 128, 0, s>>>(h);
    D2D_LAUNCHED();
    if ((rc = backward_chunk(n, params, x, x_lead, c0, c1, c, grads, inv_rows, s))) return rc;
  }
  return D2D_OK;
}

extern "C" int d2d_value_grad(d2d_net* n, const float* params, const float* x, int x_lead, int t0, int t1,
                              int padded, const float* target, int per_agent, float inv_rows, float* grads,
                              double* loss_sum, float* value_out, void* stream) {
  D2D_REQUIRE(n && params && x && target && grads && loss_sum, "d2d_value_grad: null argument");
  D2D_REQUIRE(n->O == 1 && n->out_kind == D2D_OUT_IDENTITY, "d2d_value_grad: net is not a critic (n_out 1, identity)");
  int rc = check_range(n, x_lead, t0, t1, "d2d_value_grad");
  if (rc) return rc;
  D2D_REQUIRE(padded == 1 || n->arch == D2D_NET_MLP, "d2d_value_grad: GRU critics train on padded windows");
  cudaStream_t s = as_stream(stream);
  Chunk c;
  if ((rc = plan_chunk(n, true, t1 - t0, c))) return rc;
  const long long NB = (long long)n->N * n->B;
  for (int c0 = t0; c0 < t1; c0 += c.Tc) {
    const int c1 = std::min(t1, c0 + c.Tc);
    if ((rc = forward_chunk(n, params, x, x_lead, c0, c1, 1, true, c, s))) return rc;
    MseArgs m;
    memset(&m, 0, sizeof(m));
    m.value = make_view(c.logits, NB, -c0, n->N, 1, n->B);
    m.dvalue = make_view(c.dl, NB, -c0, n->N, 1, n->B);
    m.target = target, m.per_agent = per_agent, m.tgt_t_stride = per_agent ? NB : n->B, m.tgt_t_off = 0;
    m.B = n->B, m.t0 = c0, m.t1 = c1, m.inv_rows = inv_rows, m.loss_sum = loss_sum;
    m.value_out = value_out, m.out_t_stride = NB;
    const long long rows = (long long)(c1 - c0) * n->B;
    mse_dvalue_kernel<<<dim3(grid_for(rows, 128), n->N), 128, 0, s>>>(m);
    D2D_LAUNCHED();
    if ((rc = backward_chunk(n, params, x, x_lead, c0, c1, c, grads, inv_rows, s))) return rc;
  }
  return D2D_OK;
}

extern "C" int d2d_adam_step(float* params, float* m, float* v, const float* grads, int N, int64_t per_agent,
                             float lr, int step, float max_norm, double* sqnorm, void* stream) {
  return d2d_adam_step_eps(params, m, v, grads, N, per_agent, lr, 1e-8f, step, max_norm, sqnorm, stream);
}

extern "C" int d2d_adam_step_eps(float* params, float* m, float* v, const float* grads, int N, int64_t per_agent,
                                 float lr, float eps, int step, float max_norm, double* sqnorm, void* stream) {
  D2D_REQUIRE(params && m && v && grads && N >= 1 && per_agent >= 1 && step >= 1, "d2d_adam_step: bad argument");
  D2D_REQUIRE(max_norm <= 0.f || sqnorm, "d2d_adam_step: clipping needs the sqnorm scratch buffer");
  cudaStream_t s = as_stream(stream);
  const int gx = grid_for(per_agent, 256);
  if (max_norm > 0.f) {
    D2D_CUDA(cudaMemsetAsync(sqnorm, 0, sizeof(double) * N, s));
    grad_sqnorm_kernel<<<dim3(gx, N), 256, 0, s>>>(grads, per_agent, sqnorm);
    D2D_LAUNCHED();
  }
  AdamArgs a;
  a.p = params, a.m = m, a.v = v, a.g = grads, a.sqnorm = max_norm > 0.f ? sqnorm : nullptr;
  a.per_agent = per_agent, a.lr = lr, a.beta1 = 0.9f, a.beta2 = 0.999f, a.eps = eps, a.max_norm = max_norm;
  a.bc1 = (float)(1.0 - pow(0.9, (double)step));
  a.bc2 = (float)(1.0 - pow(0.999, (double)step));
  adam_kernel<<<dim3(gx, N), 256, 0, s>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

// ------------------------------------------------------------------------------------------------
// independent recurrent DQN (algorithms/irdqn.py)
// ------------------------------------------------------------------------------------------------
extern "C" int d2d_q_select(int N, int B, int O, const float* q, int act_mode, float epsilon, int training_ready,
                            int n_random, uint8_t* action_idx, void* action_mask, int mask_bytes, uint64_t seed,
                            uint64_t env_offset, int t_abs, void* stream) {
  D2D_REQUIRE(action_idx && (q || act_mode == D2D_ACT_GIVEN), "d2d_q_select: null argument");
  D2D_REQUIRE(N >= 1 && N <= D2D_MAX_AGENTS && B >= 1 && O >= 1 && O <= kMaxOut, "d2d_q_select: bad shape");
  D2D_REQUIRE(act_mode >= 0 && act_mode <= 2, "d2d_q_select: bad act_mode");
  D2D_REQUIRE(n_random >= 1 && n_random <= O, "d2d_q_select: n_random %d not in 1..n_out", n_random);
  D2D_REQUIRE(!action_mask || ((mask_bytes == 1 || mask_bytes == 2 || mask_bytes == 4) && O <= 8 * mask_bytes),
              "d2d_q_select: mask_bytes %d cannot hold %d channels", mask_bytes, O);
  QSelectArgs a;
  memset(&a, 0, sizeof(a));
  a.q = q, a.action = action_idx, a.mask = action_mask, a.mask_bytes = mask_bytes, a.N = N, a.B = B, a.O = O;
  a.act_mode = act_mode, a.epsilon = epsilon, a.ready = training_ready != 0, a.n_random = n_random;
  a.k0 = (uint32_t)(seed & 0xFFFFFFFFull), a.k1 = (uint32_t)(seed >> 32), a.env_offset = (uint32_t)env_offset;
  a.t_abs = t_abs;
  q_select_kernel<<<grid_for((long long)N * B, 128), 128, 0, as_stream(stream)>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_q_td_target(int N, int B, int O, const float* q_next, const int32_t* reward, const uint8_t* done,
                               float gamma, float* target, void* stream) {
  D2D_REQUIRE(q_next && reward && done && target, "d2d_q_td_target: null argument");
  D2D_REQUIRE(N >= 1 && N <= D2D_MAX_AGENTS && B >= 1 && O >= 1 && O <= kMaxOut, "d2d_q_td_target: bad shape");
  q_td_target_kernel<<<grid_for((long long)N * B, 128), 128, 0, as_stream(stream)>>>(q_next, reward, done, gamma,
                                                                                       target, N, B, O);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_q_grad(d2d_net* n, const float* params, const float* x, int x_lead, int t0, int t1,
                          const uint8_t* actions, const float* target, int loss_kind, float inv_rows, float* grads,
                          double* loss_sum, float* q_out, void* stream) {
  D2D_REQUIRE(n && params && x && actions && target && grads && loss_sum, "d2d_q_grad: null argument");
  D2D_REQUIRE(n->out_kind == D2D_OUT_IDENTITY, "d2d_q_grad: a Q-network has identity outputs");
  D2D_REQUIRE(loss_kind == D2D_QLOSS_HUBER || loss_kind == D2D_QLOSS_MSE, "d2d_q_grad: unknown loss_kind");
  int rc = check_range(n, x_lead, t0, t1, "d2d_q_grad");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  Chunk c;
  if ((rc = plan_chunk(n, true, t1 - t0, c))) return rc;
  const long long NB = (long long)n->N * n->B;
  for (int c0 = t0; c0 < t1; c0 += c.Tc) {
    const int c1 = std::min(t1, c0 + c.Tc);
    if ((rc = forward_chunk(n, params, x, x_lead, c0, c1, 1, true, c, s))) return rc;
    QLossArgs q;
    memset(&q, 0, sizeof(q));
    q.q = make_view(c.logits, n->O * NB, -c0, n->N, n->O, n->B);
    q.dq = make_view(c.dl, n->O * NB, -c0, n->N, n->O, n->B);
    q.actions = actions, q.target = target, q.q_out = q_out, q.O = n->O, q.B = n->B, q.t0 = c0, q.t1 = c1;
    q.loss_kind = loss_kind, q.inv_rows = inv_rows, q.loss_sum = loss_sum;
    const long long rows = (long long)(c1 - c0) * n->B;
    q_loss_grad_kernel<<<dim3(grid_for(rows, 128), n->N), 128, 0, s>>>(q);
    D2D_LAUNCHED();
    if ((rc = backward_chunk(n, params, x, x_lead, c0, c1, c, grads, inv_rows, s))) return rc;
  }
  return D2D_OK;
}

extern "C" int d2d_replay_gather(const float* obs_ring, const uint8_t* act_ring, const int32_t* rew_ring,
                                 const int32_t* start, const int32_t* env_col, int ep0, int n_ep_slots, int T,
                                 int chunk, int rows, int N, int B, int mb, float* xs, float* xn, uint8_t* act,
                                 int32_t* rew, uint8_t* done, void* stream) {
  D2D_REQUIRE(obs_ring && act_ring && rew_ring && start && env_col && xs && xn && act && rew && done,
              "d2d_replay_gather: null argument");
  D2D_REQUIRE(n_ep_slots >= 1 && ep0 >= 0 && ep0 < n_ep_slots && T >= 1 && chunk >= 1 && rows >= 1 && N >= 1 &&
                  N <= D2D_MAX_AGENTS && B >= 1 && mb >= 1,
              "d2d_replay_gather: bad shape");
  GatherArgs a;
  memset(&a, 0, sizeof(a));
  a.obs_ring = obs_ring, a.act_ring = act_ring, a.rew_ring = rew_ring, a.start = start, a.env_col = env_col;
  a.ep0 = ep0, a.slots = n_ep_slots, a.T = T, a.chunk = chunk, a.rows = rows, a.N = N, a.B = B, a.mb = mb;
  a.xs = xs, a.xn = xn, a.act = act, a.rew = rew, a.done = done;
  replay_gather_kernel<<<grid_for((long long)chunk * rows * mb, 256), 256, 0, as_stream(stream)>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_returns_scan(const int32_t* reward, const float* value, double* adv_raw, double* ret_raw,
                                double* stats, int T, int B, int n_cols, double gamma, double lam, int last_shard,
                                void* stream) {
  D2D_REQUIRE(reward && stats && T >= 1 && B >= 1 && n_cols >= 1 && n_cols <= D2D_MAX_AGENTS,
              "d2d_returns_scan: bad argument");
  D2D_REQUIRE(!adv_raw || value, "d2d_returns_scan: lambda-returns need values");
  ScanArgs a;
  memset(&a, 0, sizeof(a));
  a.reward_i = reward, a.value = value, a.adv_raw = adv_raw, a.ret_raw = ret_raw, a.stats = stats;
  a.T = T, a.B = B, a.n_cols = n_cols, a.gamma = gamma, a.lam = lam, a.last_env_is_global_last = last_shard;
  returns_scan_kernel<kScanRaw><<<dim3(grid_for(B, 128), n_cols), 128, 0, as_stream(stream)>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

// two-pass variant: pass 1 accumulates the normalisation statistics only, pass 2 (after the caller reduced the
// statistics over ranks) repeats the scan and writes the normalised fp32 results; no fp64 intermediates in HBM
extern "C" int d2d_returns_stats(const int32_t* reward, const float* value, double* stats, int T, int B, int n_cols,
                                 double gamma, double lam, int last_shard, int want_adv, int want_ret, void* stream) {
  D2D_REQUIRE(reward && stats && T >= 1 && B >= 1 && n_cols >= 1 && n_cols <= D2D_MAX_AGENTS,
              "d2d_returns_stats: bad argument");
  D2D_REQUIRE(!want_adv || value, "d2d_returns_stats: lambda-returns need values");
  ScanArgs a;
  memset(&a, 0, sizeof(a));
  a.reward_i = reward, a.value = value, a.stats = stats, a.want_adv = want_adv, a.want_ret = want_ret;
  a.T = T, a.B = B, a.n_cols = n_cols, a.gamma = gamma, a.lam = lam, a.last_env_is_global_last = last_shard;
  returns_scan_kernel<kScanStats><<<dim3(grid_for(B, 128), n_cols), 128, 0, as_stream(stream)>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_returns_norm_stats(const double* stats, int n_cols, double rows, double* adv_mean, double* adv_std,
                                      int32_t* adv_norm, double* ret_mean, double* ret_std, int32_t* ret_norm,
                                      void* stream) {
  D2D_REQUIRE(stats && adv_mean && adv_std && adv_norm && ret_mean && ret_std && ret_norm,
              "d2d_returns_norm_stats: null argument");
  D2D_REQUIRE(n_cols >= 1 && n_cols <= D2D_MAX_AGENTS && rows >= 2.0, "d2d_returns_norm_stats: bad shape");
  norm_stats_kernel<<<1, 64, 0, as_stream(stream)>>>(stats, n_cols, rows, adv_mean, adv_std, adv_norm, ret_mean,
                                                     ret_std, ret_norm);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_returns_emit(const int32_t* reward, const float* value, float* adv_out, float* ret_out,
                                const double* adv_mean, const double* adv_std, const int32_t* adv_norm,
                                const double* ret_mean, const double* ret_std, const int32_t* ret_norm, int T, int B,
                                int n_cols, double gamma, double lam, int last_shard, void* stream) {
  D2D_REQUIRE(reward && T >= 1 && B >= 1 && n_cols >= 1 && n_cols <= D2D_MAX_AGENTS, "d2d_returns_emit: bad argument");
  D2D_REQUIRE(!adv_out || (value && adv_mean && adv_std && adv_norm),
              "d2d_returns_emit: lambda-returns need values and their statistics");
  D2D_REQUIRE(!ret_out || (ret_mean && ret_std && ret_norm), "d2d_returns_emit: returns need their statistics");
  ScanArgs a;
  memset(&a, 0, sizeof(a));
  a.reward_i = reward, a.value = value, a.adv_out = adv_out, a.ret_out = ret_out;
  a.adv_mean = adv_mean, a.adv_std = adv_std, a.adv_norm = adv_norm;
  a.ret_mean = ret_mean, a.ret_std = ret_std, a.ret_norm = ret_norm;
  a.T = T, a.B = B, a.n_cols = n_cols, a.gamma = gamma, a.lam = lam, a.last_env_is_global_last = last_shard;
  returns_scan_kernel<kScanEmit><<<dim3(grid_for(B, 128), n_cols), 128, 0, as_stream(stream)>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

extern "C" int d2d_normalize(const double* raw, float* out, const double* mean, const double* std,
                             const int32_t* do_norm, int fp32_math, int T, int B, int n_cols, void* stream) {
  D2D_REQUIRE(raw && out && mean && std && do_norm, "d2d_normalize: null argument");
  NormArgs a;
  a.raw = raw, a.out = out, a.mean = mean, a.std = std, a.do_norm = do_norm, a.fp32_math = fp32_math;
  a.per_t = (long long)n_cols * B, a.B = B, a.n = (long long)T * n_cols * B;
  normalize_kernel<<<grid_for(a.n, 256), 256, 0, as_stream(stream)>>>(a);
  D2D_LAUNCHED();
  return D2D_OK;
}

#ifdef D2D_BPTT_TRACE
extern "C" int d2d_debug_bptt_trace(long long* out) {
  return cudaMemcpyFromSymbol(out, d2d::g_bptt_trace, sizeof(long long) * 16 * 512) == cudaSuccess ? 0 : -1;
}
#endif
