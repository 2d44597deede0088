// Pointwise / gather kernels of the independent recurrent DQN learner (reference algorithms/irdqn.py):
// epsilon-greedy action selection, TD target, loss gradient w.r.t. the Q-values, replay-chunk gather.
// The Q-networks themselves run on the net-set kernels (GRU window / dense / BPTT); these kernels are the glue
// between them and are all HBM-trivial (a few bytes per row).
#pragma once
#include "learner_kernels.cuh"
#include "learner_pointwise.cuh"

namespace d2d {

// ---- DQN.act / DQN.predict (irdqn.py:150-166) for every (agent, env) ----
struct QSelectArgs {
  const float* q;        // [N][O][B]
  uint8_t* action;       // [N][B] channel index
  void* mask;            // [N][B] one-hot bitmask (mask_bytes each) or null
  int mask_bytes;
  int N, B, O;
  int act_mode;          // kActSample (epsilon-greedy) / kActGreedy / kActGiven
  float epsilon;
  int ready;             // is_training_ready (irdqn.py:233): not ready -> every action is the random draw
  int n_random;          // the random draw is uniform on {0 .. n_random - 1} (np.random.randint(0, 2) -> 2)
  PhiloxKey key;
  uint32_t env_offset;
  int t_abs;
};

__global__ void q_select_kernel(const QSelectArgs a) {
  const long long n = (long long)a.N * a.B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i / a.B), b = (int)(i % a.B);
    uint32_t act;
    if (a.act_mode == kActGiven) {
      act = a.action[i];
    } else {
      const float* q = a.q + (long long)g * a.O * a.B + b;
      float best = q[0];
      act = 0;
      for (int o = 1; o < a.O; ++o) {
        const float v = q[(long long)o * a.B];
        if (v > best) best = v, act = (uint32_t)o;      // torch.argmax: first maximum
      }
      if (a.act_mode == kActSample) {
        const uint4 r = philox(a.key, a.env_offset + (uint32_t)b, (uint32_t)a.t_abs,
                               (uint32_t)g | (kPurposePolicy << 16), 0u);
        const double u = ((double)r.x + 0.5) * (1.0 / 4294967296.0);
        const bool greedy = a.ready && u >= (double)a.epsilon;            // irdqn.py:151
        if (!greedy) act = (uint32_t)(((unsigned long long)r.y * (unsigned long long)a.n_random) >> 32);
      }
      a.action[i] = (uint8_t)act;
    }
    if (a.mask) {
      const uint32_t m = 1u << act;
      if (a.mask_bytes == 1) reinterpret_cast<uint8_t*>(a.mask)[i] = (uint8_t)m;
      else if (a.mask_bytes == 2) reinterpret_cast<uint16_t*>(a.mask)[i] = (uint16_t)m;
      else reinterpret_cast<uint32_t*>(a.mask)[i] = m;
    }
  }
}

// ---- td_target = rewards + (1 - dones) * gamma * max_a Q_target(s') (irdqn.py:137-139) ----
// fp32 in torch's evaluation order, every product and the sum rounded separately (no contraction into an FMA)
__global__ void q_td_target_kernel(const float* __restrict__ q_next, const int32_t* __restrict__ reward,
                                   const uint8_t* __restrict__ done, float gamma, float* __restrict__ target, int N,
                                   int B, int O) {
  const long long n = (long long)N * B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i / B), b = (int)(i % B);
    const float* q = q_next + (long long)g * O * B + b;
    float best = q[0];
    for (int o = 1; o < O; ++o) best = fmaxf(best, q[(long long)o * B]);
    const float nd = 1.0f - (float)(done[b] != 0);
    target[i] = __fadd_rn((float)reward[b], __fmul_rn(__fmul_rn(nd, gamma), best));
  }
}

// ---- d(loss)/d(Q) of loss = mean_rows(l(Q[action] - target)), l = smooth_l1 (beta 1) or squared error ----
struct QLossArgs {
  View q;                 // [.. O ..] chunk-local Q-values
  View dq;                // out, same shape
  const uint8_t* actions; // [t][N][B] absolute time
  const float* target;    // [t][N][B]
  float* q_out;           // optional [t][N][B]
  int O, B, t0, t1, loss_kind;
  float inv_rows;
  double* loss_sum;       // [N]
};

// part != nullptr (deterministic mode): warp w of agent g's blocks stores its sum to part[g][w] instead of the atomic
template <bool PART>
__device__ __forceinline__ void q_loss_grad_body(const QLossArgs& a, double* part) {
  const int g = blockIdx.y, N = gridDim.y;
  const long long n = (long long)(a.t1 - a.t0) * a.B;
  double local = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int t = a.t0 + (int)(i / a.B), b = (int)(i % a.B);
    const long long idx = ((long long)t * N + g) * a.B + b;
    const int act = a.actions[idx];
    const float* q = view_ptr(a.q, g, t, a.B, b);
    float* dq = view_ptr(a.dq, g, t, a.B, b);
    const float qa = q[(long long)act * a.B];
    const float d = qa - a.target[idx];
    float grad;
    if (a.loss_kind == D2D_QLOSS_MSE) {
      local += (double)d * (double)d;
      grad = 2.0f * d;
    } else {
      const float ad = fabsf(d);
      local += ad < 1.0f ? 0.5 * (double)d * (double)d : (double)ad - 0.5;
      grad = ad < 1.0f ? d : (d > 0.f ? 1.0f : -1.0f);
    }
    for (int o = 0; o < a.O; ++o) dq[(long long)o * a.B] = o == act ? grad * a.inv_rows : 0.f;
    if (a.q_out) a.q_out[idx] = qa;
  }
  for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xFFFFFFFFu, local, o);
  if ((threadIdx.x & 31) == 0) {
    if constexpr (PART) part[(long long)g * gridDim.x * (blockDim.x >> 5) + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5)] = local;
    else atomicAdd(&a.loss_sum[g], local);
  }
}
__global__ void q_loss_grad_kernel(const QLossArgs a) { q_loss_grad_body<false>(a, nullptr); }
__global__ void q_loss_grad_part_kernel(const QLossArgs a, double* part) { q_loss_grad_body<true>(a, part); }

// ---- ReplayBuffer.sample_chunk (irdqn.py:24-42) ----
struct GatherArgs {
  const float* obs_ring;     // [slots][T + 1][rows][B]
  const uint8_t* act_ring;   // [slots][T][N][B]
  const int32_t* rew_ring;   // [slots][T][B]
  const int32_t* start;      // [mb] deque index of the chunk's first transition
  const int32_t* env_col;    // [mb]
  int ep0, slots, T, chunk, rows, N, B, mb;
  float* xs;                 // [chunk][rows][mb]
  float* xn;                 // [chunk][rows][mb]
  uint8_t* act;              // [N][mb]
  int32_t* rew;              // [mb]
  uint8_t* done;             // [mb]
};

__global__ void replay_gather_kernel(const GatherArgs a) {
  const long long per_l = (long long)a.rows * a.mb;
  const long long n = (long long)a.chunk * per_l;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int l = (int)(i / per_l);
    const int row = (int)((i % per_l) / a.mb), j = (int)(i % a.mb);
    const int k = a.start[j] + l;                       // deque index of the transition
    const int slot = (a.ep0 + k / a.T) % a.slots, t = k % a.T;
    const float* p = a.obs_ring + (((long long)slot * (a.T + 1) + t) * a.rows + row) * a.B + a.env_col[j];
    a.xs[i] = p[0];
    a.xn[i] = p[(long long)a.rows * a.B];               // state_next = the following observation block
    if (l == a.chunk - 1 && row == 0) {                 // action / reward / done of the chunk's last transition
      const long long tb = (long long)slot * a.T + t;
      for (int g = 0; g < a.N; ++g) a.act[(long long)g * a.mb + j] = a.act_ring[(tb * a.N + g) * a.B + a.env_col[j]];
      a.rew[j] = a.rew_ring[tb * a.B + a.env_col[j]];
      a.done[j] = (uint8_t)(t == a.T - 1);
    }
  }
}

}  // namespace d2d
