// Fused GRU window on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
//   h_last[row] = GRU(x[t-L+1 .. t][row]; W_ih, W_hh, b_ih, b_hh)   for every row (time t, env b) of every agent
//
// replaces, for the rollout / inference direction, L x (hidden-projection GEMM + gate kernel) and the input
// projection GEMM (reference: RNN.forward, algorithms/d2d_ppo.py:46-54, called once per env step by
// PPO.select_action at :302-303).  Nothing but the observations (L x I floats per row) is read and nothing but
// h_last (H floats per row) is written: the [rows x 3H] projections live in TMEM, h lives in registers and in
// shared memory as the next step's A operand.
//
// fp32 parity on tensor cores: every fp32 operand is split into TWO fp16 planes (v = p0 + p1, p0 = rn16(v),
// p1 = rn16(v - p0): 22 significant bits, absolute error <= 2^-25 for |v| <= 1) and a product keeps the three plane
// pairs p0 q0 + p0 q1 + p1 q0 (the dropped p1 q1 term is 2^-24 relative).  Weights are pre-scaled by 2^6 so that their
// low planes stay out of the fp16 subnormal range; the accumulators then carry 64 x the pre-activation and the factor
// is folded into the gate constants.  Measured (CPU emulation on the reference's c3 weights, 6 recurrent steps):
// 1.3e-7 norm-wise, the same as fp32 itself and as the earlier 3-plane bf16 scheme, which needed 6 products per GEMM
// instead of 3 and 3 operand planes in shared memory instead of 2.  Observations are small integers (exact in fp16 up
// to 2048), so the input projection needs only x (1 plane) x W_ih (2 planes).
//
// CTA = 16 warps (512 threads: 128 registers each; a 17th warp would be charged as four and leave 96, which spills
// the prefetched observations in store mode).  Two 128-row tiles ("slots") are in flight per CTA so that the tensor
// pipe works on one slot while the other slot's gates are evaluated:
//   warps 0-7  : slot 0; warp w serves TMEM lane quadrant w % 4 (rows 32 (w % 4) + lane) and the hidden units of
//                half (w / 4) % 2: stage x, read gate pre-activations with tcgen05.ld, gate maths, write h
//                (2 fp16 planes) + next x into the canonical K-major smem layout
//   warps 8-15 : the same for slot 1
//   the first thread of each slot also issues that slot's tcgen05.mma batch once the slot's operands are in place:
//                TMEM columns [0, H) r, [H, 2H) z, [2H, 3H) gh_n, [3H, 4H) gi_n (the n gate needs gi_n and gh_n
//                separately).  x W_ih^T is ONE N = 4H MMA per (plane, k-step) over W_ih stored as [r; z; 0; n] (the zero
//                block initialises the gh_n columns); h W_hh^T is ONE N = 3H MMA per (plane pair, k-step) over W_hh's
//                natural [r; z; n] rows: 4 + 12 = 16 MMAs per step (36 with 3 bf16 planes), A tiles fetched once
// Hand-offs are mbarriers: a_ready[slot] (256 arrivals: operands staged) and d_ready[slot] (tcgen05.commit).
// The kernel is bound by the gate maths (6 MUFU per (row, unit, step)), not by the tensor pipe: sigmoid / tanh use
// ex2.approx + rcp.approx (rel. error ~2^-21).
// Shared memory (H = 64, I <= 32): W_ih planes 32 KB + W_hh planes 48 KB + h planes 2 x 32 KB + x 2 x 8 KB = 160 KB;
// TMEM: 2 slots x 4H = 512 columns.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "learner_kernels.cuh"
#include "learner_pointwise.cuh"

namespace d2d {

struct GruTcArgs {
  View x;        // observations: element (agent g, feature f, time t, env b); time blocks before 0 are zero
  View h_out;    // [.. H ..] last hidden state
  const float* w;
  long long w_agent_stride;
  int wih_off[D2D_MAX_AGENTS], whh_off[D2D_MAX_AGENTS], bih_off[D2D_MAX_AGENTS], bhh_off[D2D_MAX_AGENTS];
  int in_dim[D2D_MAX_AGENTS];
  int L, B, t0, t1;
  int padded;    // 1: steps before the episode start run on zero inputs; 0: they do not exist (rollout windows)
  // training direction (store = 1, padded = 1): every step's gate activations and hidden state are kept for BPTT
  int store;
  View acts;     // [.. 4H ..] r, z, n, gh_n of step 0; step s is acts_step floats further (p == nullptr: not kept)
  View hs;       // [.. H ..]  h after step 0; step s is hs_step floats further (h_out is not written when store = 1)
  long long acts_step, hs_step;
  // fused network head (kernel template OMAX > 0, inference direction): out = W2 relu(W1 h_last + b1) + b2 is written
  // instead of h_last (reference: the `layers` Sequential of RNN, d2d_ppo.py:36-41,54)
  View out;      // [.. O ..] pre-activation outputs
  View y1;       // [.. H ..] relu(W1 h_last + b1), kept for the backward pass (store mode with a fused head)
  // select_action fused behind the head (policy nets at rollout time): sel.actions != nullptr -> the epilogue turns the
  // outputs into probabilities, selects / reads the action and writes action + log-prob (d2d_ppo.py:159-181);
  // out.p may then be null
  DistArgs sel;
  int w1_off[D2D_MAX_AGENTS], b1_off[D2D_MAX_AGENTS], w2_off[D2D_MAX_AGENTS], b2_off[D2D_MAX_AGENTS];
  int O;
};

namespace tc {

constexpr int kM = 128;       // rows per slot
constexpr int kKx = 32;       // padded input size (I <= 32)
constexpr int kThreads = 512;
constexpr int kGateThreads = 256;   // per slot

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// canonical K-major, no-swizzle UMMA layout of a [rows][kc] bf16 tile: 8-row x 16-byte core matrices,
// K-adjacent core matrices contiguous (LBO = 128 B), 8-row groups (kc / 8) * 128 B apart (SBO)
__device__ __forceinline__ int canon16(int r, int k, int kc) {
  return ((r >> 3) * (kc >> 3) + (k >> 3)) * 64 + (r & 7) * 8 + (k & 7);
}
__device__ __forceinline__ uint64_t desc16(uint32_t saddr, int kc) {
  const uint64_t start = (saddr & 0x3FFFFu) >> 4;
  const uint64_t lbo = 128 >> 4, sbo = (uint64_t)((kc >> 3) * 128) >> 4;
  return start | (lbo << 16) | (sbo << 32) | (1ull << 46);   // version 1 (Blackwell), no swizzle, base offset 0
}
// descriptor of the tile `byte_off` bytes further (same strides): one 32-bit add on the start-address field instead of
// rebuilding the descriptor; the single issuing thread is latency bound on exactly this arithmetic
__device__ __forceinline__ uint64_t desc_adv(uint64_t base, uint32_t byte_off) {
  return (base & 0xFFFFFFFF00000000ull) | (uint64_t)((uint32_t)base + (byte_off >> 4));
}
// instruction descriptor: D = F32, A = B = BF16, both K-major, M = 128
__device__ __forceinline__ uint32_t idesc_bf16(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kM >> 4) << 24);
}
// the same with A = B = FP16 (a_format = b_format = 0)
__device__ __forceinline__ uint32_t idesc_f16(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kM >> 4) << 24);
}
constexpr float kWScale = 64.0f;              // weights are staged as 64 w: their low fp16 planes stay normal
constexpr float kInvWScale = 1.0f / 64.0f;
// (a, b) -> two fp16 planes, each as a packed half2 word (element a in the low half): v = p0 + p1 + O(2^-24 |v|)
__device__ __forceinline__ void split2h(float a, float b, uint32_t& p0, uint32_t& p1) {
  const __half2 h0 = __floats2half2_rn(a, b);
  const float2 f0 = __half22float2(h0);
  const __half2 h1 = __floats2half2_rn(a - f0.x, b - f0.y);
  p0 = *reinterpret_cast<const uint32_t*>(&h0), p1 = *reinterpret_cast<const uint32_t*>(&h1);
}
__device__ __forceinline__ void split2h1(float v, __half& p0, __half& p1) {
  p0 = __float2half_rn(v);
  p1 = __float2half_rn(v - __half2float(p0));
}
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accum) {
  const uint32_t acc = accum ? 1u : 0u;
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_u32(b)), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(r[j]);
}
__device__ __forceinline__ void split3(float v, __nv_bfloat16& p0, __nv_bfloat16& p1, __nv_bfloat16& p2) {
  p0 = __float2bfloat16_rn(v);
  float r = v - __bfloat162float(p0);
  p1 = __float2bfloat16_rn(r);
  r -= __bfloat162float(p1);
  p2 = __float2bfloat16_rn(r);
}
// v = t0 + t1 + t2 (+ < 2^-24 |v|) with every t the top 16 bits of an fp32 word, i.e. a bf16 value: cut by masking
// (ALU pipe) rather than by F2F conversions (quarter-rate XU pipe, which the gate maths already saturates)
__device__ __forceinline__ void split3_trunc(float v, uint32_t& t0, uint32_t& t1, uint32_t& t2) {
  t0 = __float_as_uint(v) & 0xFFFF0000u;
  const float r1 = v - __uint_as_float(t0);
  t1 = __float_as_uint(r1) & 0xFFFF0000u;
  t2 = __float_as_uint(r1 - __uint_as_float(t1));
}
// two fp32 words -> their top halves packed as two bf16 (element 0 in the low half)
__device__ __forceinline__ uint32_t pack_hi(uint32_t a, uint32_t b) { return __byte_perm(a, b, 0x7632); }
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

template <int H>
struct Smem {
  static constexpr int kWih = 4 * H * kKx;        // fp16 elements of one W_ih plane: rows [r; z; 0; n] (the zero block
                                                  // initialises / leaves alone the gh_n accumulator columns)
  static constexpr int kWhh = 3 * H * H;
  static constexpr int kAh = kM * H;
  static constexpr int kAx = kM * kKx;
  static constexpr size_t bytes = (size_t)(2 * kWih + 2 * kWhh + 2 * 2 * kAh + 2 * kAx) * 2 + 4 * H * 4 + 64;
  // fused head: W1 planes [2][H][H] fp16, then fp32: b1 [H], W2^T [H][OMAX], b2 [OMAX], partial sums [2 slots][128][OMAX]
  static constexpr size_t head_bytes(int omax) {
    return (size_t)2 * H * H * 2 + (size_t)(H + H * omax + omax + 2 * kM * omax) * 4 + 16;
  }
};

}  // namespace tc

// STORE: the training direction (a.store); compile time so that the rollout kernel carries none of the store code.
// 1: h and the gates (r, z, n, gh_n) of every step are kept (H 16 / 48: the FP32 gate backward reads them);
// 2: only h is kept (H 32 / 64: the recomputing BPTT kernel) and the gate maths takes the rollout's shared-reciprocal
// form.
// OMAX > 0: the network head is fused behind the last step -- Linear(H, H) as one more
// two-plane GEMM on the h planes the step already staged (12 MMAs), ReLU and Linear(H, O <= OMAX) on the CUDA cores from
// TMEM, the two unit halves of a row combined through shared memory -- and the kernel writes the O pre-activation
// outputs instead of h_last: no head kernel, no h_last round trip through HBM.
template <int H, int STORE, int OMAX = 0>
__global__ void __launch_bounds__(tc::kThreads, 1) gru_window_tc_kernel(const GruTcArgs a) {
  using namespace tc;
  using S = Smem<H>;
  static_assert(H % 16 == 0 && H >= 16 && H <= 64, "H in {16, 32, 48, 64}");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __half* wih = reinterpret_cast<__half*>(smem_raw);                    // [2 planes][4H][kKx], rows [r; z; 0; n]
  __half* whh = wih + 2 * S::kWih;                                      // [2 planes][3H][H]
  __half* ah = whh + 2 * S::kWhh;                                       // [2 slots][2 planes][128][H]
  __half* ax = ah + 2 * 2 * S::kAh;                                     // [2 slots][128][kKx]
  float* bias = reinterpret_cast<float*>(ax + 2 * S::kAx);              // [2H] b_ih + b_hh (r, z), [H] b_in, [H] b_hn
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias + 4 * H);           // a_ready[2], d_ready[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  uint64_t* a_ready = bars;
  uint64_t* d_ready = bars + 2;
  constexpr bool HEAD = OMAX > 0;
  constexpr int OP = HEAD ? OMAX : 1;
  __half* w1p = reinterpret_cast<__half*>(smem_raw + ((S::bytes + 15) & ~(size_t)15));   // [2 planes][H][H]
  float* b1s = reinterpret_cast<float*>(w1p + 2 * H * H);                                 // [H]
  float* w2t = b1s + H;                                                                   // [H][OP] = W2[o][j]
  float* b2s = w2t + H * OP;                                                              // [OP]
  float* part = b2s + OP;                                                                 // [2 slots][128][OP]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = blockIdx.y;
  const int I = a.in_dim[g];
  const float* Wih = a.w + g * a.w_agent_stride + a.wih_off[g];
  const float* Whh = a.w + g * a.w_agent_stride + a.whh_off[g];
  const float* bih = a.w + g * a.w_agent_stride + a.bih_off[g];
  const float* bhh = a.w + g * a.w_agent_stride + a.bhh_off[g];

  // ---- one-time setup: 64 x weights -> two fp16 planes in the canonical layout, biases, barriers, TMEM ----
  for (int i = tid; i < 4 * H * kKx; i += kThreads) {
    const int n4 = i / kKx, k = i % kKx;          // row of the [r; z; 0; n] arrangement
    const int n = n4 < 2 * H ? n4 : n4 - H;       // row of W_ih ([r; z; n]); rows [2H, 3H) of the arrangement are zero
    const bool zero = n4 >= 2 * H && n4 < 3 * H;
    __half p0, p1;
    split2h1((!zero && k < I) ? kWScale * Wih[(long long)n * I + k] : 0.f, p0, p1);
    const int o = canon16(n4, k, kKx);
    wih[o] = p0, wih[S::kWih + o] = p1;
  }
  for (int i = tid; i < 3 * H * H; i += kThreads) {
    const int n = i / H, k = i % H;
    __half p0, p1;
    split2h1(kWScale * Whh[i], p0, p1);
    const int o = canon16(n, k, H);
    whh[o] = p0, whh[S::kWhh + o] = p1;
  }
  if constexpr (HEAD) {
    const float* base = a.w + g * a.w_agent_stride;
    for (int i = tid; i < H * H; i += kThreads) {
      const int n = i / H, k = i % H;
      __half p0, p1;
      split2h1(kWScale * base[a.w1_off[g] + i], p0, p1);
      const int o = canon16(n, k, H);
      w1p[o] = p0, w1p[H * H + o] = p1;
    }
    for (int i = tid; i < H * OP; i += kThreads) {
      const int j = i / OP, o = i % OP;
      w2t[i] = o < a.O ? base[a.w2_off[g] + o * H + j] : 0.f;
    }
    for (int i = tid; i < H; i += kThreads) b1s[i] = base[a.b1_off[g] + i];
    for (int i = tid; i < OP; i += kThreads) b2s[i] = i < a.O ? base[a.b2_off[g] + i] : 0.f;
  }
  // biases, pre-scaled for the ex2-based gates: sigmoid(a) = 1 / (1 + 2^(-a log2 e))
  for (int i = tid; i < 4 * H; i += kThreads) {
    float v;
    if (i < 2 * H) v = -1.4426950408889634f * (bih[i] + bhh[i]);   // r, z: -(b_i + b_h) log2 e
    else if (i < 3 * H) v = bih[i];            // b_in
    else v = bhh[i - H];                       // b_hn
    bias[i] = v;
  }
  if (tid == 0) {
    mbar_init(&a_ready[0], kGateThreads), mbar_init(&a_ready[1], kGateThreads);
    mbar_init(&d_ready[0], 1), mbar_init(&d_ready[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  const int L = a.L;
  const int pairs_per_t = (a.B + 2 * kM - 1) / (2 * kM);
  const int n_pairs = (a.t1 - a.t0) * pairs_per_t;

  {
    // =================== gate warps: slot = warp / 8, lane quadrant = warp % 4, unit half = (warp / 4) % 2 ====
    constexpr int HH = H / 2;          // hidden units per thread
    constexpr int KH = kKx / 2;        // input features staged per thread
    static_assert(HH % 8 == 0 && KH % 8 == 0, "units / features per thread in groups of 8");
    const int slot = warp / 8;
    const int half = (warp >> 2) % 2;
    const int row = ((warp & 3) << 5) + lane;
    const uint32_t lane_addr = (uint32_t)((warp & 3) << 5) << 16;
    __half* my_ax = ax + slot * S::kAx;
    __half* my_ah = ah + slot * 2 * S::kAh;
    const int u0 = half * HH;
    uint32_t ph = 0, ph_a = 0;
    float h[HH];
    const bool issuer = (tid & (kGateThreads - 1)) == 0;
    const uint32_t id3 = idesc_f16(3 * H), id4 = idesc_f16(4 * H);
    // base descriptors of the slot's operand tiles, built once
    const uint32_t d_slot = tmem + (uint32_t)slot * (4 * H);
    const uint64_t dx = desc16(smem_u32(ax + slot * S::kAx), kKx), dwih = desc16(smem_u32(wih), kKx);
    const uint64_t dah = desc16(smem_u32(ah + slot * 2 * S::kAh), H), dwhh = desc16(smem_u32(whh), H);
    // the slot's MMA batch for the step whose operands were just published (first_step: h = 0, input projection only)
    auto issue = [&](bool first_step) {
      mbar_wait(&a_ready[slot], ph_a);
      ph_a ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // Accumulator columns of the slot: [0, H) r, [H, 2H) z, [2H, 3H) gh_n, [3H, 4H) gi_n (the n gate needs both
      // separately), all scaled by 64 (kWScale).
      // input projection, x exact in fp16: ONE N = 4H MMA per (plane, k-step) over W_ih stored as [r; z; 0; n]; the
      // first one initialises all 4H columns (zeros into the gh_n columns)
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int k16 = 0; k16 < kKx / 16; ++k16)
          mma_bf16(d_slot, desc_adv(dx, k16 * 256), desc_adv(dwih, j * S::kWih * 2 + k16 * 256), id4, j + k16 > 0);
      if (!first_step) {
        // hidden projection, plane pairs h0 w0, h0 w1, h1 w0: ONE N = 3H MMA per (pair, k-step) over W_hh's natural
        // [r; z; n] rows, accumulated onto the r, z and gh_n columns
#pragma unroll
        for (int pr = 0; pr < 3; ++pr) {
          const int i = pr == 2 ? 1 : 0, j = pr == 1 ? 1 : 0;
#pragma unroll
          for (int k16 = 0; k16 < H / 16; ++k16)
            mma_bf16(d_slot, desc_adv(dah, (i * S::kAh) * 2 + k16 * 256), desc_adv(dwhh, (j * S::kWhh) * 2 + k16 * 256),
                     id3, true);
        }
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                   ::"r"(smem_u32(&d_ready[slot]))
                   : "memory");
    };

    const uint64_t dw1 = desc16(smem_u32(w1p), H);
    const uint32_t idh = idesc_f16(H);
    auto issue_head = [&]() {   // Y1 = h_last W1^T (x 64) into the slot's columns [0, H): h0 w0, h0 w1, h1 w0
      mbar_wait(&a_ready[slot], ph_a);
      ph_a ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int pr = 0; pr < 3; ++pr) {
        const int i = pr == 2 ? 1 : 0, j = pr == 1 ? 1 : 0;
#pragma unroll
        for (int k16 = 0; k16 < H / 16; ++k16)
          mma_bf16(d_slot, desc_adv(dah, (i * S::kAh) * 2 + k16 * 256), desc_adv(dw1, (j * H * H) * 2 + k16 * 256), idh,
                   pr + k16 > 0);
      }
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                   ::"r"(smem_u32(&d_ready[slot]))
                   : "memory");
    };
    auto load_x = [&](int t_obs, int b, float* xr) {   // this thread's half of the row's observation -> registers
      const bool ok = b < a.B;
      const float* xp = view_ptr(a.x, g, t_obs, a.B, ok ? b : 0);
#pragma unroll
      for (int k = 0; k < KH; ++k) {
        const int kk = half * KH + k;
        xr[k] = (ok && kk < I) ? xp[(long long)kk * a.B] : 0.f;
      }
    };
    auto stage_x = [&](const float* xr) {              // integer-valued observations: exact in one fp16 plane
#pragma unroll
      for (int kc = 0; kc < KH / 8; ++kc) {
        uint4 v;
        const __half2 a0 = __floats2half2_rn(xr[kc * 8 + 0], xr[kc * 8 + 1]), a1 = __floats2half2_rn(xr[kc * 8 + 2], xr[kc * 8 + 3]);
        const __half2 a2 = __floats2half2_rn(xr[kc * 8 + 4], xr[kc * 8 + 5]), a3 = __floats2half2_rn(xr[kc * 8 + 6], xr[kc * 8 + 7]);
        v.x = *reinterpret_cast<const uint32_t*>(&a0), v.y = *reinterpret_cast<const uint32_t*>(&a1);
        v.z = *reinterpret_cast<const uint32_t*>(&a2), v.w = *reinterpret_cast<const uint32_t*>(&a3);
        *reinterpret_cast<uint4*>(my_ax + canon16(row, half * KH + kc * 8, kKx)) = v;
      }
    };
    auto publish = [&]() {   // operands of the next MMA batch are in place (and our TMEM reads are done)
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(&a_ready[slot]);
    };

    for (int p = blockIdx.x; p < n_pairs; p += gridDim.x) {
      const int t = a.t0 + p / pairs_per_t;
      const int b = (p % pairs_per_t) * (2 * kM) + slot * kM + row;
      const int s0 = a.padded ? 0 : max(0, L - 1 - t);
      float xr[KH];
      load_x(t - (L - 1 - s0), b, xr);
      stage_x(xr);
      publish();
      if (issuer) issue(true);
      __syncwarp();
#pragma unroll
      for (int u = 0; u < HH; ++u) h[u] = 0.f;
      for (int s = s0; s < L; ++s) {
        const bool has_next = s + 1 < L;
        if (has_next) load_x(t - (L - 2 - s), b, xr);   // in flight during the gate maths
        mbar_wait(&d_ready[slot], ph);
        ph ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d = tmem + (uint32_t)slot * (4 * H) + lane_addr + (uint32_t)u0;
        float* acts_row = nullptr;
        float* hs_row = nullptr;
        if (STORE && b < a.B) {   // acts.p == nullptr: only h is kept (the recomputing BPTT kernel, gru_bptt_tc.cuh)
          if constexpr (STORE == 1) acts_row = view_ptr(a.acts, g, t, a.B, b) + (long long)s * a.acts_step;
          hs_row = view_ptr(a.hs, g, t, a.B, b) + (long long)s * a.hs_step;
        }
#pragma unroll
        for (int c = 0; c < HH / 8; ++c) {
          float pr[8], pz[8], pin[8], phn[8];
          tmem_ld8(d + c * 8, pr);
          tmem_ld8(d + H + c * 8, pz);
          tmem_ld8(d + 3 * H + c * 8, pin);
          tmem_ld8(d + 2 * H + c * 8, phn);      // zero at the window's first step (written by the zero block)
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          float hv8[8];
          const float4* bz = reinterpret_cast<const float4*>(bias + u0 + c * 8);   // 16-byte aligned: u0 + 8c
          const float4 br0 = bz[0], br1 = bz[1];
          const float4 bz0 = bz[H / 4], bz1 = bz[H / 4 + 1];
          const float4 bi0 = bz[2 * H / 4], bi1 = bz[2 * H / 4 + 1];
          const float4 bh0 = bz[3 * H / 4], bh1 = bz[3 * H / 4 + 1];
          const float b_r[8] = {br0.x, br0.y, br0.z, br0.w, br1.x, br1.y, br1.z, br1.w};
          const float b_z[8] = {bz0.x, bz0.y, bz0.z, bz0.w, bz1.x, bz1.y, bz1.z, bz1.w};
          const float b_i[8] = {bi0.x, bi0.y, bi0.z, bi0.w, bi1.x, bi1.y, bi1.z, bi1.w};
          const float b_h[8] = {bh0.x, bh0.y, bh0.z, bh0.w, bh1.x, bh1.y, bh1.z, bh1.w};
          constexpr float kSig = -1.4426950408889634f * kInvWScale;   // accumulators carry 64 x the pre-activation
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            // (a reciprocal on the FMA pipe -- bit-trick seed + two cubic steps, 7 instructions -- was measured here for r:
            // 4.72e8 agent-steps/s against 4.80e8, the issue slots it takes cost more than the MUFU slot it frees)
            const float r = rcp_approx(1.0f + ex2_approx(fmaf(pr[j], kSig, b_r[j])));
            const float ghn = fmaf(phn[j], kInvWScale, b_h[j]);
            const float pre = fmaf(r, ghn, fmaf(pin[j], kInvWScale, b_i[j]));
            float hv, z = 0.f, nn = 0.f;
            if constexpr (STORE == 1) {
              z = rcp_approx(1.0f + ex2_approx(fmaf(pz[j], kSig, b_z[j])));
              // tanh(v) = 1 - 2 / (1 + 2^(2 v log2 e))
              nn = fmaf(-2.0f, rcp_approx(1.0f + ex2_approx(2.8853900817779268f * pre)), 1.0f);
              hv = fmaf(z, h[c * 8 + j] - nn, nn);             // (1 - z) n + z h
            } else {
              // rollout direction (the MUFU pipe is the busiest one): z = 1 / (1 + ez) and n = (en - 1) / (1 + en) share
              // ONE reciprocal, (1 - z) n + z h = ((en - 1) ez + h (1 + en)) / ((1 + ez)(1 + en)).  The exponents are
              // clamped at 2^40 (sigmoid < 1e-12, 1 - tanh < 2e-12: below fp32 resolution) so the product stays finite.
              const float ez = ex2_approx(fminf(fmaf(pz[j], kSig, b_z[j]), 40.0f));
              const float en = ex2_approx(fminf(2.8853900817779268f * pre, 40.0f));
              const float bn = 1.0f + en;
              const float inv = rcp_approx((1.0f + ez) * bn);
              hv = fmaf(en - 1.0f, ez, h[c * 8 + j] * bn) * inv;
            }
            h[c * 8 + j] = hv;
            hv8[j] = hv;
            if (STORE && b < a.B) {   // rows of a warp are consecutive envs: every store below is one 128-byte line
              const long long f = (long long)(u0 + c * 8 + j) * a.B;
              const long long hb = (long long)H * a.B;
              if constexpr (STORE == 1) acts_row[f] = r, acts_row[f + hb] = z, acts_row[f + 2 * hb] = nn, acts_row[f + 3 * hb] = ghn;
              hs_row[f] = hv;
            }
          }
          if (has_next || HEAD) {   // the head GEMM reads h_last from the same operand tiles
            uint32_t q0[4], q1[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) split2h(hv8[2 * j], hv8[2 * j + 1], q0[j], q1[j]);
            const int o = canon16(row, u0 + c * 8, H);
            *reinterpret_cast<uint4*>(my_ah + o) = make_uint4(q0[0], q0[1], q0[2], q0[3]);
            *reinterpret_cast<uint4*>(my_ah + S::kAh + o) = make_uint4(q1[0], q1[1], q1[2], q1[3]);
          }
        }
        if (has_next) {
          stage_x(xr);
          publish();
          if (issuer) issue(false);
          __syncwarp();
        } else if constexpr (HEAD) {
          publish();
          if (issuer) issue_head();
          __syncwarp();
          mbar_wait(&d_ready[slot], ph);
          ph ^= 1u;
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          float po[OP];
#pragma unroll
          for (int o = 0; o < OP; ++o) po[o] = 0.f;
#pragma unroll
          for (int c = 0; c < HH / 8; ++c) {
            float y[8];
            tmem_ld8(d + c * 8, y);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int u = u0 + c * 8 + j;
              const float yv = fmaxf(fmaf(y[j], kInvWScale, b1s[u]), 0.f);     // relu(W1 h + b1)
              if (STORE && b < a.B) view_ptr(a.y1, g, t, a.B, b)[(long long)u * a.B] = yv;   // for the backward pass
#pragma unroll
              for (int o = 0; o < OP; ++o) po[o] = fmaf(w2t[u * OP + o], yv, po[o]);
            }
          }
          // the row's two unit halves live in different warps: half 1 hands its partial sums to half 0 through smem
          float* pp = part + ((size_t)slot * kM + row) * OP;
          if (half == 1) {
#pragma unroll
            for (int o = 0; o < OP; ++o) pp[o] = po[o];
          }
          asm volatile("bar.sync %0, %1;" ::"r"(1 + slot), "r"(kGateThreads) : "memory");
          if (half == 0 && b < a.B) {
#pragma unroll
            for (int o = 0; o < OP; ++o) po[o] += pp[o];
#pragma unroll
            for (int o = 0; o < OP; ++o) po[o] += b2s[o];
            if (a.out.p) {
              float* op = view_ptr(a.out, g, t, a.B, b);
#pragma unroll
              for (int o = 0; o < OP; ++o)
                if (o < a.O) op[(long long)o * a.B] = po[o];
            }
            if (!STORE && OMAX > 1 && a.sel.actions) {   // PPO.select_action on the row's outputs, in registers
              float lg_[OP], pr_[kMaxOut];       // copies: the helpers index by a runtime count (local memory)
#pragma unroll
              for (int o = 0; o < OP; ++o) lg_[o] = po[o];
              head_probs(a.sel, lg_, 1, pr_);
              policy_select(a.sel, g, t, b, pr_);
            }
          }
          // TMEM reads of this tile are complete before the next tile's first MMA: its publish() fences them
        } else {
          // TMEM reads of this tile are complete before the next tile's first MMA: its publish() fences them
          if (b < a.B && !STORE) {
            float* ho = view_ptr(a.h_out, g, t, a.B, b);
#pragma unroll
            for (int u = 0; u < HH; ++u) ho[(long long)(u0 + u) * a.B] = h[u];
          }
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
}

}  // namespace d2d
