// Back-propagation through the GRU window with the forward pass RECOMPUTED on the tensor cores (tcgen05 + TMEM), sm_100a.
//
// gru_bwd_tc.cuh walks the window backwards on activations the forward kernel stored (r, z, n, gh_n, h: 5H floats per
// row and step, written once and read once: 160 of the 185 GB an iPPO epoch moved at 4,096 envs x 200 steps).  This
// kernel keeps only h of every step (H floats) and recomputes the gates of step s from (x_s, h_{s-1}) with two more
// GEMMs on the tensor pipe, which the BPTT kernel left 70 % idle:
//
//   recompute   [r | z | gh_n | gi_n] = x_s [W_ih]^T + h_{s-1} [W_hh]^T         (the forward kernel's accumulator map)
//   gates       r, z = sigmoid, n = tanh(gi_n + b_in + r (gh_n + b_hn))
//   backward    dn = dh (1 - z)(1 - n^2)    dz = dh (h_prev - n) z (1 - z)    dr = dn gh_n r (1 - r)
//               d(gh) = (dr, dz, dn r)      d(gi) = (dr, dz, dn)              dh_prev = dh z + d(gh) W_hh
//               dW_hh += d(gh)^T h_prev     db_hh += sum_rows d(gh)
//   (reference: autograd through nn.GRU inside PPO.train_step, algorithms/d2d_ppo.py:198-216, on the windows of
//   preprocess_input_for_rnn, :385-398)
//
// Operands are TWO fp16 planes per fp32 value and a product keeps p0 q0 + p0 q1 + p1 q0 (gru_tc.cuh): weights are
// staged as 64 w, d(gh) as g_scale d(gh) with g_scale the power of two that brings the chunk's largest |dh| to ~2^10
// (the loss is a mean over rows, so d(gh) ~ 1 / rows would sit in the fp16 subnormal range; a first attempt with a
// scale guessed from the row count left small elements with 15 significant bits: 2.3e-5 on a bias gradient); the
// factors are divided out when accumulators are read.
// CPU emulation on the reference's c3 weights: 5e-7 norm-wise on the data gradient (2.4e-6 with the 2 bf16 planes of
// gru_bwd_tc.cuh).
//
// CTA = 16 warps on ONE 128-row tile: thread = (row = 32 (w % 4) + lane, unit quarter w / 4).  Per step:
//   A. threads stage P = h_{s-1} (2 planes + a ones column for db_hh) and X = x_s (1 plane: integer observations);
//      thread 0 issues the 16 recompute MMAs (x: N = 4H over W_ih as [r; z; 0; n]; h: N = 3H, W_hh^T read MN-major from
//      the SAME tiles the data-gradient GEMM reads K-major);
//   B. threads read the 4H pre-activations of their units from TMEM, evaluate gates and derivatives, write G = d(gh)
//      (2 planes), add d(gi) to the observation's gradient row (red.global: up to L windows share an observation; the
//      kDgiSlices variant stores it into slice s at the window's own time instead, see dgi_slice_sum_kernel) and
//      pre-load D with the direct path dh z; lane 0 of every warp issues its share of D += G W_hh (36 MMAs) and
//      dW += G^T P (48 MMAs, both tiles read along their contiguous dimension);
//   C. threads read dh_prev from D while the next step's h and x are in flight.
// Per row and step the kernel reads H + I floats instead of 5H, and the forward kernel writes H instead of 5H.
// Shared memory (H = 64): G 96 KB + W_hh^T 48 KB + P 36 KB + W_ih 32 KB + X 8 KB = 220 KB; TMEM: 4H + H + 2 (H + 16)
// = 480 columns.
#pragma once
#include "gru_bwd_tc.cuh"

namespace d2d {

struct GruBpttArgs {
  View x;      // observations: element (agent g, feature f, time t, env b); time blocks before 0 are zero
  View hs;     // [.. H ..] h after step 0 (forward kernel, store mode); step s is hs_step floats further
  View dh;     // [.. H ..] in: d(loss) / d(h after the last step)
  View dgi;    // [.. 3H ..] accumulated at observation time t - (L - 1 - s); zeroed by the caller (the slices kernel:
               // slice 0 of the [L][..] d(gi) slices, written at time t)
  const float* w;
  long long w_agent_stride;
  int wih_off[D2D_MAX_AGENTS], whh_off[D2D_MAX_AGENTS], bih_off[D2D_MAX_AGENTS], bhh_off[D2D_MAX_AGENTS];
  int in_dim[D2D_MAX_AGENTS];
  float* partial;        // [N][gridDim.x][part_stride]: dW_hh [3H][H] then db_hh [3H], one partial per CTA
  long long part_stride;
  long long hs_step;
  const float* dh_absmax;  // device scalar: max |dh| over the chunk (absmax_kernel); d(gh) is scaled by the power of two
                           // that brings it to ~2^10 before the fp16 split, so that values down to 2^-22 of the
                           // largest one keep 22 significant bits (fp16 max 65504 leaves a factor 64 of headroom)
  int L, B, t0, t1;
  long long slice_step;    // kDgiSlices instantiation: floats between two d(gi) slices
};

#ifdef D2D_BPTT_TRACE
__device__ long long g_bptt_trace[16 * 512];
#define D2D_TR(i) do { if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0 && tr_n < 512) g_bptt_trace[tr_n * 16 + (i)] = clock64(); } while (0)
#else
#define D2D_TR(i) do { } while (0)
#endif
namespace tcr {
constexpr int kGate = 512;              // 16 gate warps
constexpr int kThreads = kGate + 32;    // + one warp whose lane 0 issues every MMA
template <int H>
struct Smem {
  static constexpr int kG = tc::kM * 3 * H;       // fp16 elements per d(gh) plane
  static constexpr int kW = H * 3 * H;            // per W_hh^T plane
  static constexpr int kP0 = tc::kM * (H + 16);   // h_prev plane 0 (+ ones column group)
  static constexpr int kP1 = tc::kM * H;          // h_prev plane 1
  static constexpr int kWih = 4 * H * tc::kKx;    // per W_ih plane, rows [r; z; 0; n]
  static constexpr int kX = tc::kM * tc::kKx;
  static constexpr size_t bytes = (size_t)(2 * kG + 2 * kW + kP0 + kP1 + 2 * kWih + kX) * 2 + 4 * H * 4 + 64;
};
// D[tmem] (+)= A[tmem] B[smem]: the A tile sits in tensor memory, lane = row, one 32-bit column = two consecutive K
// elements (K = 16 per instruction = 8 columns)
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, bool accum) {
  const uint32_t acc = accum ? 1u : 0u;
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// Warp-uniform issue: EVERY lane of the issuing warp executes these (uniform control flow, identical operands), the
// instruction itself is predicated on elect.sync.  With uniform operands ptxas keeps the descriptors in uniform
// registers and emits back-to-back UTCHMMA (3 instructions per MMA); issued from one lane of a divergent branch, each
// MMA costs two R2UR and an ELECT / BRA.U.ANY loop (~14 instructions, 80-100 cycles per MMA measured).
__device__ __forceinline__ void mma_f16_e(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void mma_f16_ts_e(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void commit_e(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(tc::smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tmem_st8u(uint32_t taddr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st4u(uint32_t taddr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
               ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3])
               : "memory");
}
// D = F32, A = B = FP16, M = 128; bit 15 / 16: A / B are MN-major
__device__ __forceinline__ uint32_t idesc_f16_major(int n, bool a_mn, bool b_mn) {
  return tc::idesc_f16(n) | (a_mn ? (1u << 15) : 0u) | (b_mn ? (1u << 16) : 0u);
}
}  // namespace tcr

// HS = H: d(gi) is added into a.dgi at the observation's time (fp32 reductions, order not fixed).
// HS = H | kDgiSlices (deterministic mode): window step s stores its d(gi) into slice s, a.slice_step floats from
// slice 0 = a.dgi, at the window's own time t; dgi_slice_sum_kernel then sums the L slices in a fixed order.
template <int HS>
__global__ void __launch_bounds__(tcr::kThreads, 1) gru_bptt_tc_kernel(const GruBpttArgs a) {
  using namespace tc;
  constexpr int H = HS & ~kDgiSlices;
  constexpr bool SLICES = (HS & kDgiSlices) != 0;
  using S = tcr::Smem<H>;
  static_assert(H == 32 || H == 64, "units per thread (H / 4) must be a multiple of 8");
  constexpr int UT = H / 4;            // hidden units per thread
  constexpr int K3 = 3 * H;            // gate rows
  constexpr int NP0 = H + 16;          // columns of h_prev plane 0 (ones column at index H)
  constexpr int NBLK = (K3 + 127) / 128;
  constexpr int XQ = kKx / 4;          // input features staged per thread
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __half* sg = reinterpret_cast<__half*>(smem_raw);                     // [2 planes][128][3H]
  __half* sw = sg + 2 * S::kG;                                          // [2 planes][H][3H]   (row = unit, k = gate row)
  __half* sp0 = sw + 2 * S::kW;                                         // [128][H + 16]
  __half* sp1 = sp0 + S::kP0;                                           // [128][H]
  __half* swih = sp1 + S::kP1;                                          // [2 planes][4H][kKx], rows [r; z; 0; n]
  __half* sx = swih + 2 * S::kWih;                                      // [128][kKx]
  float* bias = reinterpret_cast<float*>(sx + S::kX);                   // [2H] -(b_i + b_h) log2 e, [H] b_in, [H] b_hn
  uint64_t* bars = reinterpret_cast<uint64_t*>(bias + 4 * H);           // a_ready, r_ready, g_ready, d_ready, w_done
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);
  uint64_t *a_ready = bars, *r_ready = bars + 1, *g_ready = bars + 2, *d_ready = bars + 3, *w_done = bars + 4;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = blockIdx.y;
  const int I = a.in_dim[g];
  const float* Wih = a.w + g * a.w_agent_stride + a.wih_off[g];        // [3H][I]
  const float* Whh = a.w + g * a.w_agent_stride + a.whh_off[g];        // [3H][H] row-major
  const float* bih = a.w + g * a.w_agent_stride + a.bih_off[g];
  const float* bhh = a.w + g * a.w_agent_stride + a.bhh_off[g];

  // ---- one-time setup: 64 x weights -> two fp16 planes in the canonical layout ----
  for (int i = tid; i < K3 * H; i += tcr::kThreads) {
    const int j = i / H, u = i % H;                                     // coalesced read of W_hh[j][u]
    __half p0, p1;
    split2h1(kWScale * Whh[i], p0, p1);
    const int o = canon16(u, j, K3);
    sw[o] = p0, sw[S::kW + o] = p1;
  }
  for (int i = tid; i < 4 * H * kKx; i += tcr::kThreads) {
    const int n4 = i / kKx, k = i % kKx;          // row of the [r; z; 0; n] arrangement (gru_tc.cuh)
    const int n = n4 < 2 * H ? n4 : n4 - H;
    const bool zero = n4 >= 2 * H && n4 < 3 * H;
    __half p0, p1;
    split2h1((!zero && k < I) ? kWScale * Wih[(long long)n * I + k] : 0.f, p0, p1);
    const int o = canon16(n4, k, kKx);
    swih[o] = p0, swih[S::kWih + o] = p1;
  }
  // the ones column (unit index H) of h_prev plane 0 and its zero padding: constant for the whole kernel
  for (int i = tid; i < kM * 16; i += tcr::kThreads) {
    const int r = i / 16, c = i % 16;
    sp0[canon16(r, H + c, NP0)] = __float2half_rn(c == 0 ? 1.0f : 0.0f);
  }
  for (int i = tid; i < 4 * H; i += tcr::kThreads) {
    float v;
    if (i < 2 * H) v = -1.4426950408889634f * (bih[i] + bhh[i]);   // r, z: -(b_i + b_h) log2 e
    else if (i < 3 * H) v = bih[i];            // b_in
    else v = bhh[i - H];                       // b_hn
    bias[i] = v;
  }
  if (tid == 0) {
    mbar_init(a_ready, tcr::kGate), mbar_init(r_ready, 1), mbar_init(g_ready, tcr::kGate);
    mbar_init(d_ready, 1), mbar_init(w_done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr uint32_t kColsUsed = 4 * H + H + NBLK * NP0;
  constexpr uint32_t kColsAll = kColsUsed + (H == 64 ? 0 : 32);    // H = 32: h_{s-1} operand planes behind the accumulators
  constexpr uint32_t kCols = kColsAll <= 128 ? 128 : (kColsAll <= 256 ? 256 : 512);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;      // [0, 4H): recomputed pre-activations r | z | gh_n | gi_n (x 64)
  const uint32_t tmem_d = tmem + 4 * H;  // [4H, 5H): D = dh z + d(gh) W_hh (x 64 g_scale)
  const uint32_t tmem_dw = tmem + 5 * H; // weight-gradient accumulators: block blk at columns blk * NP0 (x g_scale)
  if (warp < 4) {                        // zero the weight-gradient accumulators once: every MMA accumulates
    const float zero[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int c0 = 0; c0 < NBLK * NP0; c0 += 8) tcb::tmem_st8(tmem_dw + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, zero);
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

  const int L = a.L;
  const int n_t = a.t1 - a.t0;
  const int blocks = (a.B + kM - 1) / kM;
  const int n_tiles = n_t * blocks;     // tile p = (env block p / n_t, time t0 + p % n_t): the <= L tiles that touch
                                        // one d(gi) element are processed close together (L2-resident reductions)
  const int quarter = warp >> 2;
  const int row = ((warp & 3) << 5) + lane;
  const uint32_t lane_addr = (uint32_t)((warp & 3) << 5) << 16;
  const int u0 = quarter * UT;
  const long long HB = (long long)H * a.B;
  const float gs = exp2f(10.0f - ceilf(log2f(fmaxf(*a.dh_absmax, 1e-30f))));
  const float d_scale = kWScale * gs, d_unscale = 1.0f / d_scale;
  const uint32_t id_x = idesc_f16(4 * H);                                  // x W_ih^T: both K-major, N = 4H
  const uint32_t id_h = tcr::idesc_f16_major(K3, false, true);             // h W_hh^T: B = W_hh^T tiles read MN-major
  const uint32_t id_d = idesc_f16(H);                                      // G W_hh: both K-major, N = H
  const uint32_t id_w0 = tcr::idesc_f16_major(NP0, true, true), id_w = tcr::idesc_f16_major(H, true, true);
  constexpr uint32_t ks_g = (K3 / 8) * 128, ks_p0 = (NP0 / 8) * 128, ks_p = (H / 8) * 128;   // 8-row group strides
  // h_{s-1} as the A operand of the recompute, in TENSOR memory (the shared-memory copy P is written later, in phase B,
  // for the weight-gradient GEMM only, so that GEMM can run behind the next step's recompute).  Plane i of hidden-unit
  // group j (16 units = one K step = 8 packed columns):
  //   H = 64: inside D's columns, at tmem_d + 16 j + 8 i -- the 16 columns of D that belong to the thread quarter j
  //           which also owns those units, so a thread only overwrites D columns it has read itself;
  //   H = 32: its own 32 columns behind the accumulators, at tmem_p + 16 i + 8 j (thread quarter q: 4 columns at + 4 q).
  const uint32_t tmem_p = H == 64 ? tmem_d : tmem + kColsUsed;
  int n_steps = 0;                      // window steps this CTA has staged so far
  int tr_n = 0;
  (void)tr_n;

  if (__shfl_sync(0xffffffffu, warp, 0) == tcr::kGate / 32) {
    // =================== MMA warp: issues every MMA, in the order  D(s), recompute(s - 1), dW(s)  ==================
    // so that the weight-gradient GEMM of a step runs on the tensor pipe while the CUDA cores are in the NEXT step's
    // gate phase (the pipe would idle there), and no gate warp ever blocks on a full MMA queue.  The whole warp runs
    // this code uniformly; the MMA / commit instructions are predicated on elect.sync (mma_f16_e).
    const uint32_t tm = __shfl_sync(0xffffffffu, tmem, 0);
    const uint32_t tm_d = tm + 4 * H, tm_dw = tm + 5 * H, tm_p = H == 64 ? tm_d : tm + kColsUsed;
    const uint64_t dg_k = desc16(smem_u32(sg), K3), dw_k = desc16(smem_u32(sw), K3);
    const uint64_t dw_mn = tcb::desc_mn(smem_u32(sw), ks_g, 128);            // [H rows = K][3H = N]
    const uint64_t dg_mn = tcb::desc_mn(smem_u32(sg), ks_g, 128);
    const uint64_t dp0_mn = tcb::desc_mn(smem_u32(sp0), ks_p0, 128), dp1_mn = tcb::desc_mn(smem_u32(sp1), ks_p, 128);
    const uint64_t dx_k = desc16(smem_u32(sx), kKx), dwih_k = desc16(smem_u32(swih), kKx);
    auto a_col = [&](int plane, int k16) { return H == 64 ? tm_p + 16 * k16 + 8 * plane : tm_p + 16 * plane + 8 * k16; };
    // dW += G^T P of the step whose G / P tiles are staged: both tiles read along their contiguous dimension,
    // reduction over the 128 rows; plane pairs g0 p0, g1 p0, g0 p1
    auto issue_dw = [&]() {
#pragma unroll
      for (int pr = 0; pr < 3; ++pr) {
        const int gi_ = pr == 1 ? 1 : 0;
#pragma unroll
        for (int k16 = 0; k16 < kM / 16; ++k16) {
          const uint64_t pd = pr < 2 ? desc_adv(dp0_mn, k16 * 2 * ks_p0) : desc_adv(dp1_mn, k16 * 2 * ks_p);
#pragma unroll
          for (int blk = 0; blk < NBLK; ++blk)
            tcr::mma_f16_e(tm_dw + (uint32_t)(blk * NP0), desc_adv(dg_mn, gi_ * S::kG * 2 + blk * 16 * 128 + k16 * 2 * ks_g),
                           pd, pr < 2 ? id_w0 : id_w, 1u);
        }
      }
      tcr::commit_e(w_done);
    };
    uint32_t ph_a = 0, ph_g = 0;
    bool dw_pending = false;
    for (int p = blockIdx.x; p < n_tiles; p += gridDim.x) {
#pragma unroll 1
      for (int s = L - 1; s >= 0; --s) {
        mbar_wait(a_ready, ph_a);
        ph_a ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // recompute: x W_ih^T initialises all 4H columns (zero block -> gh_n), h_{s-1} W_hh^T accumulates onto [0, 3H)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int k16 = 0; k16 < kKx / 16; ++k16)
            tcr::mma_f16_e(tm, desc_adv(dx_k, k16 * 256), desc_adv(dwih_k, j * S::kWih * 2 + k16 * 256), id_x,
                           j + k16 > 0 ? 1u : 0u);
        if (s > 0) {
#pragma unroll
          for (int pr = 0; pr < 3; ++pr) {          // h0 w0, h0 w1, h1 w0
            const int wi = pr == 1 ? 1 : 0;
#pragma unroll
            for (int k16 = 0; k16 < H / 16; ++k16)
              tcr::mma_f16_ts_e(tm, a_col(pr == 2 ? 1 : 0, k16), desc_adv(dw_mn, wi * S::kW * 2 + k16 * 2 * ks_g), id_h, 1u);
          }
        }
        tcr::commit_e(r_ready);
        if (dw_pending) issue_dw();             // the previous step's G / P tiles: behind this step's recompute
        mbar_wait(g_ready, ph_g);
        ph_g ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (s > 0) {
          // D += d(gh) W_hh : G K-major x W_hh^T K-major, plane pairs g0 w0, g0 w1, g1 w0 over 3H / 16 reduction steps
#pragma unroll
          for (int pr = 0; pr < 3; ++pr) {
            const int gi_ = pr == 2 ? 1 : 0, wi = pr == 1 ? 1 : 0;
#pragma unroll
            for (int k16 = 0; k16 < K3 / 16; ++k16)
              tcr::mma_f16_e(tm_d, desc_adv(dg_k, gi_ * S::kG * 2 + k16 * 256), desc_adv(dw_k, wi * S::kW * 2 + k16 * 256),
                             id_d, 1u);
          }
          tcr::commit_e(d_ready);
        }
        dw_pending = true;
      }
    }
    if (dw_pending) issue_dw();                 // flush: the last step staged
    __syncwarp();
  } else {
  // =================== gate warps ==================================================================================
  uint32_t ph_r = 0, ph_d = 0, ph_w = 0;
  for (int p = blockIdx.x; p < n_tiles; p += gridDim.x) {
    const int t = a.t0 + p % n_t;
    const int b = (p / n_t) * kM + row;
    const bool ok = b < a.B;
    const int bb = ok ? b : 0;
    float dh[UT], hp[UT], xq[XQ];
    {
      const float* dp = view_ptr(a.dh, g, t, a.B, bb) + (long long)u0 * a.B;
#pragma unroll
      for (int u = 0; u < UT; ++u) dh[u] = ok ? dp[(long long)u * a.B] : 0.f;
    }
    auto load_step = [&](int s) {      // h_{s-1} of this thread's units and its share of x_s
      if (s > 0) {
        const float* hq = view_ptr(a.hs, g, t, a.B, bb) + (long long)(s - 1) * a.hs_step + (long long)u0 * a.B;
#pragma unroll
        for (int u = 0; u < UT; ++u) hp[u] = ok ? hq[(long long)u * a.B] : 0.f;
      } else {
#pragma unroll
        for (int u = 0; u < UT; ++u) hp[u] = 0.f;
      }
      const float* xp = view_ptr(a.x, g, t - (L - 1 - s), a.B, bb);
#pragma unroll
      for (int k = 0; k < XQ; ++k) {
        const int kk = quarter * XQ + k;
        xq[k] = (ok && kk < I) ? xp[(long long)kk * a.B] : 0.f;
      }
    };
    load_step(L - 1);
    for (int s = L - 1; s >= 0; --s) {
      float* gp = SLICES ? view_ptr(a.dgi, g, t, a.B, bb) + s * a.slice_step + (long long)u0 * a.B
                         : view_ptr(a.dgi, g, t - (L - 1 - s), a.B, bb) + (long long)u0 * a.B;
      D2D_TR(0);
      // ---- A. h_{s-1} (2 planes) -> tensor memory, X = x_s -> shared memory ----
      // (D's columns are free: this thread read its own in phase C, the MMAs that wrote them completed before that;
      //  X was last read by the previous recompute, which completed before the previous phase B)
      if (s > 0) {
        uint32_t q0[UT / 2], q1[UT / 2];
#pragma unroll
        for (int j = 0; j < UT / 2; ++j) split2h(hp[2 * j], hp[2 * j + 1], q0[j], q1[j]);
        if constexpr (H == 64) {
          tcr::tmem_st8u(tmem_p + lane_addr + (uint32_t)(16 * quarter), q0);
          tcr::tmem_st8u(tmem_p + lane_addr + (uint32_t)(16 * quarter + 8), q1);
        } else {
          tcr::tmem_st4u(tmem_p + lane_addr + (uint32_t)(4 * quarter), q0);
          tcr::tmem_st4u(tmem_p + lane_addr + (uint32_t)(16 + 4 * quarter), q1);
        }
      }
      {
        const __half2 a0 = __floats2half2_rn(xq[0], xq[1]), a1 = __floats2half2_rn(xq[2], xq[3]);
        const __half2 a2 = __floats2half2_rn(xq[4], xq[5]), a3 = __floats2half2_rn(xq[6], xq[7]);
        uint4 v;
        v.x = *reinterpret_cast<const uint32_t*>(&a0), v.y = *reinterpret_cast<const uint32_t*>(&a1);
        v.z = *reinterpret_cast<const uint32_t*>(&a2), v.w = *reinterpret_cast<const uint32_t*>(&a3);
        *reinterpret_cast<uint4*>(sx + canon16(row, quarter * XQ, kKx)) = v;
      }
      if (s > 0) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(a_ready);
      D2D_TR(1);
      mbar_wait(r_ready, ph_r);
      ph_r ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      D2D_TR(2);
      // ---- B. gates from the recomputed pre-activations, derivatives, G = d(gh), d(gi), direct path into D ----
#pragma unroll
      for (int c = 0; c < UT / 8; ++c) {
        float pr[8], pz[8], pin[8], phn[8];
        const uint32_t d = tmem + lane_addr + (uint32_t)(u0 + c * 8);
        tmem_ld8(d, pr);
        tmem_ld8(d + H, pz);
        tmem_ld8(d + 3 * H, pin);
        tmem_ld8(d + 2 * H, phn);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const float4* bz = reinterpret_cast<const float4*>(bias + u0 + c * 8);
        const float4 br0 = bz[0], br1 = bz[1];
        const float4 bz0 = bz[H / 4], bz1 = bz[H / 4 + 1];
        const float4 bi0 = bz[2 * H / 4], bi1 = bz[2 * H / 4 + 1];
        const float4 bh0 = bz[3 * H / 4], bh1 = bz[3 * H / 4 + 1];
        const float b_r[8] = {br0.x, br0.y, br0.z, br0.w, br1.x, br1.y, br1.z, br1.w};
        const float b_z[8] = {bz0.x, bz0.y, bz0.z, bz0.w, bz1.x, bz1.y, bz1.z, bz1.w};
        const float b_i[8] = {bi0.x, bi0.y, bi0.z, bi0.w, bi1.x, bi1.y, bi1.z, bi1.w};
        const float b_h[8] = {bh0.x, bh0.y, bh0.z, bh0.w, bh1.x, bh1.y, bh1.z, bh1.w};
        constexpr float kSig = -1.4426950408889634f * kInvWScale;
        float dg[3][8], dd[8];               // dr, dz, dn r of 8 units (x g_scale); direct path (x 64 g_scale)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int u = c * 8 + j;
          const float r = rcp_approx(1.0f + ex2_approx(fmaf(pr[j], kSig, b_r[j])));
          const float z = rcp_approx(1.0f + ex2_approx(fmaf(pz[j], kSig, b_z[j])));
          const float ghn = fmaf(phn[j], kInvWScale, b_h[j]);
          const float pre = fmaf(r, ghn, fmaf(pin[j], kInvWScale, b_i[j]));
          const float nn = fmaf(-2.0f, rcp_approx(1.0f + ex2_approx(2.8853900817779268f * pre)), 1.0f);
          const float dv = ok ? dh[u] : 0.f;
          const float dn = dv * (1.0f - z) * (1.0f - nn * nn);
          const float dz = dv * (hp[u] - nn) * z * (1.0f - z);
          const float dr = dn * ghn * r * (1.0f - r);
          dg[0][j] = dr * gs, dg[1][j] = dz * gs, dg[2][j] = dn * r * gs;
          dd[j] = dv * z * d_scale;          // direct path: pre-loaded into D, d(gh) W_hh accumulates on top
          if (ok) {
            const long long f = (long long)u * a.B;
            if constexpr (SLICES) gp[f] = dr, gp[f + HB] = dz, gp[f + 2 * HB] = dn;
            else atomicAdd(gp + f, dr), atomicAdd(gp + f + HB, dz), atomicAdd(gp + f + 2 * HB, dn);
          }
        }
        if (c == 0) D2D_TR(3);
        if (c == 0 && n_steps > 0) {         // G and P are free once the previous step's weight-gradient MMAs are done
          mbar_wait(w_done, ph_w);
          ph_w ^= 1u;
        }
        if (c == 0) D2D_TR(4);
        if (s > 0) tcb::tmem_st8(tmem_d + lane_addr + (uint32_t)(u0 + c * 8), dd);
#pragma unroll
        for (int gate = 0; gate < 3; ++gate) {
          uint32_t w0[4], w1[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) split2h(dg[gate][2 * j], dg[gate][2 * j + 1], w0[j], w1[j]);
          __half* dst = sg + canon16(row, gate * H + u0 + c * 8, K3);
          *reinterpret_cast<uint4*>(dst) = make_uint4(w0[0], w0[1], w0[2], w0[3]);
          *reinterpret_cast<uint4*>(dst + S::kG) = make_uint4(w1[0], w1[1], w1[2], w1[3]);
        }
        {                                    // P = h_{s-1} (2 planes) for the weight-gradient GEMM
          uint32_t q0[4], q1[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) split2h(hp[c * 8 + 2 * j], hp[c * 8 + 2 * j + 1], q0[j], q1[j]);
          *reinterpret_cast<uint4*>(sp0 + canon16(row, u0 + c * 8, NP0)) = make_uint4(q0[0], q0[1], q0[2], q0[3]);
          *reinterpret_cast<uint4*>(sp1 + canon16(row, u0 + c * 8, H)) = make_uint4(q1[0], q1[1], q1[2], q1[3]);
        }
      }
      if (s > 0) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(g_ready);
      D2D_TR(5);
      ++n_steps;
      if (s == 0) { ++tr_n; break; }         // dh of the zero initial state is not needed
      load_step(s - 1);                      // in flight while the tensor pipe works (h_{s-1}'s registers are free now)
      D2D_TR(6);
      // ---- C. dh_prev = (dh z + d(gh) W_hh) from D ----
      mbar_wait(d_ready, ph_d);
      ph_d ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      D2D_TR(7);
#pragma unroll
      for (int c = 0; c < UT / 8; ++c) {
        float v[8];
        tmem_ld8(tmem_d + lane_addr + (uint32_t)(u0 + c * 8), v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 8; ++j) dh[c * 8 + j] = v[j] * d_unscale;
      }
      D2D_TR(8);
      ++tr_n;
    }
  }
  // the flush's weight-gradient MMAs (the accumulators are read below)
  if (n_steps > 0) {
    mbar_wait(w_done, ph_w);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  }   // gate warps
  const bool any_tile = (int)blockIdx.x < n_tiles;
  const bool staged_before = any_tile;
  // ---- partial dW_hh / db_hh of this CTA: accumulator row = gate row (TMEM lane), column = unit, column H = bias ----
  if (warp < 4) {
    float* out = a.partial + ((long long)g * gridDim.x + blockIdx.x) * a.part_stride;
    const float unscale = 1.0f / gs;
    for (int blk = 0; blk < NBLK; ++blk) {
      const int j = blk * 128 + warp * 32 + lane;      // gate row
      const uint32_t d = tmem_dw + ((uint32_t)(warp * 32) << 16) + (uint32_t)(blk * NP0);
      for (int c0 = 0; c0 < NP0; c0 += 8) {
        float v[8];
        if (staged_before) {
          tmem_ld8(d + c0, v);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) v[q] = 0.f;
        }
        if (j < K3) {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const int k = c0 + q;
            if (k < H) out[(long long)j * H + k] = v[q] * unscale;
            else if (k == H) out[(long long)K3 * H + j] = v[q] * unscale;
          }
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kCols));
}

}  // namespace d2d
