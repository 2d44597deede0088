// Fused back-propagation through the GRU window on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// For every row (agent g, time t, env b) the L steps of the training window are walked backwards with d(h) held in
// registers (reference: autograd through nn.GRU inside PPO.train_step, algorithms/d2d_ppo.py:198-216 with the
// windows of preprocess_input_for_rnn, :385-398):
//
//   dn  = dh (1 - z)(1 - n^2)      dz = dh (h_prev - n) z (1 - z)      dr = dn gh_n r (1 - r)
//   d(gh) = (dr, dz, dn r)         d(gi) = (dr, dz, dn)                dh_prev = dh z + d(gh) W_hh
//   dW_hh += d(gh)^T h_prev        db_hh += sum_rows d(gh)
//
// replaces, per step, gru_gate_bwd_kernel + the K = 3H data-gradient GEMM + the W_hh weight-gradient GEMM and their
// d(h) / d(gh) round trips through HBM.  Per row-step the kernel reads r, z, n, gh_n, h_prev (5H floats, written by
// the forward window kernel in store mode); d(gi) of the observation the step looked at is accumulated with fp32
// reductions (red.global.add: up to L windows share an observation) for the W_ih weight gradient; nothing else is
// written until the CTA stores its partial dW_hh / db_hh at the end (summed over CTAs by wreduce_kernel).
//
// CTA = 16 warps on ONE 128-row tile (512 threads leave 128 registers each): warp w serves TMEM lane quadrant w % 4
// (row = 32 (w % 4) + lane) and the hidden units of quarter w / 4.  Lane 0 of EVERY warp issues a share of the step's
// 140 MMAs: a single issuing thread needs ~18 instructions per tcgen05.mma and was the critical path (5 of 11 us per
// tile-step).  Concurrent issue needs order-free accumulation: D is pre-loaded with the direct path dh z through
// tcgen05.st and the dW accumulators are zeroed once, so every MMA accumulates.
// Per step the threads write two operand tiles in the canonical no-swizzle layout (16-byte vectors, thread = row):
//   G = d(gh)   [128 rows][3H]   2 bf16 planes (hi + lo, round to nearest: 16 significant bits, unbiased)
//   P = h_prev  [128 rows][H]    3 bf16 planes (+ a constant ones column in plane 0 for the bias gradient)
// and two GEMMs run on them:
//   D  [128 rows][H]  = G W_hh          G is K-major (gates contiguous), W_hh^T resident as [H][3H] K-major, 3 planes
//   dW [3H][H (+1)]  += G^T P           the SAME tiles read M-major / N-major (reduction over the 128 rows): no
//                                       transposition pass; accumulators stay in TMEM for the whole kernel
// with the plane products (g0 w0, g0 w1, g0 w2, g1 w0, g1 w1) resp. (g0 p0, g1 p0, g0 p1, g0 p2, g1 p1).
// The weight-gradient MMAs of step s overlap the gate maths of step s - 1; only the restaging waits for them.
// Shared memory (H = 64): G 2 x 48 KB + W_hh^T 3 x 24 KB + P 20 + 2 x 16 KB = 220 KB; TMEM: H + 2 (H + 16) columns.
#pragma once
#include "gru_tc.cuh"

namespace d2d {

struct GruBwdTcArgs {
  View acts;   // [.. 4H ..] step 0; step s is acts_step floats further: r, z, n, gh_n
  View hs;     // [.. H ..]  h after step 0; step s is hs_step floats further
  View dh;     // [.. H ..]  in: d(loss) / d(h after the last step)
  View dgi;    // [.. 3H ..] accumulated at observation time t - (L - 1 - s); zeroed by the caller (the slices kernel:
               // slice 0 of the [L][..] d(gi) slices, written at time t)
  const float* w;
  long long w_agent_stride;
  int whh_off[D2D_MAX_AGENTS];
  float* partial;        // [N][gridDim.x][part_stride]: dW_hh [3H][H] then db_hh [3H], one partial per CTA
  long long part_stride;
  long long acts_step, hs_step;
  int L, B, t0, t1;
  long long slice_step;    // kDgiSlices instantiation: floats between two d(gi) slices
};

// or-ed into the H template argument of the BPTT kernels: d(gi) per window step into slices (deterministic mode)
constexpr int kDgiSlices = 1024;

namespace tcb {
constexpr int kThreads = 512;
template <int H>
struct Smem {
  static constexpr int kG = tc::kM * 3 * H;       // bf16 elements per d(gh) plane
  static constexpr int kW = H * 3 * H;            // per W_hh^T plane
  static constexpr int kP0 = tc::kM * (H + 16);   // h_prev plane 0 (+ ones column group)
  static constexpr int kP = tc::kM * H;           // h_prev planes 1, 2
  static constexpr size_t bytes = (size_t)(2 * kG + 3 * kW + kP0 + 2 * kP) * 2 + 64;
};
// no-swizzle descriptor of an operand read along its contiguous dimension (MN-major): 8 (K) x 8 (MN) core matrices
// of 128 bytes; sbo = bytes between core matrices adjacent in MN, lbo = bytes between core matrices adjacent in K
// (verified on B200: LBO is the K-direction stride, SBO the MN-direction stride; the other assignment faults)
__device__ __forceinline__ uint64_t desc_mn(uint32_t saddr, uint32_t k_stride, uint32_t mn_stride) {
  const uint64_t start = (saddr & 0x3FFFFu) >> 4;
  const uint64_t lbo = k_stride >> 4, sbo = mn_stride >> 4;
  return start | (lbo << 16) | (sbo << 32) | (1ull << 46);
}
// D = F32, A = B = BF16, M = 128; bit 15 / 16: A / B are MN-major
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                 "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                 "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
               : "memory");
}
__device__ __forceinline__ uint32_t idesc_bf16_mn(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(tc::kM >> 4) << 24);
}
}  // namespace tcb

// HS = H | kDgiSlices (deterministic mode): d(gi) of window step s is stored into slice s (a.slice_step floats from
// slice 0 = a.dgi) at the window's own time, for dgi_slice_sum_kernel; HS = H: added atomically as described above.
template <int HS>
__global__ void __launch_bounds__(tcb::kThreads, 1) gru_bwd_tc_kernel(const GruBwdTcArgs a) {
  using namespace tc;
  constexpr int H = HS & ~kDgiSlices;
  constexpr bool SLICES = (HS & kDgiSlices) != 0;
  // MMAs that accumulate into one TMEM tile run in issue order, and the order of issue across warps is not fixed: the
  // deterministic variant issues every MMA from warp 0 in a fixed order
  constexpr int kIssuers = SLICES ? 1 : tcb::kThreads / 32;
  using S = tcb::Smem<H>;
  static_assert(H == 32 || H == 64, "units per thread (H / 4) must be a multiple of 8");
  constexpr int UT = H / 4;            // hidden units per thread
  constexpr int K3 = 3 * H;            // gate rows
  constexpr int NP0 = H + 16;          // columns of h_prev plane 0 (ones column at index H)
  constexpr int NBLK = (K3 + 127) / 128;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __nv_bfloat16* sg = reinterpret_cast<__nv_bfloat16*>(smem_raw);      // [2 planes][128][3H]
  __nv_bfloat16* sw = sg + 2 * S::kG;                                   // [3 planes][H][3H]   (n = unit, k = gate row)
  __nv_bfloat16* sp0 = sw + 3 * S::kW;                                  // [128][H + 16]
  __nv_bfloat16* sp1 = sp0 + S::kP0;                                    // [2 planes][128][H]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sp1 + 2 * S::kP);        // a_ready, d_ready, w_done
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);
  uint64_t *a_ready = bars, *d_ready = bars + 1, *w_done = bars + 2;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = blockIdx.y;
  const float* Whh = a.w + g * a.w_agent_stride + a.whh_off[g];        // [3H][H] row-major

  for (int i = tid; i < K3 * H; i += tcb::kThreads) {
    const int j = i / H, u = i % H;                                     // coalesced read of W_hh[j][u]
    __nv_bfloat16 p0, p1, p2;
    split3(Whh[i], p0, p1, p2);
    const int o = canon16(u, j, K3);
    sw[o] = p0, sw[S::kW + o] = p1, sw[2 * S::kW + o] = p2;
  }
  // the ones column (unit index H) of h_prev plane 0 and its zero padding: constant for the whole kernel
  for (int i = tid; i < kM * 16; i += tcb::kThreads) {
    const int r = i / 16, c = i % 16;
    sp0[canon16(r, H + c, NP0)] = __float2bfloat16_rn(c == 0 ? 1.0f : 0.0f);
  }
  if (tid == 0) {
    mbar_init(a_ready, tcb::kThreads), mbar_init(d_ready, kIssuers), mbar_init(w_done, kIssuers);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  constexpr uint32_t kColsUsed = H + NBLK * NP0;
  constexpr uint32_t kCols = kColsUsed <= 32 ? 32 : (kColsUsed <= 64 ? 64 : (kColsUsed <= 128 ? 128 : 256));
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(kCols));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_dw = tmem + H;     // weight-gradient accumulators: block blk at columns blk * NP0
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
  uint32_t ph_d = 0, ph_a = 0, ph_w = 0;
  bool staged_before = false;           // a weight-gradient batch is (or was) in flight on the operand tiles
  const uint32_t id_d = idesc_bf16(H);
  const uint32_t id_w0 = tcb::idesc_bf16_mn(NP0), id_w = tcb::idesc_bf16_mn(H);
  // base descriptors, built once (desc_adv moves the start address only)
  constexpr uint32_t ks_g = (K3 / 8) * 128, ks_p0 = (NP0 / 8) * 128, ks_p = (H / 8) * 128;   // K (row group) strides
  const uint64_t dg_k = desc16(smem_u32(sg), K3), dw_k = desc16(smem_u32(sw), K3);
  const uint64_t dg_mn = tcb::desc_mn(smem_u32(sg), ks_g, 128);
  const uint64_t dp0_mn = tcb::desc_mn(smem_u32(sp0), ks_p0, 128), dp1_mn = tcb::desc_mn(smem_u32(sp1), ks_p, 128);

  for (int p = blockIdx.x; p < n_tiles; p += gridDim.x) {
    const int t = a.t0 + p % n_t;
    const int b = (p / n_t) * kM + row;
    const bool ok = b < a.B;
    const int bb = ok ? b : 0;
    float dh[UT];
    float r[UT], z[UT], nn[UT], ghn[UT], hp[UT];
    {
      const float* dp = view_ptr(a.dh, g, t, a.B, bb) + (long long)u0 * a.B;
#pragma unroll
      for (int u = 0; u < UT; ++u) dh[u] = ok ? dp[(long long)u * a.B] : 0.f;
    }
    auto load_step = [&](int s) {
      const float* ap = view_ptr(a.acts, g, t, a.B, bb) + (long long)s * a.acts_step + (long long)u0 * a.B;
#pragma unroll
      for (int u = 0; u < UT; ++u) {
        const long long f = (long long)u * a.B;
        r[u] = ap[f], z[u] = ap[f + HB], nn[u] = ap[f + 2 * HB], ghn[u] = ap[f + 3 * HB];
      }
      if (s > 0) {
        const float* hq = view_ptr(a.hs, g, t, a.B, bb) + (long long)(s - 1) * a.hs_step + (long long)u0 * a.B;
#pragma unroll
        for (int u = 0; u < UT; ++u) hp[u] = hq[(long long)u * a.B];
      } else {
#pragma unroll
        for (int u = 0; u < UT; ++u) hp[u] = 0.f;
      }
    };
    load_step(L - 1);
    for (int s = L - 1; s >= 0; --s) {
      float* gp = SLICES ? view_ptr(a.dgi, g, t, a.B, bb) + s * a.slice_step + (long long)u0 * a.B
                         : view_ptr(a.dgi, g, t - (L - 1 - s), a.B, bb) + (long long)u0 * a.B;
      // the operand tiles are free once the weight-gradient MMAs of the previous staging have completed
      if (staged_before) {
        mbar_wait(w_done, ph_w);
        ph_w ^= 1u;
      }
      staged_before = true;
#pragma unroll
      for (int c = 0; c < UT / 8; ++c) {
        float dg[3][8];                      // dr, dz, dn r of 8 units
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int u = c * 8 + j;
          const float d = ok ? dh[u] : 0.f;
          const float dn = d * (1.0f - z[u]) * (1.0f - nn[u] * nn[u]);
          const float dz = d * (hp[u] - nn[u]) * z[u] * (1.0f - z[u]);
          const float dr = dn * ghn[u] * r[u] * (1.0f - r[u]);
          dg[0][j] = dr, dg[1][j] = dz, dg[2][j] = dn * r[u];
          dh[u] = d * z[u];                  // direct path: pre-loaded into D, d(gh) W_hh accumulates on top
          if (ok) {
            const long long f = (long long)u * a.B;
            if constexpr (SLICES) gp[f] = dr, gp[f + HB] = dz, gp[f + 2 * HB] = dn;
            else atomicAdd(gp + f, dr), atomicAdd(gp + f + HB, dz), atomicAdd(gp + f + 2 * HB, dn);
          }
        }
        if (s > 0) tcb::tmem_st8(tmem + lane_addr + (uint32_t)(u0 + c * 8), &dh[c * 8]);
#pragma unroll
        for (int gate = 0; gate < 3; ++gate) {
          uint32_t w0[4], w1[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float x0 = dg[gate][2 * j], x1 = dg[gate][2 * j + 1];
            const __nv_bfloat162 hi = __floats2bfloat162_rn(x0, x1);
            const __nv_bfloat162 lo = __floats2bfloat162_rn(x0 - __low2float(hi), x1 - __high2float(hi));
            w0[j] = *reinterpret_cast<const uint32_t*>(&hi), w1[j] = *reinterpret_cast<const uint32_t*>(&lo);
          }
          __nv_bfloat16* dst = sg + canon16(row, gate * H + u0 + c * 8, K3);
          *reinterpret_cast<uint4*>(dst) = make_uint4(w0[0], w0[1], w0[2], w0[3]);
          *reinterpret_cast<uint4*>(dst + S::kG) = make_uint4(w1[0], w1[1], w1[2], w1[3]);
        }
        {   // h_prev -> three planes (zero at s = 0: only the ones column contributes, i.e. the bias gradient)
          uint32_t q0[8], q1[8], q2[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) split3_trunc(ok ? hp[c * 8 + j] : 0.f, q0[j], q1[j], q2[j]);
          *reinterpret_cast<uint4*>(sp0 + canon16(row, u0 + c * 8, NP0)) =
              make_uint4(pack_hi(q0[0], q0[1]), pack_hi(q0[2], q0[3]), pack_hi(q0[4], q0[5]), pack_hi(q0[6], q0[7]));
          const int o = canon16(row, u0 + c * 8, H);
          *reinterpret_cast<uint4*>(sp1 + o) =
              make_uint4(pack_hi(q1[0], q1[1]), pack_hi(q1[2], q1[3]), pack_hi(q1[4], q1[5]), pack_hi(q1[6], q1[7]));
          *reinterpret_cast<uint4*>(sp1 + S::kP + o) =
              make_uint4(pack_hi(q2[0], q2[1]), pack_hi(q2[2], q2[3]), pack_hi(q2[4], q2[5]), pack_hi(q2[6], q2[7]));
        }
      }
      if (s > 0) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive(a_ready);
      if (lane == 0 && (!SLICES || warp == 0)) {
        mbar_wait(a_ready, ph_a);
        ph_a ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        constexpr int kWarps = kIssuers;
        if (s > 0) {
          // D += d(gh) W_hh : G K-major x W_hh^T K-major, five plane products x 3H / 16 reduction steps, dealt round
          // robin to the warps' issuing lanes
          constexpr int kPer = K3 / 16;
          for (int m = warp; m < 5 * kPer; m += kWarps) {
            const int pr = m / kPer, k16 = m % kPer;
            const int gi_ = pr < 3 ? 0 : 1, wi = pr < 3 ? pr : pr - 3;
            mma_bf16(tmem, desc_adv(dg_k, gi_ * S::kG * 2 + k16 * 256), desc_adv(dw_k, wi * S::kW * 2 + k16 * 256), id_d,
                     true);
          }
          asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                       ::"r"(smem_u32(d_ready))
                       : "memory");
        }
        // dW += G^T P : both tiles read along their contiguous dimension, reduction over the 128 rows
        constexpr int kPerW = (kM / 16) * NBLK;
        for (int m = warp; m < 5 * kPerW; m += kWarps) {
          const int pr = m / kPerW, k16 = (m % kPerW) / NBLK, blk = m % NBLK;
          const int gi_ = (pr == 1 || pr == 4) ? 1 : 0;          // (g0 p0) (g1 p0) (g0 p1) (g0 p2) (g1 p1)
          const int pi = pr < 2 ? 0 : (pr == 3 ? 2 : 1);
          const uint64_t pd = pi == 0 ? desc_adv(dp0_mn, k16 * 2 * ks_p0)
                                      : desc_adv(dp1_mn, (pi - 1) * S::kP * 2 + k16 * 2 * ks_p);
          mma_bf16(tmem_dw + (uint32_t)(blk * NP0), desc_adv(dg_mn, gi_ * S::kG * 2 + blk * 16 * 128 + k16 * 2 * ks_g),
                   pd, pi == 0 ? id_w0 : id_w, true);
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                     ::"r"(smem_u32(w_done))
                     : "memory");
      }
      __syncwarp();
      if (s == 0) break;                     // dh of the zero initial state is not needed
      load_step(s - 1);                      // in flight while the tensor pipe works
      mbar_wait(d_ready, ph_d);
      ph_d ^= 1u;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int c = 0; c < UT / 8; ++c) {
        float v[8];
        tmem_ld8(tmem + lane_addr + (uint32_t)(u0 + c * 8), v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 8; ++j) dh[c * 8 + j] = v[j];      // dh z + d(gh) W_hh
      }
    }
  }
  // ---- partial dW_hh / db_hh of this CTA: accumulator row = gate row (TMEM lane), column = unit, column H = bias ----
  if (staged_before) {
    mbar_wait(w_done, ph_w);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  }
  if (warp < 4) {
    float* out = a.partial + ((long long)g * gridDim.x + blockIdx.x) * a.part_stride;
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
            if (k < H) out[(long long)j * H + k] = v[q];
            else if (k == H) out[(long long)K3 * H + j] = v[q];
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
