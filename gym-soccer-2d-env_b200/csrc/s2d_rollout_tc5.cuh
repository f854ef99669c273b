// s2d_rollout_tc5.cuh - the closed-loop Q-network rollout of s2d_rollout.cuh with the network on the 5th-generation
// tensor cores: tcgen05.mma (kind::tf32), accumulators and the activations of layers 2 and 3 in tensor memory.
//
// A 128-thread block is exactly one M = 128 tile: thread t = episode t = TMEM lane t.  Per closed-loop cycle
//
//   obs row (registers, TF32-rounded)  --tcgen05.st-->  A1  [128 lanes x 16 columns]           (region RA of TMEM)
//   layer 1   D1 [128 x 64] = A1 . W1^T          2 x tcgen05.mma (K = 8 each), B = W1 from shared memory   -> region RD
//   epilogue  D1 --tcgen05.ld--> registers: + bias, ReLU, round to TF32 --tcgen05.st--> A2 [128 x 64]     -> region RA
//   layer 2   D2 = A2 . W2^T                     8 x tcgen05.mma, A from TMEM                              -> region RD
//   epilogue  as above -> A3
//   layer 3   Q  [128 x 16 | 32] = A3 . W3^T     8 x tcgen05.mma                                           -> region RD
//   Q row --tcgen05.ld--> registers: + bias, argmax in the thread (its own row: no cross-lane reduction) -> action -> step
//
// One elected thread issues the MMAs of a layer and commits them to an mbarrier the block waits on; the epilogues are
// block-wide (every thread its own row).  TMEM: 128 columns per block (RD 64 + RA 64), allocated once per block, so the
// four resident blocks of an SM share its 512 columns.  Weights sit in shared memory in the canonical K-major,
// no-swizzle core-matrix layout (8 rows x 16 bytes per core matrix) that the shared-memory descriptors describe:
// element (n, k) of W [N][K] at float ((k / 4) * (N / 8) + n / 8) * 32 + (n % 8) * 4 + k % 4;
// leading-dimension byte offset (the two 16-byte K chunks of one MMA) = N / 8 * 128, stride byte offset (8-row groups) = 128.
// The env half of the cycle is the code of s2d_scenarios.cuh, unchanged (bit-exact by the replay test).
#pragma once
#include "s2d_rollout.cuh"

#ifndef S2D_ROLLOUT_DRAW_MEMO
#define S2D_ROLLOUT_DRAW_MEMO true
#endif
namespace s2d {

#ifndef S2D_HOST_EMU

constexpr int kTc5Hidden = 64;

struct Tc5Shared {
  alignas(128) float w1[16 * kTc5Hidden];          // W1 [64][16]  (10 real input features, the rest zero)
  alignas(128) float w2[kTc5Hidden * kTc5Hidden];  // W2 [64][64]
  alignas(128) float w3[32 * kTc5Hidden];          // W3 [N3][64], N3 = 16 (ReachBall) or 32 (Shoot: 24 real)
  alignas(16) float b1[kTc5Hidden], b2[kTc5Hidden], b3[32];
  alignas(8) unsigned long long mbar;
  uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// float offset of W[n][k] in the core-matrix layout of an [N][K] K-major operand
__device__ __forceinline__ int tc5_core_offset(int n, int k, int N) { return ((k >> 2) * (N >> 3) + (n >> 3)) * 32 + (n & 7) * 4 + (k & 3); }

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): K-major, SWIZZLE_NONE, version 1 (Blackwell)
__device__ __forceinline__ uint64_t tc5_smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4) | (static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         (static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, M = 128
__host__ __device__ constexpr uint32_t tc5_idesc(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(128 >> 4) << 24);
}

__device__ __forceinline__ void tc5_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(static_cast<uint32_t>(accumulate))
      : "memory");
}
__device__ __forceinline__ void tc5_commit(uint32_t mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void tc5_wait(uint32_t mbar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(ok)
        : "r"(mbar), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tc5_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc5_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Round-to-nearest (ties away) to TF32 for an operand the tensor core reads: the MMA ignores the low 13 mantissa bits, so
// adding half a TF32 ulp to the bit pattern is the whole rounding (what cvt.rna.tf32.f32 takes three instructions for).
__device__ __forceinline__ float tc5_round(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }

// 16 consecutive columns of this thread's TMEM lane <-> registers
__device__ __forceinline__ void tc5_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
      "tcgen05.wait::ld.sync.aligned;"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc5_st16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
      "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
      "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
      "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
      : "memory");
}
__device__ __forceinline__ void tc5_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// weights (torch nn.Linear layout, device pointers) -> shared memory, TF32-rounded, core-matrix layout
template <int N3>
__device__ __forceinline__ void tc5_load_weights(Tc5Shared& s, const MlpWeights& w) {
  for (int idx = threadIdx.x; idx < 16 * kTc5Hidden; idx += blockDim.x) {
    const int n = idx / 16, k = idx % 16;
    s.w1[tc5_core_offset(n, k, kTc5Hidden)] = k < w.obs_dim ? to_tf32(__ldg(w.w1 + n * w.obs_dim + k)) : 0.0f;
  }
  for (int idx = threadIdx.x; idx < kTc5Hidden * kTc5Hidden; idx += blockDim.x) {
    const int n = idx / kTc5Hidden, k = idx % kTc5Hidden;
    s.w2[tc5_core_offset(n, k, kTc5Hidden)] = to_tf32(__ldg(w.w2 + idx));
  }
  for (int idx = threadIdx.x; idx < N3 * kTc5Hidden; idx += blockDim.x) {
    const int n = idx / kTc5Hidden, k = idx % kTc5Hidden;
    s.w3[tc5_core_offset(n, k, N3)] = n < w.n_actions ? to_tf32(__ldg(w.w3 + idx)) : 0.0f;
  }
  for (int idx = threadIdx.x; idx < kTc5Hidden; idx += blockDim.x) {
    s.b1[idx] = __ldg(w.b1 + idx);
    s.b2[idx] = __ldg(w.b2 + idx);
    if (idx < 32) s.b3[idx] = idx < w.n_actions ? __ldg(w.b3 + idx) : -3.0e38f;  // absent actions never win
  }
}

// one layer's MMAs (issued by ONE thread): D[128 x N] (+)= A[128 x K] . W^T, K / 8 instructions, then the commit
__device__ __forceinline__ void tc5_issue_layer(uint32_t d_tmem, uint32_t a_tmem, const float* w_smem, int n, int k_total,
                                                uint32_t mbar) {
  const uint32_t lbo = static_cast<uint32_t>(n >> 3) * 128u, w_addr = smem_u32(w_smem);
  const uint32_t idesc = tc5_idesc(n);
  tc5_fence_after();
  for (int ks = 0; ks < (k_total >> 3); ++ks)
    tc5_mma_ts(d_tmem, a_tmem + 8u * ks, tc5_smem_desc(w_addr + 2u * ks * lbo, lbo, 128u), idesc, ks > 0);
  tc5_commit(mbar);
}

// the hidden-layer epilogue of this thread's row: D (64 columns at d_tmem) -> + bias, ReLU, TF32 -> A (64 columns at a_tmem)
__device__ __forceinline__ void tc5_hidden_epilogue(uint32_t d_tmem, uint32_t a_tmem, const float* bias) {
#pragma unroll 1
  for (int c = 0; c < kTc5Hidden; c += 16) {  // (32 columns at a time: measured, no gain, 25 more registers)
    float v[16];
    tc5_ld16(d_tmem + c, v);
#pragma unroll
    for (int i = 0; i < 16; i += 4) {
      const float4 b = *reinterpret_cast<const float4*>(bias + c + i);
      v[i] = tc5_round(fmaxf(v[i] + b.x, 0.0f));
      v[i + 1] = tc5_round(fmaxf(v[i + 1] + b.y, 0.0f));
      v[i + 2] = tc5_round(fmaxf(v[i + 2] + b.z, 0.0f));
      v[i + 3] = tc5_round(fmaxf(v[i + 3] + b.w, 0.0f));
    }
    tc5_st16(a_tmem + c, v);
  }
  tc5_wait_st();
}

// K closed-loop cycles (observe, network on tcgen05, action, step) of a one-player scenario: the same contract as
// rollout_mlp_kernel<SCN, VAR, ACT>.  ACT = S2D_ACT_DISCRETE: W is a Q-network, (epsilon-)greedy action.
// ACT = S2D_ACT_CONTINUOUS / S2D_ACT_TURNING (ReachBall): W is a DDPG actor - tanh of the last layer's first 1 / 4 outputs is
// the Box(1) / Box(4) action, `epsilon` the half-width of the uniform exploration noise.  ACT = S2D_ACT_PARAMETERIZED
// (Shoot, s2d_shoot_param.cu): the first 8 outputs, translated to the command row the step kernel would make of them.
template <int SCN, int VAR, int ACT = S2D_ACT_DISCRETE>
__global__ void __launch_bounds__(kBlock, S2D_ROLLOUT_MIN_BLOCKS)
    rollout_mlp_tc5_kernel(const __grid_constant__ KernelParams P, const int K, const MlpWeights W, const float epsilon,
                           uint8_t* __restrict__ actions_out, float* __restrict__ q_out, const TrajOut T) {
  static_assert(kBlock == 128, "one block = one M = 128 tile");
  constexpr bool kActor = ACT != S2D_ACT_DISCRETE;
  constexpr int kActDim = ACT == S2D_ACT_TURNING ? 4 : ACT == S2D_ACT_PARAMETERIZED ? 8 : 1;
  // layer 3's N (a multiple of 16): 32 for Shoot's 24 Q-values, else 16; q_out rows hold 8 NT values
  constexpr int N3 = SCN == S2D_SCENARIO_SHOOT && !kActor ? 32 : 16;
  constexpr int NQ = SCN == S2D_SCENARIO_SHOOT ? 24 : 16;
  using SP = typename VariantSP<VAR>::type;
  const SP sp(P.cc);
  __shared__ Tc5Shared s;
  __shared__ __align__(16) float s_stage[kBlock / 32][32 * kObsDim];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  tc5_load_weights<N3>(s, W);
  const uint32_t mbar = smem_u32(&s.mbar);
  if (warp == 0) {  // 128 columns of tensor memory for the block: RD = [0, 64), RA = [64, 128)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(smem_u32(&s.tmem_base)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  tc5_fence_before();
  __syncthreads();
  tc5_fence_after();
  const uint32_t lane_base = s.tmem_base + (static_cast<uint32_t>(32 * warp) << 16);  // this warp's quarter of the lanes
  const uint32_t rd = lane_base, ra = lane_base + 64u;                                  // per-thread views (ld / st)
  const uint32_t rd0 = s.tmem_base, ra0 = s.tmem_base + 64u;                            // whole-tile views (mma)
  uint32_t parity = 0;

  const int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  const int64_t n = P.num_envs;
  const bool valid = i < n;
  const uint64_t gid = static_cast<uint64_t>(P.env_id_offset + i);
  const int64_t warp_first = i - lane;
  const int64_t il = valid ? i : n - 1;  // (rows past the end replay the last episode and report nothing: whole blocks)

  Episode e;
  LaunchOut out;
  float obs_row[kObsDim];
  load_episode(P.state, n, il, e);
#pragma unroll 1
  for (int k = 0; k < K; ++k) {
    scenario_obs<SCN>(e, obs_row);
    if (T.obs && warp_first < n) {
      if ((n & 1) == 0) {  // whole sectors: the warp's 32 rows go out as 512-byte stores (slices of n rows stay 16-byte aligned)
        warp_store_obs(T.obs + static_cast<int64_t>(k) * n * kObsDim, warp_first, n, obs_row, valid, s_stage[warp]);
      } else if (valid) {
        float* dst = T.obs + (static_cast<int64_t>(k) * n + i) * kObsDim;
#pragma unroll
        for (int f = 0; f < kObsDim; f += 2) *reinterpret_cast<float2*>(dst + f) = make_float2(obs_row[f], obs_row[f + 1]);
      }
    }
    {  // A1: the observation row, TF32, features 10..15 zero
      float v[16];
#pragma unroll
      for (int f = 0; f < 16; ++f) v[f] = f < kObsDim ? tc5_round(obs_row[f]) : 0.0f;
      tc5_st16(ra, v);
      tc5_wait_st();
    }
    tc5_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) tc5_issue_layer(rd0, ra0, s.w1, kTc5Hidden, 16, mbar);
    tc5_wait(mbar, parity);
    parity ^= 1u;
    tc5_fence_after();
    tc5_hidden_epilogue(rd, ra, s.b1);
    tc5_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) tc5_issue_layer(rd0, ra0, s.w2, kTc5Hidden, kTc5Hidden, mbar);
    tc5_wait(mbar, parity);
    parity ^= 1u;
    tc5_fence_after();
    tc5_hidden_epilogue(rd, ra, s.b2);
    tc5_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) tc5_issue_layer(rd0, ra0, s.w3, N3, kTc5Hidden, mbar);
    tc5_wait(mbar, parity);
    parity ^= 1u;
    tc5_fence_after();
    // the thread's own output row.  Q-network: + bias, first maximum wins (as torch.argmax); actor: tanh(. + bias)
    int a = 0;
    float4 av = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    float4 av2 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);  // components 4..7 (S2D_ACT_PARAMETERIZED)
    if (kActor) {
      float v[16];
      tc5_ld16(rd, v);
      av.x = tanh_poly(v[0] + s.b3[0]);
      if (kActDim >= 4) {
        av.y = tanh_poly(v[1] + s.b3[1]);
        av.z = tanh_poly(v[2] + s.b3[2]);
        av.w = tanh_poly(v[3] + s.b3[3]);
      }
      if constexpr (kActDim == 8) {
        av2.x = tanh_poly(v[4] + s.b3[4]);
        av2.y = tanh_poly(v[5] + s.b3[5]);
        av2.z = tanh_poly(v[6] + s.b3[6]);
        av2.w = tanh_poly(v[7] + s.b3[7]);
      }
    } else {
      float best = -3.4e38f;
#pragma unroll
      for (int c = 0; c < N3; c += 16) {
        float v[16];
        tc5_ld16(rd + c, v);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (c + j < NQ) {
            v[j] += s.b3[c + j];
            if (v[j] > best) {
              best = v[j];
              a = c + j;
            }
          }
        }
        if (q_out && k == K - 1 && valid) {
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            if (c + j < NQ) *reinterpret_cast<float4*>(q_out + i * NQ + c + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
    }
    tc5_fence_before();  // (the next cycle's A1 store and MMA re-use the regions this cycle read)
    int rs;
    const float reward_before = out.reward_sum;
    if (kActor) {  // (exploration noise and action stores as in rollout_mlp_kernel: the same counter streams)
      if (epsilon > 0.0f) {
        const uint4 w = philox4x32_10(P.seed, gid, e.cycle, RNG_ACTION, 2);
        av.x = clampf(-1.0f, av.x + epsilon * u11(w.x), 1.0f);
        av.y = clampf(-1.0f, av.y + epsilon * u11(w.y), 1.0f);
        av.z = clampf(-1.0f, av.z + epsilon * u11(w.z), 1.0f);
        av.w = clampf(-1.0f, av.w + epsilon * u11(w.w), 1.0f);
        if constexpr (kActDim == 8) {  // (counter 3 of RNG_ACTION: drawn by nothing else)
          const uint4 w2 = philox4x32_10(P.seed, gid, e.cycle, RNG_ACTION, 3);
          av2.x = clampf(-1.0f, av2.x + epsilon * u11(w2.x), 1.0f);
          av2.y = clampf(-1.0f, av2.y + epsilon * u11(w2.y), 1.0f);
          av2.z = clampf(-1.0f, av2.z + epsilon * u11(w2.z), 1.0f);
          av2.w = clampf(-1.0f, av2.w + epsilon * u11(w2.w), 1.0f);
        }
      }
      if constexpr (kActDim == 8) {
        if (T.actions_f && valid) {  // 32-byte rows of a 16-byte aligned buffer (s2d_api.cu checks)
          float4* dst = reinterpret_cast<float4*>(T.actions_f + (static_cast<int64_t>(k) * n + i) * 8);
          dst[0] = av;
          dst[1] = av2;
        }
        out.reward_sum = 0.0f;
        const float4 c = parameterized_command(av, av2);
        rs = substep<SCN, S2D_ACT_COMMAND, SP, true>(e, P, sp, gid, i, c.x, c.y, c.z, c.w, out);
      } else {
      if (T.actions_f && valid) {
        float* dst = T.actions_f + (static_cast<int64_t>(k) * n + i) * kActDim;
        dst[0] = av.x;
        if (kActDim == 4) { dst[1] = av.y; dst[2] = av.z; dst[3] = av.w; }
      }
      out.reward_sum = 0.0f;
      rs = substep<SCN, ACT, SP, true>(e, P, sp, gid, i, av.x, kActDim == 4 ? av.y : 0.f, kActDim == 4 ? av.z : 0.f,
                                       kActDim == 4 ? av.w : 0.f, out, kActDim == 1 ? P.sincos_memo : nullptr);
      }
    } else {
    if (epsilon > 0.0f) {  // exploration: the same counter stream as the mma.sync kernel
      const uint4 w = philox4x32_10(P.seed, gid, e.cycle, RNG_ACTION, 1);
      if (u32_to_unit(w.x) < epsilon) a = u32_to_int(w.y, 0, W.n_actions - 1);
    }
    if (actions_out && valid) actions_out[i * K + k] = static_cast<uint8_t>(a);
    out.reward_sum = 0.0f;
    if (SCN == S2D_SCENARIO_SHOOT) {
      const float4 tab = __ldg(P.action_table + a);
      rs = substep<SCN, S2D_ACT_DISCRETE, SP, true>(e, P, sp, gid, i, tab.x, tab.y, tab.z, tab.w, out);
    } else {
      const float2 tab = __ldg(reinterpret_cast<const float2*>(P.action_table + a) + 1);
      rs = substep<SCN, S2D_ACT_DISCRETE, SP, true>(e, P, sp, gid, i, 0.f, 0.f, tab.x, tab.y, out, P.sincos_memo);
    }
    }
    const float rw = out.reward_sum;
    out.reward_sum = reward_before + rw;
    if (valid) {
      const int64_t at = static_cast<int64_t>(k) * n + i;
      if (T.actions) T.actions[at] = static_cast<uint8_t>(a);
      if (T.reward) T.reward[at] = rw;
      if (T.done) T.done[at] = static_cast<uint8_t>(rs != S2D_RESULT_NONE);
    }
    end_of_episode<SCN, SP, false, S2D_ROLLOUT_DRAW_MEMO>(e, P, sp, gid, i, valid, rs, out);
  }
  if (valid) {
    store_episode(P.state, n, i, e);
    scenario_obs<SCN>(e, obs_row);
    P.reward[i] = out.reward_sum;
    P.done[i] = static_cast<uint8_t>(out.ended != 0);
    P.result[i] = static_cast<uint8_t>(out.last_result());
  } else {
    out = LaunchOut();
  }
  if (warp_first < n) {
    if (T.obs && (n & 1) == 0) {
      warp_store_obs(T.obs + static_cast<int64_t>(K) * n * kObsDim, warp_first, n, obs_row, valid, s_stage[warp]);
    } else if (T.obs && valid) {
      float* dst = T.obs + (static_cast<int64_t>(K) * n + i) * kObsDim;
#pragma unroll
      for (int f = 0; f < kObsDim; ++f) dst[f] = obs_row[f];
    }
    warp_store_obs(P.obs, warp_first, n, obs_row, valid, s_stage[warp]);
  }
  flush_tally(out, P.stats);
  tc5_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(s.tmem_base) : "memory");
}

// SHOOT + S2D_ACT_PARAMETERIZED (s2d_shoot_param.cu): step_kernel and rollout_mlp_tc5_kernel for the constants variant
// `var` (kVarRuntime, kVarDefault, kVarNoisy); cudaErrorInvalidValue, and no launch, for any other.
cudaError_t launch_shoot_param(int var, int grid, const KernelParams& kp, int k_substeps, cudaStream_t s);
cudaError_t launch_shoot_param_actor(int var, int grid, const KernelParams& kp, int k_substeps, const MlpWeights& w,
                                     float noise, const TrajOut& traj, cudaStream_t s);

#endif  // !S2D_HOST_EMU

}  // namespace s2d
