// K1: fused policy-in-the-loop rollout (include/trajopt_grpo.h: tg_rollout),
// plus the batched single-step kernels (tg_env_step, tg_quadrotor12_dynamics)
// and the Philox noise materialiser (tg_noise_fill).
//
// One CTA advances a tile of B environments through all T steps:
//   * the staged policy weights are copied ONCE into shared memory by the TMA
//     bulk engine (cp.async.bulk + mbarrier) and stay resident;
//   * each environment's state lives in the registers of its owner thread
//     (threadIdx.x < B) for the whole episode;
//   * per step: owners publish fp32 obs to shared memory and to the [T][O][N]
//     trajectory (coalesced: env index innermost), the CTA runs the MLP as
//     register-tiled fp32 GEMMs over the tile, owners sample the action from
//     the supplied/Philox noise, integrate the dynamics, and write
//     act/logp/reward rows;
//   * finished environments idle (zero rows) until every env of the tile is
//     done, then the CTA only zero-fills the remaining rows.
#include <math.h>

#include "tg_mlp.cuh"
#include "tg_rollout.cuh"
#include "tg_umma.cuh"

template <int KIND, typename R, int CFG, bool WG>
__global__ void __launch_bounds__(TileCfg<CFG>::NT) rollout_kernel(const __grid_constant__ RolloutArgs<tg_mlp_layout> a) {
    using Ev = RolloutEnv<KIND, R>;
    constexpr int B = TileCfg<CFG>::B, NT = TileCfg<CFG>::NT, LDX = B + 4;
    constexpr int S = Ev::S, A = Ev::A;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t wbar;
    float *Ws = reinterpret_cast<float *>(smem_raw);
    float *Xa = Ws + (WG ? 0 : a.lay.total);
    float *Xb = Xa + (size_t)a.lay.kmax * LDX;
    float *P = Xb + (size_t)a.lay.kmax * LDX;
    const float *W = WG ? a.packed : Ws;
    if (!WG) stage_weights_tma(Ws, a.packed, a.lay.total, &wbar);

    const int T = a.io.env.max_steps;
    const int64_t n = (int64_t)blockIdx.x * B + threadIdx.x;
    const bool owner = threadIdx.x < B;
    Ev ev(a.io, n, owner && n < a.io.N, true);      // only owner threads hold an env
    const int nl = a.lay.n_layers;
    int t = 0;
    for (; t < T; ++t) {
        // 1. publish the observation
        if (owner) {
            float x[S];
            ev.observe(a.io, t, x);
#pragma unroll
            for (int i = 0; i < S; ++i) Xa[i * LDX + threadIdx.x] = x[i];
        }
        __syncthreads();
        // 2. hidden layers (ping-pong Xa <-> Xb)
        float *xin = Xa, *xout = Xb;
        for (int l = 0; l < nl - 1; ++l) {
            tile_layer<CFG, 0, WG>(W + a.lay.L[l].wt, W + a.lay.L[l].bias, xin, xout, a.lay.L[l].K, a.lay.acts[l]);
            __syncthreads();
            float *tmp = xin; xin = xout; xout = tmp;
        }
        // 3. output layer -> mean action for the owner's env
        float mu[A];
        tile_output_layer<CFG, A, WG>(W + a.lay.L[nl - 1].wt, W + a.lay.L[nl - 1].bias, xin, P, a.lay.L[nl - 1].K, mu);
        // 4. sample, step the env, write the trajectory rows
        if (owner) ev.act(a.io, t, mu);
        // 5. tile-wide early exit; also the barrier that protects Xa/Xb/P reuse
        if (!__syncthreads_or(ev.alive ? 1 : 0)) { ++t; break; }
    }
    ev.finish(a.io, t);
}

template <int KIND, typename R, int CFG, bool WG>
static int launch_rollout(const RolloutArgs<tg_mlp_layout> &a, size_t smem, cudaStream_t st) {
    constexpr int B = TileCfg<CFG>::B, NT = TileCfg<CFG>::NT;
    auto kern = rollout_kernel<KIND, R, CFG, WG>;
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)((a.io.N + B - 1) / B);
    kern<<<grid, NT, smem, st>>>(a);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

template <int KIND, typename R>
static int dispatch_cfg(const RolloutArgs<tg_mlp_layout> &a, size_t smem, bool wg, cudaStream_t st) {
    if (wg) {
        switch (a.lay.cfg) {
            case 0: return launch_rollout<KIND, R, 0, true>(a, smem, st);
            case 1: return launch_rollout<KIND, R, 1, true>(a, smem, st);
            default: return launch_rollout<KIND, R, 2, true>(a, smem, st);
        }
    }
    switch (a.lay.cfg) {
        case 0: return launch_rollout<KIND, R, 0, false>(a, smem, st);
        case 1: return launch_rollout<KIND, R, 1, false>(a, smem, st);
        default: return launch_rollout<KIND, R, 2, false>(a, smem, st);
    }
}

// ---------------------------------------------------------------------------
// Tensor-core variant (TG_MATH_AUTO / TG_MATH_3XTF32, eligible policies: tg_tc_eligible).
// 128 threads, thread i = env i of the tile = TMEM lane i.  Per step each thread evaluates
// the first Linear for its own env on the FP32 pipe, writes its activation row (hi/lo
// split) straight into the core-matrix-layout A operand in shared memory, one elected
// thread issues the 3xTF32 tcgen05.mma sequence for the [128 x 64] x [64 x 64] hidden
// GEMM (weights hi/lo resident in shared memory, staged once by TMA), the accumulator
// comes back from TMEM with tcgen05.ld -- each thread receives exactly its env's row --
// and bias/activation/output layer/sampling/dynamics continue in registers.
// ---------------------------------------------------------------------------
// RELU: the activation is known at compile time (no per-element branch); otherwise a.lay.act
template <int KIND, typename R, bool RELU>
__global__ void __launch_bounds__(128) rollout_tc_kernel(const __grid_constant__ RolloutArgs<tg_tc_layout> a) {
    using Ev = RolloutEnv<KIND, R>;
    constexpr int S = Ev::S, A = Ev::A, W = TC_W, O4 = (S + 1 + 3) / 4 * 4;
    // 1024-byte alignment comes from the declaration (no integer pointer arithmetic, so the
    // compiler keeps every access below in the shared address space: LDS/STS, not generic LD)
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t wbar, mbar;
    __shared__ uint32_t tmem_slot;
    unsigned char *base = smem_raw;
    if ((smem_u32(base) & 1023u) != 0u) __trap();
    float *Wsm = reinterpret_cast<float *>(base);
    unsigned char *a_hi = base + ((size_t)a.lay.total * 4 + 1023) / 1024 * 1024;
    unsigned char *a_lo = a_hi + 128 * W * 4;
    stage_weights_tma(Wsm, a.packed, a.lay.total, &wbar);
    if (threadIdx.x == 0) {
        mbar_init(&mbar, 1);
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tmem_alloc(&tmem_slot, 64);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t idesc = umma_idesc_tf32(128, W);
    const uint32_t a_hi_u = smem_u32(a_hi), a_lo_u = smem_u32(a_lo), w_u = smem_u32(Wsm);
    const int warp = threadIdx.x >> 5;
    const uint32_t my_tmem = tmem + ((uint32_t)(warp * 32) << 16);
    // this thread's row of the [128][W] activation operand in the core-matrix layout
    const uint32_t row_off = (uint32_t)(threadIdx.x >> 3) * (uint32_t)(W / 4) * 128u + (uint32_t)(threadIdx.x & 7) * 16u;

    const int T = a.io.env.max_steps;
    const int64_t n = (int64_t)blockIdx.x * 128 + threadIdx.x;
    Ev ev(a.io, n, n < a.io.N, true);
    const int nh = a.lay.nh, act_kind = RELU ? TG_ACT_RELU : a.lay.act;
    const float *w1 = Wsm + a.lay.w1;
    uint32_t phase = 0;
    int t = 0;
    for (; t < T; ++t) {
        float x[S];
        ev.observe(a.io, t, x);
        // first Linear on the FP32 pipe (K = obs dim is tiny): h = act(W1 x + b1)
        float h[W];
#pragma unroll
        for (int nn = 0; nn < W; ++nn) {
            float wrow[O4];
#pragma unroll
            for (int q = 0; q < O4; q += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(w1 + nn * O4 + q);
                wrow[q] = v.x; wrow[q + 1] = v.y; wrow[q + 2] = v.z; wrow[q + 3] = v.w;
            }
            float acc = wrow[S];
#pragma unroll
            for (int i = 0; i < S; ++i) acc = fmaf(wrow[i], x[i], acc);
            h[nn] = act_fwd(acc, act_kind);
        }
        // hidden -> hidden Linears on the tensor cores
        for (int l = 1; l < nh; ++l) {
#pragma unroll
            for (int c = 0; c < W / 4; ++c) {
                float4 hi, lo;
                hi.x = tf32_hi(h[4 * c]); hi.y = tf32_hi(h[4 * c + 1]);
                hi.z = tf32_hi(h[4 * c + 2]); hi.w = tf32_hi(h[4 * c + 3]);
                lo.x = h[4 * c] - hi.x; lo.y = h[4 * c + 1] - hi.y;
                lo.z = h[4 * c + 2] - hi.z; lo.w = h[4 * c + 3] - hi.w;
                const uint32_t off = row_off + (uint32_t)c * 128u;      // core_offset(W, row, 4c)
                *reinterpret_cast<float4 *>(a_hi + off) = hi;
                *reinterpret_cast<float4 *>(a_lo + off) = lo;
            }
            fence_proxy_async();
            tc_fence_before();
            __syncthreads();
            if (threadIdx.x < 32) {        // warp 0 issues with warp-uniform operands, one elected lane per MMA
                tc_fence_after();
                umma_gemm_3xtf32_w(tmem, a_hi_u, a_lo_u, W, false, w_u + (uint32_t)a.lay.whi[l] * 4u,
                                   w_u + (uint32_t)a.lay.wlo[l] * 4u, W, false, W, idesc, false, 3);
                umma_commit_w(&mbar);
            }
            mbar_wait(&mbar, phase);
            phase ^= 1u;
            tc_fence_after();
            const float *bl = Wsm + a.lay.bias[l];
#pragma unroll
            for (int c0 = 0; c0 < W; c0 += 32) {
                float z[32];
                tmem_ld32(my_tmem + (uint32_t)c0, z);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b4 = *reinterpret_cast<const float4 *>(bl + c0 + j);
                    h[c0 + j] = act_fwd(z[j] + b4.x, act_kind);
                    h[c0 + j + 1] = act_fwd(z[j + 1] + b4.y, act_kind);
                    h[c0 + j + 2] = act_fwd(z[j + 2] + b4.z, act_kind);
                    h[c0 + j + 3] = act_fwd(z[j + 3] + b4.w, act_kind);
                }
            }
        }
        // output Linear (A <= 4 neurons) on the FP32 pipe
        float mu[A];
        {
            const float *wo = Wsm + a.lay.wo, *bo = Wsm + a.lay.bo;
#pragma unroll
            for (int j = 0; j < A; ++j) {
                float acc = bo[j];
#pragma unroll
                for (int q = 0; q < W; q += 4) {
                    const float4 v = *reinterpret_cast<const float4 *>(wo + j * W + q);
                    acc = fmaf(h[q], v.x, acc); acc = fmaf(h[q + 1], v.y, acc);
                    acc = fmaf(h[q + 2], v.z, acc); acc = fmaf(h[q + 3], v.w, acc);
                }
                mu[j] = acc;
            }
        }
        ev.act(a.io, t, mu);
        if (!__syncthreads_or(ev.alive ? 1 : 0)) { ++t; break; }
    }
    ev.finish(a.io, t);
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 64);
}

// ---------------------------------------------------------------------------
// Tensor-core variant with TWO threads per env (256 threads per 128-env tile) for hidden width
// 128: env e = TMEM lane e is served by warps q and q+4 of lane quadrant q, each owning one
// half (HW = W/2 columns) of every activation row, so a 128-wide row costs 64 registers per thread.
// The hidden activation goes to the tensor core as the A operand straight from registers through
// tensor memory (tcgen05.st, hi/lo split; tcgen05.mma with A in TMEM), the [W x W] weight (hi/lo,
// core-matrix K-major, staged once by TMA) is the B operand in shared memory, the accumulator comes
// back with tcgen05.ld.  Both threads of an env integrate its dynamics redundantly (cheap next to
// the MLP) so that `alive` and the state never have to be exchanged; only the two halves of the
// output-layer dot product meet in shared memory (fixed order -> deterministic).
// ---------------------------------------------------------------------------
template <int KIND, typename R, bool RELU, int W>
__global__ void __launch_bounds__(256, 1) rollout_tc2_kernel(const __grid_constant__ RolloutArgs<tg_tc_layout> a) {
    using Ev = RolloutEnv<KIND, R>;
    constexpr int S = Ev::S, A = Ev::A, HW = W / 2, O4 = (S + 1 + 3) / 4 * 4;
    constexpr uint32_t TM_D = 0u, TM_AHI = (uint32_t)W, TM_ALO = 2u * (uint32_t)W;
    constexpr uint32_t TM_COLS = 512u;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t wbar, mbar;
    __shared__ uint32_t tmem_slot;
    __shared__ float muS[2][A][128];
    if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();
    float *Wsm = reinterpret_cast<float *>(smem_raw);
    stage_weights_tma(Wsm, a.packed, a.lay.total, &wbar);
    if (threadIdx.x == 0) {
        mbar_init(&mbar, 1);
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tmem_alloc(&tmem_slot, TM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t idesc = umma_idesc_tf32(128, W);
    const uint32_t w_u = smem_u32(Wsm);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = warp & 3, hf = warp >> 2;       // lane quadrant, column half
    const int e = q * 32 + lane;                  // env row of this thread = TMEM lane
    const int c0 = hf * HW;                       // first column of this thread's half
    const uint32_t my_tm = tmem + ((uint32_t)(q * 32) << 16);

    const int T = a.io.env.max_steps;
    const int64_t n = (int64_t)blockIdx.x * 128 + e;
    Ev ev(a.io, n, n < a.io.N, hf == 0);          // both threads step the env, the hf == 0 one records it
    const int nh = a.lay.nh, act_kind = RELU ? TG_ACT_RELU : a.lay.act;
    const float *w1 = Wsm + a.lay.w1 + (size_t)c0 * O4;
    uint32_t phase = 0;
    int t = 0;
    for (; t < T; ++t) {
        float x[S];
        ev.observe(a.io, t, x);
        // first Linear on the FP32 pipe, this thread's HW neurons: h = act(W1 x + b1)
        float h[HW];
#pragma unroll
        for (int nn = 0; nn < HW; ++nn) {
            float wrow[O4];
#pragma unroll
            for (int c = 0; c < O4; c += 4) {
                const float4 v = *reinterpret_cast<const float4 *>(w1 + nn * O4 + c);
                wrow[c] = v.x; wrow[c + 1] = v.y; wrow[c + 2] = v.z; wrow[c + 3] = v.w;
            }
            float acc = wrow[S];
#pragma unroll
            for (int i = 0; i < S; ++i) acc = fmaf(wrow[i], x[i], acc);
            h[nn] = act_fwd(acc, act_kind);
        }
        // hidden -> hidden Linears on the tensor cores
        for (int l = 1; l < nh; ++l) {
#pragma unroll
            for (int cc = 0; cc < HW; cc += 32) {
                float hi[32], lo[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    hi[j] = tf32_hi(h[cc + j]);
                    lo[j] = h[cc + j] - hi[j];
                }
                tmem_st32(my_tm + TM_AHI + (uint32_t)(c0 + cc), hi);
                tmem_st32(my_tm + TM_ALO + (uint32_t)(c0 + cc), lo);
            }
            tmem_st_wait();
            tc_fence_before();
            __syncthreads();
            if (threadIdx.x < 32) {        // warp 0 issues with warp-uniform operands, one elected lane per MMA
                tc_fence_after();
                const uint32_t b_hi = w_u + (uint32_t)a.lay.whi[l] * 4u, b_lo = w_u + (uint32_t)a.lay.wlo[l] * 4u;
                uint32_t acc = 0;
#pragma unroll 1
                for (int pass = 0; pass < 3; ++pass) {
                    uint32_t acol = tmem + (pass == 2 ? TM_ALO : TM_AHI);
                    uint64_t b = umma_operand_desc(pass == 1 ? b_lo : b_hi, W, false, 0);
#pragma unroll 2
                    for (int k = 0; k < W; k += 8) {
                        umma_tf32_ts_w(tmem + TM_D, acol, b, idesc, acc);
                        acc = 1u;
                        acol += 8u;
                        b += 16;               // one K step = 256 B in the K-major core-matrix layout (16-byte units)
                    }
                }
                umma_commit_w(&mbar);
            }
            mbar_wait(&mbar, phase);
            phase ^= 1u;
            tc_fence_after();
            const float *bl = Wsm + a.lay.bias[l] + c0;
#pragma unroll
            for (int cc = 0; cc < HW; cc += 32) {
                float z[32];
                tmem_ld32(my_tm + TM_D + (uint32_t)(c0 + cc), z);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b4 = *reinterpret_cast<const float4 *>(bl + cc + j);
                    h[cc + j] = act_fwd(z[j] + b4.x, act_kind);
                    h[cc + j + 1] = act_fwd(z[j + 1] + b4.y, act_kind);
                    h[cc + j + 2] = act_fwd(z[j + 2] + b4.z, act_kind);
                    h[cc + j + 3] = act_fwd(z[j + 3] + b4.w, act_kind);
                }
            }
            tc_fence_before();      // orders these TMEM reads before the next layer's / step's MMA
        }
        // output Linear (A <= 4 neurons): each thread sums its half, the halves meet in shared memory
        {
            const float *wo = Wsm + a.lay.wo + c0;
#pragma unroll
            for (int j = 0; j < A; ++j) {
                float acc = 0.0f;
#pragma unroll
                for (int c = 0; c < HW; c += 4) {
                    const float4 v = *reinterpret_cast<const float4 *>(wo + j * W + c);
                    acc = fmaf(h[c], v.x, acc); acc = fmaf(h[c + 1], v.y, acc);
                    acc = fmaf(h[c + 2], v.z, acc); acc = fmaf(h[c + 3], v.w, acc);
                }
                muS[hf][j][e] = acc;
            }
        }
        asm volatile("bar.sync %0, 64;" ::"r"(q + 1) : "memory");   // the two warps of this lane quadrant
        float mu[A];
        {
            const float *bo = Wsm + a.lay.bo;
#pragma unroll
            for (int j = 0; j < A; ++j) mu[j] = (bo[j] + muS[0][j][e]) + muS[1][j][e];
        }
        ev.act(a.io, t, mu);
        if (!__syncthreads_or(ev.alive ? 1 : 0)) { ++t; break; }
    }
    ev.finish(a.io, t);
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, TM_COLS);
}

// width 64: rollout_tc_kernel; width 128: rollout_tc2_kernel
static int launch_rollout_tc(int kind, int precision, const RolloutArgs<tg_tc_layout> &a, cudaStream_t st) {
    const bool w128 = a.lay.W == 128;
    const size_t wbytes = ((size_t)a.lay.total * 4 + 1023) / 1024 * 1024;
    const size_t smem = w128 ? wbytes : 1024 + wbytes + 2 * 128 * TC_W * 4;
    auto kern = tg_with_env_kind(kind, [&](auto k) {
        return tg_with_prec_relu(precision, a.lay.act, [&](auto r, auto relu) {
            return w128 ? rollout_tc2_kernel<decltype(k)::value, decltype(r), decltype(relu)::value, 128>
                        : rollout_tc_kernel<decltype(k)::value, decltype(r), decltype(relu)::value>;
        });
    });
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)((a.io.N + 127) / 128), w128 ? 256 : 128, smem, st>>>(a);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

int tg_fill_env_params(const tg_env_cfg *env, EnvParams *p) {
    TG_REQUIRE(env != nullptr, TG_ERR_ARG, "env cfg is null");
    TG_REQUIRE(env->kind >= 0 && env->kind <= 3, TG_ERR_ARG, "unknown env kind %d", env->kind);
    TG_REQUIRE(env->max_steps > 0 && env->dt > 0, TG_ERR_SHAPE, "max_steps and dt must be positive");
    p->dt = env->dt;
    p->max_steps = env->max_steps;
    p->time_limit_step = env->time_limit_step;
    p->balanced_limit = env->balanced_limit;
    for (int i = 0; i < 5; ++i) p->k[i] = 0.0;
    const bool dflt = env->phys[0] == 0.0 && env->phys[1] == 0.0 && env->phys[2] == 0.0 && env->phys[3] == 0.0;
    if (env->kind == TG_ENV_CARTPOLE) {                 // cartpole_env.py:7-16
        const double mc = dflt ? 1.0 : env->phys[0], mp = dflt ? 1.0 : env->phys[1], l = dflt ? 0.5 : env->phys[2];
        const double g = dflt ? TG_G : env->phys[3];
        TG_REQUIRE(mc + mp > 0 && l > 0, TG_ERR_ARG, "CartPole masses and length must be positive");
        p->k[0] = mc + mp; p->k[1] = mp * l; p->k[2] = l; p->k[3] = g; p->k[4] = mp;
    } else if (env->kind == TG_ENV_PENDULUM) {          // pendulum_env.py:8-17
        const double m = dflt ? 1.0 : env->phys[0], l = dflt ? 0.5 : env->phys[1], g = dflt ? TG_G : env->phys[2];
        TG_REQUIRE(m > 0 && l > 0, TG_ERR_ARG, "Pendulum mass and length must be positive");
        p->k[0] = 1.0 / (m * (l * l)); p->k[1] = m * g * l;
    } else {
        TG_REQUIRE(dflt, TG_ERR_UNSUPPORTED, "the quadrotor envs take no physical constructor arguments in the reference");
    }
    return TG_OK;
}

extern "C" int tg_rollout(tg_ctx *ctx, const tg_env_cfg *env, const tg_mlp_cfg *mlp, int precision, int64_t N,
                          const void *init_state, const float *params, const float *cov_diag, const float *noise,
                          uint64_t seed, int64_t env_offset, float *out_obs, float *out_act, float *out_rew, float *out_logp,
                          int32_t *out_len, float *out_ret, void *stream) {
    TgRange nvtx_range("tg_rollout (K1: fused policy-in-the-loop rollout)");
    TG_REQUIRE(ctx && env && mlp && init_state && params && cov_diag && out_obs && out_act && out_rew && out_len,
               TG_ERR_ARG, "tg_rollout: null argument");
    TG_REQUIRE(N > 0, TG_ERR_SHAPE, "tg_rollout: N must be positive");
    TG_REQUIRE(precision == TG_PREC_F32 || precision == TG_PREC_F64, TG_ERR_ARG, "bad precision %d", precision);
    RolloutIo io;
    memset(&io, 0, sizeof(io));
    int rc = tg_fill_env_params(env, &io.env);
    if (rc) return rc;
    int O, A;
    tg_env_dims(env->kind, &O, &A);
    TG_REQUIRE(mlp->n_layers >= 1 && mlp->n_layers <= TG_MAX_LAYERS, TG_ERR_SHAPE, "n_layers %d not in [1,%d]",
               mlp->n_layers, TG_MAX_LAYERS);
    TG_REQUIRE(mlp->dims[0] == O && mlp->dims[mlp->n_layers] == A, TG_ERR_SHAPE,
               "policy dims (%d -> %d) do not match env obs/act dims (%d/%d)", mlp->dims[0], mlp->dims[mlp->n_layers], O, A);
    rc = tg_gauss_consts(cov_diag, A, io.sd, nullptr, nullptr, &io.log_norm);
    if (rc) return rc;
    io.N = N;
    io.init_state = init_state;
    io.noise = noise;
    io.seed = seed;
    io.env_offset = env_offset;
    io.obs = out_obs; io.act = out_act; io.rew = out_rew; io.logp = out_logp; io.len = out_len; io.ret = out_ret;
    cudaStream_t st = (cudaStream_t)stream;
    TG_CUDA(cudaSetDevice(ctx->device));
    // ---- tensor-core paths (3xTF32 tcgen05) for eligible policies
    if (tg_tc256_eligible(mlp) && ctx->math_mode != TG_MATH_FP32)      // 256-wide: weights streamed from L2
        return tg_rollout_tc256(ctx, mlp, precision, env->kind, params, io, st);
    const bool tc_ok = tg_tc_eligible(mlp);
    TG_REQUIRE(ctx->math_mode != TG_MATH_3XTF32 || tc_ok, TG_ERR_UNSUPPORTED,
               "TG_MATH_3XTF32 requested but the policy shape is not eligible (>= 2 hidden layers of equal width 64 or 128)");
    if (tc_ok && ctx->math_mode != TG_MATH_FP32) {
        RolloutArgs<tg_tc_layout> b;
        memset(&b, 0, sizeof(b));
        b.io = io;
        rc = tg_build_tc_layout(mlp, &b.lay);
        if (rc) return rc;
        rc = tg_pack_weights_tc(ctx, b.lay, params, st);
        if (rc) return rc;
        b.packed = ctx->packed_tc;
        TG_REQUIRE(((size_t)b.lay.total * 4 + 1023) / 1024 * 1024 + 4096 <= (size_t)ctx->smem_optin, TG_ERR_UNSUPPORTED,
                   "staged tensor-core weights need %zu B of shared memory", (size_t)b.lay.total * 4);
        return launch_rollout_tc(env->kind, precision, b, st);
    }
    RolloutArgs<tg_mlp_layout> a;
    memset(&a, 0, sizeof(a));
    a.io = io;
    rc = tg_build_layout(mlp, false, &a.lay);
    if (rc) return rc;
    rc = tg_pack_weights(ctx, a.lay, params, st);
    if (rc) return rc;
    a.packed = ctx->packed;
    const int B = a.lay.B, NT = a.lay.NT;
    const size_t act_bytes = (2 * (size_t)a.lay.kmax * (B + 4) + (size_t)(NT / B) * TG_MAX_ACT * B) * sizeof(float);
    size_t smem = act_bytes + (size_t)a.lay.total * sizeof(float);
    // weights resident in shared memory when they fit next to the activation
    // tiles; otherwise they stay in global memory (read-only path, L2-resident)
    const bool wg = smem > (size_t)ctx->smem_optin;
    if (wg) smem = act_bytes;
    TG_REQUIRE(smem <= (size_t)ctx->smem_optin, TG_ERR_UNSUPPORTED, "activation tiles need %zu B of shared memory", smem);
    return tg_with_env_kind(env->kind, [&](auto kind) {
        return precision == TG_PREC_F64 ? dispatch_cfg<decltype(kind)::value, double>(a, smem, wg, st)
                                        : dispatch_cfg<decltype(kind)::value, float>(a, smem, wg, st);
    });
}

// ---------------------------------------------------------------------------
// tg_noise_fill
// ---------------------------------------------------------------------------
__global__ void noise_fill_kernel(uint64_t seed, int64_t env_offset, int64_t N, int T, int A, float *out) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int t = blockIdx.y;
    if (n >= N) return;
    float z[4];
    philox_normal4(seed, (uint64_t)(env_offset + n), (uint32_t)t, z);
    for (int j = 0; j < A; ++j) out[((int64_t)t * A + j) * N + n] = z[j];
}

extern "C" int tg_noise_fill(tg_ctx *ctx, uint64_t seed, int64_t env_offset, int64_t N, int T, int A, float *noise,
                             void *stream) {
    TG_REQUIRE(ctx && noise, TG_ERR_ARG, "tg_noise_fill: null argument");
    TG_REQUIRE(N > 0 && T > 0 && T <= 65535 && A >= 1 && A <= 4, TG_ERR_SHAPE, "tg_noise_fill: bad shape");
    TG_CUDA(cudaSetDevice(ctx->device));
    dim3 grid((unsigned)((N + 255) / 256), (unsigned)T);
    noise_fill_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(seed, env_offset, N, T, A, noise);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

// ---------------------------------------------------------------------------
// tg_env_step: one Env.step for N independent envs
// ---------------------------------------------------------------------------
template <int KIND, typename R>
__global__ void env_step_kernel(EnvParams p, int64_t N, const R *state, const float *raw_action,
                                const int32_t *steps_done, const int32_t *bal_in, R *next, R *reward, int32_t *done,
                                int32_t *bal_out) {
    using E = Env<KIND>;
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    R s[E::S];
    float a[E::A];
#pragma unroll
    for (int i = 0; i < E::S; ++i) s[i] = state[(int64_t)i * N + n];
#pragma unroll
    for (int j = 0; j < E::A; ++j) a[j] = raw_action[(int64_t)j * N + n];
    int bal = bal_in ? bal_in[n] : 0;
    R r;
    const bool d = E::template step<R>(s, a, p, steps_done ? steps_done[n] : 0, bal, r);
#pragma unroll
    for (int i = 0; i < E::S; ++i) next[(int64_t)i * N + n] = s[i];
    reward[n] = r;
    done[n] = d ? 1 : 0;
    if (bal_out) bal_out[n] = bal;
}

template <int KIND>
static int launch_env_step(int precision, const EnvParams &p, int64_t N, const void *state, const float *raw_action,
                           const int32_t *steps_done, const int32_t *bal, void *next, void *reward, int32_t *done,
                           int32_t *bal_out, cudaStream_t st) {
    const unsigned grid = (unsigned)((N + 127) / 128);
    if (precision == TG_PREC_F64)
        env_step_kernel<KIND, double><<<grid, 128, 0, st>>>(p, N, (const double *)state, raw_action, steps_done, bal,
                                                            (double *)next, (double *)reward, done, bal_out);
    else
        env_step_kernel<KIND, float><<<grid, 128, 0, st>>>(p, N, (const float *)state, raw_action, steps_done, bal,
                                                           (float *)next, (float *)reward, done, bal_out);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

extern "C" int tg_env_step(tg_ctx *ctx, const tg_env_cfg *env, int precision, int64_t N, const void *state,
                           const float *raw_action, const int32_t *steps_done, const int32_t *bal_count,
                           void *next_state, void *reward, int32_t *done, int32_t *bal_out, void *stream) {
    TG_REQUIRE(ctx && env && state && raw_action && next_state && reward && done, TG_ERR_ARG,
               "tg_env_step: null argument");
    TG_REQUIRE(N > 0, TG_ERR_SHAPE, "tg_env_step: N must be positive");
    TG_REQUIRE(precision == TG_PREC_F32 || precision == TG_PREC_F64, TG_ERR_ARG, "bad precision %d", precision);
    EnvParams p;
    int rc = tg_fill_env_params(env, &p);
    if (rc) return rc;
    TG_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    return tg_with_env_kind(env->kind, [&](auto kind) {
        return launch_env_step<decltype(kind)::value>(precision, p, N, state, raw_action, steps_done, bal_count,
                                                      next_state, reward, done, bal_out, st);
    });
}

template <typename R>
__global__ void quadrotor12_kernel(int64_t N, R dt, const R *state, const R *control, R *next) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    R s[12], u[4];
#pragma unroll
    for (int i = 0; i < 12; ++i) s[i] = state[(int64_t)i * N + n];
#pragma unroll
    for (int i = 0; i < 4; ++i) u[i] = control[(int64_t)i * N + n];
    quadrotor12_step<R>(s, u, dt);
#pragma unroll
    for (int i = 0; i < 12; ++i) next[(int64_t)i * N + n] = s[i];
}

extern "C" int tg_quadrotor12_dynamics(tg_ctx *ctx, int precision, int64_t N, double dt, const void *state,
                                       const void *control, void *next, void *stream) {
    TG_REQUIRE(ctx && state && control && next, TG_ERR_ARG, "tg_quadrotor12_dynamics: null argument");
    TG_REQUIRE(N > 0, TG_ERR_SHAPE, "N must be positive");
    TG_CUDA(cudaSetDevice(ctx->device));
    const unsigned grid = (unsigned)((N + 127) / 128);
    if (precision == TG_PREC_F64)
        quadrotor12_kernel<double><<<grid, 128, 0, (cudaStream_t)stream>>>(N, dt, (const double *)state,
                                                                           (const double *)control, (double *)next);
    else
        quadrotor12_kernel<float><<<grid, 128, 0, (cudaStream_t)stream>>>(N, (float)dt, (const float *)state,
                                                                          (const float *)control, (float *)next);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}
