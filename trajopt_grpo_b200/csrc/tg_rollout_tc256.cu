// K1 on the tensor cores for 256-wide policies (BASELINE cfg 4/5: obs -> 256 -> 256 -> act).
//
// A [256 x 256] weight split into tf32 hi + lo parts is 512 KB: it fits neither in the 227 KB of shared
// memory nor, as the A operand, in tensor memory next to a [128 x 256] accumulator.  So the weight is
// STREAMED: it sits in HBM/L2 as 16 contiguous 32 KB chunks (8 K-chunks of 32 columns, hi and lo,
// pre-arranged in the K-major core-matrix layout the tensor core reads), and every step of every tile a
// producer warp pulls the chunks through a 4-stage shared-memory ring with the TMA bulk engine
// (cp.async.bulk + mbarrier expect_tx); the MMA warp consumes a chunk as soon as it lands and frees its
// stage with tcgen05.commit.  All CTAs read the same 512 KB, so the stream is served by L2.
//
// 18 warps: 16 compute warps (env e = TMEM lane e is served by 4 threads, each owning 64 of the 256
// columns), 1 TMA producer warp, 1 MMA issuer warp.  Tensor memory (512 columns): accumulator D
// [128 x 256] in columns 0..255, the A operand of HALF the reduction (128 columns hi, 128 columns lo) in
// 256..511 -- the 256-wide reduction runs as two K halves so that hi and lo of the activation are both
// resident and every weight chunk is streamed exactly once per step (3 MMAs per chunk pair:
// A_hi.B_hi, A_lo.B_hi, A_hi.B_lo).
// Per step:
//   part-0 threads publish obs (hi/lo, plus a constant ones column that carries the bias) as the K-major
//     A operand of the FIRST Linear, which also runs on the tensor core (K = obs dim + 1 padded to 8);
//   epilogue 1: tcgen05.ld -> activation -> hi/lo split -> tcgen05.st into the A region (K half 0 by
//     parts 0-1, K half 1 by parts 2-3 once the MMAs of half 0 have released it);
//   epilogue 2: tcgen05.ld -> bias, activation -> partial output-layer dot products (FP32 pipe), exchanged
//     through shared memory; the part-0 thread samples the action, integrates the env, writes the rows.
#include <math.h>

#include "tg_mlp.cuh"
#include "tg_rollout.cuh"
#include "tg_umma.cuh"

#define W256 256
#define RING_STAGES 4
#define CHUNK_K 32
#define CHUNK_FLOATS (W256 * CHUNK_K)           // 8192 floats = 32 KB
#define N_CHUNKS (2 * W256 / CHUNK_K)           // 16: (hi, lo) x 8 K-chunks

bool tg_tc256_eligible(const tg_mlp_cfg *mlp) {
    return mlp && mlp->n_layers == 3 && mlp->dims[1] == W256 && mlp->dims[2] == W256 && mlp->dims[0] >= 1 &&
           mlp->dims[0] <= 23 && mlp->dims[3] >= 1 && mlp->dims[3] <= TG_MAX_ACT && mlp->activation >= 0 &&
           mlp->activation <= 2;
}

#define BAR_L1 5
#define BAR_K0 6
#define BAR_K1 7

template <int KIND, typename R, bool RELU>
__global__ void __launch_bounds__(576, 1) rollout_tc256_kernel(const __grid_constant__ RolloutArgs<TcwLayout> a) {
    using Ev = RolloutEnv<KIND, R>;
    constexpr int S = Ev::S, A = Ev::A, W = W256, HW = 64, OKP = (S + 1 + 7) / 8 * 8;
    constexpr uint32_t TM_D = 0u, TM_AHI = 256u, TM_ALO = 384u;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t wbar, bar_d, bar_k0, full_bar[RING_STAGES], empty_bar[RING_STAGES];
    __shared__ uint32_t tmem_slot;
    __shared__ float muS[4][A][128];
    if ((smem_u32(smem_raw) & 1023u) != 0u) __trap();
    unsigned char *ring = smem_raw;                                           // RING_STAGES x 32 KB
    float *Rsm = reinterpret_cast<float *>(smem_raw + RING_STAGES * CHUNK_FLOATS * 4);
    unsigned char *O_hi = reinterpret_cast<unsigned char *>(Rsm + a.lay.resident);   // obs A operand [128][OKP], K-major
    unsigned char *O_lo = O_hi + 128 * OKP * 4;
    stage_weights_tma(Rsm, a.packed, a.lay.resident, &wbar);
    if (threadIdx.x == 0) {
        mbar_init(&bar_d, 1);
        mbar_init(&bar_k0, 1);
        for (int i = 0; i < RING_STAGES; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tmem_alloc(&tmem_slot, 512);
    // obs operand: zero, then the constant ones column (it multiplies the bias row of W0)
    for (int i = threadIdx.x; i < 128 * OKP; i += blockDim.x) {
        const int r = i / OKP, c = i % OKP;
        *reinterpret_cast<float *>(O_hi + core_offset(OKP, r, c)) = c == S ? 1.0f : 0.0f;
        *reinterpret_cast<float *>(O_lo + core_offset(OKP, r, c)) = 0.0f;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int T = a.io.env.max_steps;

    if (warp == 16) {
        // ===== TMA producer: streams the 16 weight chunks of every step through the ring =====
        uint32_t gi = 0;
        const float *src = a.packed + a.lay.chunks_f;
        for (int t = 0; t < T; ++t) {
            if (lane == 0) {
                for (int i = 0; i < N_CHUNKS; ++i, ++gi) {
                    const uint32_t st = gi % RING_STAGES, ph = (gi / RING_STAGES) & 1u;
                    mbar_wait(&empty_bar[st], ph ^ 1u);
                    mbar_expect_tx(&full_bar[st], CHUNK_FLOATS * 4);
                    tma_bulk_g2s(ring + (size_t)st * CHUNK_FLOATS * 4, src + (size_t)i * CHUNK_FLOATS, CHUNK_FLOATS * 4,
                                 &full_bar[st]);
                }
            }
            __syncwarp();
            if (!__syncthreads_or(0)) break;
        }
    } else if (warp == 17) {
        // ===== MMA issuer =====
        const uint32_t idesc1 = umma_idesc_tf32(128, W, false, false);
        const uint32_t r_u = smem_u32(Rsm), ring_u = smem_u32(ring);
        const uint32_t w0hi = r_u + (uint32_t)a.lay.w0hi * 4u, w0lo = r_u + (uint32_t)a.lay.w0lo * 4u;
        const uint32_t ohi = smem_u32(O_hi), olo = smem_u32(O_lo);
        uint32_t gi = 0;
        for (int t = 0; t < T; ++t) {
            // ---- first Linear: D = [obs, 1] . [W0, b0]^T  (3xTF32, both operands K-major in smem)
            named_sync(BAR_L1, 544);
            tc_fence_after();
            if (lane == 0) {
                uint32_t acc = 0;
#pragma unroll
                for (int pass = 0; pass < 3; ++pass) {
                    const uint32_t aa = pass == 2 ? olo : ohi, bb = pass == 1 ? w0lo : w0hi;
#pragma unroll
                    for (int k = 0; k < OKP; k += 8) {
                        umma_tf32(tmem + TM_D, umma_operand_desc(aa, OKP, false, k), umma_operand_desc(bb, OKP, false, k),
                                  idesc1, acc);
                        acc = 1u;
                    }
                }
                umma_commit(&bar_d);
            }
            __syncwarp();
            // ---- second Linear, two K halves; each (hi, lo) chunk pair: A_hi.B_hi, A_lo.B_hi, A_hi.B_lo
            for (int half = 0; half < 2; ++half) {
                if (half == 0) named_sync(BAR_K0, 544);
                else named_sync(BAR_K1, 288);
                tc_fence_after();
                if (lane == 0) {
                    for (int c = 0; c < 4; ++c) {
                        const uint32_t st_hi = gi % RING_STAGES, ph_hi = (gi / RING_STAGES) & 1u;
                        ++gi;
                        const uint32_t st_lo = gi % RING_STAGES, ph_lo = (gi / RING_STAGES) & 1u;
                        ++gi;
                        const uint32_t bhi = ring_u + st_hi * (CHUNK_FLOATS * 4), blo = ring_u + st_lo * (CHUNK_FLOATS * 4);
                        const uint32_t acol = (uint32_t)(c * CHUNK_K);
                        mbar_wait(&full_bar[st_hi], ph_hi);
                        tc_fence_after();
#pragma unroll
                        for (int ks = 0; ks < CHUNK_K; ks += 8)
                            umma_tf32_ts(tmem + TM_D, tmem + TM_AHI + acol + (uint32_t)ks,
                                         umma_operand_desc(bhi, CHUNK_K, false, ks), idesc1, (half | c | ks) ? 1u : 0u);
#pragma unroll
                        for (int ks = 0; ks < CHUNK_K; ks += 8)
                            umma_tf32_ts(tmem + TM_D, tmem + TM_ALO + acol + (uint32_t)ks,
                                         umma_operand_desc(bhi, CHUNK_K, false, ks), idesc1, 1u);
                        umma_commit(&empty_bar[st_hi]);
                        mbar_wait(&full_bar[st_lo], ph_lo);
                        tc_fence_after();
#pragma unroll
                        for (int ks = 0; ks < CHUNK_K; ks += 8)
                            umma_tf32_ts(tmem + TM_D, tmem + TM_AHI + acol + (uint32_t)ks,
                                         umma_operand_desc(blo, CHUNK_K, false, ks), idesc1, 1u);
                        umma_commit(&empty_bar[st_lo]);
                    }
                    umma_commit(half == 0 ? &bar_k0 : &bar_d);
                }
                __syncwarp();
            }
            if (!__syncthreads_or(0)) break;
        }
    } else {
        // ===== compute warps =====
        const int q = warp & 3, part = warp >> 2;     // lane quadrant, column part (64 columns each)
        const int e = q * 32 + lane;                  // env row = TMEM lane
        const int c0 = part * HW;
        const uint32_t my_tm = tmem + ((uint32_t)(q * 32) << 16);
        const int64_t n = (int64_t)blockIdx.x * 128 + e;
        const int act_kind = RELU ? TG_ACT_RELU : a.lay.act;
        const float *b1 = Rsm + a.lay.b1 + c0, *wo = Rsm + a.lay.wo + c0, *bo = Rsm + a.lay.bo;
        Ev ev(a.io, n, n < a.io.N && part == 0, true);      // only part 0 holds, steps and records the env
        uint32_t ph_d = 0, ph_k0 = 0;
        int t = 0;
        for (; t < T; ++t) {
            if (part == 0) {
                float x[S];
                ev.observe(a.io, t, x);
#pragma unroll
                for (int i = 0; i < S; ++i) {
                    const float xh = tf32_hi(x[i]);
                    *reinterpret_cast<float *>(O_hi + core_offset(OKP, e, i)) = xh;
                    *reinterpret_cast<float *>(O_lo + core_offset(OKP, e, i)) = x[i] - xh;
                }
            }
            fence_proxy_async();
            tc_fence_before();
            named_arrive(BAR_L1, 544);
            mbar_wait(&bar_d, ph_d);
            ph_d ^= 1u;
            tc_fence_after();
            // ---- epilogue 1: H1 = act(D) (bias folded into the GEMM), split, A operand of this thread's K half
            float h[HW];
#pragma unroll
            for (int cc = 0; cc < HW; cc += 32) {
                float z[32];
                tmem_ld32(my_tm + TM_D + (uint32_t)(c0 + cc), z);
#pragma unroll
                for (int j = 0; j < 32; ++j) h[cc + j] = act_fwd(z[j], act_kind);
            }
            tc_fence_before();
            if (part >= 2) {
                named_arrive(BAR_K0, 544);               // this thread has read D; its K half waits for half 0
                mbar_wait(&bar_k0, ph_k0);
                tc_fence_after();
            }
            ph_k0 ^= 1u;
            {
                const uint32_t acol = (uint32_t)((part & 1) * HW);
#pragma unroll
                for (int cc = 0; cc < HW; cc += 32) {
                    float hi[32], lo[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        hi[j] = tf32_hi(h[cc + j]);
                        lo[j] = h[cc + j] - hi[j];
                    }
                    tmem_st32(my_tm + TM_AHI + acol + (uint32_t)cc, hi);
                    tmem_st32(my_tm + TM_ALO + acol + (uint32_t)cc, lo);
                }
                tmem_st_wait();
                tc_fence_before();
            }
            if (part >= 2) named_arrive(BAR_K1, 288);
            else named_arrive(BAR_K0, 544);
            mbar_wait(&bar_d, ph_d);
            ph_d ^= 1u;
            tc_fence_after();
            // ---- epilogue 2: H2 = act(D + b1); partial output-layer dot products
            float pm[A];
#pragma unroll
            for (int j = 0; j < A; ++j) pm[j] = 0.0f;
#pragma unroll
            for (int cc = 0; cc < HW; cc += 32) {
                float z[32];
                tmem_ld32(my_tm + TM_D + (uint32_t)(c0 + cc), z);
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    const float4 b4 = *reinterpret_cast<const float4 *>(b1 + cc + j);
                    const float h0 = act_fwd(z[j] + b4.x, act_kind), h1 = act_fwd(z[j + 1] + b4.y, act_kind);
                    const float h2 = act_fwd(z[j + 2] + b4.z, act_kind), h3 = act_fwd(z[j + 3] + b4.w, act_kind);
#pragma unroll
                    for (int o = 0; o < A; ++o) {
                        const float4 v = *reinterpret_cast<const float4 *>(wo + o * W + cc + j);
                        pm[o] = fmaf(h0, v.x, pm[o]); pm[o] = fmaf(h1, v.y, pm[o]);
                        pm[o] = fmaf(h2, v.z, pm[o]); pm[o] = fmaf(h3, v.w, pm[o]);
                    }
                }
            }
            tc_fence_before();
#pragma unroll
            for (int j = 0; j < A; ++j) muS[part][j][e] = pm[j];
            named_sync(q + 1, 128);                      // the four warps of this lane quadrant
            if (part == 0) {
                float mu[A];
#pragma unroll
                for (int j = 0; j < A; ++j) mu[j] = (((bo[j] + muS[0][j][e]) + muS[1][j][e]) + muS[2][j][e]) + muS[3][j][e];
                ev.act(a.io, t, mu);
            }
            if (!__syncthreads_or(ev.alive ? 1 : 0)) { ++t; break; }
        }
        ev.finish(a.io, t);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 512);
}

// Called by tg_rollout (tg_rollout.cu) for eligible 256-wide policies; io.init_state is `precision`.
int tg_rollout_tc256(tg_ctx *ctx, const tg_mlp_cfg *mlp, int precision, int kind, const float *params, const RolloutIo &io,
                     cudaStream_t st) {
    RolloutArgs<TcwLayout> a;
    memset(&a, 0, sizeof(a));
    a.io = io;
    tg_build_tcw_layout(mlp, &a.lay, false);      // without the backward chunks
    int rc = tg_pack_weights_tcw(ctx, a.lay, params, st);
    if (rc) return rc;
    a.packed = ctx->packed_tc;
    const size_t smem = (size_t)RING_STAGES * CHUNK_FLOATS * 4 + (size_t)a.lay.resident * 4 + 2 * (size_t)128 * a.lay.OKP * 4;
    TG_REQUIRE(smem + 12 * 1024 <= (size_t)ctx->smem_optin, TG_ERR_UNSUPPORTED, "tc256 rollout needs %zu B of shared memory", smem);
    auto kern = tg_with_env_kind(kind, [&](auto k) {
        return tg_with_prec_relu(precision, a.lay.act, [](auto r, auto relu) {
            return rollout_tc256_kernel<decltype(k)::value, decltype(r), decltype(relu)::value>;
        });
    });
    TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)((io.N + 127) / 128), 576, smem, st>>>(a);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}
