// K3: fused clipped-surrogate objective + MLP backward (tg_policy_grad), the
// critic regression gradient (tg_value_grad), the batched forward / log-prob
// (tg_policy_forward) and Adam (tg_adam_step).
//
// Persistent CTAs walk tiles of B samples (one step t, B consecutive envs --
// every trajectory row is then a coalesced 128 B-per-warp read).  Per tile, all
// in shared memory: forward through the MLP keeping every hidden activation,
// the per-sample objective and d objective / d mu, then the backward sweep:
//   dW_l  = dZ_l . H_{l-1}^T   (register-tiled, reduction over the B samples)
//   dZ_{l-1} = (W_l^T dZ_l) * act'(H_{l-1})   (same tiled GEMM as the forward)
// Each CTA adds its tile's dW into a CTA-private copy of the flat gradient
// (plain read-modify-write by a fixed owner thread, L2-resident), and a second
// kernel sums the private copies in a fixed order: the result is deterministic
// and has the flat torch layout the NCCL allreduce and Adam consume.
#include <math.h>

#include "tg_mlp.cuh"

#define HEAD_POLICY 0
#define HEAD_VALUE 1
#define HEAD_FORWARD 2

struct UpdArgs {
    tg_mlp_layout lay;
    int64_t N;
    int T;
    int head;
    const float *obs, *act, *adv, *oldlp, *target;
    const float *reflp;   // log-prob under a frozen reference policy (GRPO's KL term) or null
    const int32_t *len;
    // length order (tg_order.cu) or null: sorted position j of step t is env perm[j], live iff j < cnt[t]
    const int32_t *perm, *cnt;
    // minibatch mode (PPO with batch_size, ppo.py:147-157) or null: the launch covers the n_sidx samples
    // whose flat slot ids t*N + n are listed in sidx, in that order
    const int64_t *sidx;
    int64_t n_sidx;
    const float *packed;
    float inv_sd[TG_MAX_ACT], inv_var[TG_MAX_ACT], log_norm;
    float eps_clip, scale, kl_scale, ref_coef;
    float *gpart;   // [grid][n_params]
    double *spart;  // [grid][TG_SPART_LD]
    float *out_mu, *out_logp;
};

// Fire-and-forget accumulation into the CTA-private gradient copy (SASS RED.E.ADD.F32): every element has
// one fixed owner thread, so the additions to an address are issued by one thread in program order and the
// sum stays deterministic -- but unlike a load/add/store the thread never waits for the L2 round trip.
TG_D void red_add(float *p, float v) { asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }

// dW[n][k] (+)= sum_b dZ[n][b] * H[k][b] for a BIxBJ register block per thread;
// rows are interleaved (n = nb + i*NBI, k = kb + j*KBJ) so that the 8 lanes of a
// quarter warp read 8 consecutive shared-memory rows (conflict-free LDS.128) and
// the global read-modify-write of gW is coalesced along k.
template <int CFG, int BI, int BJ>
TG_D void tile_dw_blk(const float *dZ, int Nn, const float *Hin, int Kk, float *__restrict__ gW) {
    constexpr int B = TileCfg<CFG>::B, NT = TileCfg<CFG>::NT, LDX = B + 4;
    const int NBI = (Nn + BI - 1) / BI, KBJ = (Kk + BJ - 1) / BJ;
    const int nblk = NBI * KBJ;
    for (int blk = threadIdx.x; blk < nblk; blk += NT) {
        const int kb = blk % KBJ, nb = blk / KBJ;
        float acc[BI][BJ];
#pragma unroll
        for (int i = 0; i < BI; ++i)
#pragma unroll
            for (int j = 0; j < BJ; ++j) acc[i][j] = 0.0f;
#pragma unroll 2
        for (int b = 0; b < B; b += 4) {
            float4 dz[BI], h[BJ];
#pragma unroll
            for (int i = 0; i < BI; ++i) dz[i] = *reinterpret_cast<const float4 *>(dZ + (nb + i * NBI) * LDX + b);
#pragma unroll
            for (int j = 0; j < BJ; ++j) h[j] = *reinterpret_cast<const float4 *>(Hin + (kb + j * KBJ) * LDX + b);
#pragma unroll
            for (int i = 0; i < BI; ++i)
#pragma unroll
                for (int j = 0; j < BJ; ++j) {
                    acc[i][j] = fmaf(dz[i].x, h[j].x, acc[i][j]);
                    acc[i][j] = fmaf(dz[i].y, h[j].y, acc[i][j]);
                    acc[i][j] = fmaf(dz[i].z, h[j].z, acc[i][j]);
                    acc[i][j] = fmaf(dz[i].w, h[j].w, acc[i][j]);
                }
        }
#pragma unroll
        for (int i = 0; i < BI; ++i) {
            const int n = nb + i * NBI;
            if (n < Nn) {
#pragma unroll
                for (int j = 0; j < BJ; ++j) {
                    const int k = kb + j * KBJ;
                    if (k < Kk) red_add(gW + (int64_t)n * Kk + k, acc[i][j]);
                }
            }
        }
    }
}

// The buffers have at least roundup(Nn,8) and roundup(Kk,8) rows (zero/finite padding).
template <int CFG>
TG_D void tile_dw(const float *dZ, int Nn, const float *Hin, int Kk, float *__restrict__ gW, float *__restrict__ gB) {
    constexpr int B = TileCfg<CFG>::B, NT = TileCfg<CFG>::NT, LDX = B + 4;
    const int n88 = ((Nn + 7) / 8) * ((Kk + 7) / 8);
    if (n88 >= NT) tile_dw_blk<CFG, 8, 8>(dZ, Nn, Hin, Kk, gW);
    else if (2 * n88 >= NT) tile_dw_blk<CFG, 8, 4>(dZ, Nn, Hin, Kk, gW);
    else tile_dw_blk<CFG, 4, 4>(dZ, Nn, Hin, Kk, gW);
    // bias gradient: row sums of dZ
    for (int n = threadIdx.x; n < Nn; n += NT) {
        float s = 0.0f;
        for (int b = 0; b < B; b += 4) {
            const float4 v = *reinterpret_cast<const float4 *>(dZ + n * LDX + b);
            s += (v.x + v.y) + (v.z + v.w);
        }
        red_add(gB + n, s);
    }
}

template <int CFG, int A, bool WG>
__global__ void __launch_bounds__(TileCfg<CFG>::NT) update_kernel(const __grid_constant__ UpdArgs a) {
    constexpr int B = TileCfg<CFG>::B, NT = TileCfg<CFG>::NT, NP = TileCfg<CFG>::NP, LDX = B + 4;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t wbar;
    __shared__ double sred[TG_NSTAT][NT / 32];
    __shared__ int32_t tile_env[B];      // env index of each sample of the tile, -1 = padding
    __shared__ int32_t tile_t[B];        // its step index (tile-uniform except in minibatch mode)
    const int nl = a.lay.n_layers, nh = nl - 1;
    const int O = a.lay.O, O8 = tg_round_up(O, 8);
    float *Ws = reinterpret_cast<float *>(smem_raw);
    float *X0 = Ws + (WG ? 0 : a.lay.total);        // [O8][LDX]
    float *H = X0 + (size_t)O8 * LDX;               // nh buffers of [NP][LDX]
    float *D = H + (size_t)nh * NP * LDX;           // [8][LDX]  d objective / d mu
    float *P = D + 8 * LDX;                         // output-layer partials
    const float *W = WG ? a.packed : Ws;
    if (!WG) stage_weights_tma(Ws, a.packed, a.lay.total, &wbar);
    for (int i = threadIdx.x; i < 8 * LDX; i += NT) D[i] = 0.0f;
    for (int i = threadIdx.x; i < O8 * LDX; i += NT) X0[i] = 0.0f;
    __syncthreads();

    const int64_t N = a.N;
    const int64_t NB = a.sidx ? (a.n_sidx + B - 1) / B : (N + B - 1) / B;
    const int64_t ntiles = a.sidx ? NB : NB * a.T;
    float *gp = a.gpart ? a.gpart + (int64_t)blockIdx.x * a.lay.n_params : nullptr;
    const bool owner = threadIdx.x < B;
    double s_obj = 0.0, s_cnt = 0.0, s_ratio = 0.0, s_clip = 0.0, s_kl = 0.0;
    const tg_layer_layout &LO = a.lay.L[nl - 1];

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int t = (int)(tile / NB);
        const int64_t nb0 = (tile % NB) * B;
        // ---- 1. load the tile's observations (rows of obs[t][o][:]; coalesced when the tile is a run of
        //         consecutive envs, a gather through perm when the rollout is walked in length order)
        bool valid = false;
        int64_t n_own = 0;
        int t_own = t;
        if (a.sidx == nullptr && a.cnt != nullptr && nb0 >= a.cnt[t]) continue;   // whole tile is padding (CTA-uniform)
        if (owner) {
            const int64_t j = nb0 + threadIdx.x;
            if (a.sidx != nullptr) {
                valid = j < a.n_sidx;
                if (valid) {
                    const int64_t id = a.sidx[j];
                    t_own = (int)(id / N);
                    n_own = id % N;
                }
            } else if (a.cnt != nullptr) {
                valid = j < a.cnt[t];
                n_own = valid ? a.perm[j] : 0;
            } else {
                n_own = j;
                valid = j < N && (a.len == nullptr || t < a.len[j]);
            }
            tile_env[threadIdx.x] = valid ? (int32_t)n_own : -1;
            tile_t[threadIdx.x] = t_own;
        }
        if (!__syncthreads_or(valid ? 1 : 0)) continue;   // whole tile is padding
        for (int idx = threadIdx.x; idx < O * B; idx += NT) {
            const int o = idx / B, b = idx % B;
            const int32_t n = tile_env[b];
            X0[o * LDX + b] = n >= 0 ? a.obs[((int64_t)tile_t[b] * O + o) * N + n] : 0.0f;
        }
        __syncthreads();
        // ---- 2. forward, keeping H_1..H_nh
        for (int l = 0; l < nh; ++l) {
            tile_layer<CFG, 0, WG>(W + a.lay.L[l].wt, W + a.lay.L[l].bias, l == 0 ? X0 : H + (size_t)(l - 1) * NP * LDX,
                                   H + (size_t)l * NP * LDX, a.lay.L[l].K, a.lay.acts[l]);
            __syncthreads();
        }
        const float *Hlast = nh > 0 ? H + (size_t)(nh - 1) * NP * LDX : X0;
        float mu[A];
        tile_output_layer<CFG, A, WG>(W + LO.wt, W + LO.bias, Hlast, P, LO.K, mu);
        // ---- 3. per-sample objective and d/dmu
        if (owner) {
            const int64_t n = n_own;
            float dmu[A];
#pragma unroll
            for (int j = 0; j < A; ++j) dmu[j] = 0.0f;
            if (valid) {
                const int64_t row = (int64_t)t_own * N + n;
                if (a.head == HEAD_VALUE) {
                    const float err = mu[0] - a.target[row];       // ppo.py:168-169 MSELoss
                    s_obj += (double)err * err;
                    s_cnt += 1.0;
                    dmu[0] = 2.0f * a.scale * err;
                } else {
                    float av[A], m2 = 0.0f;
                    bool have_act = a.act != nullptr;
#pragma unroll
                    for (int j = 0; j < A; ++j) {
                        av[j] = have_act ? a.act[((int64_t)t_own * A + j) * N + n] : mu[j];
                        const float z = (av[j] - mu[j]) * a.inv_sd[j];
                        m2 += z * z;
                    }
                    const float lp = -0.5f * m2 - a.log_norm;       // MultivariateNormal.log_prob
                    if (a.head == HEAD_FORWARD) {
                        if (a.out_logp) a.out_logp[row] = lp;
#pragma unroll
                        for (int j = 0; j < A; ++j)
                            if (a.out_mu) a.out_mu[((int64_t)t_own * A + j) * N + n] = mu[j];
                    } else {
                        const float adv = a.adv[row], olp = a.oldlp[row];
                        const float ratio = expf(lp - olp);          // grpo.py:125 / ppo.py:160
                        const float lo = 1.0f - a.eps_clip, hi = 1.0f + a.eps_clip;
                        const float s1 = ratio * adv;
                        const float s2 = fminf(fmaxf(ratio, lo), hi) * adv;
                        const bool in_range = ratio >= lo && ratio <= hi;   // clamp backward mask
                        // torch.min backward: the smaller branch takes the gradient, ties split 50/50
                        float g;
                        if (s1 < s2) g = adv;
                        else if (s1 > s2) g = in_range ? adv : 0.0f;
                        else g = 0.5f * (adv + (in_range ? adv : 0.0f));
                        s_obj += (double)fminf(s1, s2) * a.scale;
                        float dlp = a.scale * g * ratio;
                        if (a.kl_scale != 0.0f) {                   // ppo.py:175-176
                            const float eo = expf(olp);
                            s_obj += (double)a.kl_scale * eo * (olp - lp);
                            dlp -= a.kl_scale * eo;
                        }
                        if (a.reflp) {                              // k3 KL to the reference policy
                            const float u = a.reflp[row] - lp, em = expm1f(u);
                            const float d = em - u;
                            s_obj -= (double)a.ref_coef * d;
                            s_kl += d;
                            dlp += a.ref_coef * em;
                        }
                        s_cnt += 1.0;
                        s_ratio += ratio;
                        s_clip += in_range ? 0.0 : 1.0;
#pragma unroll
                        for (int j = 0; j < A; ++j) dmu[j] = dlp * (av[j] - mu[j]) * a.inv_var[j];
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < A; ++j) D[j * LDX + threadIdx.x] = dmu[j];
        }
        __syncthreads();
        if (a.head == HEAD_FORWARD) continue;
        // ---- 4. output layer: dWo, dbo, then dZ_nh in place over H_nh
        tile_dw<CFG>(D, A, Hlast, LO.K, gp + LO.flat_w, gp + LO.flat_w + (int64_t)LO.N * LO.K);
        if (nh > 0) {
            __syncthreads();
            float *Hl = H + (size_t)(nh - 1) * NP * LDX;
            const float *Wo = W + LO.wt;
            const int K = LO.K;
            for (int idx = threadIdx.x; idx < NP * B; idx += NT) {
                const int k = idx / B, b = idx % B;
                float s = 0.0f;
                if (k < K) {
#pragma unroll
                    for (int j = 0; j < A; ++j) s = fmaf(ldw1<WG>(Wo + j * K + k), D[j * LDX + b], s);
                    s *= act_bwd_from_out(Hl[k * LDX + b], a.lay.acts[nh - 1]);
                }
                Hl[k * LDX + b] = s;
            }
            __syncthreads();
            // ---- 5. hidden layers, last to first
            for (int l = nh - 1; l >= 0; --l) {
                const tg_layer_layout &L = a.lay.L[l];
                const float *dZ = H + (size_t)l * NP * LDX;
                float *Hin = l == 0 ? X0 : H + (size_t)(l - 1) * NP * LDX;
                tile_dw<CFG>(dZ, L.N, Hin, L.K, gp + L.flat_w, gp + L.flat_w + (int64_t)L.N * L.K);
                __syncthreads();
                if (l > 0) {
                    tile_layer<CFG, 1, WG>(W + L.wn, nullptr, dZ, Hin, L.N, a.lay.acts[l - 1]);
                    __syncthreads();
                }
            }
        } else {
            __syncthreads();
        }
    }
    // ---- statistics: warp shuffle, then a fixed-order sum over the warps
    if (a.spart) {
        double v[TG_NSTAT] = {s_obj, s_cnt, s_ratio, s_clip, s_kl};
#pragma unroll
        for (int q = 0; q < TG_NSTAT; ++q) {
            for (int off = 16; off > 0; off >>= 1) v[q] += __shfl_down_sync(0xffffffffu, v[q], off);
            if ((threadIdx.x & 31) == 0) sred[q][threadIdx.x >> 5] = v[q];
        }
        __syncthreads();
        if (threadIdx.x < TG_NSTAT) {
            double s = 0.0;
            for (int w = 0; w < NT / 32; ++w) s += sred[threadIdx.x][w];
            a.spart[(int64_t)blockIdx.x * TG_SPART_LD + threadIdx.x] = s;
        }
    }
}

// sum the CTA-private gradient copies in a fixed order; the first nstat statistics go to out_stats
__global__ void grad_reduce_kernel(int grid, int64_t n_params, const float *__restrict__ gpart,
                                   const double *__restrict__ spart, float *__restrict__ out_grad,
                                   float *__restrict__ out_stats, int nstat) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_params) {
        float s = 0.0f;
        for (int c = 0; c < grid; ++c) s += gpart[(int64_t)c * n_params + i];
        out_grad[i] = s;
    }
    if (out_stats && blockIdx.x == 0 && threadIdx.x < nstat) {
        double s = 0.0;
        for (int c = 0; c < grid; ++c) s += spart[(int64_t)c * TG_SPART_LD + threadIdx.x];
        out_stats[threadIdx.x] = (float)s;
    }
}

static size_t update_smem_bytes(const tg_mlp_layout &lay, bool with_weights) {
    return tg_update_smem_bytes(lay, with_weights);
}

static int update_grid(const tg_ctx *ctx, const tg_mlp_layout &lay) {
    const size_t act = update_smem_bytes(lay, false);
    int per_sm = (int)((size_t)ctx->smem_optin / (act + (size_t)lay.total * 4 + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 2) per_sm = 2;
    return ctx->sm_count * per_sm;
}

template <int CFG, int A>
static int launch_update(const tg_ctx *ctx, const UpdArgs &a, int grid, cudaStream_t st) {
    constexpr int NT = TileCfg<CFG>::NT;
    size_t smem = update_smem_bytes(a.lay, true);
    const bool wg = smem > (size_t)ctx->smem_optin;
    if (wg) smem = update_smem_bytes(a.lay, false);
    TG_REQUIRE(smem <= (size_t)ctx->smem_optin, TG_ERR_UNSUPPORTED,
               "update tiles need %zu B of shared memory (%d hidden layers of width <= %d)", smem, a.lay.n_layers - 1,
               a.lay.NP);
    if (wg) {
        auto kern = update_kernel<CFG, A, true>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, NT, smem, st>>>(a);
    } else {
        auto kern = update_kernel<CFG, A, false>;
        TG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, NT, smem, st>>>(a);
    }
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

template <int A>
static int dispatch_update_cfg(const tg_ctx *ctx, const UpdArgs &a, int grid, cudaStream_t st) {
    switch (a.lay.cfg) {
        case 0: return launch_update<0, A>(ctx, a, grid, st);
        case 1: return launch_update<1, A>(ctx, a, grid, st);
        case 3: return launch_update<3, A>(ctx, a, grid, st);
        default: return launch_update<2, A>(ctx, a, grid, st);
    }
}

static int dispatch_update(const tg_ctx *ctx, const UpdArgs &a, int grid, cudaStream_t st) {
    switch (a.lay.A) {
        case 1: return dispatch_update_cfg<1>(ctx, a, grid, st);
        case 2: return dispatch_update_cfg<2>(ctx, a, grid, st);
        case 4: return dispatch_update_cfg<4>(ctx, a, grid, st);
        default:
            tg_set_error("output dim %d has no update kernel instance (1, 2 and 4 are built)", a.lay.A);
            return TG_ERR_UNSUPPORTED;
    }
}

extern "C" int64_t tg_policy_grad_workspace_bytes(const tg_ctx *ctx, const tg_mlp_cfg *mlp) {
    if (!ctx || !mlp) return -1;
    tg_mlp_layout lay;
    if (tg_build_layout(mlp, true, &lay, ctx->smem_optin)) return -1;
    const int64_t grid = update_grid(ctx, lay);
    return grid * lay.n_params * (int64_t)sizeof(float) + grid * TG_SPART_LD * (int64_t)sizeof(double) + 256;
}

// The gradient of every update path: the workspace holds one partial gradient per CTA, gpart [grid][n_params], and
// the statistics spart [grid][TG_SPART_LD] (256-byte aligned); both are zeroed, `update(gpart, spart)` launches the
// kernels that fill them, and grad_reduce_kernel sums the copies in a fixed order into out_grad and the first
// `nstat` statistics into out_stats.
template <typename Update>
static int grad_via_partials(int grid, int64_t n_params, void *workspace, float *out_grad, float *out_stats, int nstat,
                             cudaStream_t st, Update update) {
    const size_t gbytes = ((size_t)grid * n_params * sizeof(float) + 255) / 256 * 256;
    float *gpart = reinterpret_cast<float *>(workspace);
    double *spart = reinterpret_cast<double *>(reinterpret_cast<char *>(workspace) + gbytes);
    TG_CUDA(cudaMemsetAsync(workspace, 0, gbytes + (size_t)grid * TG_SPART_LD * sizeof(double), st));
    int rc = update(gpart, spart);
    if (rc) return rc;
    grad_reduce_kernel<<<(unsigned)((n_params + 255) / 256), 256, 0, st>>>(grid, n_params, gpart, spart, out_grad,
                                                                          out_stats, nstat);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

static int run_grad(tg_ctx *ctx, UpdArgs &a, const float *params, float *out_grad, float *out_stats, int nstat,
                    void *workspace, cudaStream_t st) {
    TG_CUDA(cudaSetDevice(ctx->device));
    int rc = tg_pack_weights(ctx, a.lay, params, st);
    if (rc) return rc;
    a.packed = ctx->packed;
    if (a.len != nullptr && a.sidx == nullptr) {  // ragged episodes: walk the samples in length order
        rc = tg_len_order(ctx, a.N, a.T, a.len, st);
        if (rc) return rc;
        a.perm = ctx->perm;
        a.cnt = ctx->cnt;
    }
    const int grid = update_grid(ctx, a.lay);
    return grad_via_partials(grid, a.lay.n_params, workspace, out_grad, out_stats, nstat, st, [&](float *gpart, double *spart) {
        a.gpart = gpart;
        a.spart = spart;
        return dispatch_update(ctx, a, grid, st);
    });
}

// tg_policy_grad and tg_policy_grad_ref: ref_logp == null leaves out the KL term and writes 4 statistics
static int policy_grad_impl(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *act,
                            const float *adv, const float *old_logp, const float *ref_logp, const int32_t *len,
                            const float *params, const float *cov_diag, float eps_clip, float scale, float kl_coef,
                            float ref_coef, float *out_grad, float *out_stats, void *workspace, void *stream) {
    TgRange nvtx_range("tg_policy_grad (K3: clipped surrogate + MLP backward)");
    TG_REQUIRE(ctx && mlp && obs && act && adv && old_logp && len && params && cov_diag && out_grad && workspace,
               TG_ERR_ARG, "tg_policy_grad: null argument");
    TG_REQUIRE(N > 0 && T > 0, TG_ERR_SHAPE, "tg_policy_grad: N and T must be positive");
    const int nstat = ref_logp ? TG_NSTAT : 4;
    UpdArgs a;
    memset(&a, 0, sizeof(a));
    int rc = tg_build_layout(mlp, true, &a.lay, ctx->smem_optin);
    if (rc) return rc;
    rc = tg_gauss_consts(cov_diag, a.lay.A, nullptr, a.inv_sd, a.inv_var, &a.log_norm);
    if (rc) return rc;
    a.N = N; a.T = T; a.head = HEAD_POLICY;
    a.obs = obs; a.act = act; a.adv = adv; a.oldlp = old_logp; a.reflp = ref_logp; a.len = len;
    a.eps_clip = eps_clip; a.scale = scale; a.kl_scale = kl_coef; a.ref_coef = ref_coef;
    // ---- tensor-core paths (3xTF32 tcgen05) for eligible policies
    if (tg_update_tcw_shape_built(mlp) && ctx->math_mode != TG_MATH_FP32) {      // 128 / 256 wide: streamed, two kernels
        cudaStream_t st = (cudaStream_t)stream;
        TG_CUDA(cudaSetDevice(ctx->device));
        const int grid = ctx->sm_count;
        return grad_via_partials(grid, a.lay.n_params, workspace, out_grad, out_stats, nstat, st,
                                 [&](float *gpart, double *spart) {
            return tg_policy_grad_tcw(ctx, mlp, N, T, obs, act, adv, old_logp, nullptr, len, params, a.inv_sd, a.inv_var,
                                      a.log_norm, eps_clip, scale, kl_coef, gpart, spart, grid, st, nullptr, nullptr,
                                      ref_logp, ref_coef);
        });
    }
    const bool tc_ok = tg_update_tc_eligible(mlp);
    TG_REQUIRE(ctx->math_mode != TG_MATH_3XTF32 || tc_ok, TG_ERR_UNSUPPORTED,
               "TG_MATH_3XTF32 requested but the policy shape has no tensor-core update kernel "
               "(obs -> %d -> %d -> act for the four environments)", TC_W, TC_W);
    if (tc_ok && ctx->math_mode != TG_MATH_FP32) {
        cudaStream_t st = (cudaStream_t)stream;
        TG_CUDA(cudaSetDevice(ctx->device));
        const int grid = tg_update_tc_grid(ctx);
        return grad_via_partials(grid, a.lay.n_params, workspace, out_grad, out_stats, nstat, st,
                                 [&](float *gpart, double *spart) {
            return tg_policy_grad_tc(ctx, mlp, N, T, obs, act, adv, old_logp, ref_logp, len, params, a.inv_sd, a.inv_var,
                                     a.log_norm, eps_clip, scale, kl_coef, ref_coef, gpart, spart, grid, st);
        });
    }
    return run_grad(ctx, a, params, out_grad, out_stats, nstat, workspace, (cudaStream_t)stream);
}

extern "C" int tg_policy_grad(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *act,
                              const float *adv, const float *old_logp, const int32_t *len, const float *params,
                              const float *cov_diag, float eps_clip, float scale, float kl_coef, float *out_grad,
                              float *out_stats, void *workspace, void *stream) {
    return policy_grad_impl(ctx, mlp, N, T, obs, act, adv, old_logp, nullptr, len, params, cov_diag, eps_clip, scale,
                            kl_coef, 0.0f, out_grad, out_stats, workspace, stream);
}

extern "C" int tg_policy_grad_ref(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs,
                                  const float *act, const float *adv, const float *old_logp, const float *ref_logp,
                                  const int32_t *len, const float *params, const float *cov_diag, float eps_clip,
                                  float scale, float kl_coef, float ref_coef, float *out_grad, float *out_stats,
                                  void *workspace, void *stream) {
    return policy_grad_impl(ctx, mlp, N, T, obs, act, adv, old_logp, ref_logp, len, params, cov_diag, eps_clip, scale,
                            kl_coef, ref_coef, out_grad, out_stats, workspace, stream);
}

// Minibatch forms (PPO with batch_size != None, algorithms/ppo.py:147-183): the gradient of the same
// objective over an explicit list of samples.  Always the FP32-pipe kernel (a minibatch is a few tiles).
extern "C" int tg_policy_grad_batch(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs,
                                    const float *act, const float *adv, const float *old_logp,
                                    const int64_t *sample_ids, int64_t n_samples, const float *params,
                                    const float *cov_diag, float eps_clip, float scale, float kl_coef, float *out_grad,
                                    float *out_stats, void *workspace, void *stream) {
    TG_REQUIRE(ctx && mlp && obs && act && adv && old_logp && sample_ids && params && cov_diag && out_grad && workspace,
               TG_ERR_ARG, "tg_policy_grad_batch: null argument");
    TG_REQUIRE(N > 0 && T > 0 && n_samples > 0, TG_ERR_SHAPE, "tg_policy_grad_batch: N, T, n_samples must be positive");
    UpdArgs a;
    memset(&a, 0, sizeof(a));
    int rc = tg_build_layout(mlp, true, &a.lay, ctx->smem_optin);
    if (rc) return rc;
    rc = tg_gauss_consts(cov_diag, a.lay.A, nullptr, a.inv_sd, a.inv_var, &a.log_norm);
    if (rc) return rc;
    a.N = N; a.T = T; a.head = HEAD_POLICY;
    a.obs = obs; a.act = act; a.adv = adv; a.oldlp = old_logp;
    a.sidx = sample_ids; a.n_sidx = n_samples;
    a.eps_clip = eps_clip; a.scale = scale; a.kl_scale = kl_coef;
    return run_grad(ctx, a, params, out_grad, out_stats, 4, workspace, (cudaStream_t)stream);
}

extern "C" int tg_value_grad_batch(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs,
                                   const float *target, const int64_t *sample_ids, int64_t n_samples,
                                   const float *params, float scale, float *out_grad, float *out_stats,
                                   void *workspace, void *stream) {
    TG_REQUIRE(ctx && mlp && obs && target && sample_ids && params && out_grad && workspace, TG_ERR_ARG,
               "tg_value_grad_batch: null argument");
    TG_REQUIRE(N > 0 && T > 0 && n_samples > 0, TG_ERR_SHAPE, "tg_value_grad_batch: N, T, n_samples must be positive");
    TG_REQUIRE(mlp->dims[mlp->n_layers] == 1, TG_ERR_SHAPE, "critic output dim must be 1");
    UpdArgs a;
    memset(&a, 0, sizeof(a));
    int rc = tg_build_layout(mlp, true, &a.lay, ctx->smem_optin);
    if (rc) return rc;
    a.N = N; a.T = T; a.head = HEAD_VALUE;
    a.obs = obs; a.target = target; a.scale = scale;
    a.sidx = sample_ids; a.n_sidx = n_samples;
    return run_grad(ctx, a, params, out_grad, out_stats, 4, workspace, (cudaStream_t)stream);
}

extern "C" int tg_value_grad(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs,
                             const float *target, const int32_t *len, const float *params, float scale,
                             float *out_grad, float *out_stats, void *workspace, void *stream) {
    TgRange nvtx_range("tg_value_grad (K3: critic regression gradient)");
    TG_REQUIRE(ctx && mlp && obs && target && len && params && out_grad && workspace, TG_ERR_ARG,
               "tg_value_grad: null argument");
    TG_REQUIRE(N > 0 && T > 0, TG_ERR_SHAPE, "tg_value_grad: N and T must be positive");
    TG_REQUIRE(mlp->dims[mlp->n_layers] == 1, TG_ERR_SHAPE, "critic output dim must be 1");
    UpdArgs a;
    memset(&a, 0, sizeof(a));
    int rc = tg_build_layout(mlp, true, &a.lay, ctx->smem_optin);
    if (rc) return rc;
    a.N = N; a.T = T; a.head = HEAD_VALUE;
    a.obs = obs; a.target = target; a.len = len; a.scale = scale;
    if (tg_update_tcw_shape_built(mlp) && ctx->math_mode != TG_MATH_FP32) {      // wide critic: streamed tensor-core path
        cudaStream_t st = (cudaStream_t)stream;
        TG_CUDA(cudaSetDevice(ctx->device));
        const int grid = ctx->sm_count;
        return grad_via_partials(grid, a.lay.n_params, workspace, out_grad, out_stats, 4, st, [&](float *gpart, double *spart) {
            return tg_policy_grad_tcw(ctx, mlp, N, T, obs, nullptr, nullptr, nullptr, target, len, params, nullptr, nullptr,
                                      0.0f, 0.0f, scale, 0.0f, gpart, spart, grid, st);
        });
    }
    return run_grad(ctx, a, params, out_grad, out_stats, 4, workspace, (cudaStream_t)stream);
}

extern "C" int tg_policy_forward(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t M, const float *x, const float *params,
                                 const float *cov_diag, const float *act, float *out_mu, float *out_logp,
                                 void *stream) {
    TG_REQUIRE(ctx && mlp && x && params, TG_ERR_ARG, "tg_policy_forward: null argument");
    TG_REQUIRE(out_mu || out_logp, TG_ERR_ARG, "tg_policy_forward: no output requested");
    TG_REQUIRE(!out_logp || (act && cov_diag), TG_ERR_ARG, "log-prob needs act and cov_diag");
    TG_REQUIRE(M > 0, TG_ERR_SHAPE, "M must be positive");
    UpdArgs a;
    memset(&a, 0, sizeof(a));
    int rc = tg_build_layout(mlp, false, &a.lay, ctx->smem_optin);
    if (rc) return rc;
    if (cov_diag) {
        rc = tg_gauss_consts(cov_diag, a.lay.A, nullptr, a.inv_sd, a.inv_var, &a.log_norm);
        if (rc) return rc;
    } else {
        for (int j = 0; j < TG_MAX_ACT; ++j) a.inv_sd[j] = a.inv_var[j] = 1.0f;
    }
    a.N = M; a.T = 1; a.head = HEAD_FORWARD;
    a.obs = x; a.act = act; a.out_mu = out_mu; a.out_logp = out_logp;
    cudaStream_t st = (cudaStream_t)stream;
    TG_CUDA(cudaSetDevice(ctx->device));
    rc = tg_pack_weights(ctx, a.lay, params, st);
    if (rc) return rc;
    a.packed = ctx->packed;
    int grid = update_grid(ctx, a.lay);
    const int64_t ntiles = (M + a.lay.B - 1) / a.lay.B;
    if (grid > ntiles) grid = (int)ntiles;
    return dispatch_update(ctx, a, grid, st);
}

extern "C" int tg_policy_forward_traj(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs,
                                      const float *act, const int32_t *len, const float *params,
                                      const float *cov_diag, float *out_mu, float *out_logp, void *stream) {
    TgRange nvtx_range("tg_policy_forward_traj (old log-probs / critic values)");
    TG_REQUIRE(ctx && mlp && obs && params, TG_ERR_ARG, "tg_policy_forward_traj: null argument");
    TG_REQUIRE(out_mu || out_logp, TG_ERR_ARG, "tg_policy_forward_traj: no output requested");
    TG_REQUIRE(!out_logp || (act && cov_diag), TG_ERR_ARG, "log-prob needs act and cov_diag");
    TG_REQUIRE(N > 0 && T > 0, TG_ERR_SHAPE, "N and T must be positive");
    UpdArgs a;
    memset(&a, 0, sizeof(a));
    int rc = tg_build_layout(mlp, false, &a.lay, ctx->smem_optin);
    if (rc) return rc;
    if (cov_diag) {
        rc = tg_gauss_consts(cov_diag, a.lay.A, nullptr, a.inv_sd, a.inv_var, &a.log_norm);
        if (rc) return rc;
    } else {
        for (int j = 0; j < TG_MAX_ACT; ++j) a.inv_sd[j] = a.inv_var[j] = 1.0f;
    }
    a.N = N; a.T = T; a.head = HEAD_FORWARD;
    a.obs = obs; a.act = act; a.len = len; a.out_mu = out_mu; a.out_logp = out_logp;
    cudaStream_t st = (cudaStream_t)stream;
    TG_CUDA(cudaSetDevice(ctx->device));
    if (len != nullptr && tg_update_tcw_shape_built(mlp) && ctx->math_mode != TG_MATH_FP32)   // wide: streamed tensor-core forward
        return tg_policy_grad_tcw(ctx, mlp, N, T, obs, act, nullptr, nullptr, nullptr, len, params, a.inv_sd, a.inv_var,
                                  a.log_norm, 0.0f, 0.0f, 0.0f, nullptr, nullptr, ctx->sm_count, st, out_mu, out_logp);
    rc = tg_pack_weights(ctx, a.lay, params, st);
    if (rc) return rc;
    a.packed = ctx->packed;
    if (len != nullptr) {
        rc = tg_len_order(ctx, N, T, len, st);
        if (rc) return rc;
        a.perm = ctx->perm;
        a.cnt = ctx->cnt;
    }
    int grid = update_grid(ctx, a.lay);
    const int64_t ntiles = ((N + a.lay.B - 1) / a.lay.B) * T;
    if (grid > ntiles) grid = (int)ntiles;
    return dispatch_update(ctx, a, grid, st);
}

// ---------------------------------------------------------------------------
// Adam (torch.optim.Adam defaults, single-tensor formula)
// ---------------------------------------------------------------------------
__global__ void adam_kernel(int64_t n, float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                            float *__restrict__ v, float step_size, float sqrt_bc2, float w1, float b2, float w2,
                            float eps) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float gi = g[i];
    const float mi = __fadd_rn(m[i], __fmul_rn(w1, __fsub_rn(gi, m[i])));            // exp_avg.lerp_(grad, 1-beta1)
    const float vi = __fadd_rn(__fmul_rn(v[i], b2), __fmul_rn(__fmul_rn(w2, gi), gi));  // mul_(b2).addcmul_(g,g,1-b2)
    m[i] = mi;
    v[i] = vi;
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), sqrt_bc2), eps);              // sqrt(v)/sqrt(bc2) + eps
    p[i] = __fsub_rn(p[i], __fmul_rn(step_size, __fdiv_rn(mi, denom)));             // addcdiv_(m, denom, -step_size)
}

extern "C" int tg_adam_step(tg_ctx *ctx, int64_t n, float *params, const float *grad, float *exp_avg,
                            float *exp_avg_sq, int64_t step, double lr, double beta1, double beta2, double eps,
                            void *stream) {
    TgRange nvtx_range("tg_adam_step");
    TG_REQUIRE(ctx && params && grad && exp_avg && exp_avg_sq, TG_ERR_ARG, "tg_adam_step: null argument");
    TG_REQUIRE(n > 0 && step >= 1, TG_ERR_SHAPE, "tg_adam_step: n>0 and step>=1 required");
    TG_CUDA(cudaSetDevice(ctx->device));
    // scalar prefactors in double, as torch computes them in Python before casting to fp32
    const double bc1 = 1.0 - pow(beta1, (double)step);
    const double bc2 = 1.0 - pow(beta2, (double)step);
    adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        n, params, grad, exp_avg, exp_avg_sq, (float)(lr / bc1), (float)sqrt(bc2), (float)(1.0 - beta1), (float)beta2,
        (float)(1.0 - beta2), (float)eps);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}
