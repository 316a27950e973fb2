// Shared host/device definitions for the sm_100a engine behind include/trajopt_grpo.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/trajopt_grpo.h"

#define TG_HD __host__ __device__ __forceinline__
#define TG_D __device__ __forceinline__

// ---- error plumbing ---------------------------------------------------------
void tg_set_error(const char *fmt, ...);
#define TG_CUDA(expr)                                                              \
    do {                                                                           \
        cudaError_t _e = (expr);                                                   \
        if (_e != cudaSuccess) {                                                   \
            tg_set_error("%s:%d %s -> cudaError %d (%s)", __FILE__, __LINE__, #expr, (int)_e, cudaGetErrorString(_e)); \
            return TG_ERR_CUDA;                                                    \
        }                                                                          \
    } while (0)
#define TG_REQUIRE(cond, code, ...)                                                \
    do {                                                                           \
        if (!(cond)) {                                                             \
            tg_set_error(__VA_ARGS__);                                             \
            return (code);                                                         \
        }                                                                          \
    } while (0)

// NVTX range over the host side of an entry point (nsys attributes the kernels launched inside it to the range):
// K1 = tg_rollout, K2 = tg_advantage*, K3 = tg_policy_grad / tg_value_grad.  Header-only nvtx3: a no-op unless a
// profiler injects itself.
#ifndef TG_NO_NVTX
#include <nvtx3/nvToolsExt.h>
struct TgRange {
    explicit TgRange(const char *name) { nvtxRangePushA(name); }
    ~TgRange() { nvtxRangePop(); }
};
#else
struct TgRange { explicit TgRange(const char *) {} };
#endif

// Device buffers owned by the ctx are grown with tg_ctx_grow and freed by tg_ctx_destroy.
struct tg_ctx {
    int device;
    int sm_count;
    int smem_optin;  // max dynamic shared memory per block (bytes)
    float *packed;   // staged (transposed / padded) policy weights, device
    size_t packed_cap;
    float *packed_tc;  // staged tensor-core operands (hi/lo split, core-matrix / SW128_32B layouts), device
    size_t packed_tc_cap;
    int math_mode;     // TG_MATH_*
    void *scratch;     // HBM scratch of the wide tensor-core update (tg_update_tcw.cu), device
    size_t scratch_cap;
    // length order of the rollout being updated (tg_order.cu): env indices sorted by episode length,
    // longest first, and the number of live envs per step; device, in order_buf
    void *order_buf;
    size_t order_cap;
    int32_t *perm, *cnt;
    // tg_len_order_hold: the order built for (held_len, held_N, held_T) stays valid until tg_len_order_release --
    // the episode lengths do not change between the updates of one learn() (grpo.py:106, ppo.py:147)
    const int32_t *held_len;
    int64_t held_N;
    int held_T;
};
// fills ctx->perm [N] and ctx->cnt [T] for `len` (asynchronous on `st`)
int tg_len_order(tg_ctx *ctx, int64_t N, int T, const int32_t *len, cudaStream_t st);
// makes *buf (capacity *cap, a device buffer of ctx) hold at least `bytes`; a smaller buffer is freed after a
// device synchronise (kernels in flight may still read it) and replaced, its contents are not kept
int tg_ctx_grow(tg_ctx *ctx, void **buf, size_t *cap, size_t bytes);
// constants of the diagonal Gaussian policy N(mu, diag(cov_diag)) over A actions: sd = sqrtf(cov_diag) (fp32, as
// torch's cholesky of diag(c)), inv_sd = 1 / sd, inv_var = 1 / sd^2, log_norm = A/2 log(2 pi) + sum log sd
// (summed in double).  Null outputs are skipped; TG_ERR_ARG unless every cov_diag[j] > 0.
int tg_gauss_consts(const float *cov_diag, int A, float *sd, float *inv_sd, float *inv_var, float *log_norm);

// ---- MLP tile configurations --------------------------------------------------
// A CTA advances B environments (rollout) / B samples (update) at a time with NT
// threads; the hidden GEMMs use an 8x8 register tile per thread, threads laid out
// (B/8) x (NT/(B/8)), so one pass covers NP = NT/(B/8)*8 neurons.
//   cfg 0: B=128 NT=128 NP= 64   hidden width <= 64
//   cfg 1: B=128 NT=256 NP=128   hidden width <= 128
//   cfg 2: B= 64 NT=256 NP=256   hidden width <= 256
template <int CFG> struct TileCfg;
template <> struct TileCfg<0> { static constexpr int B = 128, NT = 128, NP = 64; };
template <> struct TileCfg<1> { static constexpr int B = 128, NT = 256, NP = 128; };
template <> struct TileCfg<2> { static constexpr int B = 64, NT = 256, NP = 256; };
//   cfg 3: B= 64 NT=128 NP=128   width <= 128, update kernels of deep nets (activation tiles of cfg 1 too large)
template <> struct TileCfg<3> { static constexpr int B = 64, NT = 128, NP = 128; };

// Staged weight layout (built on the device by tg_pack_kernel from the flat
// torch-order vector).  For every hidden Linear l (input K_l, output N_l<=NP):
//   Wt[K_l][NP]  k-major copy, zero padded to NP neurons (forward operand)
//   bias[NP]
//   Wn[N_l][NPK] n-major copy (torch layout), rows padded to NPK=roundup(K_l,8)... (backward-data operand)
// and for the output Linear (K_L -> A): Wo[A][K_L] (torch layout) + bo[A] padded to 4.
struct tg_layer_layout {
    int K, N;          // true dims
    int64_t flat_w;    // offset of W (and flat_w + N*K = bias) in the flat vector
    int64_t wt, bias;  // offsets (floats) in the staged buffer
    int64_t wn;        // n-major copy [N][KP] (update kernels only), -1 if absent
    int KP;            // padded K of the n-major copy
};
struct tg_mlp_layout {
    int n_layers, act, cfg, NP, B, NT;
    int acts[TG_MAX_LAYERS];  // activation after hidden Linear l (all equal to `act` unless TG_ACT_PER_LAYER)
    int O, A, kmax;  // kmax = max input width over layers (activation buffer rows)
    tg_layer_layout L[TG_MAX_LAYERS];
    int64_t total;   // floats in the staged buffer
    int64_t n_params;
};
// smem_limit > 0 (update kernels): pick the tile configuration whose activation tiles fit
int tg_build_layout(const tg_mlp_cfg *mlp, bool with_backward, tg_mlp_layout *out, int smem_limit = 0);
size_t tg_update_smem_bytes(const tg_mlp_layout &lay, bool with_weights);
int tg_pack_weights(tg_ctx *ctx, const tg_mlp_layout &lay, const float *params, cudaStream_t st);

TG_HD int tg_round_up(int x, int m) { return (x + m - 1) / m * m; }

// ---- tensor-core (tcgen05, 3xTF32) staging ----------------------------------------
// Eligible policies: >= 2 hidden layers of equal width W = 64 or 128 (TC_W = 64 is the width the
// update kernel and the one-thread-per-env rollout kernel are built for).  The first
// Linear (K = obs dim) and the output Linear (N = act dim <= 4) stay on the FP32 pipe;
// every hidden->hidden Linear is a [128 x 64] x [64 x 64] UMMA per tile.
// Staged buffer (floats; the kernel bulk-copies it to a 1024-byte aligned smem base):
//   w1   [TC_W][O4]            row n = (W1[n][0..O), b1[n], 0...)   O4 = roundup(O+1, 4)
//   per hidden->hidden layer l (1024-byte aligned):
//        w_hi [TC_W x TC_W] core-matrix layout of tg_umma.cuh, w_lo same, bias [TC_W]
//   wo   [A][TC_W], bo [4]
#define TC_W 64
struct tg_tc_layout {
    int n_layers, nh, act, O, O4, A;
    int W;                             // hidden width: 64 or 128
    int64_t flat_w[TG_MAX_LAYERS];     // offsets of each Linear in the flat torch vector
    int64_t w1, whi[TG_MAX_LAYERS], wlo[TG_MAX_LAYERS], bias[TG_MAX_LAYERS], wo, bo;
    // update kernels only: W[out][in] again in the MN-major (SW128_32B) layout, the B operand of
    // the backward-data GEMM dH = dZ * W (reduction over `out`); -1 when absent
    int64_t wbhi[TG_MAX_LAYERS], wblo[TG_MAX_LAYERS];
    int64_t total;                     // floats
    int64_t n_params;
};
bool tg_tc_eligible(const tg_mlp_cfg *mlp);
int tg_build_tc_layout(const tg_mlp_cfg *mlp, tg_tc_layout *out, bool with_backward = false);
int tg_pack_weights_tc(tg_ctx *ctx, const tg_tc_layout &lay, const float *params, cudaStream_t st);

// Wide staging (obs -> W -> W -> act, W = 128 or 256): the 256-wide rollout (tg_rollout_tc256.cu) and the wide
// update (tg_update_tcw.cu).  The hidden [W x W] weight does not fit in shared memory next to the rest; it is
// streamed from L2 in chunks of 32 reduction columns (32 KB at W = 256).  Staged buffer (floats):
//   resident block, copied once into shared memory (multiple of 256 floats):
//     w0hi, w0lo [W x OKP]  first Linear rows (W0[n][:], b0[n], 0..), core-matrix layout, OKP = roundup(O + 1, 8)
//     b1 [W], wo [A][W], bo [4]
//   chunks_f: forward chunks hi(0), lo(0), hi(1), .. of W1 [W rows out][32 cols in], K-major core-matrix layout
//   chunks_b: backward chunks (update only) of W1 [32 rows out][W cols in], MN-major SW128_32B layout
struct TcwLayout {
    int O, OKP, A, act, W;
    int64_t w0hi, w0lo, b1, wo, bo;      // offsets (floats) in the resident block
    int64_t resident;                     // floats, multiple of 256
    int64_t chunks_f, chunks_b;           // forward (K-major) / backward (MN-major) chunk streams
    int64_t chunk_floats;                 // W * 32
    int64_t total;                        // floats; = chunks_b without the backward chunks
    int64_t flat_w[3], n_params;
};
void tg_build_tcw_layout(const tg_mlp_cfg *mlp, TcwLayout *out, bool with_backward);
int tg_pack_weights_tcw(tg_ctx *ctx, const TcwLayout &lay, const float *params, cudaStream_t st);
// statistics each update CTA leaves in its row of spart [grid][TG_SPART_LD]: objective, n_valid, sum ratio, n_clipped,
// and the sum of GRPO's k3 KL estimator (0 without a reference policy).  The row is padded to 8 doubles: with a
// stride of 5, ptxas spilled more in the tensor-core kernels without the KL term (W = 256 kernel A 44 -> 72 B).
#define TG_NSTAT 5
#define TG_SPART_LD 8
// wide (128 / 256) tensor-core update, two streamed kernels per batch of tiles (tg_update_tcw.cu)
bool tg_update_tcw_shape_built(const tg_mlp_cfg *mlp);
int tg_policy_grad_tcw(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *act,
                       const float *adv, const float *old_logp, const float *target, const int32_t *len, const float *params,
                       const float *inv_sd, const float *inv_var, float log_norm, float eps_clip, float scale,
                       float kl_scale, float *gpart, double *spart, int grid, cudaStream_t st, float *out_mu = nullptr,
                       float *out_logp = nullptr,    // out_mu / out_logp non-null: forward only (no gradients)
                       const float *ref_logp = nullptr, float ref_coef = 0.0f);   // GRPO's k3 KL term
// tensor-core update kernel (tg_update_tc.cu)
bool tg_update_tc_eligible(const tg_mlp_cfg *mlp);
int tg_update_tc_grid(const tg_ctx *ctx);
int tg_policy_grad_tc(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *act,
                      const float *adv, const float *old_logp, const float *ref_logp, const int32_t *len,
                      const float *params, const float *inv_sd, const float *inv_var, float log_norm, float eps_clip,
                      float scale, float kl_scale, float ref_coef, float *gpart, double *spart, int grid, cudaStream_t st);
