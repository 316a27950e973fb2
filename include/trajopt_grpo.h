/*
 * trajopt_grpo.h -- C ABI of the B200-native rollout-and-update engine.
 *
 * Drop-in boundary for the hot loop of Dyllon-Preston/trajopt-grpo.  The
 * reference has no FFI; its boundary is a Python object protocol, so each entry
 * point below names the Python call (reference file:line) it replaces.  The
 * Python host in trajopt_grpo_b200/ binds these with ctypes (see
 * INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - every function returns an int status: 0 ok, <0 a TG_ERR_* code (a failing CUDA runtime call
 *     is TG_ERR_CUDA; its cudaError_t name and string are in the message); tg_last_error()
 *     returns the message of the last failure on the calling thread;
 *   - the CALLER allocates every buffer (device pointers unless stated), the
 *     library never frees caller memory; calls are asynchronous on `stream`
 *     (a cudaStream_t passed as void*);
 *   - trajectories are struct-of-arrays with the env index innermost:
 *     obs[T][O][N], act[T][A][N], rew/logp/adv[T][N]; env n = group*E + episode;
 *     the host exposes them as strided views of logical shape [G,E,T,.];
 *   - policy parameters are ONE flat fp32 vector in torch.nn order
 *     (W0[out][in], b0, W1, b1, ...) -- the layout of
 *     models/neural_network.py:50-65's Sequential -- so that the gradient is a
 *     flat vector of the same layout (one NCCL allreduce) and Adam is one launch.
 *   - there is NO CPU fallback: without an sm_100a device every compute call fails.
 */
#ifndef TRAJOPT_GRPO_H
#define TRAJOPT_GRPO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TG_ABI_VERSION 2

/* status codes */
#define TG_OK 0
#define TG_ERR_ARG (-1)         /* null pointer / bad enum */
#define TG_ERR_SHAPE (-2)       /* dimension out of the supported range */
#define TG_ERR_UNSUPPORTED (-3) /* configuration the kernels do not cover */
#define TG_ERR_NO_DEVICE (-4)   /* no CUDA device / not sm_100 */
#define TG_ERR_CUDA (-5)        /* a CUDA runtime call failed; tg_last_error() carries cudaGetErrorString */

/* environments (environments/*.py) */
#define TG_ENV_CARTPOLE 0   /* cartpole_env.py:6-182   obs 5  act 1 */
#define TG_ENV_PENDULUM 1   /* pendulum_env.py:7-162   obs 3  act 1 */
#define TG_ENV_QUADPOLE2D 2 /* quadrotor_env.py:867-1223 obs 10 act 2 */
#define TG_ENV_QUADPOLE 3   /* quadrotor_env.py:353-713  obs 20 act 4 */

/* hidden-layer activations (models/neural_network.py:36-55: torch.nn class name) */
#define TG_ACT_RELU 0
#define TG_ACT_TANH 1
#define TG_ACT_SIGMOID 2
#define TG_ACT_PER_LAYER (-1) /* tg_mlp_cfg.activation: read layer_activation[l] per hidden layer instead */

/* arithmetic of the env state */
#define TG_PREC_F32 0 /* throughput mode: state, dynamics and reward in fp32 */
#define TG_PREC_F64 1 /* parity mode: float64 state as the reference's numpy envs */

/* advantage modes */
#define TG_ADV_GRPO 0    /* grpo.py:66-74,108-115: per-group pooled z-score of RTG */
#define TG_ADV_PPO_MC 1  /* ppo.py:100-111,138-139: RTG - V, global z-scores */
#define TG_ADV_PPO_GAE 2 /* ppo.py:112-124,138-139 */

#define TG_MAX_LAYERS 8
#define TG_MAX_WIDTH 256
#define TG_MAX_OBS 20
#define TG_MAX_ACT 4

typedef struct tg_ctx tg_ctx; /* opaque: device id, SM count, scratch */

/* Constructor arguments of the reference env classes plus the two integer
 * thresholds that stand in for its float64 time accumulators (SURVEY.md s7):
 *   time_limit_step : first step count k at which `_time > max_time` fires
 *                     (cartpole_env.py:153,168; pendulum_env.py:137,154)
 *   balanced_limit  : consecutive balanced steps at which `_time_balanced > 5`
 *                     fires (pendulum_env.py:138,155)
 * Both are computed on the host by replaying the float64 accumulation. */
typedef struct tg_env_cfg {
    int32_t kind;            /* TG_ENV_* */
    int32_t max_steps;       /* T, env.max_steps */
    double dt;               /* env.timestep */
    int32_t time_limit_step; /* CartPole, Pendulum */
    int32_t balanced_limit;  /* Pendulum */
    /* physical constructor arguments (all zero = the reference's defaults):
     *   CartPole (cartpole_env.py:7-16): masscart, masspole, length, gravity
     *   Pendulum (pendulum_env.py:8-17): mass, length, gravity, -
     * QuadPole2D / QuadPole take none in the reference (quadrotor_env.py:353-357, 867-872). */
    double phys[4];
} tg_env_cfg;

/* models/neural_network.py:36-65 -- n_layers Linear layers, dims[0]=input_dim,
 * dims[n_layers]=output_dim; `activation` is the torch.nn class applied after every hidden Linear
 * (a string in the reference), or TG_ACT_PER_LAYER with layer_activation[l] = the activation after
 * hidden Linear l (the reference's list form, neural_network.py:41-45).  Per-layer lists run on the
 * FP32-pipe kernels; the tensor-core kernels take one activation for all layers. */
typedef struct tg_mlp_cfg {
    int32_t n_layers;
    int32_t dims[TG_MAX_LAYERS + 1];
    int32_t activation; /* TG_ACT_* or TG_ACT_PER_LAYER */
    int32_t layer_activation[TG_MAX_LAYERS]; /* read only when activation == TG_ACT_PER_LAYER */
} tg_mlp_cfg;

int tg_abi_version(void);
const char *tg_last_error(void);

int tg_ctx_create(int device, tg_ctx **out);
void tg_ctx_destroy(tg_ctx *ctx);
int tg_ctx_sm_count(const tg_ctx *ctx);

/* Arithmetic of the hidden->hidden MLP GEMMs inside tg_rollout / tg_policy_grad:
 *   TG_MATH_AUTO   tensor cores (tcgen05.mma kind::tf32 with the 3xTF32 hi/lo split, fp32
 *                  accumulation in TMEM) when the policy shape is eligible, FP32 FMA pipe otherwise
 *   TG_MATH_FP32   always the FP32 FMA pipe (register-tiled GEMMs)
 *   TG_MATH_3XTF32 require the tensor-core path (TG_ERR_UNSUPPORTED if the shape is not eligible)
 * Default: TG_MATH_AUTO. */
#define TG_MATH_AUTO 0
#define TG_MATH_FP32 1
#define TG_MATH_3XTF32 2
int tg_ctx_set_math(tg_ctx *ctx, int math_mode);

/* Measured FP32 FMA-pipe throughput of the device (TFLOP/s), the roofline of the
 * register-tiled MLP GEMMs; bench.py reports K1/K3 against it. */
int tg_fp32_peak(tg_ctx *ctx, double *out_tflops);

/* Microbenchmark behind a design rule of the tensor-core kernels (DESIGN.md): clocks taken by a tcgen05.ld and
 * a tcgen05.st issued right after n_mma tcgen05.mma (M=128, N=64, K=8) were put in flight by another thread.
 * out[0] = ld, out[1] = st (+wait::st), out[2] = issue-to-retire of the MMAs, out[3] = issue time (host array of 4). */
int tg_tmem_probe(tg_ctx *ctx, int n_mma, long long *out_host4);

/* Tensor-core self test (row-major fp32 in/out) through tcgen05.mma kind::tf32 with fp32 TMEM
 * accumulation; passes = 1 (plain TF32) or 3 (3xTF32 hi/lo split, fp32-faithful):
 *   mode 0  D[128][N] = A[128][K] * B[N][K]^T   (forward layer: both operands K-major)
 *   mode 1  D[128][N] = A[128][K] * B[K][N]     (backward-data: B MN-major)
 *   mode 2  D[ 64][N] = A[K][64]^T * B[K][N]    (weight gradient: both MN-major, reduction over K rows)
 * Exercises the UMMA descriptor / TMEM helpers of the fused kernels. */
int tg_umma_selftest(tg_ctx *ctx, const float *A, const float *B, float *D, int K, int N, int passes,
                     int mode, void *stream);

/* dims of an env kind: returns 0 or TG_ERR_ARG */
int tg_env_dims(int kind, int *obs_dim, int *act_dim);

/* number of fp32 parameters of an MLP in flat torch order */
int64_t tg_mlp_param_count(const tg_mlp_cfg *mlp);

/* ---- K1: fused policy-in-the-loop rollout ---------------------------------
 * Replaces RolloutManager.rollout (rollout/rollout_manager.py:85-125) =
 * G x RolloutWorker.run_episodes (rollout/rollout_worker.py:19-84) =
 * per step policy.forward (policies/actor_critic.py:107-138) + env.step.
 *
 *   init_state : [S][N] (S = obs_dim) float (TG_PREC_F32) or double (TG_PREC_F64)
 *   params     : flat fp32 policy (actor) parameters, torch order
 *   cov_diag   : HOST pointer, A floats, diagonal of policy.cov
 *   noise      : [T][A][N] fp32 standard normals (one [A] slice per policy
 *                call), or NULL to draw them in-kernel from Philox4x32-10 keyed
 *                by (seed, env_offset + n, step t) -- tg_noise_fill materialises the
 *                identical stream; env_offset is the global index of this
 *                shard's first env, so a sharded run draws the single-GPU stream
 *   out_obs    : [T][O][N] fp32  observation stored BEFORE acting (rollout_worker.py:53)
 *   out_act    : [T][A][N] fp32  UNCLIPPED sample (rollout_worker.py:58)
 *   out_rew    : [T][N]    fp32
 *   out_logp   : [T][N]    fp32  log pi(a|s) at rollout time (may be NULL)
 *   out_len    : [N]       int32 episode length (rollout_worker.py:67)
 *   out_ret    : [N]       fp32  sum of rewards of the episode (may be NULL)
 * Steps past the end of an episode are written as zeros (rollout_worker.py:64-68).
 */
int tg_rollout(tg_ctx *ctx, const tg_env_cfg *env, const tg_mlp_cfg *mlp, int precision,
               int64_t N, const void *init_state, const float *params, const float *cov_diag,
               const float *noise, uint64_t seed, int64_t env_offset,
               float *out_obs, float *out_act, float *out_rew, float *out_logp,
               int32_t *out_len, float *out_ret, void *stream);

/* Fill noise[T][A][N] with the Philox stream tg_rollout(noise=NULL, seed) uses. */
int tg_noise_fill(tg_ctx *ctx, uint64_t seed, int64_t env_offset, int64_t N, int T, int A, float *noise,
                  void *stream);

/* ---- batched single env step -----------------------------------------------
 * Replaces Env.step (cartpole_env.py:138-182, pendulum_env.py:125-162,
 * quadrotor_env.py:625-713, 1132-1223) for N independent envs.
 *   state [S][N] (float|double per precision), raw_action [A][N] fp32,
 *   steps_done [N] int32 (= env._steps before the call), bal_count [N] int32
 *   (Pendulum: consecutive balanced steps before the call; may be NULL)
 *   -> next_state [S][N], reward [N] (same type as state), done [N] int32
 *   (terminated OR truncated), bal_out [N] int32 (may be NULL)
 */
int tg_env_step(tg_ctx *ctx, const tg_env_cfg *env, int precision, int64_t N,
                const void *state, const float *raw_action, const int32_t *steps_done,
                const int32_t *bal_count, void *next_state, void *reward, int32_t *done,
                int32_t *bal_out, void *stream);

/* Env._dynamics(state, control) (cartpole_env.py:51-92, pendulum_env.py:48-75, quadrotor_env.py:417-528,
 * 1044-1130): the state transition alone, for N independent envs, with the control ALREADY wrapped
 * (what step() passes after _wrap_action; float32 like the reference's wrapped action).
 *   state [S][N] (float|double per precision), control [A][N] fp32 -> next_state [S][N] */
int tg_env_dynamics(tg_ctx *ctx, const tg_env_cfg *env, int precision, int64_t N, const void *state,
                    const float *control, void *next_state, void *stream);

/* Quadrotor._dynamics (quadrotor_env.py:113-169): state [12][N], control [4][N]
 * (both float|double per precision) -> next [12][N]. */
int tg_quadrotor12_dynamics(tg_ctx *ctx, int precision, int64_t N, double dt,
                            const void *state, const void *control, void *next, void *stream);

/* ---- policy forward / log-prob over a batch --------------------------------
 * Replaces GaussianActor_NeuralNetwork.log_prob (policies/actor_critic.py:140-160)
 * and NeuralNetwork.forward (models/neural_network.py:67-77) for M rows.
 *   x [K0][M] fp32 (feature-major), act [A][M] or NULL
 *   -> out_mu [A][M] (or NULL), out_logp [M] (or NULL; needs act and cov_diag)
 */
int tg_policy_forward(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t M, const float *x,
                      const float *params, const float *cov_diag, const float *act,
                      float *out_mu, float *out_logp, void *stream);

/* Same, reading a trajectory in place: obs [T][O][N], act [T][A][N] or NULL,
 * len [N] or NULL (rows with t >= len[n] are skipped and left unwritten)
 *   -> out_mu [T][A][N] (or NULL), out_logp [T][N] (or NULL).
 * Used for the frozen old-policy log-prob (grpo.py:118-119, ppo.py:142-143) and
 * the critic values over a rollout (ppo.py:93-94). */
int tg_policy_forward_traj(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs,
                           const float *act, const int32_t *len, const float *params,
                           const float *cov_diag, float *out_mu, float *out_logp, void *stream);

/* ---- K2: reward-to-go + advantages -----------------------------------------
 * Replaces the RTG loop and per-group normalisation of GRPO.learn
 * (algorithms/grpo.py:66-74, 108-115) and PPO.learn's MC/GAE + global z-scores
 * (algorithms/ppo.py:100-139).
 *   rew [T][N], len [N] int32, values [T][N] or NULL (PPO), N = G*E
 *   -> out_adv [T][N] (zeros in padding), out_rtg [T][N] or NULL
 *      (GRPO: raw RTG; PPO: z-scored returns = critic targets)
 *   workspace: tg_advantage_workspace_bytes(N) bytes of device scratch
 */
int64_t tg_advantage_workspace_bytes(int64_t N, int G);
int tg_advantage(tg_ctx *ctx, int mode, int64_t G, int E, int T, double gamma, double lam,
                 const float *rew, const int32_t *len, const float *values,
                 float *out_adv, float *out_rtg, void *workspace, void *stream);

/* The two halves of tg_advantage's PPO modes, for a rollout sharded over several GPUs (whole
 * groups per GPU): PPO.learn z-scores advantages and returns over EVERY valid step of the rollout
 * (algorithms/ppo.py:138-139), so a rank computes its raw values and the five additive sums
 *   out_sums[5] (device, float64) = (sum adv, sum adv^2, sum ret, sum ret^2, n valid),
 * the host allreduces them (SUM) and every rank normalises with the global sums.
 * tg_advantage(mode = PPO_*) is exactly raw followed by normalize with the local sums. */
int tg_advantage_ppo_raw(tg_ctx *ctx, int mode, int64_t G, int E, int T, double gamma, double lam,
                         const float *rew, const int32_t *len, const float *values,
                         float *out_adv, float *out_rtg, double *out_sums, void *workspace, void *stream);
int tg_advantage_ppo_normalize(tg_ctx *ctx, int64_t N, int T, const int32_t *len, const double *sums,
                               float *adv, float *rtg, void *stream);

/* ---- trajectory export ---------------------------------------------------------
 * Replaces the host loop of Rollout_Buffer.save_trajectory (buffers/rollout_buffer.py:72-102):
 * compacts the valid steps of a rollout into a dense table on the device.
 *   obs [T][O][N], act [T][A][N], len [N]; row0 [N] int64 = exclusive prefix sum of len
 *   -> out_episode_id [n_valid] int32 (= env index n = worker*E + episode, rollout_buffer.py:88),
 *      out_rows [n_valid][O + A] fp32 (observation_0.., action_0..), row row0[n] + t = step t of episode n */
int tg_export_trajectory(tg_ctx *ctx, int64_t N, int T, int O, int A, const float *obs, const float *act,
                         const int32_t *len, const int64_t *row0, int32_t *out_episode_id, float *out_rows,
                         void *stream);

/* ---- K3: clipped-surrogate objective + flat gradient ------------------------
 * Replaces one iteration of the update loop of GRPO.learn
 * (algorithms/grpo.py:106-145: J = (1/G) sum_g sum_valid min(rho A, clamp(rho) A),
 * J.backward()) -- and, with a critic, of PPO.learn (algorithms/ppo.py:147-183).
 *   obs [T][O][N], act [T][A][N], adv [T][N], old_logp [T][N], len [N]
 *   params: flat actor parameters
 *   scale : multiplies the objective (GRPO: 1/G_global; PPO: -1/n_valid)
 *   kl_coef: weight of mean(exp(old)*(old-lp)) (ppo.py:175-176), 0 for GRPO
 *   -> out_grad [n_params] fp32 (d objective / d params), out_stats [4] fp32:
 *      {objective, n_valid, sum ratio, n_clipped}
 *   workspace: tg_policy_grad_workspace_bytes(ctx, mlp) bytes
 */
int64_t tg_policy_grad_workspace_bytes(const tg_ctx *ctx, const tg_mlp_cfg *mlp);
int tg_policy_grad(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T,
                   const float *obs, const float *act, const float *adv, const float *old_logp,
                   const int32_t *len, const float *params, const float *cov_diag,
                   float eps_clip, float scale, float kl_coef,
                   float *out_grad, float *out_stats, void *workspace, void *stream);
/* tg_policy_grad with GRPO's KL penalty to a frozen reference policy (Shao et al. 2024, eq. 4; the k3 estimator):
 * per valid sample, u = ref_logp - lp and D = exp(u) - u - 1 >= 0; the objective gains -ref_coef * sum D, so
 * d objective / d lp gains ref_coef * expm1(u).  ref_coef = beta * scale.
 *   ref_logp [T][N]: log-prob of act under the reference policy (its own covariance)
 *   -> out_stats [5] fp32: {objective (with the KL term), n_valid, sum ratio, n_clipped, sum D}
 * ref_logp == NULL is tg_policy_grad: no KL term, out_stats [4].  Same workspace as tg_policy_grad. */
int tg_policy_grad_ref(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T,
                       const float *obs, const float *act, const float *adv, const float *old_logp,
                       const float *ref_logp, const int32_t *len, const float *params, const float *cov_diag,
                       float eps_clip, float scale, float kl_coef, float ref_coef,
                       float *out_grad, float *out_stats, void *workspace, void *stream);

/* The update kernels walk a ragged rollout in LENGTH ORDER (env indices sorted by episode length, live envs per
 * step), built from `len` at the start of every tg_policy_grad / tg_value_grad / tg_policy_forward_traj call.
 * The lengths do not change between the updates of one learn() (grpo.py:106, ppo.py:147): tg_len_order_hold
 * builds the order once and later calls with the same (len pointer, N, T) reuse it until tg_len_order_release.
 * The caller must not modify `len` while it is held. */
int tg_len_order_hold(tg_ctx *ctx, int64_t N, int T, const int32_t *len, void *stream);
int tg_len_order_release(tg_ctx *ctx);

/* HBM scratch traffic of one tg_policy_grad call beyond the algorithmic trajectory reads (host-side arithmetic,
 * no device work): the streamed 128 / 256-wide tensor-core path hands H1, dZ2, dZ1 and [x, 1] from its
 * forward/backward kernel to its weight-gradient kernel through an HBM scratch.  n_tiles = number of live
 * 128-sample tiles (sum over steps of ceil(live envs / 128)).  Both outputs are 0 for the fused paths. */
int tg_policy_grad_scratch_bytes(const tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t n_tiles,
                                 int64_t *bytes_written, int64_t *bytes_read);

/* Critic regression gradient (ppo.py:168-169: MSELoss(V(obs), rtg_norm)):
 *   target [T][N]; scale = c1 / n_valid  -> out_grad [n_params(critic)], out_stats[0] = sum sq err */
int tg_value_grad(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T,
                  const float *obs, const float *target, const int32_t *len, const float *params,
                  float scale, float *out_grad, float *out_stats, void *workspace, void *stream);

/* Minibatch forms of tg_policy_grad / tg_value_grad (PPO with batch_size != None, algorithms/ppo.py:147-183:
 * `permutation[start:start+batch_size]` over the valid steps).  sample_ids [n_samples] int64 (device) lists the
 * samples of the minibatch as flat slot ids t*N + n into the [T][.][N] buffers; `scale` is the caller's
 * 1/len(batch) (the reference's .mean() over the batch).  Same outputs and workspace as the full forms. */
int tg_policy_grad_batch(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *act,
                         const float *adv, const float *old_logp, const int64_t *sample_ids, int64_t n_samples,
                         const float *params, const float *cov_diag, float eps_clip, float scale, float kl_coef,
                         float *out_grad, float *out_stats, void *workspace, void *stream);
int tg_value_grad_batch(tg_ctx *ctx, const tg_mlp_cfg *mlp, int64_t N, int T, const float *obs, const float *target,
                        const int64_t *sample_ids, int64_t n_samples, const float *params, float scale,
                        float *out_grad, float *out_stats, void *workspace, void *stream);

/* Minibatch plan of one PPO epoch (algorithms/ppo.py:147-157) over a rollout sharded by whole groups.
 *   perm [n_total] int64 (device): the epoch's torch.randperm over the valid steps of the WHOLE rollout,
 *        in the reference's flattening order (global env index major, step minor)
 *   len [N] int32, row0 [N] int64 = exclusive prefix sum of len (as tg_export_trajectory): the shard's local
 *        valid step row0[n] + t is step t of env n
 *   base: global index of this shard's first valid step; n_local = sum(len)
 *   -> out_ids [max_ids] int64: flat slot ids t*N + n of the perm entries in [base, base + n_local), in perm order
 *      out_offsets [n_batches + 1] int64, n_batches = ceil(n_total / batch_size):
 *      out_offsets[b] = number of this shard's entries in perm[0 : b*batch_size]
 *      (minibatch b = out_ids[out_offsets[b] : out_offsets[b+1]]).  No write at or past out_ids[max_ids];
 *      out_offsets still counts every entry, so the caller detects a perm that is not a permutation.
 *   workspace: tg_minibatch_plan_workspace_bytes(n_total) bytes of device scratch (8 per perm entry + 8 per 4096)
 * Deterministic: positions come from per-chunk counts and their prefix sum, never from atomics. */
int64_t tg_minibatch_plan_workspace_bytes(int64_t n_total);
int tg_minibatch_plan(tg_ctx *ctx, int64_t N, const int32_t *len, const int64_t *row0, const int64_t *perm,
                      int64_t n_total, int64_t batch_size, int64_t base, int64_t n_local, int64_t max_ids,
                      int64_t *out_ids, int64_t *out_offsets, void *workspace, void *stream);

/* ---- Adam --------------------------------------------------------------------
 * torch.optim.Adam defaults as the reference constructs it
 * (pipelines/cartpole_pipeline_grpo.py:65): p -= lr/(1-b1^t) * m/(sqrt(v)/sqrt(1-b2^t)+eps).
 * `step` is the 1-based step count AFTER this update. */
int tg_adam_step(tg_ctx *ctx, int64_t n, float *params, const float *grad, float *exp_avg,
                 float *exp_avg_sq, int64_t step, double lr, double beta1, double beta2, double eps,
                 void *stream);

/* ---- gradient allreduce fused with Adam over NVLink peer memory -----------------
 * Replaces, for a rollout sharded over several GPUs (one process per GPU, whole GRPO groups per GPU), the
 * `torch.distributed.all_reduce(grad)` + `optimizer.step()` pair of every update (grpo.py:143-145, ppo.py:181-183
 * on the summed gradient): each rank owns a cudaMalloc'ed window that its peers map through CUDA IPC; one kernel
 * waits until every rank has published its gradient, sums the ranks' gradients with peer loads in rank order
 * (bit-identical on every rank) and applies Adam in the same pass.  No NCCL call, no separate Adam launch.
 *
 *   tg_comm_create   allocates this rank's window for gradients of up to n_floats and writes its IPC handle
 *                    (tg_comm_handle_bytes() bytes, host) to handle_out; the host exchanges the handles
 *                    (e.g. torch.distributed.all_gather_object) ...
 *   tg_comm_connect  ... and passes all `world` handles, rank-major; maps every peer window
 *   tg_comm_grad_slot  device pointer where the NEXT step's local gradient has to be written: pass it as
 *                    tg_policy_grad's out_grad (no copy)
 *   tg_allreduce_adam_step  params -= Adam(sum over ranks of the gradient slots); `step` as tg_adam_step;
 *                    out_grad_sum (may be NULL) receives the summed gradient
 * All ranks must call tg_allreduce_adam_step the same number of times (it is a collective). */
typedef struct tg_comm tg_comm;
int tg_comm_handle_bytes(void);
int tg_comm_create(tg_ctx *ctx, int rank, int world, int64_t n_floats, tg_comm **out, void *handle_out);
int tg_comm_connect(tg_comm *comm, const void *all_handles);
int tg_comm_destroy(tg_comm *comm);
int tg_comm_grad_slot(tg_comm *comm, float **out);
int tg_allreduce_adam_step(tg_ctx *ctx, tg_comm *comm, int64_t n, float *params, float *exp_avg, float *exp_avg_sq,
                           int64_t step, double lr, double beta1, double beta2, double eps, float *out_grad_sum,
                           void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TRAJOPT_GRPO_H */
