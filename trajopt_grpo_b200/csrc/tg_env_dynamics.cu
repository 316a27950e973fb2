// tg_env_dynamics: Env._dynamics(state, control) for N independent envs -- the state transition of
// Env<KIND>::step with the control taken as already wrapped (cartpole_env.py:51-92,
// pendulum_env.py:48-75, quadrotor_env.py:417-528, 1044-1130).  Reward and termination are discarded.
#include "tg_env.cuh"

template <int KIND, typename R>
__global__ void env_dynamics_kernel(EnvParams p, int64_t N, const R *__restrict__ state, const float *__restrict__ control,
                                    R *__restrict__ next) {
    using E = Env<KIND>;
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    R s[E::S];
    float u[E::A];
#pragma unroll
    for (int i = 0; i < E::S; ++i) s[i] = state[(int64_t)i * N + n];
#pragma unroll
    for (int j = 0; j < E::A; ++j) u[j] = control[(int64_t)j * N + n];
    int bal = 0;
    R r;
    E::template step<R, true>(s, u, p, 0, bal, r);
#pragma unroll
    for (int i = 0; i < E::S; ++i) next[(int64_t)i * N + n] = s[i];
}

template <int KIND>
static int launch(int precision, const EnvParams &p, int64_t N, const void *state, const float *control, void *next,
                  cudaStream_t st) {
    const unsigned grid = (unsigned)((N + 127) / 128);
    if (precision == TG_PREC_F64)
        env_dynamics_kernel<KIND, double><<<grid, 128, 0, st>>>(p, N, (const double *)state, control, (double *)next);
    else
        env_dynamics_kernel<KIND, float><<<grid, 128, 0, st>>>(p, N, (const float *)state, control, (float *)next);
    TG_CUDA(cudaGetLastError());
    return TG_OK;
}

extern "C" int tg_env_dynamics(tg_ctx *ctx, const tg_env_cfg *env, int precision, int64_t N, const void *state,
                               const float *control, void *next_state, void *stream) {
    TG_REQUIRE(ctx && env && state && control && next_state, TG_ERR_ARG, "tg_env_dynamics: null argument");
    TG_REQUIRE(N > 0, TG_ERR_SHAPE, "tg_env_dynamics: N must be positive");
    TG_REQUIRE(precision == TG_PREC_F32 || precision == TG_PREC_F64, TG_ERR_ARG, "bad precision %d", precision);
    EnvParams p;
    int rc = tg_fill_env_params(env, &p);
    if (rc) return rc;
    TG_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    return tg_with_env_kind(env->kind, [&](auto kind) {
        return launch<decltype(kind)::value>(precision, p, N, state, control, next_state, st);
    });
}
