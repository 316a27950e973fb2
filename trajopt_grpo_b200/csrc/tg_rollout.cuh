// The environment half of K1, shared by the four rollout kernels (tg_rollout.cu, tg_rollout_tc256.cu): their
// trajectory/env arguments and the per-environment step (observe, sample, integrate, record, pad).  Each kernel
// keeps only its own MLP, barriers and thread roles.
#pragma once
#include "tg_env.cuh"

// the trajectory and env arguments of tg_rollout, filled once on the host
struct RolloutIo {
    EnvParams env;
    int64_t N;
    const void *init_state;        // [S][N] float or double
    const float *noise;            // [T][A][N], or null: Philox keyed by (seed, env_offset + n, t)
    uint64_t seed;
    int64_t env_offset;
    float sd[TG_MAX_ACT], log_norm;
    float *obs, *act, *rew, *logp, *ret;   // logp and ret may be null
    int32_t *len;
};

// kernel argument block: the trajectory/env arguments plus the kernel's own staged-weight layout
template <typename Layout> struct RolloutArgs {
    RolloutIo io;
    Layout lay;
    const float *packed;
};

// tg_rollout_tc256.cu
bool tg_tc256_eligible(const tg_mlp_cfg *mlp);
int tg_rollout_tc256(tg_ctx *ctx, const tg_mlp_cfg *mlp, int precision, int kind, const float *params, const RolloutIo &io,
                     cudaStream_t st);

// The state of env n held by one thread for the whole episode.  `holds`: this thread holds a real env (n < N and
// its kernel's role); only such a thread integrates it, the others keep alive = false and a zero state.  `writer`:
// this holding thread also writes env n's trajectory rows (several threads may step one env redundantly).
// Every call takes the kernel's RolloutIo instead of the struct keeping a reference to it: with the reference,
// ptxas gave some FP32-pipe rollout_kernel instances more spills.
template <int KIND, typename R> struct RolloutEnv {
    using E = Env<KIND>;
    static constexpr int S = E::S, A = E::A;
    const int64_t n;
    const bool writes;
    bool alive;
    R s[S];
    int steps = 0, bal = 0;
    float ret = 0.0f;

    TG_D RolloutEnv(const RolloutIo &io, int64_t n_, bool holds, bool writer)
        : n(n_), writes(holds && writer), alive(holds) {
        if (holds) {
            const R *init = reinterpret_cast<const R *>(io.init_state);
#pragma unroll
            for (int i = 0; i < S; ++i) s[i] = init[(int64_t)i * io.N + n];
        } else {
#pragma unroll
            for (int i = 0; i < S; ++i) s[i] = (R)0;
        }
    }

    // the policy input of step t (zero once the env is done), stored BEFORE acting (rollout_worker.py:53)
    TG_D void observe(const RolloutIo &io, int t, float (&x)[S]) const {
#pragma unroll
        for (int i = 0; i < S; ++i) {
            x[i] = alive ? (float)s[i] : 0.0f;
            if (writes) io.obs[((int64_t)t * S + i) * io.N + n] = x[i];
        }
    }

    // samples the action around the policy mean mu, evaluates its log-prob, steps the env, writes the rows of step t
    TG_D void act(const RolloutIo &io, int t, const float (&mu)[A]) {
        float a[A], lp = 0.0f, rw = 0.0f;
        if (alive) {
            float eps[4];
            if (io.noise != nullptr) {
#pragma unroll
                for (int j = 0; j < A; ++j) eps[j] = io.noise[((int64_t)t * A + j) * io.N + n];
            } else {
                philox_normal4(io.seed, (uint64_t)(io.env_offset + n), (uint32_t)t, eps);
            }
            float m2 = 0.0f;
#pragma unroll
            for (int j = 0; j < A; ++j) {
                a[j] = mu[j] + io.sd[j] * eps[j];               // MultivariateNormal.rsample
                const float z = (a[j] - mu[j]) / io.sd[j];
                m2 += z * z;
            }
            lp = -0.5f * m2 - io.log_norm;
            R r;
            const bool done = E::template step<R>(s, a, io.env, steps, bal, r);
            rw = (float)r;
            ret += rw;
            steps += 1;
            alive = !done;
        } else {
#pragma unroll
            for (int j = 0; j < A; ++j) a[j] = 0.0f;
        }
        if (writes) {
#pragma unroll
            for (int j = 0; j < A; ++j) io.act[((int64_t)t * A + j) * io.N + n] = a[j];
            io.rew[(int64_t)t * io.N + n] = rw;
            if (io.logp) io.logp[(int64_t)t * io.N + n] = lp;
        }
    }

    // zero rows from step t on, once every env of the tile is done (rollout_worker.py:64-68 padding), then len / ret
    TG_D void finish(const RolloutIo &io, int t) const {
        const int T = io.env.max_steps;
        if (writes) {
            for (; t < T; ++t) {
#pragma unroll
                for (int i = 0; i < S; ++i) io.obs[((int64_t)t * S + i) * io.N + n] = 0.0f;
#pragma unroll
                for (int j = 0; j < A; ++j) io.act[((int64_t)t * A + j) * io.N + n] = 0.0f;
                io.rew[(int64_t)t * io.N + n] = 0.0f;
                if (io.logp) io.logp[(int64_t)t * io.N + n] = 0.0f;
            }
            io.len[n] = steps;
            if (io.ret) io.ret[n] = ret;
        }
    }
};

// Calls f(R(), std::bool_constant<RELU>()) for the env state type of `precision` and whether the activation is
// ReLU: the kernels take both as template parameters.
template <typename F> auto tg_with_prec_relu(int precision, int act, F &&f) {
    const bool relu = act == TG_ACT_RELU;
    if (precision == TG_PREC_F64) return relu ? f(double(), std::true_type()) : f(double(), std::false_type());
    return relu ? f(float(), std::true_type()) : f(float(), std::false_type());
}
