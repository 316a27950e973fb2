"""Parity of the sm_100a kernels (called through the C ABI) against the oracle
and against the fixtures generated from the unmodified reference."""
import os

import numpy as np
import pytest
import torch

import philox
import restate as R

pytestmark = pytest.mark.gpu

MAXS = {0: 120, 1: 200, 2: 150, 3: 150}


def load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name), allow_pickle=False))


def dev(x, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return t if dtype is None else t.to(dtype)


@pytest.fixture(scope="module")
def E():
    from trajopt_grpo_b200 import engine
    return engine


def _weights(g, prefix=""):
    Ws, bs, i = [], [], 0
    while f"{prefix}W{i}" in g:
        Ws.append(g[f"{prefix}W{i}"]); bs.append(g[f"{prefix}b{i}"]); i += 1
    return Ws, bs


def _flat(Ws, bs):
    return np.concatenate([np.concatenate([w.reshape(-1), b.reshape(-1)]) for w, b in zip(Ws, bs)]).astype(np.float32)


def _dims(Ws):
    return [Ws[0].shape[1]] + [w.shape[0] for w in Ws]


# ----------------------------------------------------------------------------
# env transitions (teacher-forced single steps on the reference's own states)
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_env_step_float64_matches_reference(E, golden_dir, kind):
    g = load(golden_dir, f"transitions_env{kind}.npz")
    nxt, rew, done, _ = E.env_step(kind, MAXS[kind], R.DEFAULT_DT[kind], dev(g["state"].T.copy()),
                                   dev(g["action"].T.copy()), dev(g["steps_done"].astype(np.int32)),
                                   dev(g["bal_count"].astype(np.int32)))
    # float64 kernel vs float64 reference: only FMA contraction / libm differ (1e-12 relative)
    np.testing.assert_allclose(nxt.cpu().numpy().T, g["next"], rtol=1e-11, atol=1e-12)
    np.testing.assert_allclose(rew.cpu().numpy(), g["reward"], rtol=1e-10, atol=1e-11)
    assert np.array_equal(done.cpu().numpy().astype(bool), g["done"])       # flags bit-exact


@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_env_step_float32_tolerance(E, golden_dir, kind):
    g = load(golden_dir, f"transitions_env{kind}.npz")
    nxt, rew, done, _ = E.env_step(kind, MAXS[kind], R.DEFAULT_DT[kind], dev(g["state"].T.copy(), torch.float32),
                                   dev(g["action"].T.copy()), dev(g["steps_done"].astype(np.int32)),
                                   dev(g["bal_count"].astype(np.int32)))
    # stated tolerance of the throughput mode: rel 1e-5 per step (+ abs 1e-5 where terms cancel)
    np.testing.assert_allclose(nxt.cpu().numpy().T, g["next"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(rew.cpu().numpy(), g["reward"], rtol=1e-4, atol=2e-4)
    # flags may only flip where a threshold sits inside fp32 rounding of the state: count them
    flips = int((done.cpu().numpy().astype(bool) != g["done"]).sum())
    assert flips <= 1


def test_quadrotor12_dynamics(E, golden_dir):
    g = load(golden_dir, "quadrotor12_dynamics.npz")
    out = E.quadrotor12_dynamics(dev(g["state"].T.copy()), dev(g["control"].T.copy()))
    np.testing.assert_allclose(out.cpu().numpy().T, g["next"], rtol=1e-11, atol=1e-12)
    out32 = E.quadrotor12_dynamics(dev(g["state"].T.copy(), torch.float32), dev(g["control"].T.copy(), torch.float32))
    np.testing.assert_allclose(out32.cpu().numpy().T, g["next"], rtol=1e-4, atol=1e-5)


# ----------------------------------------------------------------------------
# noise
# ----------------------------------------------------------------------------
def test_philox_stream_matches_host_restatement(E):
    N, T, A = 1000, 7, 4
    z = E.noise_fill(0x1234_5678_9ABC_DEF0, N, T, A).cpu().numpy()
    ref = philox.normals(0x1234_5678_9ABC_DEF0, N, T, A)
    np.testing.assert_allclose(z, ref, rtol=0, atol=2e-6)
    big = E.noise_fill(7, 1 << 18, 8, 2).cpu().numpy()
    assert abs(big.mean()) < 5e-3 and abs(big.std() - 1) < 5e-3


# ----------------------------------------------------------------------------
# rollouts vs the reference's RolloutManager (injected states and noise)
# ----------------------------------------------------------------------------
ROLLOUTS = ["cartpole", "pendulum", "quadpole2d", "quadpole"]


def _run_rollout(E, g, dtype, noise=True, seed=0):
    kind, T = int(g["kind"]), int(g["T"])
    Ws, bs = _weights(g)
    cov = [float(g["cov"])] * R.ACT_DIM[kind]
    nz = dev(np.ascontiguousarray(g["noise"].transpose(0, 2, 1))) if noise else None
    out = E.rollout(kind, T, R.DEFAULT_DT[kind], _dims(Ws), "ReLU", dev(_flat(Ws, bs)), cov,
                    dev(g["init"].T.copy(), dtype), noise=nz, seed=seed)
    torch.cuda.synchronize()
    return out


def _to_ref_shape(x, G, Eps):
    # [T,D,N] -> [G,E,T,D] ; [T,N] -> [G,E,T]
    x = x.cpu().numpy()
    if x.ndim == 3:
        return x.transpose(2, 0, 1).reshape(G, Eps, x.shape[0], x.shape[1])
    return x.T.reshape(G, Eps, x.shape[0])


@pytest.mark.parametrize("name", ROLLOUTS)
def test_rollout_float64_matches_reference(E, golden_dir, name):
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    G, Eps = int(g["G"]), int(g["E"])
    out = _run_rollout(E, g, torch.float64)
    ln = out["len"].cpu().numpy().reshape(G, Eps)
    assert np.array_equal(ln, g["len"].astype(np.int32))                     # lengths bit-exact
    mask = (np.arange(int(g["T"]))[None, None, :] < ln[:, :, None]).astype(np.float32)
    assert np.array_equal(mask, g["mask"])
    # free-running: float64 env, fp32 policy -- the only difference to the reference is
    # the fp32 summation order inside the MLP, amplified over the horizon
    np.testing.assert_allclose(_to_ref_shape(out["obs"], G, Eps), g["obs"], rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(_to_ref_shape(out["act"], G, Eps), g["act"], rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(_to_ref_shape(out["rew"], G, Eps), g["rew"], rtol=2e-4, atol=5e-4)
    sel = g["mask"] > 0
    np.testing.assert_allclose(_to_ref_shape(out["logp"], G, Eps)[sel], g["logp_valid"], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(out["ret"].cpu().numpy().reshape(G, Eps), g["rew"].sum(2), rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("name", ROLLOUTS)
def test_rollout_float32_drift_bound(E, golden_dir, name):
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    G, Eps, T = int(g["G"]), int(g["E"]), int(g["T"])
    out = _run_rollout(E, g, torch.float32)
    obs = _to_ref_shape(out["obs"], G, Eps)
    ln = out["len"].cpu().numpy().reshape(G, Eps)
    # padding is exactly zero and lengths are sane
    pad = np.arange(T)[None, None, :] >= ln[:, :, None]
    assert np.all(obs[pad] == 0) and np.all(_to_ref_shape(out["rew"], G, Eps)[pad] == 0)
    assert ln.min() >= 1 and ln.max() <= T
    # first step is teacher-forced by construction: 1e-5
    np.testing.assert_allclose(obs[:, :, 0], g["obs"][:, :, 0], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(_to_ref_shape(out["rew"], G, Eps)[:, :, 0], g["rew"][:, :, 0], rtol=1e-4, atol=2e-4)
    # drift bound over the (short) horizon where both are still running
    both = (~pad) & (g["mask"] > 0)
    err = np.abs(obs - g["obs"])[both].max()
    assert err < 5e-2, f"fp32 free-running drift {err}"
    assert np.abs(ln - g["len"]).max() <= 3        # an OOB crossing can move by a few steps under drift


def test_rollout_philox_equals_explicit_noise(E, golden_dir):
    g = load(golden_dir, "rollout_grpo_quadpole.npz")
    kind, T = 3, int(g["T"])
    N = g["init"].shape[0]
    z = E.noise_fill(99, N, T, 4)
    g2 = dict(g)
    g2["noise"] = z.cpu().numpy().transpose(0, 2, 1)
    a = _run_rollout(E, g2, torch.float32)
    b = _run_rollout(E, g, torch.float32, noise=False, seed=99)
    for k in ("obs", "act", "rew", "logp", "len", "ret"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.parametrize("hidden", [[32, 32], [64, 64], [128, 128], [256, 256]],
                         ids=["fp32", "tc64", "tc128", "tc256"])
def test_rollout_kernels_philox_and_without_logp(E, hidden):
    """Each of the four rollout kernels (FP32 pipe, tensor cores at width 64, 128 and 256) draws in-kernel Philox
    noise exactly as tg_noise_fill materialises it, and leaves its other outputs bit-identical when it writes no
    log-probs (PPO.learn_streamed rolls out without them)."""
    kind, T, N, A = 3, 60, 300, 4
    rng = np.random.default_rng(17)
    dims = [R.OBS_DIM[kind]] + hidden + [A]
    Ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32) for i in range(len(dims) - 1)]
    bs = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(dims) - 1)]
    params, init = dev(_flat(Ws, bs)), dev(R.reset_states(kind, N, rng).T.copy(), torch.float32)

    def run(**kw):
        out = E.rollout(kind, T, R.DEFAULT_DT[kind], dims, "ReLU", params, [0.3] * A, init, env_offset=5, **kw)
        torch.cuda.synchronize()
        return out

    a = run(noise=E.noise_fill(99, N, T, A, env_offset=5))
    b = run(seed=99)
    c = run(seed=99, want_logp=False)
    for k in ("obs", "act", "rew", "logp", "len", "ret"):
        assert torch.equal(a[k], b[k]), k
    assert c["logp"] is None
    for k in ("obs", "act", "rew", "len", "ret"):
        assert torch.equal(b[k], c[k]), k


@pytest.mark.parametrize("hidden,kind", [([64, 64], 1), ([128, 128], 2), ([256, 256], 3), ([128, 128, 128, 128], 0),
                                         ([40, 24], 2), ([], 1)])
def test_rollout_matches_oracle_all_tile_configs(E, hidden, kind):
    """Every tile configuration (width<=64/128/256, smem-resident and global
    weights, odd widths, no hidden layer) against the fp32-mode oracle."""
    rng = np.random.default_rng(5)
    O, A = R.OBS_DIM[kind], R.ACT_DIM[kind]
    dims = [O] + hidden + [A]
    Ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32) for i in range(len(dims) - 1)]
    bs = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(dims) - 1)]
    N, T = 200, 12
    init = R.reset_states(kind, N, rng)
    noise = rng.standard_normal((T, N, A)).astype(np.float32)
    cfg = R.EnvCfg.make(kind, T)
    cov = np.full(A, 0.3, np.float32)
    o, a, r, lp, ln, m = R.rollout(cfg, init, Ws, bs, cov, noise, dtype=np.float64)
    out = E.rollout(kind, T, cfg.dt, dims, "ReLU", dev(_flat(Ws, bs)), cov.tolist(), dev(init.T.copy()),
                    noise=dev(np.ascontiguousarray(noise.transpose(0, 2, 1))))
    assert np.array_equal(out["len"].cpu().numpy(), ln)
    np.testing.assert_allclose(out["obs"].cpu().numpy().transpose(2, 0, 1), o, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(out["act"].cpu().numpy().transpose(2, 0, 1), a, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(out["rew"].cpu().numpy().T, r, rtol=1e-4, atol=1e-3)
    np.testing.assert_allclose(out["logp"].cpu().numpy().T, lp, rtol=1e-4, atol=1e-4)


# ----------------------------------------------------------------------------
# policy forward / log-prob
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("hidden,act", [([64, 64], "ReLU"), ([128, 96], "Tanh"), ([256, 256], "Sigmoid"), ([32], "ReLU")])
def test_policy_forward_and_logp(E, hidden, act):
    rng = np.random.default_rng(3)
    dims = [10] + hidden + [2]
    Ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32) for i in range(len(dims) - 1)]
    bs = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(dims) - 1)]
    M = 777
    x = rng.standard_normal((M, 10)).astype(np.float32)
    a = rng.standard_normal((M, 2)).astype(np.float32)
    cov = np.array([0.5, 0.2], np.float32)
    mu_ref = R.mlp_forward(x, Ws, bs, R.ACT_IDS[act], np.float64)
    lp_ref = R.gaussian_log_prob(mu_ref, cov, a, np.float64)
    mu, lp = E.policy_forward(dims, act, dev(_flat(Ws, bs)), dev(x.T.copy()), cov.tolist(), dev(a.T.copy()),
                              want_mu=True, want_logp=True)
    np.testing.assert_allclose(mu.cpu().numpy().T, mu_ref, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(lp.cpu().numpy(), lp_ref, rtol=1e-5, atol=2e-5)


# ----------------------------------------------------------------------------
# advantages
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("name", ROLLOUTS)
def test_grpo_advantage_matches_oracle(E, golden_dir, name):
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    G, Eps, T = int(g["G"]), int(g["E"]), int(g["T"])
    rtg_ref, adv_ref = R.grpo_advantage(g["rew"], g["mask"], float(g["gamma"]))
    rew = dev(np.ascontiguousarray(g["rew"].reshape(G * Eps, T).T))
    ln = dev(g["len"].reshape(-1).astype(np.int32))
    adv, rtg = E.advantage(0, G, Eps, T, float(g["gamma"]), 0.0, rew, ln, want_rtg=True)
    assert np.array_equal(rtg.cpu().numpy().T.reshape(G, Eps, T), rtg_ref)   # same fp32 recurrence: bit-exact
    np.testing.assert_allclose(adv.cpu().numpy().T.reshape(G, Eps, T), adv_ref, rtol=1e-5, atol=1e-6)


def test_grpo_advantage_ragged_and_degenerate(E):
    rng = np.random.default_rng(11)
    G, Eps, T = 37, 10, 23                       # E=10 does not divide a warp (cfg 1's group size)
    ln = rng.integers(1, T + 1, (G, Eps)).astype(np.int32)
    ln[3, :] = 1
    mask = (np.arange(T)[None, None, :] < ln[:, :, None]).astype(np.float32)
    rew = (rng.standard_normal((G, Eps, T)).astype(np.float32)) * mask
    rew[5] = 0.0                                 # zero-variance group -> division by zero std (SURVEY q2)
    rtg_ref, adv_ref = R.grpo_advantage(rew, mask, 0.9)
    adv, rtg = E.advantage(0, G, Eps, T, 0.9, 0.0, dev(np.ascontiguousarray(rew.reshape(G * Eps, T).T)),
                           dev(ln.reshape(-1)), want_rtg=True)
    got = adv.cpu().numpy().T.reshape(G, Eps, T)
    assert np.array_equal(rtg.cpu().numpy().T.reshape(G, Eps, T), rtg_ref)
    ok = np.isfinite(adv_ref)
    np.testing.assert_allclose(got[ok], adv_ref[ok], rtol=2e-5, atol=2e-6)
    assert np.array_equal(np.isnan(got), np.isnan(adv_ref))
    assert np.all(got[mask == 0] == 0)


# ----------------------------------------------------------------------------
# GRPO objective gradient and Adam vs the reference's GRPO.learn
# ----------------------------------------------------------------------------
def _soa(g):
    G, Eps, T = int(g["G"]), int(g["E"]), int(g["T"])
    N = G * Eps
    obs = dev(np.ascontiguousarray(g["obs"].reshape(N, T, -1).transpose(1, 2, 0)))
    act = dev(np.ascontiguousarray(g["act"].reshape(N, T, -1).transpose(1, 2, 0)))
    rew = dev(np.ascontiguousarray(g["rew"].reshape(N, T).T))
    ln = dev(g["len"].reshape(-1).astype(np.int32))
    return G, Eps, T, N, obs, act, rew, ln


@pytest.mark.parametrize("name", ROLLOUTS)
def test_grpo_gradient_matches_reference(E, golden_dir, name):
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    G, Eps, T, N, obs, act, rew, ln = _soa(g)
    Ws, bs = _weights(g)
    dims = _dims(Ws)
    cov = [float(g["cov"])] * dims[-1]
    params = dev(_flat(Ws, bs))
    adv, _ = E.advantage(0, G, Eps, T, float(g["gamma"]), 0.0, rew, ln)
    _, old_lp = E.policy_forward(dims, "ReLU", params, obs.permute(1, 0, 2).reshape(dims[0], T * N).contiguous(),
                                 cov, act.permute(1, 0, 2).reshape(dims[-1], T * N).contiguous(), want_mu=False, want_logp=True)
    old_lp = old_lp.reshape(T, N).contiguous()
    grad, stats = E.policy_grad(dims, "ReLU", params, cov, obs, act, adv, old_lp, ln, float(g["eps_clip"]), 1.0 / G)
    grad = grad.cpu().numpy()
    off = 0
    for i in range(len(Ws)):
        for ref in (g[f"grpo_grad{2 * i}"], g[f"grpo_grad{2 * i + 1}"]):
            got = grad[off:off + ref.size].reshape(ref.shape)
            off += ref.size
            scale = max(np.abs(ref).max(), 1e-6)
            assert np.abs(got - ref).max() <= 3e-4 * scale + 1e-5, (i, np.abs(got - ref).max(), scale)
    assert int(stats[1].item()) == int(g["mask"].sum())


@pytest.mark.parametrize("name", ROLLOUTS)
def test_grpo_adam_updates_match_reference(E, golden_dir, name):
    """updates_per_iter=3 twice (old policy synced in between), Adam lr 3e-4: final
    weights against the unmodified GRPO.learn; exercises ratio != 1 and the clip."""
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    G, Eps, T, N, obs, act, rew, ln = _soa(g)
    Ws, bs = _weights(g)
    dims = _dims(Ws)
    cov = [float(g["cov"])] * dims[-1]
    params = dev(_flat(Ws, bs))
    m, v = torch.zeros_like(params), torch.zeros_like(params)
    adv, _ = E.advantage(0, G, Eps, T, float(g["gamma"]), 0.0, rew, ln)
    x = obs.permute(1, 0, 2).reshape(dims[0], T * N).contiguous()
    a = act.permute(1, 0, 2).reshape(dims[-1], T * N).contiguous()
    step = 0
    for key in ("grpo_adam3_p", "grpo_adam6_p"):
        _, old_lp = E.policy_forward(dims, "ReLU", params, x, cov, a, want_mu=False, want_logp=True)
        old_lp = old_lp.reshape(T, N).contiguous()
        for _ in range(3):
            step += 1
            grad, _ = E.policy_grad(dims, "ReLU", params, cov, obs, act, adv, old_lp, ln, float(g["eps_clip"]), 1.0 / G)
            E.adam_step(params, grad, m, v, step, 3e-4)
        got = params.cpu().numpy()
        off = 0
        for i in range(2 * len(Ws)):
            ref = g[f"{key}{i}"]
            np.testing.assert_allclose(got[off:off + ref.size].reshape(ref.shape), ref, rtol=2e-4, atol=3e-6)
            off += ref.size


def test_adam_step_bitwise_formula(E):
    rng = np.random.default_rng(2)
    n = 5000
    p = rng.standard_normal(n).astype(np.float32)
    gr = rng.standard_normal(n).astype(np.float32)
    tp = torch.nn.Parameter(torch.from_numpy(p.copy()))
    opt = torch.optim.Adam([tp], lr=3e-4)
    P, M, V = dev(p), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    for step in range(1, 4):
        tp.grad = torch.from_numpy(gr * step)
        opt.step()
        E.adam_step(P, dev(gr * step), M, V, step, 3e-4)
    np.testing.assert_allclose(P.cpu().numpy(), tp.detach().numpy(), rtol=1e-6, atol=1e-7)


# ----------------------------------------------------------------------------
# size-independent properties at larger shapes
# ----------------------------------------------------------------------------
def test_large_rollout_properties(E):
    """65,536 Pendulum envs x 200 steps (BASELINE config 2 shape): determinism,
    zero padding, group-sharding invariance of rollout and advantages."""
    rng = np.random.default_rng(1)
    kind, T, G, Eps = 1, 200, 4096, 16
    N = G * Eps
    dims = [3, 64, 64, 1]
    Ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32) for i in range(3)]
    bs = [np.zeros(dims[i + 1], np.float32) for i in range(3)]
    params = dev(_flat(Ws, bs))
    init = np.repeat(R.reset_states(kind, G, rng), Eps, axis=0)
    init_d = dev(init.T.copy(), torch.float32)
    a = E.rollout(kind, T, 0.05, dims, "ReLU", params, [0.5], init_d, seed=5)
    b = E.rollout(kind, T, 0.05, dims, "ReLU", params, [0.5], init_d, seed=5)
    for k in ("obs", "act", "rew", "logp", "len"):
        assert torch.equal(a[k], b[k])
    ln = a["len"]
    assert int(ln.min()) >= 1 and int(ln.max()) <= T
    pad = torch.arange(T, device="cuda")[:, None] >= ln[None, :]
    assert bool((a["rew"][pad] == 0).all()) and bool((a["obs"].permute(0, 2, 1)[pad] == 0).all())
    adv, _ = E.advantage(0, G, Eps, T, 0.99, 0.0, a["rew"], ln)
    # pooled z-score: every group has mean 0 / unbiased std 1 over its valid steps
    av = adv.T.reshape(G, Eps * T).double()
    mv = (~pad).T.reshape(G, Eps * T)
    cnt = mv.sum(1)
    mean = (av * mv).sum(1) / cnt
    var = (((av - mean[:, None]) ** 2) * mv).sum(1) / (cnt - 1)
    assert float(mean.abs().max()) < 1e-4 and float((var.sqrt() - 1).abs().max()) < 1e-4
    # sharding invariance: the second half of the groups rolled out alone, as rank 1 of 2 does
    half = N // 2
    c = E.rollout(kind, T, 0.05, dims, "ReLU", params, [0.5], init_d[:, half:].contiguous(), seed=5, env_offset=half)
    assert torch.equal(c["rew"], a["rew"][:, half:]) and torch.equal(c["len"], a["len"][half:])
    adv_h, _ = E.advantage(0, G // 2, Eps, T, 0.99, 0.0, c["rew"], c["len"])
    assert torch.equal(adv_h, adv[:, half:])


# ----------------------------------------------------------------------------
# PPO over a sharded rollout: raw advantages + additive sums per shard, "allreduce" = sum of the
# shards' sums, normalise with the global statistics, gradients scaled by the global step count --
# the two ranks of a world-size-2 run emulated one after the other on one GPU (SURVEY 8e)
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("mode_name,width", [pytest.param("mc", 32, id="mc"), pytest.param("gae", 32, id="gae"),
                                             pytest.param("mc", 128, id="mc-w128"), pytest.param("gae", 128, id="gae-w128")])
def test_ppo_sharded_equals_single_rollout(E, mode_name, width):
    """32 wide: FP32-pipe kernels; 128 wide: the streamed tensor-core critic forward and actor / critic gradients."""
    from trajopt_grpo_b200 import _lib as L
    rng = np.random.default_rng(11)
    G, Eg, T, O, A = 6, 8, 20, 10, 2
    N = G * Eg
    a_dims, c_dims = [O, width, width, A], [O, width, width, 1]
    mk = lambda dims: dev(_flat([(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32)
                                 for i in range(3)], [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(3)]))
    a_flat, c_flat = mk(a_dims), mk(c_dims)
    lens = rng.integers(1, T + 1, N).astype(np.int32)
    mask = (np.arange(T)[:, None] < lens[None, :])
    obs = (rng.standard_normal((T, O, N)) * mask[:, None, :]).astype(np.float32)
    act = (rng.standard_normal((T, A, N)) * mask[:, None, :]).astype(np.float32)
    rew = (rng.standard_normal((T, N)) * mask).astype(np.float32)
    mode = L.ADV_PPO_MC if mode_name == "mc" else L.ADV_PPO_GAE
    cov, eps, c1, kl = [0.4, 0.4], 0.2, 0.5, 0.5

    def run(sl, sums_global=None, n_global=None):
        o, a, r, ln = (dev(np.ascontiguousarray(x[..., sl])) for x in (obs, act, rew, lens))
        g_loc = (sl.stop - sl.start) // Eg
        vals, _ = E.policy_forward_traj(c_dims, "ReLU", c_flat, o, None, None, ln, want_mu=True, want_logp=False)
        adv, rtg, sums = E.advantage_ppo_raw(mode, g_loc, Eg, T, 0.99, 0.95, r, ln, vals.view(T, -1))
        if sums_global is None:
            return sums
        E.advantage_ppo_normalize(T, ln, sums_global, adv, rtg)
        _, olp = E.policy_forward_traj(a_dims, "ReLU", a_flat, o, cov, a, ln)
        ga, _ = E.policy_grad(a_dims, "ReLU", a_flat, cov, o, a, adv, olp, ln, eps, -1.0 / n_global, kl / n_global)
        gc, _ = E.value_grad(c_dims, "ReLU", c_flat, o, rtg, ln, c1 / n_global)
        return torch.cat([ga, gc]).double()

    full = slice(0, N)
    s_full = run(full)
    n = int(round(float(s_full[4])))
    assert n == int(lens.sum())
    g_full = run(full, s_full, n)
    shards = [slice(0, N // 2), slice(N // 2, N)]
    s_sum = sum(run(sl) for sl in shards)
    np.testing.assert_allclose(s_sum.cpu().numpy(), s_full.cpu().numpy(), rtol=1e-12, atol=1e-9)
    g_sum = sum(run(sl, s_sum, n) for sl in shards)
    err = (g_sum - g_full).abs().max().item()
    assert err <= 2e-5 * g_full.abs().max().item() + 1e-7, err
    # and the one-call form equals raw + normalize with the local sums
    o, r, ln = dev(obs), dev(rew), dev(lens)
    vals, _ = E.policy_forward_traj(c_dims, "ReLU", c_flat, o, None, None, ln, want_mu=True, want_logp=False)
    adv1, rtg1 = E.advantage(mode, G, Eg, T, 0.99, 0.95, r, ln, vals.view(T, N))
    adv2, rtg2, s2 = E.advantage_ppo_raw(mode, G, Eg, T, 0.99, 0.95, r, ln, vals.view(T, N))
    E.advantage_ppo_normalize(T, ln, s2, adv2, rtg2)
    assert torch.equal(adv1, adv2) and torch.equal(rtg1, rtg2)


# ----------------------------------------------------------------------------
# fp32 (throughput mode) vs float64 (the reference's env arithmetic) over the FULL benchmark horizons
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("workload,bound", [("pendulum", 0.5), ("quadpole_cfg4", 1e-3), ("quadpole2d_cfg3", 2e-2)])
def test_fp32_drift_over_benchmark_horizons(E, workload, bound):
    """North star: 'rel 1e-5 fp32 per step, with drift bounds stated over the horizon'.  The per-step bound is
    test_env_step_float32_tolerance; this is the free-running drift of the fp32 rollout against the float64 one on the
    SAME policy, initial states and Philox noise over the benchmark's own horizon (200 / 1000 / 500 steps) and start
    policy.  Stated bounds (measured values are printed): max |obs32 - obs64| over all steps both runs are alive, and
    episode lengths equal for >= 99.9 % of the envs.  Measured on B200: 3-D QuadPole, 1000 steps: 7.5e-5 (the closed loop
    under the stabilising start policy is contracting); QuadPole2D, 500 steps: 1.2e-3 (its pole swings undamped);
    Pendulum, 200 steps under a random-init policy: 0.13 -- the episodes start 0.05 rad from an equilibrium the policy
    does not stabilise, so rounding differences are amplified exponentially by the dynamics themselves (a property of
    the system, not of the arithmetic: the per-step error stays at 1e-5).  Lengths were equal for 100 % of the envs."""
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    w = bench.WORKLOADS[workload]
    kind, T = w["kind"], w["T"]
    dims, Ws, bs = bench.start_policy_arrays(w)
    params = dev(_flat(Ws, bs))
    rng = np.random.default_rng(0)
    G, Eg = 32, w["E"]
    N = G * Eg
    init = np.repeat(R.reset_states(kind, G, rng), Eg, axis=0)
    cov = [w["cov"]] * R.ACT_DIM[kind]
    o32 = E.rollout(kind, T, R.DEFAULT_DT[kind], dims, "ReLU", params, cov, dev(init.T.copy(), torch.float32), seed=11)
    o64 = E.rollout(kind, T, R.DEFAULT_DT[kind], dims, "ReLU", params, cov, dev(init.T.copy(), torch.float64), seed=11)
    l32, l64 = o32["len"].cpu().numpy(), o64["len"].cpu().numpy()
    same = float((l32 == l64).mean())
    both = (torch.arange(T, device="cuda")[:, None] < torch.minimum(o32["len"], o64["len"])[None, :])
    d = (o32["obs"] - o64["obs"]).abs().permute(0, 2, 1)[both]
    drift = float(d.max())
    rdiff = float((o32["rew"] - o64["rew"]).abs()[both].max())
    print(f"[fp32-drift] {workload:16s} T={T} N={N}: max |obs32-obs64| {drift:.2e}, max |rew32-rew64| {rdiff:.2e}, "
          f"lengths equal {100 * same:.2f} %, mean length {l64.mean():.1f}")
    assert drift <= bound, drift
    assert same >= 0.999, same
