"""The oracle (oracle/restate.py) pinned against fixtures produced by the
UNMODIFIED reference (oracle/make_golden.py -> tests/golden/*.npz)."""
import os

import numpy as np
import pytest

import restate as R

ENVS = [0, 1, 2, 3]


def load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name), allow_pickle=False))


@pytest.mark.parametrize("kind", ENVS)
def test_transitions_float64(golden_dir, kind):
    g = load(golden_dir, f"transitions_env{kind}.npz")
    cfg = R.EnvCfg.make(kind, {0: 120, 1: 200, 2: 150, 3: 150}[kind])
    nxt, rew, done, _ = R.env_step(cfg, g["state"], g["action"], g["steps_done"], g["bal_count"], np.float64)
    # float64 restatement of float64 arithmetic: agreement to rounding of the
    # few re-associated sums (np.sum order) -- 1e-12 relative
    np.testing.assert_allclose(nxt, g["next"], rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(rew, g["reward"], rtol=1e-11, atol=1e-12)
    assert np.array_equal(done, g["done"])          # flags bit-exact
    assert g["done"].sum() > 0


@pytest.mark.parametrize("kind", ENVS)
def test_transitions_float32_mode_close(golden_dir, kind):
    g = load(golden_dir, f"transitions_env{kind}.npz")
    cfg = R.EnvCfg.make(kind, {0: 120, 1: 200, 2: 150, 3: 150}[kind])
    nxt, rew, _, _ = R.env_step(cfg, g["state"], g["action"], g["steps_done"], g["bal_count"], np.float32)
    np.testing.assert_allclose(nxt, g["next"], rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(rew, g["reward"], rtol=1e-4, atol=2e-4)


@pytest.mark.parametrize("name,kind,keys", [("cartpole", 0, ("masscart", "masspole", "length", "gravity")),
                                            ("pendulum", 1, ("mass", "length", "gravity"))])
def test_transitions_non_default_physical_parameters(golden_dir, name, kind, keys):
    """CartPole / Pendulum constructed with non-default masses, lengths, gravity and timestep."""
    g = load(golden_dir, f"transitions_{name}_params.npz")
    cfg = R.EnvCfg.make(kind, 100, float(g["timestep"]), phys=[float(g[k]) for k in keys])
    nxt, rew, done, _ = R.env_step(cfg, g["state"], g["action"], g["steps_done"], g["bal_count"], np.float64)
    np.testing.assert_allclose(nxt, g["next"], rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(rew, g["reward"], rtol=1e-11, atol=1e-12)
    assert np.array_equal(done, g["done"])


def test_quadrotor12_dynamics(golden_dir):
    g = load(golden_dir, "quadrotor12_dynamics.npz")
    out = R.quadrotor12_dynamics(g["state"], g["control"])
    np.testing.assert_allclose(out, g["next"], rtol=1e-12, atol=1e-13)


def test_survey_known_answers():
    # SURVEY.md section 8c seeds (probe of the unmodified reference)
    s = np.array([[0.1, -0.2, np.sin(0.3), np.cos(0.3), 0.5]])
    nxt, rew, _ = R.cartpole_step(s, np.array([[0.25]], np.float32), 0.02)
    np.testing.assert_allclose(nxt[0], [0.09575993016964922, -0.2120034915175395, 0.3070415499754497,
                                        0.9516961104200613, 0.6041429572050855], rtol=1e-13)
    np.testing.assert_allclose(rew[0], 0.42912246516789815, rtol=1e-12)
    s = np.array([[np.sin(3.0), np.cos(3.0), 0.2]])
    nxt, rew, _ = R.pendulum_step(s, np.array([[0.4]], np.float32), 0.05, np.zeros(1, np.int64))
    np.testing.assert_allclose(nxt[0], [0.13410695933245298, -0.9909668629467908, 0.14160854729597033], rtol=1e-7)
    assert abs(R.gaussian_entropy(np.array([0.5]), 1) - 1.0723649263) < 1e-7   # the survey value is an fp32 tensor print


def test_time_thresholds():
    # SURVEY.md section 7 "hard parts": float64 accumulation facts
    assert R.balanced_limit_count(0.05) == 101
    assert R.time_limit_step(0.05, 200) == 200
    assert R.time_limit_step(0.02, 500) == 501
    assert R.time_limit_step(0.02, 1000) == 1001


def _weights(g, prefix=""):
    Ws, bs, i = [], [], 0
    while f"{prefix}W{i}" in g:
        Ws.append(g[f"{prefix}W{i}"]); bs.append(g[f"{prefix}b{i}"]); i += 1
    return Ws, bs


ROLLOUTS = ["cartpole", "pendulum", "quadpole2d", "quadpole",
            # round 2: BASELINE shapes (cfg 1 at full size with the shipped weights, cfg 3 / cfg 4 policy widths),
            # depth 0 / 1 / 3, Tanh and a per-layer activation list
            "cartpole_cfg1", "quadpole2d_w128", "quadpole_w256", "pendulum_h1", "cartpole_h3", "pendulum_h0",
            "cartpole_tanh", "pendulum_mixed_act"]


def _act(g):
    return R.acts_from_names(g["activation"]) if "activation" in g else R.ACT_RELU


@pytest.mark.parametrize("name", ROLLOUTS)
def test_rollout_matches_reference(golden_dir, name):
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    kind, G, E, T = int(g["kind"]), int(g["G"]), int(g["E"]), int(g["T"])
    Ws, bs = _weights(g)
    cfg = R.EnvCfg.make(kind, T)
    cov = np.full(R.ACT_DIM[kind], g["cov"], np.float32)
    obs, act, rew, logp, ln, mask = R.rollout(cfg, g["init"], Ws, bs, cov, g["noise"], act=_act(g))
    sh = lambda x: x.reshape((G, E) + x.shape[1:])
    assert np.array_equal(sh(ln), g["len"].astype(np.int32))       # lengths bit-exact
    assert np.array_equal(sh(mask), g["mask"])
    # free-running float64 env + fp32 policy; only the fp32 MLP summation order
    # (batched numpy matmul vs torch single-row GEMV) differs
    np.testing.assert_allclose(sh(obs), g["obs"], rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(sh(act), g["act"], rtol=2e-4, atol=2e-4)
    np.testing.assert_allclose(sh(rew), g["rew"], rtol=2e-4, atol=5e-4)
    sel = g["mask"] > 0
    np.testing.assert_allclose(sh(logp)[sel], g["logp_valid"], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("name", ROLLOUTS)
def test_grpo_gradient_matches_reference(golden_dir, name):
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    Ws, bs = _weights(g)
    kind = int(g["kind"])
    cov = np.full(R.ACT_DIM[kind], g["cov"], np.float32)
    rtg, adv = R.grpo_advantage(g["rew"], g["mask"], float(g["gamma"]))
    J, dW, db, lp, old_lp = R.grpo_objective_and_grad(g["obs"], g["act"], adv, g["mask"], Ws, bs, Ws, bs,
                                                       cov, float(g["eps_clip"]), act=_act(g), dtype="float32")
    for i in range(len(Ws)):
        gw, gb = g[f"grpo_grad{2 * i}"], g[f"grpo_grad{2 * i + 1}"]
        scale = max(np.abs(gw).max(), 1e-6)
        assert np.abs(dW[i] - gw).max() <= 2e-4 * scale + 1e-5
        assert np.abs(db[i] - gb).max() <= 2e-4 * max(np.abs(gb).max(), 1e-6) + 1e-5


@pytest.mark.parametrize("name", ROLLOUTS)
def test_grpo_adam_updates_match_reference(golden_dir, name):
    g = load(golden_dir, f"rollout_grpo_{name}.npz")
    Ws, bs = _weights(g)
    kind = int(g["kind"])
    cov = np.full(R.ACT_DIM[kind], g["cov"], np.float32)
    rtg, adv = R.grpo_advantage(g["rew"], g["mask"], float(g["gamma"]))
    params = []
    for w, b in zip(Ws, bs):
        params += [w.copy(), b.copy()]
    m = [np.zeros_like(p) for p in params]
    v = [np.zeros_like(p) for p in params]
    old = [p.copy() for p in params]
    step = 0
    for learn_call, key in ((0, "grpo_adam3_p"), (1, "grpo_adam6_p")):
        for it in range(3):
            step += 1
            J, dW, db, _, _ = R.grpo_objective_and_grad(g["obs"], g["act"], adv, g["mask"], params[0::2], params[1::2],
                                                       old[0::2], old[1::2], cov, float(g["eps_clip"]), act=_act(g),
                                                       dtype="float32")
            grads = []
            for a, b in zip(dW, db):
                grads += [a, b]
            params = R.adam_step(params, grads, m, v, step, 3e-4)
        old = [p.copy() for p in params]
        for i, p in enumerate(params):
            np.testing.assert_allclose(p, g[f"{key}{i}"], rtol=1e-4, atol=2e-6)


PPO_FIXTURES = ["ppo_mc_quadpole2d", "ppo_gae_quadpole2d", "ppo_mc_ragged_quadpole2d", "ppo_gae_ragged_quadpole2d",
                "ppo_mc_quadpole2d_shipped", "ppo_gae_cartpole_shipped"]


def _ppo_setup(g):
    """Actor / critic weights and the start-of-learn() quantities of PPO.learn (ppo.py:85-143) in float32."""
    import torch
    Ws, bs = _weights(g)
    cWs, cbs = _weights(g, "c")
    kind = int(g["kind"])
    cov = np.full(R.ACT_DIM[kind], g["cov"], np.float32)
    t = lambda x: torch.tensor(np.asarray(x))
    with torch.no_grad():
        values = R._torch_mlp(t(g["obs"]), [t(w) for w in cWs], [t(b) for b in cbs], R.ACT_RELU)[..., 0].numpy()
        old_logp = R._torch_logp(R._torch_mlp(t(g["obs"]), [t(w) for w in Ws], [t(b) for b in bs], R.ACT_RELU),
                                 t(cov), t(g["act"])).numpy()
    return Ws, bs, cWs, cbs, cov, values, old_logp


def _pairs(flat, shapes):
    out, off = [], 0
    for s in shapes:
        n = int(np.prod(s))
        out.append(flat[off:off + n].reshape(s))
        off += n
    return out


@pytest.mark.parametrize("name", PPO_FIXTURES)
def test_ppo_restatement_matches_reference(golden_dir, name):
    """R.ppo_advantages + R.ppo_objective_and_grad in float32 against PPO.learn full batch: one SGD(lr=1) update
    (the gradient) and three Adam updates with the old log-probs fixed at the start of learn() (ppo.py:142-143)."""
    g = load(golden_dir, f"{name}.npz")
    Ws, bs, cWs, cbs, cov, values, old_logp = _ppo_setup(g)
    mask = g["mask"]
    _, _, adv, ret = R.ppo_advantages(g["rew"], mask, values, float(g["gamma"]), float(g["lam"]),
                                      bool(g["monte_carlo"]))
    shapes = [p.shape for wb in zip(Ws, bs) for p in wb] + [p.shape for wb in zip(cWs, cbs) for p in wb]
    params = [p.copy() for wb in zip(Ws, bs) for p in wb] + [p.copy() for wb in zip(cWs, cbs) for p in wb]
    na = 2 * len(Ws)
    m = [np.zeros_like(p) for p in params]
    v = [np.zeros_like(p) for p in params]
    for step in range(1, 4):
        o = R.ppo_objective_and_grad(g["obs"], g["act"], adv, ret, mask, params[0:na:2], params[1:na:2],
                                     params[na::2], params[na + 1::2], old_logp, cov, float(g["eps_clip"]), 0.5, 0.5,
                                     dtype="float32")
        grads = _pairs(np.concatenate([o["actor_grad"], o["critic_grad"]]), shapes)
        if step == 1:
            assert o["n"] == int(mask.sum())
            for i, gr in enumerate(grads):
                ref = g[f"ppo_grad{i}"]
                assert np.abs(gr - ref).max() <= 2e-4 * max(np.abs(ref).max(), 1e-6) + 1e-5, (i, np.abs(gr - ref).max())
        params = R.adam_step(params, grads, m, v, step, 2e-4)
    for i, p in enumerate(params):
        np.testing.assert_allclose(p, g[f"ppo_adam3_p{i}"], rtol=1e-4, atol=2e-6, err_msg=str(i))


def test_ppo_minibatch_restatement_matches_reference(golden_dir):
    """batch_size=64: one torch.randperm over the valid rows per epoch, drawn from torch's default generator seeded
    right before learn() (ppo.py:147-157), the rows in the reference's flattening order (env-major, step-minor), each
    minibatch's means over its own rows, one Adam step per minibatch."""
    import torch
    g = load(golden_dir, "ppo_minibatch_quadpole2d.npz")
    Ws, bs, cWs, cbs, cov, values, old_logp = _ppo_setup(g)
    mask = g["mask"]
    _, _, adv, ret = R.ppo_advantages(g["rew"], mask, values, float(g["gamma"]), float(g["lam"]),
                                      bool(g["monte_carlo"]))
    sel = mask > 0
    rows = {k: np.asarray(x)[sel] for k, x in (("obs", g["obs"]), ("act", g["act"]), ("adv", adv), ("ret", ret),
                                                ("olp", old_logp))}
    n, bsz = int(sel.sum()), int(g["batch_size"])
    shapes = [p.shape for wb in zip(Ws, bs) for p in wb] + [p.shape for wb in zip(cWs, cbs) for p in wb]
    params = [p.copy() for wb in zip(Ws, bs) for p in wb] + [p.copy() for wb in zip(cWs, cbs) for p in wb]
    na = 2 * len(Ws)
    m = [np.zeros_like(p) for p in params]
    v = [np.zeros_like(p) for p in params]
    step = 0
    torch.manual_seed(int(g["torch_seed"]))
    for _ in range(int(g["updates"])):
        perm = torch.randperm(n).numpy()
        for s in range(0, n, bsz):
            idx = perm[s:s + bsz]
            o = R.ppo_objective_and_grad(rows["obs"][idx], rows["act"][idx], rows["adv"][idx], rows["ret"][idx],
                                         np.ones(idx.size), params[0:na:2], params[1:na:2], params[na::2],
                                         params[na + 1::2], rows["olp"][idx], cov, float(g["eps_clip"]), 0.5, 0.5,
                                         dtype="float32")
            step += 1
            params = R.adam_step(params, _pairs(np.concatenate([o["actor_grad"], o["critic_grad"]]), shapes), m, v,
                                 step, 2e-4)
    for i, p in enumerate(params):
        np.testing.assert_allclose(p, g[f"ppo_mb_adam_p{i}"], rtol=1e-4, atol=2e-6, err_msg=str(i))


def test_gae_gamma_lambda_is_one_rounded_scalar():
    """The GAE recurrence multiplies by fp32(gamma*lam) (the float64 product, ppo.py:123), which for 0.99 / 0.99
    differs from fp32(0.99)*fp32(0.99): a restatement that rounds the factors separately disagrees in the last bit."""
    assert np.float32(0.99 * 0.99) != np.float32(0.99) * np.float32(0.99)
    rew = np.array([[0.0, 0.0, 1.0]], np.float32)
    adv, _ = R.gae(rew, np.ones_like(rew), np.zeros_like(rew), 0.99, 0.99)
    f = np.float32(0.99 * 0.99)
    assert adv[0, 0] == f * (f * np.float32(1.0))


def test_rtg_reference_example():
    # the one numeric expectation the reference's tests hold (tests/test_rollout_buffer.py:78-92),
    # evaluated in floating point (its expected array is int-typed, SURVEY section 4)
    rew = np.array([[[1, 2, 3], [0, 1, 2]], [[3, 2, 1], [1, 0, 1]]], np.float32)
    rtg = R.reward_to_go(rew, np.ones_like(rew), 0.99)
    np.testing.assert_allclose(rtg[0, 0], [1 + 0.99 * (2 + 0.99 * 3), 2 + 0.99 * 3, 3], rtol=1e-6)
    mask = np.ones_like(rew); mask[0, 1, 2] = 0
    rtg = R.reward_to_go(rew, mask, 0.99)
    np.testing.assert_allclose(rtg[0, 1], [0 + 0.99 * 1, 1, 0], rtol=1e-6)
