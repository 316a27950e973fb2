"""PPO on the tensor-core kernels against the float64 PPO restatement (oracle/restate.py: ppo_advantages,
ppo_objective_and_grad, themselves pinned on the reference's PPO fixtures by tests/test_oracle_golden.py).

  K3 objective   tg_policy_grad at PPO (scale -1/n, KL 0.5/n) and GRPO (+-1/G, no KL) settings, every built
                 tensor-core (O, A) instance at width 64 (K3-TC), 128 and 256 (K3-TCW), ReLU and Tanh, with inputs
                 that populate every branch of the clipped surrogate (asserted)
  forward-only   tg_policy_forward_traj on the wide path: critic values and log-probs
  K2             tg_advantage in its PPO modes (raw Monte-Carlo / GAE scan, sums, z-score) over several blocks
  PPO.learn      end to end at actor + critic widths 64 / 128 / 256, MC and GAE
  GRPO           maximize=True at width 256 is the exact negation of maximize=False

Every kernel-level case runs on the FP32 pipe and on the 3xTF32 tensor cores; the measured errors are printed next to
their bounds ([ppo-parity]).
"""
import functools

import numpy as np
import pytest
import torch

import restate as R
from test_gpu_baseline_shapes import GRAD_TOL_F64, KINK, _adam_close, _load_actor, _make_buffer

pytestmark = pytest.mark.gpu

EPS = 0.2
INSTANCES = [(3, 1), (5, 1), (10, 2), (20, 4)]     # (obs, act) of the four environments
MODES = ("fp32", "3xtf32")
ACT_FN = {"ReLU": R.ACT_RELU, "Tanh": R.ACT_TANH}


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.fixture(scope="module")
def E():
    from trajopt_grpo_b200 import engine
    return engine


def _policy(rng, dims):
    Ws = [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32) for i in range(len(dims) - 1)]
    bs = [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(len(dims) - 1)]
    return Ws, bs


def _flat(Ws, bs):
    return np.concatenate([np.concatenate([w.reshape(-1), b.reshape(-1)]) for w, b in zip(Ws, bs)]).astype(np.float32)


def _ragged_lengths(rng, N, T):
    """Exactly 128 envs run all T steps (the last step holds exactly one full 128-env tile), the others end earlier."""
    ln = np.concatenate([np.full(128, T), rng.integers(1, T, N - 128)]).astype(np.int32)
    return rng.permutation(ln)


def _kink_free(dims, act_name, seed, draw):
    """Weights and inputs from `seed`, with the biases of ReLU units that have a valid sample within KINK of the kink
    moved off it (R.kink_free_biases), so that a tolerance measures arithmetic and not which side of a kink fp32
    summation noise lands on."""
    rng = np.random.default_rng(seed)
    Ws, bs = _policy(rng, dims)
    x = draw(rng)
    if act_name == "ReLU":
        bs = R.kink_free_biases(x[0], Ws, bs, R.ACT_RELU, KINK)
    return rng, Ws, bs, x


def _mmul(x, Ws, bs, act_name):
    return R.mlp_forward(x, Ws, bs, ACT_FN[act_name], np.float64)


# ----------------------------------------------------------------------------
# a. the K3 objective at PPO and GRPO settings
# ----------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _k3_case(O, A, W, act_name):
    """Inputs in the kernels' [T, ., N] layout that populate every branch of the clipped surrogate: the ratio
    r = exp(lp - old_logp) is SET through old_logp = lp64 - log r with r spread over [0.6, 1.5] and none within 1e-3
    of 1 +- eps (the clip decision is then the same in every arithmetic), adv of both signs with ~5 % exact zeros."""
    N, T = 300, 9
    dims = [O, W, W, A]

    def draw(rng):
        ln = _ragged_lengths(rng, N, T)
        mask = np.arange(T)[:, None] < ln[None, :]
        obs = rng.standard_normal((T, O, N)).astype(np.float32)
        return obs.transpose(0, 2, 1)[mask], obs, ln, mask

    rng, Ws, bs, (_, obs, ln, mask) = _kink_free(dims, act_name, 1000 * O + W + (7 if act_name == "Tanh" else 0), draw)
    cov = np.full(A, 0.4, np.float32)
    rows = obs.transpose(0, 2, 1)                                          # [T, N, O]
    mu = _mmul(rows.reshape(-1, O), Ws, bs, act_name).reshape(T, N, A)
    act = (mu + np.sqrt(cov.astype(np.float64)) * rng.standard_normal((T, N, A))).astype(np.float32)
    lp64 = R.gaussian_log_prob(mu, cov, act, np.float64)
    r = rng.uniform(0.6, 1.5, (T, N))
    r = np.where((np.abs(r - (1 - EPS)) < 1e-3) | (np.abs(r - (1 + EPS)) < 1e-3), r + 5e-3, r)
    old_logp = (lp64 - np.log(r)).astype(np.float32)
    adv = rng.normal(0.4, 1.0, (T, N)).astype(np.float32)
    adv[rng.random((T, N)) < 0.05] = 0.0
    # every (sign of A) x (clip side) cell holds a few percent of the valid samples
    rv, av = r[mask], adv[mask]
    for s in (av > 0, av < 0):
        for side in (rv < 1 - EPS, (rv >= 1 - EPS) & (rv <= 1 + EPS), rv > 1 + EPS):
            assert (s & side).mean() >= 0.03
    assert 0.03 <= (av == 0).mean() <= 0.08
    return dict(dims=dims, Ws=Ws, bs=bs, cov=cov, obs=obs, act=act, adv=adv, old_logp=old_logp, ln=ln, mask=mask,
                rows=rows)


# The KL term's gradient sums exp(old_logp) (a - mu) / var over samples with exp(old_logp) > 0 and (a - mu) averaging
# ~0, so it grows like sqrt(n) while a systematic error in mu enters n-fold.  The 3xTF32 forward's truncating split
# leaves such a bias (~1e-6 of mu): the KL-only gradient measured 4.6e-5 .. 1.2e-4 of its max on B200 (FP32 pipe
# 3e-7), mostly in the output layer, and the PPO objective's gradient 1.2e-5 .. 1.5e-5 for the one-action instances
# ((3,1) W 256, (5,1) W 128 / 256) against <= 6.6e-6 for everything else.  Bound for that case, 2x the measurement:
KL_TOL_3XTF32 = 3e-5

SETTINGS = {   # name -> (scale, kl_scale) as functions of n valid samples (G = 5 groups for GRPO)
    "ppo": lambda n: (-1.0 / n, 0.5 / n),             # algorithms.py PPO.learn: actor + kl_coeff * KL, kl_coeff 0.5
    "grpo": lambda n: (1.0 / 5, 0.0),                 # GRPO.learn
    "grpo_max": lambda n: (-1.0 / 5, 0.0),            # GRPO(maximize=True)
}


@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("act_name", ["ReLU", "Tanh"])
@pytest.mark.parametrize("W", [64, 128, 256])
@pytest.mark.parametrize("O,A", INSTANCES)
def test_policy_grad_tensor_core_matches_float64_ppo_objective(E, O, A, W, act_name, setting):
    c = _k3_case(O, A, W, act_name)
    mask = c["mask"]
    n = int(mask.sum())
    scale, kl_scale = SETTINGS[setting](n)
    # the kernel's objective is scale * sum(min(...)) + kl_scale * sum(exp(old) (old - lp)) = f * (actor + k * KL)
    # with the restatement's means: f = -n * scale, k = kl_scale / -scale
    f, k = -n * scale, kl_scale / -scale
    o = R.ppo_objective_and_grad(c["rows"], c["act"], c["adv"], None, mask, c["Ws"], c["bs"], None, None,
                                 c["old_logp"], c["cov"], EPS, 0.5, k, act=ACT_FN[act_name])
    ref = f * o["actor_grad"]
    J = f * (o["actor"] + k * o["kl"])
    args = (dev(c["obs"]), dev(c["act"].transpose(0, 2, 1)), dev(c["adv"]), dev(c["old_logp"]), dev(c["ln"]))
    params = dev(_flat(c["Ws"], c["bs"]))
    out = {}
    try:
        for mode in MODES:
            E.set_math(mode)
            g, st = E.policy_grad(c["dims"], act_name, params, c["cov"].tolist(), *args, EPS, scale, kl_scale)
            torch.cuda.synchronize()
            out[mode] = (g.cpu().numpy(), st.cpu().numpy().astype(np.float64))
    finally:
        E.set_math("auto")
    for mode, (g, st) in out.items():
        tol = KL_TOL_3XTF32 if (kl_scale and mode == "3xtf32") else GRAD_TOL_F64[mode]
        err = float(np.abs(g - ref).max() / np.abs(ref).max())
        e_obj = abs(st[0] - J) / abs(J)
        e_rat = abs(st[2] - o["ratio_sum"]) / o["ratio_sum"]
        print(f"[ppo-parity] K3 ({O},{A}) W {W:3d} {act_name:4s} {setting:8s} {mode:6s} grad {err:.2e} "
              f"(<= {tol:.0e})  objective {e_obj:.1e}  sum ratio {e_rat:.1e} (<= 1e-5)  "
              f"clipped {int(st[3])}/{n}")
        assert err <= tol, (mode, err)
        assert int(st[1]) == n and int(st[3]) == o["n_clipped"], (mode, st, o["n_clipped"])
        assert e_obj <= 1e-5 and e_rat <= 1e-5, (mode, st, J, o["ratio_sum"])


# ----------------------------------------------------------------------------
# c. forward-only mode of kernel A (critic values, old log-probs) against float64
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("O,A,W,act_name", [(10, 1, 128, "ReLU"), (20, 1, 256, "ReLU"), (3, 1, 256, "Tanh"),
                                            (10, 2, 128, "ReLU"), (20, 4, 256, "Tanh"), (5, 1, 128, "ReLU")])
def test_policy_forward_traj_wide_matches_float64(E, O, A, W, act_name):
    """Values (mu of an A = 1 net) and log-probs on valid rows within 1e-5 relative (atol 1e-5 of the largest
    magnitude, for entries that cancel to ~0); rows past an episode's end exactly 0."""
    N, T = 333, 6
    dims = [O, W, W, A]

    def draw(rng):
        ln = _ragged_lengths(rng, N, T)
        mask = np.arange(T)[:, None] < ln[None, :]
        obs = rng.standard_normal((T, O, N)).astype(np.float32)
        return obs.transpose(0, 2, 1)[mask], obs, ln, mask

    rng, Ws, bs, (_, obs, ln, mask) = _kink_free(dims, act_name, 31 * O + W, draw)
    act = rng.standard_normal((T, A, N)).astype(np.float32)
    cov = np.full(A, 0.3, np.float32)
    mu64 = _mmul(obs.transpose(0, 2, 1).reshape(-1, O), Ws, bs, act_name).reshape(T, N, A)
    lp64 = R.gaussian_log_prob(mu64, cov, act.transpose(0, 2, 1), np.float64)
    out = {}
    try:
        for mode in MODES:
            E.set_math(mode)
            mu, lp = E.policy_forward_traj(dims, act_name, dev(_flat(Ws, bs)), dev(obs), cov.tolist(), dev(act), dev(ln),
                                           want_mu=True, want_logp=True)
            torch.cuda.synchronize()
            out[mode] = (mu.cpu().numpy().transpose(0, 2, 1), lp.cpu().numpy())
    finally:
        E.set_math("auto")
    for mode, (mu, lp) in out.items():
        for what, got, ref in (("value" if A == 1 else "mu", mu[mask], mu64[mask]), ("logp", lp[mask], lp64[mask])):
            err = float((np.abs(got - ref) / (np.abs(ref) + np.abs(ref).max())).max())
            print(f"[ppo-parity] forward ({O},{A}) W {W} {act_name:4s} {mode:6s} {what:5s} {err:.1e}")
            np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-5 * np.abs(ref).max(), err_msg=f"{mode} {what}")
        assert np.all(mu[~mask] == 0) and np.all(lp[~mask] == 0), mode


# ----------------------------------------------------------------------------
# d. K2 in its PPO modes
# ----------------------------------------------------------------------------
def _k2_lengths(rng, N, T):
    """Block 0: two warps of length T, one warp of one shorter common length, one ragged warp holding 1 and T;
    the rest (two more blocks and a 37-env partial block) ragged."""
    ln = rng.integers(1, T + 1, N)
    ln[0:64] = T
    ln[64:96] = max(1, T // 2)
    ln[96] = 1
    ln[97] = T
    return ln.astype(np.int32)


@pytest.mark.parametrize("T", [1, 8, 37])
@pytest.mark.parametrize("mc", [True, False], ids=["mc", "gae"])
def test_ppo_advantages_match_restatement(E, T, mc):
    """Raw adv / returns bit-exact against the fp32 recurrence (gamma = lam = 0.99: fp32(gamma*lam) differs from
    fp32(gamma)*fp32(lam)), the five sums to 1e-12 of the float64 sums (the count exact), the z-scores within 1e-6
    (relative to max(|z|, 1)) of the float64 z-score, padding 0.  Padding rows of rew / values hold garbage: the kernel
    must not read them."""
    from trajopt_grpo_b200 import _lib as L
    rng = np.random.default_rng(T + 100 * mc)
    N = 3 * 128 + 37
    gamma, lam = 0.99, 0.99
    ln = _k2_lengths(rng, N, T)
    mask = np.arange(T)[:, None] < ln[None, :]                          # [T, N]
    rew = rng.standard_normal((T, N)).astype(np.float32)
    val = (0.5 + rng.standard_normal((T, N))).astype(np.float32)
    adv, ret, adv_z, ret_z = R.ppo_advantages(rew.T, mask.T, val.T, gamma, lam, mc, np.float32)
    mode = L.ADV_PPO_MC if mc else L.ADV_PPO_GAE
    dr, dl, dv = dev(rew), dev(ln), dev(val)
    ka, kr, sums = E.advantage_ppo_raw(mode, N, 1, T, gamma, lam, dr, dl, dv)
    ka, kr, sums = ka.cpu().numpy(), kr.cpu().numpy(), sums.cpu().numpy()
    assert np.array_equal(ka[mask], adv.T[mask]) and np.array_equal(kr[mask], ret.T[mask])
    assert np.all(ka[~mask] == 0) and np.all(kr[~mask] == 0)
    a64, r64 = adv.T[mask].astype(np.float64), ret.T[mask].astype(np.float64)
    ref = np.array([a64.sum(), (a64 * a64).sum(), r64.sum(), (r64 * r64).sum()])
    np.testing.assert_allclose(sums[:4], ref, rtol=1e-12)
    assert sums[4] == mask.sum()
    za, zr = E.advantage(mode, N, 1, T, gamma, lam, dr, dl, dv)
    na, nr = dev(ka), dev(kr)
    E.advantage_ppo_normalize(T, dl, dev(sums), na, nr)
    for what, got, z in (("adv", za, adv_z), ("ret", zr, ret_z), ("adv raw+norm", na, adv_z), ("ret raw+norm", nr, ret_z)):
        got = got.cpu().numpy()
        err = float((np.abs(got[mask] - z.T[mask]) / np.maximum(np.abs(z.T[mask]), 1.0)).max())
        print(f"[ppo-parity] K2 {'mc' if mc else 'gae'} T {T:2d} {what:12s} z-score {err:.1e} (<= 1e-6)")
        assert err <= 1e-6, (what, err)
        assert np.all(got[~mask] == 0), what


# ----------------------------------------------------------------------------
# e. PPO.learn end to end at tensor-core widths
# ----------------------------------------------------------------------------
# max |g - g_float64| / max |g_float64| of the whole update (actor + critic) against the float64 chain (values, raw
# advantages, z-scores, old log-probs and gradients all in float64), measured on B200: FP32 pipe 1.5e-7 .. 5.2e-7,
# 3xTF32 7.5e-7 (W 64), 1.9e-6 (W 128), 2.7e-6 (W 256).  Bound with a ~4x margin:
LEARN_TOL_F64 = 1e-5


def _rollout_case(kind, W, seed):
    """A reference-semantics rollout (R.rollout, float64 env, fp32 policy) of 3 x 100 envs, T = 12, with episodes cut
    at random steps so that the lengths are ragged (an episode's prefix is itself a valid episode)."""
    O, A = R.OBS_DIM[kind], R.ACT_DIM[kind]
    G, Eg, T = 3, 100, 12
    N = G * Eg
    hidden = [W, W]

    def draw(rng):
        obs, act, rew, _, ln, _ = R.rollout(R.EnvCfg.make(kind, T), R.reset_states(kind, N, rng),
                                            *_policy(np.random.default_rng(rng.integers(1 << 30)), [O] + hidden + [A]),
                                            np.full(A, 0.5, np.float32), rng.standard_normal((T, N, A)).astype(np.float32))
        return obs, act, rew, ln

    rng = np.random.default_rng(seed)
    obs, act, rew, ln = draw(rng)
    ln = np.minimum(ln, rng.integers(1, T + 1, N)).astype(np.int32)
    mask = (np.arange(T)[None, :] < ln[:, None])
    obs, act, rew = obs * mask[..., None], act * mask[..., None], rew * mask
    x = obs[mask]
    Ws, bs = _policy(rng, [O] + hidden + [A])
    cWs, cbs = _policy(rng, [O] + hidden + [1])
    bs, cbs = R.kink_free_biases(x, Ws, bs, R.ACT_RELU, KINK), R.kink_free_biases(x, cWs, cbs, R.ACT_RELU, KINK)
    sh = lambda a: a.reshape((G, Eg) + a.shape[1:])
    return dict(kind=kind, O=O, A=A, hidden=hidden, G=G, Eg=Eg, T=T, obs=sh(obs).astype(np.float32),
                act=sh(act).astype(np.float32), rew=sh(rew).astype(np.float32), len=sh(ln), mask=sh(mask.astype(np.float32)),
                Ws=Ws, bs=bs, cWs=cWs, cbs=cbs)


def _oracle_chain(c, mc, dtype):
    """PPO.learn's start (values, advantages, z-scores, old log-probs) and its first full-batch loss, in `dtype`."""
    td = getattr(torch, dtype)
    t = lambda x: torch.tensor(np.asarray(x), dtype=td)
    cov = np.full(c["A"], 0.5, np.float32)
    with torch.no_grad():
        values = R._torch_mlp(t(c["obs"]), [t(w) for w in c["cWs"]], [t(b) for b in c["cbs"]], R.ACT_RELU)[..., 0].numpy()
        old_logp = R._torch_logp(R._torch_mlp(t(c["obs"]), [t(w) for w in c["Ws"]], [t(b) for b in c["bs"]], R.ACT_RELU),
                                 t(cov), t(c["act"])).numpy()
    _, _, adv, ret = R.ppo_advantages(c["rew"], c["mask"], values, 0.99, 0.95, mc, np.dtype(dtype).type)
    return adv, ret, old_logp, cov


def _pol(tg, c):
    pol = tg.GaussianActorCritic_NeuralNetwork(c["O"], c["A"], c["hidden"], "ReLU", 0.5)
    _load_actor(pol.actor, c["Ws"], c["bs"])
    _load_actor(pol.critic, c["cWs"], c["cbs"])
    return pol


PPO_KW = dict(c1=0.5, kl_coeff=0.5, gamma=0.99, lam=0.95, entropy=0.01, batch_size=None)


@pytest.mark.parametrize("mc", [True, False], ids=["mc", "gae"])
@pytest.mark.parametrize("kind,W", [(1, 64), (2, 128), (3, 256)])
def test_ppo_learn_tensor_core_widths_match_oracle(E, kind, W, mc):
    import trajopt_grpo_b200 as tg
    c = _rollout_case(kind, W, 40 + kind)
    buf = _make_buffer(tg, c)
    assert len(set(c["len"].reshape(-1).tolist())) > 3
    params = [p for wb in zip(c["Ws"], c["bs"]) for p in wb] + [p for wb in zip(c["cWs"], c["cbs"]) for p in wb]
    na = 2 * len(c["Ws"])
    chains = {}
    for dtype in ("float32", "float64"):
        adv, ret, old_logp, cov = _oracle_chain(c, mc, dtype)
        o = R.ppo_objective_and_grad(c["obs"], c["act"], adv, ret, c["mask"], c["Ws"], c["bs"], c["cWs"], c["cbs"],
                                     old_logp, cov, EPS, 0.5, 0.5, dtype=dtype)
        chains[dtype] = (o, np.concatenate([o["actor_grad"], o["critic_grad"]]), adv, ret, old_logp, cov)
    o32, g32 = chains["float32"][:2]
    o64, g64 = chains["float64"][:2]
    grads, stats = {}, {}
    try:
        for mode in ("fp32", "auto"):
            E.set_math(mode)
            pol = _pol(tg, c)
            algo = tg.PPO(EPS, pol, torch.optim.SGD(pol.parameters(), lr=1.0), None, 1, monte_carlo=mc, **PPO_KW)
            algo.learn(buf)
            torch.cuda.synchronize()
            grads[mode] = torch.cat([p.grad.reshape(-1) for p in pol.parameters()]).cpu().numpy()
            stats[mode] = algo.last_stats.cpu().numpy().astype(np.float64)
    finally:
        E.set_math("auto")
    n = o64["n"]
    for mode, g in grads.items():
        off = 0
        for i, p in enumerate(params):                   # vs the float32 chain, tensor by tensor (the fixtures' bound)
            ref = g32[off:off + p.size]
            assert np.abs(g[off:off + p.size] - ref).max() <= 5e-4 * max(np.abs(ref).max(), 1e-6) + 1e-6, (mode, i)
            off += p.size
        e64 = float(np.abs(g - g64).max() / np.abs(g64).max())
        st = stats[mode]
        # the first update's ratios are 1 and the z-scored advantages average 0, so the objective is ~0: compare it
        # on the scale of its terms (mean |A| = mean |min(r A, clip(r) A)| at r = 1)
        J = o64["actor"] + 0.5 * o64["kl"]
        e_obj = abs(st[0] - J) / np.abs(chains["float64"][2][c["mask"] > 0]).mean()
        print(f"[ppo-parity] PPO.learn kind {kind} W {W} {'mc' if mc else 'gae'} {mode:5s} vs float64 chain {e64:.2e} "
              f"(<= {LEARN_TOL_F64:.0e})  objective {e_obj:.1e} (<= 1e-5)")
        assert e64 <= LEARN_TOL_F64, (mode, e64)
        assert int(st[1]) == n and int(st[3]) == o64["n_clipped"]
        assert e_obj <= 1e-5 and abs(st[2] - o64["ratio_sum"]) <= 1e-5 * n, (mode, st, J, o64["ratio_sum"])
    assert np.abs(grads["auto"] - grads["fp32"]).max() <= 5e-5 * np.abs(grads["fp32"]).max()
    # three Adam updates (old log-probs and advantages fixed at the start of learn()) vs the float32 chain
    _, _, adv, ret, old_logp, cov = chains["float32"]
    ref = [p.copy() for p in params]
    m = [np.zeros_like(p) for p in ref]
    v = [np.zeros_like(p) for p in ref]
    x = c["obs"][c["mask"] > 0]
    margin = np.inf                      # smallest distance of a ReLU pre-activation from its kink along the path
    for step in range(1, 4):
        margin = min(margin, R.kink_margin(x, ref[0:na:2], ref[1:na:2]), R.kink_margin(x, ref[na::2], ref[na + 1::2]))
        o = R.ppo_objective_and_grad(c["obs"], c["act"], adv, ret, c["mask"], ref[0:na:2], ref[1:na:2], ref[na::2],
                                     ref[na + 1::2], old_logp, cov, EPS, 0.5, 0.5, dtype="float32")
        flat = np.concatenate([o["actor_grad"], o["critic_grad"]])
        gl, off = [], 0
        for p in ref:
            gl.append(flat[off:off + p.size].reshape(p.shape))
            off += p.size
        ref = R.adam_step(ref, gl, m, v, step, 2e-4)
    pol = _pol(tg, c)
    tg.PPO(EPS, pol, torch.optim.Adam(pol.parameters(), lr=2e-4), None, 3, monte_carlo=mc, **PPO_KW).learn(buf)
    for i, (p, r) in enumerate(zip(pol.parameters(), ref)):
        _adam_close(p.detach().cpu().numpy(), r, margin, 2e-4, 3, f"adam3 p{i}")


# ----------------------------------------------------------------------------
# g. GRPO maximize=True at 256 wide (the headline workload's objective)
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "auto"])
def test_grpo_maximize_is_the_exact_negation_at_width_256(E, mode):
    """Negating the scale negates every product and sum the kernels form, exactly: one SGD(lr=1) GRPO.learn with
    maximize=True must produce the bitwise negated gradient (and objective) of maximize=False."""
    import trajopt_grpo_b200 as tg
    c = _rollout_case(3, 256, 60)
    buf = _make_buffer(tg, c)
    out = {}
    try:
        E.set_math(mode)
        for maximize in (False, True):
            pol = tg.GaussianActor_NeuralNetwork(c["O"], c["A"], c["hidden"], "ReLU", 0.5)
            _load_actor(pol.actor, c["Ws"], c["bs"])
            algo = tg.GRPO(EPS, 0.0, 0.99, pol, torch.optim.SGD(pol.parameters(), lr=1.0), None, updates_per_iter=1,
                           maximize=maximize)
            algo.learn(buf)
            torch.cuda.synchronize()
            out[maximize] = (torch.cat([p.grad.reshape(-1) for p in pol.parameters()]).clone(), algo.last_stats.clone())
    finally:
        E.set_math("auto")
    (g0, s0), (g1, s1) = out[False], out[True]
    assert float(g0.abs().max()) > 0
    assert torch.equal(g1, -g0)
    assert torch.equal(s1[0], -s0[0]) and torch.equal(s1[1:], s0[1:])
