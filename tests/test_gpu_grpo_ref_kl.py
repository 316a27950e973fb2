"""GRPO's KL penalty to a frozen reference policy (GRPO(ref_model=..., beta=...)) against the float64 restatement
(tests/helpers/grpo_kl_restate.py, pinned by central differences in tests/test_grpo_ref_kl_oracle.py).

  K3 + KL        tg_policy_grad_ref on every built tensor-core (obs, act) instance at widths 64, 128, 256 and on
                 FP32-only shapes, ReLU and Tanh, both signs of scale; u = ref_logp - lp over [-2, 2] with a band of
                 |u| < 1e-3 (asserted); gradient and all 5 statistics
  NULL ref       tg_policy_grad_ref(ref_logp = NULL) is bit-identical to tg_policy_grad and writes 4 statistics
  GRPO.learn     ref_model at widths 64 / 128 / 256, 2 updates, a reference with its own width and covariance, against
                 the restatement + restate.adam_step; maximize=True is the exact negation; beta = 0 changes nothing
  learn_streamed one chunk bit-identical to sample() + learn(), several chunks within the streamed-epoch bound
  refusals, guard bands around every buffer of the new call, 2 GPUs on both exchange paths

Every kernel-level case runs on the FP32 pipe and on the 3xTF32 tensor cores; measured errors print next to their
bounds ([grpo-kl]).
"""
import ctypes as C
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import restate as R
from test_gpu_baseline_shapes import GRAD_TOL_F64, _adam_close, _load_actor, _make_buffer
from test_gpu_ppo_tensor_core import _flat, _kink_free, _mmul, _policy, _ragged_lengths, _rollout_case

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "helpers"))
from grpo_kl_restate import grpo_kl_objective_and_grad  # noqa: E402

pytestmark = pytest.mark.gpu

EPS = 0.2
MODES = ("fp32", "3xtf32")
ACT_FN = {"ReLU": R.ACT_RELU, "Tanh": R.ACT_TANH}
INSTANCES = [(3, 1), (5, 1), (10, 2), (20, 4)]
BETA = 0.04


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.fixture(scope="module")
def E():
    from trajopt_grpo_b200 import engine
    return engine


@pytest.fixture(scope="module")
def tg():
    import trajopt_grpo_b200 as pkg
    return pkg


# ----------------------------------------------------------------------------
# 1. K3 with the KL term against float64
# ----------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _k3_case(dims, act_name, small_u=False):
    """[T, ., N] inputs: ratios set through old_logp over [0.6, 1.5] (none within 1e-3 of 1 +- eps), advantages of both
    signs, and reference log-probs set through u = ref_logp - lp64 uniform over [-2, 2], 10 % of them over
    [-1e-3, 1e-3].  300 envs (a partial last tile), ragged lengths."""
    N, T = 300, 9
    O, A = dims[0], dims[-1]

    def draw(rng):
        ln = _ragged_lengths(rng, N, T)
        mask = np.arange(T)[:, None] < ln[None, :]
        obs = rng.standard_normal((T, O, N)).astype(np.float32)
        return obs.transpose(0, 2, 1)[mask], obs, ln, mask

    rng, Ws, bs, (_, obs, ln, mask) = _kink_free(list(dims), act_name, 77 * O + sum(dims[1:-1]) + len(dims)
                                                 + (5 if act_name == "Tanh" else 0), draw)
    cov = np.full(A, 0.4, np.float32)
    rows = obs.transpose(0, 2, 1)                                          # [T, N, O]
    mu = _mmul(rows.reshape(-1, O), Ws, bs, act_name).reshape(T, N, A)
    act = (mu + np.sqrt(cov.astype(np.float64)) * rng.standard_normal((T, N, A))).astype(np.float32)
    lp64 = R.gaussian_log_prob(mu, cov, act, np.float64)
    r = rng.uniform(0.6, 1.5, (T, N))
    r = np.where((np.abs(r - (1 - EPS)) < 1e-3) | (np.abs(r - (1 + EPS)) < 1e-3), r + 5e-3, r)
    old_logp = (lp64 - np.log(r)).astype(np.float32)
    u = rng.uniform(-2.0, 2.0, (T, N))
    small = rng.random((T, N)) < 0.1
    u[small] = rng.uniform(-1e-3, 1e-3, small.sum())
    if small_u:
        u = rng.choice([-1.0, 1.0], (T, N)) * rng.uniform(1e-4, 1e-3, (T, N))
    ref_logp = (lp64 + u).astype(np.float32)
    adv = rng.normal(0.4, 1.0, (T, N)).astype(np.float32)
    uv = (ref_logp.astype(np.float64) - lp64)[mask]
    assert small_u or ((uv > 1e-3).mean() > 0.3 and (uv < -1e-3).mean() > 0.3)
    assert ((np.abs(uv) < 1e-3) & (uv > 0)).sum() > 20 and ((np.abs(uv) < 1e-3) & (uv < 0)).sum() > 20
    return dict(dims=list(dims), Ws=Ws, bs=bs, cov=cov, obs=obs, act=act, adv=adv, old_logp=old_logp, ref_logp=ref_logp,
                ln=ln, mask=mask, rows=rows)


def _restated(c, act_name, scale):
    """The kernel's objective scale * (sum min(...) - beta sum D) and its gradient, float64 (G = 1: a plain sum)."""
    J, dW, db, lp, _, sD = grpo_kl_objective_and_grad(
        c["rows"][None], c["act"][None], c["adv"][None], c["mask"][None], c["Ws"], c["bs"], None, None, c["cov"], EPS,
        act=ACT_FN[act_name], ref_logp=c["ref_logp"][None], beta=BETA, old_logp=c["old_logp"][None])
    g = scale * np.concatenate([np.concatenate([w.reshape(-1), b.reshape(-1)]) for w, b in zip(dW, db)])
    r = np.exp(lp - c["old_logp"][c["mask"]].astype(np.float64))
    return scale * J, g, sD, r.sum(), int(((r < 1 - EPS) | (r > 1 + EPS)).sum())


# Measured on B200 (1000 W): max |g - g_float64| / max |g_float64| 1.1e-6 on the FP32 pipe and 7.8e-6 on 3xTF32
# (5-256-256-1), inside the global bounds; the objective and the sum of D within 3.3e-7.
K3_SHAPES = [((O, W, W, A), act, modes) for O, A in INSTANCES for W in (64, 128, 256) for act in ("ReLU", "Tanh")
             for modes in [MODES]]
K3_SHAPES += [((10, 64, 64, 64, 2), "ReLU", ("fp32",)), ((5, 33, 33, 1), "Tanh", ("fp32",)),
              ((20, 96, 96, 4), "ReLU", ("fp32",))]


@pytest.mark.parametrize("sign", [1.0, -1.0], ids=["min", "max"])
@pytest.mark.parametrize("dims,act_name,modes", K3_SHAPES,
                         ids=["-".join(map(str, d)) + f"-{a}" for d, a, _ in K3_SHAPES])
def test_policy_grad_ref_matches_float64(E, dims, act_name, modes, sign):
    c = _k3_case(tuple(dims), act_name)
    n = int(c["mask"].sum())
    scale = sign / 5
    J, ref, sD, rsum, nclip = _restated(c, act_name, scale)
    args = (dev(c["obs"]), dev(c["act"].transpose(0, 2, 1)), dev(c["adv"]), dev(c["old_logp"]), dev(c["ln"]))
    params = dev(_flat(c["Ws"], c["bs"]))
    out = {}
    try:
        for mode in modes:
            E.set_math(mode)
            g, st = E.policy_grad(c["dims"], act_name, params, c["cov"].tolist(), *args, EPS, scale,
                                  ref_logp=dev(c["ref_logp"]), ref_scale=BETA * scale)
            torch.cuda.synchronize()
            out[mode] = (g.cpu().numpy(), st.cpu().numpy().astype(np.float64))
    finally:
        E.set_math("auto")
    for mode, (g, st) in out.items():
        tol = GRAD_TOL_F64[mode]
        err = float(np.abs(g - ref).max() / np.abs(ref).max())
        e_obj, e_rat, e_kl = abs(st[0] - J) / abs(J), abs(st[2] - rsum) / rsum, abs(st[4] - sD) / sD
        print(f"[grpo-kl] K3 {'-'.join(map(str, dims)):14s} {act_name:4s} {'+' if sign > 0 else '-'}scale {mode:6s} "
              f"grad {err:.2e} (<= {tol:.0e})  objective {e_obj:.1e}  sum ratio {e_rat:.1e}  sum D {e_kl:.1e} (<= 1e-5)")
        assert st.shape == (5,)
        assert err <= tol, (mode, err)
        assert int(st[1]) == n and int(st[3]) == nclip, (mode, st, nclip)
        assert e_obj <= 1e-5 and e_rat <= 1e-5 and e_kl <= 1e-5, (mode, st, J, rsum, sD)


@pytest.mark.parametrize("dims,act_name,modes", [((10, 64, 64, 2), "ReLU", MODES), ((3, 128, 128, 1), "Tanh", MODES),
                                                  ((20, 256, 256, 4), "ReLU", MODES), ((5, 33, 33, 1), "Tanh", ("fp32",))])
def test_small_u_divergence(E, dims, act_name, modes):
    """Every |u| in [1e-4, 1e-3]: D ~ u^2 / 2 is 5e-9 .. 5e-7, where expf(u) - 1 (rounding error ~6e-8) would be wrong by
    up to ~50 % per sample and expm1f is not.  The sum of D is checked to 1e-3; the fp32 rounding of the log-probs
    themselves (~5e-7 absolute) moves it by ~3e-5."""
    c = _k3_case(tuple(dims), act_name, small_u=True)
    scale = 1.0 / 5
    J, ref, sD, _, _ = _restated(c, act_name, scale)
    args = (dev(c["obs"]), dev(c["act"].transpose(0, 2, 1)), dev(c["adv"]), dev(c["old_logp"]), dev(c["ln"]))
    try:
        for mode in modes:
            E.set_math(mode)
            g, st = E.policy_grad(c["dims"], act_name, dev(_flat(c["Ws"], c["bs"])), c["cov"].tolist(), *args, EPS, scale,
                                  ref_logp=dev(c["ref_logp"]), ref_scale=BETA * scale)
            g, st = g.cpu().numpy(), st.cpu().numpy().astype(np.float64)
            err, e_kl = float(np.abs(g - ref).max() / np.abs(ref).max()), abs(st[4] - sD) / sD
            print(f"[grpo-kl] small u {'-'.join(map(str, dims)):14s} {mode:6s} grad {err:.2e} (<= {GRAD_TOL_F64[mode]:.0e})"
                  f"  sum D {e_kl:.1e} (<= 1e-3)")
            assert err <= GRAD_TOL_F64[mode] and e_kl <= 1e-3, (mode, err, e_kl)
    finally:
        E.set_math("auto")


# ----------------------------------------------------------------------------
# 2. ref_logp = NULL is tg_policy_grad
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("dims,mode", [((10, 64, 64, 2), "auto"), ((20, 128, 128, 4), "auto"), ((3, 256, 256, 1), "auto"),
                                       ((10, 64, 64, 2), "fp32"), ((5, 33, 33, 1), "fp32")])
def test_null_ref_is_bit_identical_to_policy_grad(E, dims, mode):
    from trajopt_grpo_b200 import _lib as L
    c = _k3_case(tuple(dims), "ReLU" if dims[1] != 33 else "Tanh")
    act_name = "ReLU" if dims[1] != 33 else "Tanh"
    lib = L.load()
    T, O, N = c["obs"].shape
    obs, act, adv, olp, ln = (dev(c["obs"]), dev(c["act"].transpose(0, 2, 1)), dev(c["adv"]), dev(c["old_logp"]),
                              dev(c["ln"]))
    params = dev(_flat(c["Ws"], c["bs"]))
    mcfg = L.mlp_cfg(list(dims), act_name)
    outs = []
    try:
        E.set_math(mode)
        ctx = L.ctx(0)
        ws = torch.empty(lib.tg_policy_grad_workspace_bytes(ctx, C.byref(mcfg)), dtype=torch.uint8, device="cuda")
        for fn in ("plain", "null"):
            g = torch.full_like(params, 7.0)
            st = torch.full((6,), 123.0, device="cuda")
            common = (ctx, C.byref(mcfg), N, T, L.ptr(obs), L.ptr(act), L.ptr(adv), L.ptr(olp))
            tail = (L.ptr(ln), L.ptr(params), L.cov_array(c["cov"].tolist()), EPS, 0.2, 0.01)
            if fn == "plain":
                rc = lib.tg_policy_grad(*common, *tail, L.ptr(g), L.ptr(st), L.ptr(ws), L.stream_ptr())
            else:
                rc = lib.tg_policy_grad_ref(*common, None, *tail, 0.5, L.ptr(g), L.ptr(st), L.ptr(ws), L.stream_ptr())
            L.check(rc, fn)
            torch.cuda.synchronize()
            outs.append((g, st))
    finally:
        E.set_math("auto")
    (g0, s0), (g1, s1) = outs
    assert float(g0.abs().max()) > 0
    assert torch.equal(g0, g1) and torch.equal(s0, s1)
    assert torch.all(s1[4:] == 123.0)                    # exactly 4 statistics written


# ----------------------------------------------------------------------------
# 3-4. GRPO.learn with ref_model
# ----------------------------------------------------------------------------
REF_HIDDEN = {64: [128, 128], 128: [64, 64], 256: [128, 128]}
LR = 3e-3                  # large enough that the second update clips some ratios


def _grpo_case(kind, W, seed):
    c = _rollout_case(kind, W, seed)
    rng = np.random.default_rng(seed + 1000)
    c["rWs"], c["rbs"] = _policy(rng, [c["O"]] + REF_HIDDEN[W] + [c["A"]])
    return c


def _ref_logp64(c, cov_ref):
    t = lambda x: torch.tensor(np.asarray(x), dtype=torch.float64)
    with torch.no_grad():
        mu = R._torch_mlp(t(c["obs"]), [t(w) for w in c["rWs"]], [t(b) for b in c["rbs"]], R.ACT_RELU)
        return R._torch_logp(mu, t(cov_ref), t(c["act"])).numpy()


def _grpo_algo(tg, c, beta, ref=True, maximize=False, opt="adam", updates=2):
    pol = tg.GaussianActor_NeuralNetwork(c["O"], c["A"], c["hidden"], "ReLU", 0.5)
    _load_actor(pol.actor, c["Ws"], c["bs"])
    rm = None
    if ref:
        rm = tg.GaussianActor_NeuralNetwork(c["O"], c["A"], REF_HIDDEN[c["hidden"][0]], "ReLU", 0.8)
        _load_actor(rm.actor, c["rWs"], c["rbs"])
    o = torch.optim.Adam(pol.parameters(), lr=LR) if opt == "adam" else torch.optim.SGD(pol.parameters(), lr=1.0)
    return pol, tg.GRPO(EPS, beta, 0.99, pol, o, rm, updates_per_iter=updates, maximize=maximize)


@pytest.mark.parametrize("kind,W", [(1, 64), (2, 128), (3, 256)])
def test_grpo_learn_with_ref_model_matches_restatement(tg, kind, W):
    c = _grpo_case(kind, W, 70 + kind)
    buf = _make_buffer(tg, c)
    cov, cov_ref = np.full(c["A"], 0.5), np.full(c["A"], 0.8)
    ref_logp = _ref_logp64(c, cov_ref)
    _, adv = R.grpo_advantage(c["rew"], c["mask"], 0.99)
    pol, algo = _grpo_algo(tg, c, BETA)
    algo.learn(buf)
    torch.cuda.synchronize()
    # the chain: 2 updates, old log-probs of the start weights, Adam in float32
    ref = [p.astype(np.float32) for wb in zip(c["Ws"], c["bs"]) for p in wb]
    m = [np.zeros_like(p) for p in ref]
    v = [np.zeros_like(p) for p in ref]
    x = c["obs"][c["mask"] > 0]
    margin, n_clip, sD = np.inf, 0, 0.0
    for step in (1, 2):
        margin = min(margin, R.kink_margin(x, ref[0::2], ref[1::2]))
        _, dW, db, lp, olp, sD = grpo_kl_objective_and_grad(c["obs"], c["act"], adv, c["mask"], ref[0::2], ref[1::2],
                                                            c["Ws"], c["bs"], cov, EPS, ref_logp=ref_logp, beta=BETA)
        r = np.exp(lp - olp)
        n_clip = int(((r < 1 - EPS) | (r > 1 + EPS)).sum())
        ref = R.adam_step(ref, [g for wb in zip(dW, db) for g in wb], m, v, step, LR)
    assert n_clip > 0                                  # the second update clips
    st = algo.last_stats.cpu().numpy().astype(np.float64)
    e_kl = abs(st[4] - sD) / sD
    print(f"[grpo-kl] GRPO.learn kind {kind} W {W}: clipped {int(st[3])}/{int(st[1])}  sum D {e_kl:.1e} (<= 1e-4)  "
          f"kink margin {margin:.1e}")
    # a ratio within fp32 noise of 1 +- eps may land on either side
    assert st.shape == (5,) and abs(int(st[3]) - n_clip) <= max(2, n_clip // 100) and e_kl <= 1e-4
    for i, (p, r_) in enumerate(zip(pol.parameters(), ref)):
        _adam_close(p.detach().cpu().numpy(), r_, margin, LR, 2, f"W {W} p{i}")


@pytest.mark.parametrize("mode", ["fp32", "auto"])
def test_maximize_negates_and_beta_zero_changes_nothing(tg, E, mode):
    c = _grpo_case(3, 256, 90)
    buf = _make_buffer(tg, c)
    try:
        E.set_math(mode)
        out = {}
        for maximize in (False, True):
            pol, algo = _grpo_algo(tg, c, BETA, maximize=maximize, opt="sgd", updates=1)
            algo.learn(buf)
            torch.cuda.synchronize()
            out[maximize] = (torch.cat([p.grad.reshape(-1) for p in pol.parameters()]).clone(), algo.last_stats.clone())
        (g0, s0), (g1, s1) = out[False], out[True]
        assert float(g0.abs().max()) > 0 and float(s0[4]) > 0
        assert torch.equal(g1, -g0)
        assert torch.equal(s1[0], -s0[0]) and torch.equal(s1[1:], s0[1:])
        w = {}
        for ref in (False, True):
            pol, algo = _grpo_algo(tg, c, 0.0, ref=ref)
            algo.learn(buf)
            w[ref] = (pol.flat_parameters().clone(), algo.last_stats.clone())
        assert torch.equal(w[False][0], w[True][0]) and torch.equal(w[False][1], w[True][1])
        assert w[True][1].shape == (4,)
    finally:
        E.set_math("auto")


# ----------------------------------------------------------------------------
# 5. GRPO.learn_streamed with ref_model
# ----------------------------------------------------------------------------
def _streamed_setup(tg, updates=2):
    torch.manual_seed(5)
    pol = tg.GaussianActor_NeuralNetwork(20, 4, [256, 256], "ReLU", 0.3)
    rm = tg.GaussianActor_NeuralNetwork(20, 4, [128, 128], "Tanh", 0.5)
    algo = tg.GRPO(0.2, BETA, 0.999, pol, torch.optim.Adam(pol.parameters(), lr=3e-4), rm, updates_per_iter=updates,
                   maximize=True)
    mgr = tg.RolloutManager(lambda: tg.QuadPole(max_steps=60), pol, restart=True, num_workers=12,
                            num_episodes_per_worker=16, use_multiprocessing=False, seed=11)
    return pol, algo, mgr


def test_learn_streamed_with_ref_model(tg):
    rng = np.random.default_rng(2)
    env = tg.QuadPole(max_steps=60)
    init = torch.from_numpy(np.ascontiguousarray(np.repeat(env.sample_initial_states(12, rng), 16, axis=0).T)).float().cuda()
    pol_a, algo_a, mgr_a = _streamed_setup(tg)
    buf = tg.Rollout_Buffer(mgr_a)
    buf.sample(init_state=init)
    algo_a.learn(buf)
    pol_b, algo_b, mgr_b = _streamed_setup(tg)
    algo_b.learn_streamed(mgr_b, init_state=init, chunk_groups=12)              # one chunk
    assert torch.equal(pol_a.flat_parameters(), pol_b.flat_parameters())
    assert torch.equal(algo_a.last_stats, algo_b.last_stats) and algo_b.last_stats.shape == (5,)
    pol_c, algo_c, mgr_c = _streamed_setup(tg)
    algo_c.learn_streamed(mgr_c, init_state=init, chunk_groups=5)               # chunks of 5, 5 and 2 groups
    d = (pol_a.flat_parameters() - pol_c.flat_parameters()).abs()
    print(f"[grpo-kl] learn_streamed 3 chunks vs sample()+learn(): max {float(d.max()):.1e} (<= {2 * 3e-4 * 2 + 1e-7:.1e}),"
          f" within 1e-6: {float((d <= 1e-6).float().mean()):.4f} (>= 0.999)")
    assert float(d.max()) <= 2 * 3e-4 * 2 + 1e-7
    assert float((d <= 1e-6).float().mean()) >= 0.999


# ----------------------------------------------------------------------------
# 6. refusals
# ----------------------------------------------------------------------------
def test_refusals_raise_at_construction(tg):
    from trajopt_grpo_b200 import _lib as L
    pol = tg.GaussianActor_NeuralNetwork(10, 2, [64, 64], "ReLU", 0.5)
    mgr = tg.RolloutManager(lambda: tg.QuadPole2D(max_steps=10), pol, restart=True, num_workers=2,
                            num_episodes_per_worker=4, use_multiprocessing=False, seed=1)
    opt = torch.optim.Adam(pol.parameters(), lr=1e-3)
    shared = tg.GaussianActor_NeuralNetwork(10, 2, [64, 64], "ReLU", 0.5)
    shared.actor.bind_flat(pol.flat_parameters())
    for bad, what in ((pol, "policy itself"), (tg.GaussianActor_NeuralNetwork(10, 1, [64, 64]), "obs"),
                      (tg.GaussianActor_NeuralNetwork(5, 2, [64, 64]), "obs"), (object(), "GaussianActor"),
                      (pol.actor, "GaussianActor"), (shared, "storage")):
        with pytest.raises(L.EngineError, match=what):
            tg.GRPO(EPS, BETA, 0.99, pol, opt, bad)
    assert mgr._epoch == 0
    ac = tg.GaussianActorCritic_NeuralNetwork(10, 2, [32], "Tanh", 0.2)             # an actor-critic: its actor is used
    tg.GRPO(EPS, BETA, 0.99, pol, opt, ac)


# ----------------------------------------------------------------------------
# 7. guard bands around every buffer of the new call
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("dims,mode", [((10, 64, 64, 2), "auto"), ((20, 256, 256, 4), "auto"), ((5, 33, 33, 1), "fp32")])
def test_guard_bands(E, monkeypatch, dims, mode):
    from test_gpu_guard_bands import GuardedTorch
    act_name = "ReLU" if dims[1] != 33 else "Tanh"
    c = _k3_case(tuple(dims), act_name)
    guard = GuardedTorch()
    monkeypatch.setattr(E, "torch", guard)
    E._ws_cache.clear()

    def g(x, dtype):
        t = guard.empty(x.shape, dtype=dtype, device="cuda")
        t.copy_(torch.from_numpy(np.ascontiguousarray(x)))
        return t

    try:
        E.set_math(mode)
        obs, act = g(c["obs"], torch.float32), g(c["act"].transpose(0, 2, 1), torch.float32)
        adv, olp, rlp = g(c["adv"], torch.float32), g(c["old_logp"], torch.float32), g(c["ref_logp"], torch.float32)
        ln, params = g(c["ln"], torch.int32), g(_flat(c["Ws"], c["bs"]), torch.float32)
        out_lp = guard.empty(c["adv"].shape, dtype=torch.float32, device="cuda")
        E.policy_forward_traj(list(dims), act_name, params, obs, c["cov"].tolist(), act, ln, out_logp=out_lp)
        _, st = E.policy_grad(list(dims), act_name, params, c["cov"].tolist(), obs, act, adv, olp, ln, EPS, 0.2,
                              ref_logp=rlp, ref_scale=0.2 * BETA)
        torch.cuda.synchronize()
        bad = guard.check()
    finally:
        E.set_math("auto")
        E._ws_cache.clear()
    assert float(st[4]) > 0
    assert not bad, f"guard bands overwritten: {bad}"


# ----------------------------------------------------------------------------
# 8. 2 GPUs
# ----------------------------------------------------------------------------
@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_ranks_reproduce_single_gpu(tmp_path, peer):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    helper = os.path.join(HERE, "helpers", "mgpu_grpo_ref_case.py")
    import mgpu_grpo_ref_case
    ref = mgpu_grpo_ref_case.run_case(0, 1)
    ref.pop("_peer")
    ref_path = str(tmp_path / "ref.npz")
    np.savez(ref_path, **ref)
    env = dict(os.environ, TG_PEER_ALLREDUCE=peer)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29561" if peer == "1" else "29562", helper,
                        ref_path], capture_output=True, text=True, timeout=600, env=env)
    print(r.stdout[-1500:])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert ("peer-memory allreduce: True" in r.stdout) == (peer == "1"), r.stdout[-2000:]
