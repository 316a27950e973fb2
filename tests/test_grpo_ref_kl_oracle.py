"""The float64 restatement of GRPO's KL penalty to a reference policy (tests/helpers/grpo_kl_restate.py), pinned
without a reference fixture: its gradient against central finite differences, D >= 0 with D and its gradient exactly
0 when the reference is the policy, and beta = 0 identical to the restatement without the term.  CPU only."""
import os
import sys

import numpy as np
import pytest

import restate as R

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "helpers"))
from grpo_kl_restate import grpo_kl_objective_and_grad  # noqa: E402

EPS = 0.2


def _case(seed, act=R.ACT_TANH):
    """A small net (3 -> 5 -> 4 -> 2), 2 groups x 3 envs x 4 steps with ragged masks, and reference log-probs set
    through u = lr - lp over [-2, 2] with a band |u| < 1e-3 (both signs of u present)."""
    rng = np.random.default_rng(seed)
    dims = [3, 5, 4, 2]
    Ws = [rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i]) for i in range(3)]
    bs = [0.1 * rng.standard_normal(dims[i + 1]) for i in range(3)]
    G, E, T = 2, 3, 4
    obs = rng.standard_normal((G, E, T, 3))
    act_ = rng.standard_normal((G, E, T, 2))
    adv = rng.standard_normal((G, E, T))
    mask = (np.arange(T)[None, None, :] < rng.integers(1, T + 1, (G, E))[..., None]).astype(np.float64)
    cov = np.array([0.4, 0.7])
    lp = R._torch_logp(R._torch_mlp(*_t(obs, Ws, bs), act), _tt(cov), _tt(act_)).numpy()
    u = rng.uniform(-2, 2, (G, E, T))
    u.reshape(-1)[:4] = [3e-4, -5e-4, 2e-5, -1e-4]
    return dict(obs=obs, act_=act_, adv=adv, mask=mask, Ws=Ws, bs=bs, cov=cov, ref_logp=lp + u, u=u, act=act)


def _tt(x):
    import torch
    return torch.tensor(np.asarray(x), dtype=torch.float64)


def _t(obs, Ws, bs):
    return _tt(obs), [_tt(w) for w in Ws], [_tt(b) for b in bs]


def _J(c, Ws, bs, beta, ref_logp=None):
    return grpo_kl_objective_and_grad(c["obs"], c["act_"], c["adv"], c["mask"], Ws, bs, c["Ws"], c["bs"], c["cov"], EPS,
                                      act=c["act"], ref_logp=c["ref_logp"] if ref_logp is None else ref_logp, beta=beta)


@pytest.mark.parametrize("seed", [0, 1])
def test_gradient_matches_central_finite_differences(seed):
    """Every weight and bias: autograd against (J(p + h) - J(p - h)) / 2h in float64.  The old policy is the policy, so
    every ratio is 1 and stays inside the clip interval under the perturbation: J is smooth there (Tanh)."""
    c = _case(seed)
    m = c["mask"] > 0
    assert (c["u"][m] > 0).any() and (c["u"][m] < 0).any() and (np.abs(c["u"][m]) < 1e-3).any()
    beta, h = 0.7, 1e-6
    _, dW, db, _, _, _ = _J(c, c["Ws"], c["bs"], beta)
    worst = 0.0
    for which, grads in (("W", dW), ("b", db)):
        for li, g in enumerate(grads):
            for idx in np.ndindex(g.shape):
                Ws = [w.copy() for w in c["Ws"]]
                bs = [b.copy() for b in c["bs"]]
                p = (Ws if which == "W" else bs)[li]
                p[idx] += h
                jp = _J(c, Ws, bs, beta)[0]
                p[idx] -= 2 * h
                jm = _J(c, Ws, bs, beta)[0]
                fd = (jp - jm) / (2 * h)
                worst = max(worst, abs(fd - g[idx]))
    scale = max(np.abs(g).max() for g in dW + db)
    print(f"[grpo-kl] restatement vs central differences: max err {worst:.1e} of max |g| {scale:.2e}")
    assert worst <= 1e-7 * max(scale, 1.0)


def test_kl_term_gradient_alone_matches_finite_differences():
    """The KL term isolated (adv = 0): the surrogate contributes nothing, so this pins -(beta/G) dD/dtheta itself."""
    c = _case(3)
    c["adv"] = np.zeros_like(c["adv"])
    beta, h = 1.3, 1e-6
    J0, dW, db, _, _, sD = _J(c, c["Ws"], c["bs"], beta)
    assert J0 == pytest.approx(-beta * sD / 2, rel=1e-12)
    assert np.abs(dW[-1]).max() > 0
    for li in range(3):
        for idx in [(0, 0), (1, 1)]:
            Ws = [w.copy() for w in c["Ws"]]
            Ws[li][idx] += h
            jp = _J(c, Ws, c["bs"], beta)[0]
            Ws[li][idx] -= 2 * h
            jm = _J(c, Ws, c["bs"], beta)[0]
            assert abs((jp - jm) / (2 * h) - dW[li][idx]) <= 1e-7 * max(abs(dW[li][idx]), 1.0)


def test_divergence_is_nonnegative_and_zero_at_the_policy():
    c = _case(4, act=R.ACT_RELU)
    m = c["mask"] > 0
    u = c["u"][m]
    assert np.all(np.expm1(u) - u >= 0)
    _, _, _, lp, _, sD = _J(c, c["Ws"], c["bs"], 0.5)
    assert sD > 0
    # the reference IS the policy: u == 0 exactly on every valid row, so D and its gradient vanish exactly
    ref = np.zeros_like(c["ref_logp"])
    ref[m] = lp
    J1, dW1, db1, _, _, sD1 = _J(c, c["Ws"], c["bs"], 0.5, ref_logp=ref)
    J0, dW0, db0, _, _ = R.grpo_objective_and_grad(c["obs"], c["act_"], c["adv"], c["mask"], c["Ws"], c["bs"], c["Ws"],
                                                   c["bs"], c["cov"], EPS, act=c["act"], dtype="float64")
    assert sD1 == 0.0 and J1 == J0
    for a, b in zip(dW1 + db1, dW0 + db0):
        assert np.array_equal(a, b)


def test_beta_zero_is_the_restatement_without_the_term():
    c = _case(5, act=R.ACT_RELU)
    a = _J(c, c["Ws"], c["bs"], 0.0)
    b = R.grpo_objective_and_grad(c["obs"], c["act_"], c["adv"], c["mask"], c["Ws"], c["bs"], c["Ws"], c["bs"], c["cov"],
                                  EPS, act=c["act"], dtype="float64")
    assert a[0] == b[0] and a[5] == 0.0
    for x, y in zip(a[1] + a[2] + [a[3], a[4]], b[1] + b[2] + [b[3], b[4]]):
        assert np.array_equal(x, y)
