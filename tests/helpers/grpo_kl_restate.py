"""GRPO's objective with the KL penalty to a frozen reference policy, restated in float64 torch autograd.

    u = log pi_ref(a|s) - log pi_theta(a|s),   D = exp(u) - u - 1 >= 0   (the k3 estimator, Shao et al. 2024, eq. 4)
    J = (1/G) sum_g sum_valid [ min(rho A, clamp(rho, 1-eps, 1+eps) A) - beta D ]

It is oracle/restate.py's grpo_objective_and_grad (grpo.py:118-140) with the term grpo.py:129-134 intended; D uses
torch.expm1, because the term is evaluated where u is tiny.  With ref_logp None or beta 0 it returns exactly what
restate.grpo_objective_and_grad returns, and a sum D of 0.
"""
import numpy as np
import torch

import restate as R


def grpo_kl_objective_and_grad(obs, act_, adv, mask, weights, biases, old_weights, old_biases, cov_diag, epsilon,
                               act=R.ACT_RELU, dtype="float64", ref_logp=None, beta=0.0, old_logp=None):
    """obs [G,E,T,O], act_ [G,E,T,A], adv / mask / ref_logp [G,E,T].  `old_logp` [G,E,T], when given, stands in for
    the old policy's log-probs (the kernels' input); old_weights / old_biases are then unused.
    Returns (J, [dW...], [db...], lp, old_lp, sum D), lp / old_lp over the valid rows."""
    if (ref_logp is None or beta == 0) and old_logp is None:
        return R.grpo_objective_and_grad(obs, act_, adv, mask, weights, biases, old_weights, old_biases, cov_diag,
                                         epsilon, act=act, dtype=dtype) + (0.0,)
    td = getattr(torch, dtype)
    G = obs.shape[0]
    Ws = [torch.tensor(np.asarray(w), dtype=td, requires_grad=True) for w in weights]
    bs = [torch.tensor(np.asarray(b), dtype=td, requires_grad=True) for b in biases]
    cd = torch.tensor(np.asarray(cov_diag), dtype=td)
    sel = torch.tensor(np.asarray(mask) > 0)
    o = torch.tensor(np.asarray(obs), dtype=td)[sel]
    a = torch.tensor(np.asarray(act_), dtype=td)[sel]
    A = torch.tensor(np.asarray(adv), dtype=td)[sel]
    if old_logp is not None:
        old_lp = torch.tensor(np.asarray(old_logp), dtype=td)[sel]
    else:
        oWs = [torch.tensor(np.asarray(w), dtype=td) for w in old_weights]
        obs_ = [torch.tensor(np.asarray(b), dtype=td) for b in old_biases]
        with torch.no_grad():
            old_lp = R._torch_logp(R._torch_mlp(o, oWs, obs_, act), cd, a)
    lp = R._torch_logp(R._torch_mlp(o, Ws, bs, act), cd, a)
    ratio = torch.exp(lp - old_lp)
    D = torch.zeros((), dtype=td)
    if ref_logp is not None and beta != 0:
        u = torch.tensor(np.asarray(ref_logp), dtype=td)[sel] - lp
        D = torch.expm1(u) - u
    J = (torch.min(ratio * A, torch.clamp(ratio, 1 - epsilon, 1 + epsilon) * A).sum() - beta * D.sum()) / G
    J.backward()
    return (float(J.detach()), [w.grad.numpy().copy() for w in Ws], [b.grad.numpy().copy() for b in bs],
            lp.detach().numpy(), old_lp.numpy(), float(D.detach().sum()))
