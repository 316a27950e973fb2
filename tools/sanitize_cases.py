"""Small-shape exercise of every kernel family for compute-sanitizer (SURVEY section 5 hygiene):

    compute-sanitizer --tool memcheck  python tools/sanitize_cases.py
    compute-sanitizer --tool racecheck python tools/sanitize_cases.py
    compute-sanitizer --tool synccheck python tools/sanitize_cases.py

Each case goes through the C ABI (trajopt_grpo_b200.engine) at shapes that leave a partial last tile and ragged
episode lengths; `--only a,b` restricts the families.  The logs are kept under profiles/.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from trajopt_grpo_b200 import engine as E  # noqa: E402

OBS = {0: 5, 1: 3, 2: 10, 3: 20}
ACT = {0: 1, 1: 1, 2: 2, 3: 4}


def policy(rng, dims):
    parts = []
    for i in range(len(dims) - 1):
        parts.append((rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32).reshape(-1))
        parts.append((0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32))
    return torch.from_numpy(np.concatenate(parts)).cuda()


def init_state(kind, N):
    s = torch.zeros(OBS[kind], N, device="cuda")
    if kind == 0:
        s[3] = 1.0
    elif kind == 1:
        s[1] = -1.0
    elif kind == 2:
        s[5] = 1.0; s[8] = -1.0
    else:
        s[6] = 1.0; s[13] = 1.0
    return s


def case_rollout_update(kind, hidden, N, T, math):
    rng = np.random.default_rng(0)
    dims = [OBS[kind]] + hidden + [ACT[kind]]
    p = policy(rng, dims)
    cov = [0.3] * ACT[kind]
    E.set_math(math)
    try:
        out = E.rollout(kind, T, 0.02 if kind != 1 else 0.05, dims, "ReLU", p, cov, init_state(kind, N), seed=3)
        Eg = 5
        G = N // Eg
        n = G * Eg
        sl = lambda x: x[..., :n].contiguous()
        adv, _ = E.advantage(0, G, Eg, T, 0.99, 0.0, sl(out["rew"]), sl(out["len"]))
        g, st = E.policy_grad(dims, "ReLU", p, cov, sl(out["obs"]), sl(out["act"]), adv, sl(out["logp"]), sl(out["len"]),
                              0.2, 1.0 / G)
        _, lp = E.policy_forward_traj(dims, "ReLU", p, sl(out["obs"]), cov, sl(out["act"]), sl(out["len"]))
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        E.adam_step(p, g, m, v, 1, 3e-4)
        torch.cuda.synchronize()
        assert bool(torch.isfinite(g).all())
    finally:
        E.set_math("auto")


def case_ppo(N=70, T=9):
    rng = np.random.default_rng(1)
    a_dims, c_dims = [10, 128, 128, 2], [10, 128, 128, 1]
    pa, pc = policy(rng, a_dims), policy(rng, c_dims)
    out = E.rollout(2, T, 0.02, a_dims, "ReLU", pa, [0.3, 0.3], init_state(2, N), seed=5)
    vals, _ = E.policy_forward_traj(c_dims, "ReLU", pc, out["obs"], None, None, out["len"], want_mu=True, want_logp=False)
    for mode in (1, 2):
        adv, rtg = E.advantage(mode, N // 7, 7, T, 0.99, 0.95, out["rew"], out["len"], vals.view(T, N))
    gc, _ = E.value_grad(c_dims, "ReLU", pc, out["obs"], rtg, out["len"], 0.5 / N)
    sid = torch.arange(0, 3 * N, 2, device="cuda", dtype=torch.int64)
    ok = (sid // N) < out["len"][sid % N]
    sid = sid[ok].contiguous()
    E.policy_grad_batch(a_dims, "ReLU", pa, [0.3, 0.3], out["obs"], out["act"], adv, out["logp"], sid, 0.2, -1.0 / sid.numel())
    E.value_grad_batch(c_dims, "ReLU", pc, out["obs"], rtg, sid, 0.5 / sid.numel())
    E.export_trajectory(out["obs"], out["act"], out["len"])
    torch.cuda.synchronize()


def case_ppo_shard(T=11):
    """Minibatch plans of a ragged rollout (N = 70, lengths 1..T) split into 1, 2 and 3 emulated ranks of uneven
    size, then the batch gradients on every planned minibatch of each rank."""
    rng = np.random.default_rng(2)
    a_dims, c_dims = [10, 32, 32, 2], [10, 32, 32, 1]
    pa, pc = policy(rng, a_dims), policy(rng, c_dims)
    N = 70
    lens = torch.from_numpy(rng.integers(1, T + 1, N).astype(np.int32)).cuda()
    obs = torch.randn(T, 10, N, device="cuda")
    act = torch.randn(T, 2, N, device="cuda")
    adv, olp, rtg = (torch.randn(T, N, device="cuda") for _ in range(3))
    n = int(lens.sum())
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(3)).cuda()
    for cuts in ((0, N), (0, 33, N), (0, 5, 48, N)):
        base = 0
        for e0, e1 in zip(cuts[:-1], cuts[1:]):
            ln = lens[e0:e1].contiguous()
            ids, offs = E.minibatch_plan(perm, ln, 37, base)
            base += int(ln.sum())
            o, a = obs[..., e0:e1].contiguous(), act[..., e0:e1].contiguous()
            ad, lp, rt = (x[:, e0:e1].contiguous() for x in (adv, olp, rtg))
            for b in range(len(offs) - 1):
                sid = ids[offs[b]:offs[b + 1]]
                if sid.numel():
                    E.policy_grad_batch(a_dims, "ReLU", pa, [0.3, 0.3], o, a, ad, lp, sid, 0.2, -1.0 / 37, 0.5 / 37)
                    E.value_grad_batch(c_dims, "ReLU", pc, o, rt, sid, 0.5 / 37)
    torch.cuda.synchronize()


def case_grpo_ref(N=200, T=6):
    """GRPO's KL term: the reference forward and tg_policy_grad_ref on the three K3 families."""
    rng = np.random.default_rng(4)
    for kind, hidden, math in ((1, [64, 64], "3xtf32"), (3, [256, 256], "3xtf32"), (1, [40, 24], "fp32")):
        dims = [OBS[kind]] + hidden + [ACT[kind]]
        p, pr = policy(rng, dims), policy(rng, [OBS[kind]] + [32, 32] + [ACT[kind]])
        cov = [0.3] * ACT[kind]
        E.set_math(math)
        try:
            out = E.rollout(kind, T, 0.02 if kind != 1 else 0.05, dims, "ReLU", p, cov, init_state(kind, N), seed=3)
            G = N // 5
            adv, _ = E.advantage(0, G, 5, T, 0.99, 0.0, out["rew"], out["len"])
            _, rlp = E.policy_forward_traj([OBS[kind], 32, 32, ACT[kind]], "Tanh", pr, out["obs"], [0.5] * ACT[kind],
                                           out["act"], out["len"])
            g, st = E.policy_grad(dims, "ReLU", p, cov, out["obs"], out["act"], adv, out["logp"], out["len"], 0.2,
                                  -1.0 / G, ref_logp=rlp, ref_scale=-0.04 / G)
            torch.cuda.synchronize()
            assert bool(torch.isfinite(g).all()) and float(st[4]) >= 0
        finally:
            E.set_math("auto")


def case_env():
    for kind in range(4):
        s = init_state(kind, 33).double()
        a = torch.zeros(ACT[kind], 33, device="cuda")
        E.env_step(kind, 50, 0.02, s, a)
        E.env_dynamics(kind, 0.02, s, a + 1.0)
    E.quadrotor12_dynamics(torch.zeros(12, 9, device="cuda", dtype=torch.float64), torch.ones(4, 9, device="cuda", dtype=torch.float64))
    E.noise_fill(1, 100, 3, 4)
    torch.cuda.synchronize()


CASES = {
    "fp32_small": lambda: case_rollout_update(1, [40, 24], 70, 7, "fp32"),
    "fp32_deep128": lambda: case_rollout_update(0, [128, 128, 128, 128], 70, 5, "auto"),
    "tc64": lambda: case_rollout_update(1, [64, 64], 200, 6, "3xtf32"),
    "tc128": lambda: case_rollout_update(2, [128, 128], 200, 6, "3xtf32"),
    "tc256": lambda: case_rollout_update(3, [256, 256], 200, 6, "3xtf32"),
    "ppo": case_ppo,
    "ppo_shard": case_ppo_shard,
    "grpo_ref": case_grpo_ref,
    "env": case_env,
}

if __name__ == "__main__":
    only = None
    if "--only" in sys.argv:
        only = set(sys.argv[sys.argv.index("--only") + 1].split(","))
    for name, fn in CASES.items():
        if only is None or name in only:
            fn()
            print("case", name, "ok", flush=True)
