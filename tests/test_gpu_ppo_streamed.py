"""PPO.learn_streamed: a full-batch PPO epoch whose rollout is rematerialised chunk by chunk (whole groups) from the
initial states and the Philox seed.  With one chunk it must train bit-identically to sample() + learn(); with several,
every chunk's data must be the matching columns of the whole rollout and the weights must agree up to the fp32 order
of the per-chunk gradient sums.  Also: a second epoch, memory that does not grow with the env count, the minibatch
refusal, and 2 GPUs on both exchange paths against one GPU."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "helpers"))

pytestmark = pytest.mark.gpu
HELPER = os.path.join(HERE, "helpers", "mgpu_ppo_streamed_case.py")

T, G, E = 60, 20, 16                 # 320 envs: several 128-env tiles per step
LR, UPDATES = 3e-4, 3
# env class, obs dim, act dim, hidden widths
CASES = {
    "qp2d_w64": ("QuadPole2D", 10, 2, [64, 64]),               # TC-64 update
    "qp2d_w128": ("QuadPole2D", 10, 2, [128, 128]),            # streamed tensor-core update
    "qp2d_w128x3": ("QuadPole2D", 10, 2, [128, 128, 128]),     # the shipped architecture: FP32-pipe update
    "qp3d_w256": ("QuadPole", 20, 4, [256, 256]),
}


@pytest.fixture(scope="module")
def tg():
    import trajopt_grpo_b200 as pkg
    return pkg


def _make(tg, case, monte_carlo, updates=UPDATES, batch_size=None, groups=G, seed=11):
    env_name, O, A, hidden = CASES[case]
    torch.manual_seed(3)
    pol = tg.GaussianActorCritic_NeuralNetwork(O, A, hidden, "ReLU", 0.3)
    with torch.no_grad():                 # tilt the thrust so that episodes leave the box at different steps (ragged)
        pol.actor.network[-1].bias.add_(torch.tensor([0.5, -0.5, 0.5, -0.5][:A], device=pol.device))
    algo = tg.PPO(0.2, pol, torch.optim.Adam(pol.parameters(), lr=LR), None, updates, c1=0.5, kl_coeff=0.5,
                  gamma=0.999, lam=0.95, entropy=0.01, batch_size=batch_size, monte_carlo=monte_carlo)
    mgr = tg.RolloutManager(lambda: getattr(tg, env_name)(max_steps=T), pol, restart=False, num_workers=groups,
                            num_episodes_per_worker=E, use_multiprocessing=False, seed=seed)
    return pol, algo, mgr


def _init_states(tg, case):
    env = getattr(tg, CASES[case][0])(max_steps=T)
    s0 = env.sample_initial_states(G * E, np.random.default_rng(2))
    return torch.from_numpy(np.ascontiguousarray(s0.T)).float().cuda()


def _sample_and_learn(tg, case, monte_carlo, init):
    pol, algo, mgr = _make(tg, case, monte_carlo)
    buf = tg.Rollout_Buffer(mgr)
    buf.sample(init_state=init)
    n_valid = int(buf.device_rollout.len.sum())
    assert 0 < n_valid < G * E * T                                  # ragged
    algo.learn(buf)
    return pol, algo, buf, n_valid


@pytest.mark.parametrize("monte_carlo", [True, False], ids=["mc", "gae"])
@pytest.mark.parametrize("case", list(CASES))
def test_one_chunk_is_bit_identical_to_sample_plus_learn(tg, case, monte_carlo):
    init = _init_states(tg, case)
    pol_a, algo_a, buf, n_ref = _sample_and_learn(tg, case, monte_carlo, init)
    pol_b, algo_b, mgr_b = _make(tg, case, monte_carlo)
    n_valid = algo_b.learn_streamed(mgr_b, init_state=init, chunk_groups=G)
    assert n_valid.dim() == 0 and n_valid.is_cuda and int(n_valid) == n_ref
    assert mgr_b._epoch == 1
    assert torch.equal(pol_a.flat_parameters(), pol_b.flat_parameters())
    assert torch.equal(algo_a.last_stats, algo_b.last_stats)
    assert torch.equal(algo_b.old_policy.flat_parameters(), pol_b.flat_parameters())
    ref_ret = float(buf.avg_reward[-1])
    assert abs(float(algo_b.last_mean_return) - ref_ret) <= 1e-5 * max(1.0, abs(ref_ret))


def test_drawn_initial_states_match_sample(tg):
    """Without init_state the streamed epoch draws the initial states and the seed as sample() does."""
    pol_a, algo_a, mgr_a = _make(tg, "qp2d_w64", False)
    buf = tg.Rollout_Buffer(mgr_a)
    buf.sample()
    algo_a.learn(buf)
    pol_b, algo_b, mgr_b = _make(tg, "qp2d_w64", False)
    algo_b.learn_streamed(mgr_b, chunk_groups=G)
    assert torch.equal(pol_a.flat_parameters(), pol_b.flat_parameters())
    assert mgr_a._epoch == mgr_b._epoch == 1


class _Capture:
    """Wraps the engine calls of an epoch and keeps copies of their inputs and outputs."""

    def __init__(self, monkeypatch, engine):
        self.raw, self.pg, self.vg = [], [], []
        raw, pg, vg = engine.advantage_ppo_raw, engine.policy_grad, engine.value_grad

        def c(x):
            return x.detach().clone()

        def raw_w(mode, G_, E_, T_, gamma, lam, rew, length, values, **kw):
            adv, rtg, sums = raw(mode, G_, E_, T_, gamma, lam, rew, length, values, **kw)
            self.raw.append(dict(values=c(values), adv=c(adv), rtg=c(rtg), len=c(length)))
            return adv, rtg, sums

        def pg_w(dims, act_name, params, cov, obs, act, adv, old_logp, length, *a, **kw):
            grad, stats = pg(dims, act_name, params, cov, obs, act, adv, old_logp, length, *a, **kw)
            self.pg.append(dict(obs=c(obs), act=c(act), adv=c(adv), old_logp=c(old_logp), len=c(length),
                                stats=c(stats)))
            return grad, stats

        def vg_w(dims, act_name, params, obs, target, length, *a, **kw):
            self.vg.append(dict(rtg=c(target)))
            return vg(dims, act_name, params, obs, target, length, *a, **kw)

        monkeypatch.setattr(engine, "advantage_ppo_raw", raw_w)
        monkeypatch.setattr(engine, "policy_grad", pg_w)
        monkeypatch.setattr(engine, "value_grad", vg_w)


def _within_ulps(a, b, k):
    a, b = a.cpu().numpy(), b.cpu().numpy()
    return bool((np.abs(a - b) <= k * np.spacing(np.maximum(np.abs(a), np.abs(b)))).all())


MULTI = [(c, "auto") for c in CASES] + [("qp2d_w128", "fp32")]


@pytest.mark.parametrize("monte_carlo", [True, False], ids=["mc", "gae"])
@pytest.mark.parametrize("case,math", MULTI, ids=[f"{c}-{m}" for c, m in MULTI])
def test_chunks_agree_with_the_whole_rollout(tg, monkeypatch, case, math, monte_carlo):
    from trajopt_grpo_b200 import engine
    chunk_groups = 8                                                # chunks of 8, 8 and 4 groups
    chunks = [(g0, min(G, g0 + chunk_groups)) for g0 in range(0, G, chunk_groups)]
    engine.set_math(math)
    try:
        init = _init_states(tg, case)
        cap_a = _Capture(monkeypatch, engine)
        pol_a, algo_a, buf, n_ref = _sample_and_learn(tg, case, monte_carlo, init)
        monkeypatch.undo()
        cap_b = _Capture(monkeypatch, engine)
        pol_b, algo_b, mgr_b = _make(tg, case, monte_carlo)
        n_valid = algo_b.learn_streamed(mgr_b, init_state=init, chunk_groups=chunk_groups)
        monkeypatch.undo()
    finally:
        engine.set_math("auto")
    C = len(chunks)
    assert len(cap_a.raw) == 1 and len(cap_a.pg) == UPDATES
    assert len(cap_b.raw) == (UPDATES + 1) * C and len(cap_b.pg) == len(cap_b.vg) == UPDATES * C
    whole, whole_pg, whole_vg = cap_a.raw[0], cap_a.pg[0], cap_a.vg[0]
    mask = torch.arange(T, device="cuda")[:, None] < whole["len"][None, :]
    for i, got in enumerate(cap_b.raw):                             # statistics pass + every rematerialisation
        g0, g1 = chunks[i % C]
        cols = slice(g0 * E, g1 * E)
        m = mask[:, cols]
        assert torch.equal(got["len"], whole["len"][cols])
        assert torch.equal(got["adv"], whole["adv"][:, cols])       # raw advantages (K2 writes every row)
        assert torch.equal(got["rtg"], whole["rtg"][:, cols])
        assert torch.equal(got["values"][m], whole["values"][:, cols][m])   # K2 reads the valid rows only
    for i, (pg, vg) in enumerate(zip(cap_b.pg, cap_b.vg)):
        g0, g1 = chunks[i % C]
        cols = slice(g0 * E, g1 * E)
        m = mask[:, cols]
        assert torch.equal(pg["obs"], whole_pg["obs"][..., cols])
        assert torch.equal(pg["act"], whole_pg["act"][..., cols])
        assert torch.equal(pg["len"], whole_pg["len"][cols])
        assert torch.equal(pg["old_logp"][m], whole_pg["old_logp"][:, cols][m])   # the start-of-learn actor
        assert _within_ulps(pg["adv"], whole_pg["adv"][:, cols], 2)            # z-scored with the summed sums
        assert _within_ulps(vg["rtg"], whole_vg["rtg"][:, cols], 2)
    assert int(n_valid) == n_ref
    ref_ret = float(buf.avg_reward[-1])
    assert abs(float(algo_b.last_mean_return) - ref_ret) <= 1e-5 * max(1.0, abs(ref_ret))
    # last_stats: the last update's statistics summed over its chunks, i.e. the whole rollout's up to fp32 order
    total = cap_b.pg[-C]["stats"].clone()
    for p in cap_b.pg[-C + 1:]:
        total.add_(p["stats"])
    assert torch.equal(algo_b.last_stats, total)
    sa, sb = algo_a.last_stats.double().cpu(), algo_b.last_stats.double().cpu()
    assert sb[1] == sa[1] == n_ref
    assert abs(sb[0] - sa[0]) <= 1e-5
    assert abs(sb[2] - sa[2]) <= 1e-5 * sa[2]
    assert abs(sb[3] - sa[3]) <= max(1.0, 1e-4 * n_ref)             # a sample on the clip boundary may change sides
    # Adam's first steps move every element by ~lr; a summation-order difference in the gradient flips a step only
    # where the gradient is ~0 (the bound of test_streamed_epoch_equals_sample_plus_learn)
    d = (pol_a.flat_parameters() - pol_b.flat_parameters()).abs()
    assert float(d.max()) <= 2 * LR * UPDATES + 1e-7
    assert float((d <= 1e-6).float().mean()) >= 0.999


def test_second_epoch_continues_from_synced_old_policy(tg):
    pol, algo, mgr = _make(tg, "qp2d_w128", False)
    algo.learn_streamed(mgr, chunk_groups=7)
    assert torch.equal(algo.old_policy.flat_parameters(), pol.flat_parameters())
    w1 = pol.flat_parameters().clone()
    n2 = algo.learn_streamed(mgr, chunk_groups=7)
    assert mgr._epoch == 2 and int(n2) > 0
    assert bool(torch.isfinite(pol.flat_parameters()).all())
    assert not torch.equal(pol.flat_parameters(), w1)
    assert torch.equal(algo.old_policy.flat_parameters(), pol.flat_parameters())
    assert algo._flat_opt.step_count == 2 * UPDATES


def test_peak_memory_does_not_grow_with_env_count(tg):
    """Warmed up, with a fixed chunk size: doubling the env count adds at most 256 B per added env to the peak
    allocated by an epoch (the initial states are 40 B per env here), against 3.4 KB per env of one trajectory."""
    pol, algo, _ = _make(tg, "qp2d_w64", True, updates=2)
    O, A = 10, 2
    assert T * (O + A + 2) * 4 >= 3000                              # obs, act, rew, log-prob of one env
    mgrs = {g: tg.RolloutManager(lambda: tg.QuadPole2D(max_steps=T), pol, num_workers=g, num_episodes_per_worker=16,
                                 use_multiprocessing=False, seed=4) for g in (64, 128)}
    for m in mgrs.values():
        algo.learn_streamed(m, chunk_groups=16)
    peak = {}
    for g, m in mgrs.items():
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        algo.learn_streamed(m, chunk_groups=16)
        torch.cuda.synchronize()
        peak[g] = torch.cuda.max_memory_allocated() - base
    added_envs = (128 - 64) * 16
    assert peak[128] - peak[64] <= 256 * added_envs, peak


def test_minibatches_are_refused_before_anything_runs(tg):
    from trajopt_grpo_b200 import _lib as L
    pol, algo, mgr = _make(tg, "qp2d_w64", True, batch_size=64)
    w0 = pol.flat_parameters().clone()
    with pytest.raises(L.EngineError, match="batch_size=None"):
        algo.learn_streamed(mgr)
    assert mgr._epoch == 0
    assert torch.equal(pol.flat_parameters(), w0)


def test_wrong_init_state_is_refused_before_anything_runs(tg):
    """An init_state that is not this rank's [S, local envs] block on the policy's device raises EngineError before
    the manager's epoch advances (a narrower one would otherwise leave chunks without initial states, a wider one
    would train on other envs' states)."""
    from trajopt_grpo_b200 import _lib as L
    pol, algo, mgr = _make(tg, "qp2d_w64", True)
    init = _init_states(tg, "qp2d_w64")
    w0 = pol.flat_parameters().clone()
    wider = torch.cat([init, init[:, :E]], 1)
    for bad in (init[:, :-E], wider, init[:-1], init.cpu(), init.to(torch.float16), init.cpu().numpy()):
        with pytest.raises(L.EngineError, match="init_state must be"):
            algo.learn_streamed(mgr, init_state=bad, chunk_groups=7)
        assert mgr._epoch == 0
    assert torch.equal(pol.flat_parameters(), w0)
    algo.learn_streamed(mgr, init_state=init, chunk_groups=7)          # the right block still runs
    assert mgr._epoch == 1


def _torchrun(nproc, port, args, env=None):
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
                           "--master-addr", "127.0.0.1", "--master-port", str(port), HELPER] + args,
                          capture_output=True, text=True, timeout=900, env=dict(os.environ, **(env or {})))


@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_ranks_train_like_one_gpu(tmp_path, peer):
    """2 ranks, peer-memory allreduce + Adam (peer = "1") or NCCL + tg_adam_step ("0"): bit-identical weights on both
    ranks and the single-GPU streamed weights up to the Adam amplification of fp32 summation-order differences."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import mgpu_ppo_streamed_case as M
    ref = M.run_case(0, 1)
    ref_path = str(tmp_path / "ref.npz")
    np.savez(ref_path, w=ref["w"], n_valid=ref["n_valid"])
    r = _torchrun(2, 29551 if peer == "1" else 29552, [ref_path], {"TG_PEER_ALLREDUCE": peer})
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-4000:]
    assert ("peer-memory allreduce: True" in r.stdout) == (peer == "1"), r.stdout[-2000:]
    print(r.stdout[-2000:])
