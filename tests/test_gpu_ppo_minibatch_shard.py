"""Minibatched PPO over a rollout sharded by whole groups: the planner kernel (tg_minibatch_plan) against its numpy
restatement, its behaviour on a perm that is not a permutation, a sharded epoch emulated rank by rank on one GPU
against the single-rollout minibatch gradients, and PPO.learn on 2 and 3 GPUs against the single-GPU run and the
reference's fixture."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "helpers"))
from minibatch_restate import ppo_minibatch_plan, split_groups  # noqa: E402

pytestmark = pytest.mark.gpu
HELPER = os.path.join(HERE, "helpers", "mgpu_ppo_minibatch_case.py")


@pytest.fixture(scope="module")
def E():
    from trajopt_grpo_b200 import engine
    return engine


def _lens(rng, N, T, kind):
    if kind == "ones":
        return np.ones(N, np.int32)
    if kind == "full":
        return np.full(N, T, np.int32)
    return rng.integers(1, T + 1, N).astype(np.int32)


def _old_world1_ids(perm_d, length):
    """The searchsorted translation the single-GPU minibatch path used before the planner."""
    lens = length.to(torch.int64)
    csum = torch.cumsum(lens, 0)
    row0 = csum - lens
    n_of = torch.searchsorted(csum, perm_d, right=True)
    return ((perm_d - row0[n_of]) * length.numel() + n_of).contiguous()


# (G envs-per-group E, T, lengths, batch sizes): batch 1, a non-divisor, exactly n_total, larger than n_total
PLAN_CASES = [
    ("ragged", 10, 7, 13, "ragged", [1, 5, None, "over"]),
    ("len1", 6, 5, 9, "ones", [1, 4, None, "over"]),
    ("lenT", 6, 5, 9, "full", [7, None, "over"]),
    ("N70", 14, 5, 11, "ragged", [1, 3, 64, None, "over"]),     # N = 70 envs: partial 128-wide tiles
    ("3e6", 1500, 8, 500, "ragged", [4096, 100_003, 65_536]),   # ~3e6 valid steps, boundaries inside 4096-entry chunks
]


@pytest.mark.parametrize("name,G,Eg,T,lk,sizes", PLAN_CASES, ids=[c[0] for c in PLAN_CASES])
def test_plan_matches_restatement_exactly(E, name, G, Eg, T, lk, sizes):
    rng = np.random.default_rng(len(name) * 7 + G)
    lens = _lens(rng, G * Eg, T, lk)
    n = int(lens.sum())
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(G))
    perm_d = perm.cuda()
    perm_np = perm.numpy()
    for world in (1, 2, 3):
        base = 0
        for g0, g1 in split_groups(G, world):
            l_loc = lens[g0 * Eg:g1 * Eg]
            ln = torch.from_numpy(l_loc).cuda()
            for bs in sizes:
                bs = n if bs is None else (n + 5 if bs == "over" else bs)
                ids, offs = E.minibatch_plan(perm_d, ln, bs, base)
                ref_ids, ref_offs = ppo_minibatch_plan(perm_np, l_loc, base, bs)
                assert np.array_equal(offs.numpy(), ref_offs), (world, g0, bs)
                assert np.array_equal(ids.cpu().numpy(), ref_ids), (world, g0, bs)
                if world == 1:
                    assert torch.equal(ids, _old_world1_ids(perm_d, ln))
            base += int(l_loc.sum())


def test_plan_of_a_perm_that_is_not_a_permutation(E, monkeypatch):
    """Duplicates put more entries in a shard than it has valid steps: the planner writes nothing past out_ids[max_ids],
    out_offsets still counts every entry, and engine.minibatch_plan raises."""
    from test_gpu_guard_bands import GuardedTorch
    from trajopt_grpo_b200 import _lib as L
    rng = np.random.default_rng(5)
    N, T, bs = 70, 9, 11
    lens = rng.integers(1, T + 1, N).astype(np.int32)
    n_local = int(lens.sum())
    base = 37
    perm = rng.permutation(n_local + 80).astype(np.int64)
    perm[perm >= base + n_local] = base + 3                       # every out-of-shard entry above it lands in it
    ref_ids, ref_offs = ppo_minibatch_plan(perm, lens, base, bs)
    assert ref_offs[-1] > n_local
    guard = GuardedTorch()
    monkeypatch.setattr(E, "torch", guard)
    E._ws_cache.clear()
    try:
        ln = torch.from_numpy(lens).cuda()
        perm_d = torch.from_numpy(perm).cuda()
        with pytest.raises(L.EngineError, match="not a permutation"):
            E.minibatch_plan(perm_d, ln, bs, base)
        # the raw entry point: offsets report the overflow, the ids that fit are the first max_ids of the plan
        lib = L.load()
        row0 = torch.from_numpy(np.cumsum(lens, dtype=np.int64) - lens).cuda()
        nb = -(-perm.size // bs)
        ids = guard.empty((n_local,), dtype=torch.int64, device="cuda")
        offs = guard.empty((nb + 1,), dtype=torch.int64, device="cuda")
        ws = guard.empty((lib.tg_minibatch_plan_workspace_bytes(perm.size),), dtype=torch.uint8, device="cuda")
        rc = lib.tg_minibatch_plan(L.ctx(), N, L.ptr(ln), L.ptr(row0), L.ptr(perm_d), perm.size, bs, base, n_local,
                                   n_local, L.ptr(ids), L.ptr(offs), L.ptr(ws), L.stream_ptr())
        L.check(rc, "tg_minibatch_plan")
        assert np.array_equal(offs.cpu().numpy(), ref_offs)
        assert np.array_equal(ids.cpu().numpy(), ref_ids[:n_local])
        bad = guard.check()
    finally:
        E._ws_cache.clear()
    assert not bad, f"guard bands overwritten: {bad}"


def test_ppo_shard_case_writes_inside_its_buffers(monkeypatch):
    """The guard-band check of tests/test_gpu_guard_bands.py over the planner + batch-gradient case."""
    from test_gpu_guard_bands import GuardedTorch, _cases
    from trajopt_grpo_b200 import engine
    guard = GuardedTorch()
    monkeypatch.setattr(engine, "torch", guard)
    engine._ws_cache.clear()
    try:
        _cases()["ppo_shard"]()
        bad = guard.check()
    finally:
        engine._ws_cache.clear()
    assert guard.allocs
    assert not bad, f"guard bands overwritten: {bad}"


def _flat(Ws, bs):
    return np.concatenate([np.concatenate([w.reshape(-1), b]) for w, b in zip(Ws, bs)])


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("mode_name", ["mc", "gae"])
@pytest.mark.parametrize("width", [32, 128])
def test_sharded_epoch_emulated_on_one_gpu(E, world, mode_name, width):
    """Every minibatch of one epoch: the float64 sum over the emulated ranks of their partial gradients (their own
    samples, global 1/m scale) equals the minibatch gradient of the whole rollout within 2e-5 of max|g|."""
    from trajopt_grpo_b200 import _lib as L
    rng = np.random.default_rng(world * 10 + width)
    G, Eg, T, O, A = 7, 6, 16, 10, 2
    N = G * Eg
    a_dims, c_dims = [O, width, width, A], [O, width, width, 1]
    mk = lambda dims: torch.from_numpy(_flat(
        [(rng.standard_normal((dims[i + 1], dims[i])) / np.sqrt(dims[i])).astype(np.float32) for i in range(3)],
        [(0.1 * rng.standard_normal(dims[i + 1])).astype(np.float32) for i in range(3)])).cuda()
    a_flat, c_flat = mk(a_dims), mk(c_dims)
    lens = rng.integers(1, T + 1, N).astype(np.int32)
    mask = np.arange(T)[:, None] < lens[None, :]
    obs = (rng.standard_normal((T, O, N)) * mask[:, None, :]).astype(np.float32)
    act = (rng.standard_normal((T, A, N)) * mask[:, None, :]).astype(np.float32)
    rew = (rng.standard_normal((T, N)) * mask).astype(np.float32)
    mode = L.ADV_PPO_MC if mode_name == "mc" else L.ADV_PPO_GAE
    cov, eps, c1, kl = [0.4, 0.4], 0.2, 0.5, 0.5
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()

    def shard(e0, e1):
        o, a, r, ln = (dev(x[..., e0:e1]) for x in (obs, act, rew, lens))
        vals, _ = E.policy_forward_traj(c_dims, "ReLU", c_flat, o, None, None, ln, want_mu=True, want_logp=False)
        adv, rtg, sums = E.advantage_ppo_raw(mode, (e1 - e0) // Eg, Eg, T, 0.99, 0.95, r, ln, vals.view(T, -1))
        return dict(o=o, a=a, ln=ln, adv=adv, rtg=rtg, sums=sums)

    full = shard(0, N)
    ranks = [shard(g0 * Eg, g1 * Eg) for g0, g1 in split_groups(G, world)]
    s_sum = sum(s["sums"] for s in ranks)
    n = int(lens.sum())
    for s in [full] + ranks:
        E.advantage_ppo_normalize(T, s["ln"], s_sum, s["adv"], s["rtg"])
        _, s["olp"] = E.policy_forward_traj(a_dims, "ReLU", a_flat, s["o"], cov, s["a"], s["ln"])

    def grad(s, sid, m):
        ga, _ = E.policy_grad_batch(a_dims, "ReLU", a_flat, cov, s["o"], s["a"], s["adv"], s["olp"], sid, eps,
                                    -1.0 / m, kl / m)
        gc, _ = E.value_grad_batch(c_dims, "ReLU", c_flat, s["o"], s["rtg"], sid, c1 / m)
        return torch.cat([ga, gc]).double()

    bs = 3                                                          # small enough that some rank holds none of a minibatch
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(world)).cuda()
    ids_f, offs_f = E.minibatch_plan(perm, full["ln"], bs, 0)
    base = 0
    for s in ranks:
        s["ids"], s["offs"] = E.minibatch_plan(perm, s["ln"], bs, base)
        base += int(s["ln"].sum())
    empty_seen = 0
    for b in range(len(offs_f) - 1):
        m = min(bs, n - b * bs)
        g_full = grad(full, ids_f[offs_f[b]:offs_f[b + 1]], m)
        g_sum = torch.zeros_like(g_full)
        for s in ranks:
            lo, hi = int(s["offs"][b]), int(s["offs"][b + 1])
            if hi > lo:
                g_sum += grad(s, s["ids"][lo:hi], m)
            else:
                empty_seen += 1
        err = (g_sum - g_full).abs().max().item()
        assert err <= 2e-5 * g_full.abs().max().item() + 1e-7, (b, err)
    assert empty_seen > 0                                           # some rank had no sample of some minibatch


def _torchrun(nproc, port, args, env=None):
    return subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc),
                           "--master-addr", "127.0.0.1", "--master-port", str(port), HELPER] + args,
                          capture_output=True, text=True, timeout=900, env=dict(os.environ, **(env or {})))


@pytest.mark.parametrize("peer", ["1", "0"])
def test_two_ranks_train_like_one_gpu(tmp_path, peer):
    """2 ranks, peer-memory allreduce + Adam (peer = "1") or NCCL + tg_adam_step ("0"), batch sizes 64 and 3, two updates:
    bit-identical weights on both ranks, the single-GPU step count, and the single-GPU weights up to the Adam
    amplification of fp32 summation-order differences."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import mgpu_ppo_minibatch_case as M
    ref = {f"bs{bs}": M.run_case(0, 1, bs) for bs in M.BATCH_SIZES}
    ref_path = str(tmp_path / "ref.npz")
    np.savez(ref_path, **{f"{k}_{f}": v[f] for k, v in ref.items() for f in ("w", "steps")})
    r = _torchrun(2, 29541 if peer == "1" else 29542, ["pair", ref_path], {"TG_PEER_ALLREDUCE": peer})
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-4000:]
    assert ("peer-memory allreduce: True" in r.stdout) == (peer == "1"), r.stdout[-2000:]
    print(r.stdout[-2000:])


def test_three_ranks_match_the_reference_fixture(golden_dir):
    """ppo_minibatch_quadpole2d.npz (batch 64, two epochs, G = 3 groups of 273 / 323 / 258 valid steps) with one group
    per rank: the post-Adam weights of the unmodified reference at the single-GPU test's tolerance."""
    if torch.cuda.device_count() < 3:
        pytest.skip("needs 3 GPUs")
    r = _torchrun(3, 29543, ["fixture", os.path.join(golden_dir, "ppo_minibatch_quadpole2d.npz")])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-4000:]
    print(r.stdout[-2000:])
