"""CPU checks of bench.py --dump-outputs: what dump_outputs() writes for a rollout in the kernels' layout, and that
the dump of every workload's last epoch stays under 64 MB."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from trajopt_grpo_b200.rollout import DeviceRollout  # noqa: E402


class _Policy:
    def __init__(self, flat):
        self.flat = flat

    def flat_parameters(self):
        return self.flat


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_writes_the_rollout_sample_and_weights(tmp_path):
    G, E, T, O, A = 40, 10, 30, 20, 4
    N = G * E
    g = torch.Generator().manual_seed(0)
    r = DeviceRollout(obs=torch.randn(T, O, N, generator=g), act=torch.randn(T, A, N, generator=g),
                      rew=torch.randn(T, N, generator=g), logp=torch.randn(T, N, generator=g),
                      len=torch.randint(1, T + 1, (N,), dtype=torch.int32, generator=g), ret=torch.randn(N, generator=g),
                      G=G, E=E, T=T)
    flat = torch.randn(1000, generator=g)
    valid = torch.tensor(2 ** 40 + 1, dtype=torch.int64)
    bench.dump_outputs(str(tmp_path / "a"), _Policy(flat), r, torch.tensor(1.5), valid)
    got = _load(str(tmp_path / "a"))
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    idx = got["sample_env_index"].astype(np.int64)
    assert len(idx) == bench.DUMP_SAMPLE_ENVS and len(set(idx.tolist())) == len(idx) and idx.max() < N
    np.testing.assert_array_equal(got["sample_observations"], r.obs.permute(2, 0, 1).numpy()[idx])
    np.testing.assert_array_equal(got["sample_actions"], r.act.permute(2, 0, 1).numpy()[idx])
    np.testing.assert_array_equal(got["sample_rewards"], r.rew.t().numpy()[idx])
    np.testing.assert_array_equal(got["sample_log_probs"], r.logp.t().numpy()[idx])
    np.testing.assert_array_equal(got["lengths"], r.len.numpy())
    np.testing.assert_array_equal(got["policy_params"], flat.numpy())
    assert got["mean_return"] == np.float32(1.5) and got["valid_env_steps"] == 2 ** 40 + 1    # counts stay exact
    # the sample is fixed: the same envs on every run
    bench.dump_outputs(str(tmp_path / "b"), _Policy(flat), r, torch.tensor(1.5), valid)
    np.testing.assert_array_equal(_load(str(tmp_path / "b"))["sample_env_index"], got["sample_env_index"])


def test_streamed_epoch_dumps_weights_and_counts(tmp_path):
    bench.dump_outputs(str(tmp_path), _Policy(torch.ones(7)), None, torch.tensor(2.0, dtype=torch.float64),
                       torch.tensor(5))
    assert sorted(_load(str(tmp_path))) == ["mean_return", "policy_params", "valid_env_steps"]


PER_ENV = {"lengths"}                # the only arrays that grow with the number of envs
FIXED = {"policy_params", "mean_return", "valid_env_steps", "sample_env_index", "sample_observations",
         "sample_actions", "sample_rewards", "sample_log_probs"}


def test_dump_of_every_workload_fits_64_mb(tmp_path):
    """dump_outputs() on a CPU rollout of each workload's shape with the sampled number of envs and the workload's
    policy class; the per-env arrays are then scaled to the workload's env count."""
    import trajopt_grpo_b200 as tg
    for name, w in bench.WORKLOADS.items():
        if w.get("chunk_groups") is not None:
            continue                    # streamed: weights and counts only (test_streamed_epoch_dumps_weights_and_counts)
        O, A, T, N = bench.OBS[w["kind"]], bench.ACT[w["kind"]], w["T"], w["G"] * w["E"]
        n = min(N, bench.DUMP_SAMPLE_ENVS)
        assert n % w["E"] == 0, name
        r = DeviceRollout(obs=torch.zeros(T, O, n), act=torch.zeros(T, A, n), rew=torch.zeros(T, n),
                          logp=torch.zeros(T, n), len=torch.full((n,), T, dtype=torch.int32), ret=torch.zeros(n),
                          G=n // w["E"], E=w["E"], T=T)
        cls = tg.GaussianActorCritic_NeuralNetwork if w.get("algo") == "ppo" else tg.GaussianActor_NeuralNetwork
        policy = cls(O, A, w["hidden"], "ReLU", w["cov"], device="cpu")
        d = str(tmp_path / name)
        bench.dump_outputs(d, policy, r, torch.tensor(0.0), torch.tensor(N * T))
        sizes = {f[:-4]: os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)}
        assert set(sizes) == PER_ENV | FIXED, (name, sorted(sizes))
        total = sum(s * (N / n if k in PER_ENV else 1) for k, s in sizes.items())
        assert total <= 64 << 20, (name, total)
