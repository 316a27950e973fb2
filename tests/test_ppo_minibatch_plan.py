"""CPU check of the numpy restatement of the sharded PPO minibatch plan (tests/helpers/minibatch_restate.py), the
reference tg_minibatch_plan is pinned against: united over the shards of a rollout, the shards' minibatches are exactly
the reference's `rows[perm[s:s+bs]]` of the mask-flattened rollout (algorithms/ppo.py:147-157)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "helpers"))
from minibatch_restate import ppo_minibatch_plan, split_groups  # noqa: E402


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("batch_size", [1, 7, 64, 10_000])
def test_sharded_plans_unite_to_the_reference_minibatches(world, batch_size):
    rng = np.random.default_rng(100 * world + batch_size)
    G, E, T = 7, 5, 23
    lens = rng.integers(1, T + 1, (G, E))
    lens[0, 1] = 1
    lens[-1, -1] = T
    if world == 3:
        lens[2, :] = 0                                                  # a group with no valid step at all
    mask = np.arange(T)[None, None, :] < lens[..., None]
    # the reference's rows: (global env, step) of every valid step, flattened [G, E, T] env-major, step-minor
    env_of = np.broadcast_to(np.arange(G * E).reshape(G, E, 1), mask.shape)[mask]
    t_of = np.broadcast_to(np.arange(T), mask.shape)[mask]
    n = int(mask.sum())
    perm = rng.permutation(n)
    shards = split_groups(G, world)
    base = 0
    plans = []
    for g0, g1 in shards:
        l_loc = lens[g0:g1].reshape(-1)
        ids, offs = ppo_minibatch_plan(perm, l_loc, base, batch_size)
        assert offs[0] == 0 and offs[-1] == l_loc.sum() == ids.size
        N_loc = l_loc.size
        plans.append((g0 * E, N_loc, base, ids, offs))
        base += int(l_loc.sum())
    assert base == n
    n_batches = -(-n // batch_size)
    for b in range(n_batches):
        idx = perm[b * batch_size:(b + 1) * batch_size]
        ref = list(zip(env_of[idx].tolist(), t_of[idx].tolist()))
        owner = np.searchsorted(np.array([p[2] for p in plans]), idx, side="right") - 1
        for r, (env0, N_loc, _, ids, offs) in enumerate(plans):
            mine = ids[offs[b]:offs[b + 1]]
            got = list(zip((env0 + mine % N_loc).tolist(), (mine // N_loc).tolist()))
            want = [x for x, o in zip(ref, owner) if o == r]
            assert got == want, (b, r)
