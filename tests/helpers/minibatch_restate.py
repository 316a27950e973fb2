"""numpy restatement of one PPO epoch's minibatch plan over a rollout sharded by whole groups (algorithms/ppo.py:147-157).

The reference flattens the valid steps of the whole rollout env-major, step-minor, draws one torch.randperm over them and
takes minibatch b = perm[b*bs : (b+1)*bs].  A shard holding envs with episode lengths `lens` owns the global valid steps
[base, base + sum(lens)).  Its plan lists, in perm order, the flat slot ids t*N + n (N = len(lens)) of the perm entries
it owns, and offsets[b] = how many of them lie in perm[0 : b*bs].  tg_minibatch_plan is pinned against this."""
import numpy as np


def ppo_minibatch_plan(perm, lens, base, batch_size):
    perm = np.asarray(perm, np.int64)
    lens = np.asarray(lens, np.int64)
    N, n_local = lens.size, int(lens.sum())
    # slot id of every local valid step, in the reference's flattening order
    env = np.repeat(np.arange(N, dtype=np.int64), lens)
    step = np.concatenate([np.arange(l, dtype=np.int64) for l in lens]) if n_local else np.zeros(0, np.int64)
    slots = step * N + env
    k = perm - base
    mine = (k >= 0) & (k < n_local)
    ids = slots[k[mine]]
    n_batches = -(-perm.size // batch_size)
    before = np.concatenate([[0], np.cumsum(mine)])                 # own entries in perm[0:i]
    offsets = before[np.minimum(np.arange(n_batches + 1, dtype=np.int64) * batch_size, perm.size)]
    return ids, offsets.astype(np.int64)


def split_groups(G, world):
    """Whole groups per rank, as RolloutManager(rank=, world_size=) shards them when G divides evenly, and an uneven
    split otherwise (the planner does not need equal shards): group ranges [g0, g1) per rank."""
    cuts = np.linspace(0, G, world + 1).round().astype(int)
    return [(int(cuts[r]), int(cuts[r + 1])) for r in range(world)]
