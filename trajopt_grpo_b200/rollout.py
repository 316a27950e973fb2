"""Host-side mirror of rollout/rollout_manager.py and rollout/rollout_worker.py.

`RolloutManager.rollout()` keeps the reference's signature and return value
(five tensors of logical shape [G,E,T,.], rollout_manager.py:85-125) but the
G worker processes x E sequential episodes are ONE launch of the fused rollout
kernel (tg_rollout): env n = worker*E + episode.  Semantics follow the
reference's single-process path (use_multiprocessing=False), which is the only
one whose semantics are right on Linux (SURVEY section 5): current weights,
`restart` honoured (one initial state per group, shared by its E episodes).

The returned tensors are strided VIEWS of the kernels' struct-of-arrays buffers
(obs[T][O][N] -> [G,E,T,O]); nothing is copied or transposed.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib as L
from . import engine


@dataclass
class DeviceRollout:
    """One rollout in the kernels' native layout (all CUDA tensors)."""
    obs: torch.Tensor      # [T,O,N] f32
    act: torch.Tensor      # [T,A,N] f32
    rew: torch.Tensor      # [T,N]   f32
    logp: torch.Tensor     # [T,N]   f32  log pi(a|s) under the rollout weights
    len: torch.Tensor      # [N]     i32
    ret: torch.Tensor      # [N]     f32  episodic return
    G: int
    E: int
    T: int
    policy_tag: tuple = None   # policy.param_tag() of the weights that produced `logp`

    @property
    def N(self):
        return self.G * self.E

    # reference-shaped strided views ------------------------------------------------
    def group_observations(self):
        return self.obs.permute(2, 0, 1).unflatten(0, (self.G, self.E))

    def group_actions(self):
        return self.act.permute(2, 0, 1).unflatten(0, (self.G, self.E))

    def group_rewards(self):
        return self.rew.t().unflatten(0, (self.G, self.E))

    def group_lengths(self):
        # the reference stores the int lengths in a float tensor (rollout_manager.py:89, SURVEY q16)
        return self.len.to(torch.float32).view(self.G, self.E)

    def group_masks(self):
        m = (torch.arange(self.T, device=self.len.device)[:, None] < self.len[None, :]).to(torch.float32)
        return m.t().unflatten(0, (self.G, self.E))


class RolloutWorker:
    """rollout/rollout_worker.py:4-84: one worker = one GRPO group of E episodes.
    Kept for API compatibility; it runs its group through the same fused kernel."""

    def __init__(self, worker_id: int, env, policy, episodes_completed):
        self.worker_id, self.env, self.policy = worker_id, env, policy
        self.episodes_completed = episodes_completed
        self._rng = np.random.default_rng()

    def run_episodes(self, num_episodes: int = 5, restart: bool = False):
        roll = _device_rollout(self.env, self.policy, 1, num_episodes, restart, self._rng,
                               seed=int(self._rng.integers(0, 2 ** 63 - 1)))
        self.episodes_completed[self.worker_id] = num_episodes
        return (roll.group_observations()[0], roll.group_actions()[0], roll.group_rewards()[0],
                roll.len.view(-1).clone(), roll.group_masks()[0])


def _device_rollout(env, policy, G, E, restart, rng, seed, precision="f32", init_state=None, noise=None,
                    env_offset=0, device=None, out=None) -> DeviceRollout:
    kind = getattr(env, "_tg_kind", -1)
    if kind < 0:
        raise L.EngineError(f"{type(env).__name__} has no fused kernel (supported: CartPole, Pendulum, "
                            "QuadPole2D, QuadPole)")
    if not hasattr(policy, "actor"):
        raise L.EngineError("the fused rollout needs a GaussianActor(Critic)_NeuralNetwork policy")
    flat = policy.actor.flat_params()
    dev = flat.device if device is None else torch.device(device)
    N = G * E
    if init_state is None:
        if restart:
            # one reset() per worker, every episode restarts from it (rollout_worker.py:31,70-71)
            s0 = np.repeat(env.sample_initial_states(G, rng), E, axis=0)
        else:
            s0 = env.sample_initial_states(N, rng)
        dtype = torch.float64 if precision == "f64" else torch.float32
        host = torch.from_numpy(np.ascontiguousarray(s0.T)).to(dtype).pin_memory()
        init_state = host.to(dev, non_blocking=True)
    out = engine.rollout(kind, env.max_steps, env.timestep, policy.actor.dims, policy.actor.activation_name, flat,
                         policy.cov_diag, init_state, noise=noise, seed=seed, env_offset=env_offset,
                         phys=getattr(env, "_tg_phys", None), out=out)
    tag = policy.param_tag() if hasattr(policy, "param_tag") else None
    return DeviceRollout(out["obs"], out["act"], out["rew"], out["logp"], out["len"], out["ret"], G, E,
                         int(env.max_steps), tag)


def plan_shard(num_workers: int, group_size: int, rank: int, world_size: int):
    """Whole GRPO groups per GPU (SURVEY 8e): rank r owns the contiguous block of
    `num_workers / world_size` groups; returns (local groups, first global env index)."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise L.EngineError(f"bad rank/world_size {rank}/{world_size}")
    if num_workers % world_size != 0:
        raise L.EngineError(f"num_workers={num_workers} must be divisible by world_size={world_size} "
                            "(whole GRPO groups per GPU)")
    g_local = num_workers // world_size
    return g_local, rank * g_local * group_size


def shard_initial_states(env, num_workers: int, group_size: int, restart: bool, rng, rank: int, world_size: int):
    """Every rank draws the SAME global initial states from the same generator state and
    keeps its block, so a sharded rollout equals the matching slice of the single-GPU one.
    Returns [local envs, S] float64."""
    g_local, first = plan_shard(num_workers, group_size, rank, world_size)
    if restart:
        s0 = np.repeat(env.sample_initial_states(num_workers, rng), group_size, axis=0)
    else:
        s0 = env.sample_initial_states(num_workers * group_size, rng)
    return s0[first:first + g_local * group_size]


class RolloutManager:
    """rollout/rollout_manager.py:22-133."""

    def __init__(self, env_fn: callable, policy, worker_class=RolloutWorker, restart=False, num_workers: int = 4,
                 num_episodes_per_worker: int = 5, use_multiprocessing: bool = True, *, seed: int = None,
                 precision: str = "f32", rank: int = 0, world_size: int = 1, reuse_buffers: bool = False):
        self.env_fn, self.worker_class, self.policy = env_fn, worker_class, policy
        self.restart = restart
        self.num_workers = num_workers
        self.num_episodes_per_worker = num_episodes_per_worker
        # accepted and ignored: there are no worker processes, the kernel is the worker pool
        self.use_multiprocessing = use_multiprocessing
        self.env = env_fn()
        self.obs_dim = self.env.observation_space.shape[0]
        self.act_dim = self.env.action_space.shape[0]
        self.max_steps = self.env.max_steps
        self.episodes_completed = [0] * num_workers      # no workers to poll: stays zero (rollout_manager.py:52)
        self.precision = precision
        # multi-GPU: this rank owns a contiguous block of whole groups
        self.rank, self.world_size = rank, world_size
        self.local_workers, self.env_offset = plan_shard(num_workers, num_episodes_per_worker, rank, world_size)
        self._seed = self._resolve_seed(seed, world_size)
        self._rng = np.random.default_rng(self._seed)
        self._epoch = 0
        self.last: DeviceRollout | None = None
        # reuse_buffers: every rollout overwrites ONE set of trajectory buffers instead of allocating a fresh
        # one (a cfg-4 shard is 57 GB); tensors returned by an earlier rollout()/sample() then alias the new data
        self.reuse_buffers = reuse_buffers
        self._out = None

    @staticmethod
    def _resolve_seed(seed, world_size: int) -> int:
        """One 64-bit seed for the initial-state generator and the Philox stream.  Sharded runs rely on every
        rank drawing the SAME global initial states and noise stream (shard_initial_states), so with
        seed=None rank 0's OS-entropy seed is broadcast; without a process group that cannot work."""
        if seed is not None:
            return int(np.random.SeedSequence(seed).generate_state(1, np.uint64)[0])
        own = int(np.random.SeedSequence().generate_state(1, np.uint64)[0])
        if world_size == 1:
            return own
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            raise L.EngineError("RolloutManager(world_size > 1, seed=None) needs an initialised torch.distributed "
                                "process group to share rank 0's seed; pass an explicit seed otherwise")
        box = [own]
        dist.broadcast_object_list(box, src=0)
        return int(box[0])

    def print_progress(self):  # rollout_manager.py:63-83: nothing to poll, a rollout is one launch
        pass

    def next_epoch(self, init_state=None, dtype=None):
        """Starts the next epoch: returns (init_state [S, local envs] on the policy's device, Philox seed) and advances
        the epoch counter.  Without `init_state` this rank's block of the global initial states is drawn from the
        manager's generator (float64 when precision == "f64", else float32, unless `dtype` says otherwise).  Every
        rollout of an epoch -- rollout_device() or a streamed epoch -- takes its inputs from here, so the same seed
        gives the same trajectories either way."""
        if init_state is None:
            blk = shard_initial_states(self.env, self.num_workers, self.num_episodes_per_worker, self.restart,
                                       self._rng, self.rank, self.world_size)
            if dtype is None:
                dtype = torch.float64 if self.precision == "f64" else torch.float32
            dev = self.policy.actor.flat_params().device                 # the policy's device, not the current one
            init_state = torch.from_numpy(np.ascontiguousarray(blk.T)).to(dtype).pin_memory().to(dev, non_blocking=True)
        seed = (self._seed + 0x9E3779B97F4A7C15 * (self._epoch + 1)) & (2 ** 64 - 1)
        self._epoch += 1
        return init_state, seed

    def rollout_device(self, init_state=None, noise=None) -> DeviceRollout:
        """The fast path: launch the fused kernel for this rank's groups and return
        the struct-of-arrays result without materialising masks."""
        G, E = self.local_workers, self.num_episodes_per_worker
        init_state, seed = self.next_epoch(init_state)
        self.last = _device_rollout(self.env, self.policy, G, E, self.restart, self._rng, seed, self.precision,
                                    init_state=init_state, noise=noise, env_offset=self.env_offset,
                                    out=self._out if self.reuse_buffers else None)
        if self.reuse_buffers:
            r = self.last
            self._out = {"obs": r.obs, "act": r.act, "rew": r.rew, "logp": r.logp, "len": r.len, "ret": r.ret}
        return self.last

    def rollout(self):
        """rollout_manager.py:85-125 -> (obs [G,E,T,O], act [G,E,T,A], rew [G,E,T], len [G,E], mask [G,E,T])."""
        r = self.rollout_device()
        return r.group_observations(), r.group_actions(), r.group_rewards(), r.group_lengths(), r.group_masks()

    def shutdown(self):  # rollout_manager.py:127-133: no processes to join
        pass
