"""Host-side mirror of algorithms/algorithm.py, grpo.py and ppo.py.

Same constructors, `learn(buffer)`, `save/load/metadata` and `old_policy`
attribute as the reference; `learn` is a short sequence of kernel launches:

  GRPO.learn (grpo.py:50-148):
      tg_advantage(GRPO)                         RTG + per-group z-score
      [tg_policy_forward_traj]                   frozen old-policy log-prob (skipped when
                                                 the rollout's own log-prob is that value)
      [tg_policy_forward_traj]                   reference-policy log-prob (ref_model, beta != 0)
      updates_per_iter x { tg_policy_grad[_ref]  ->  [NCCL allreduce]  ->  tg_adam_step }

The objective keeps the reference's sign: `J.backward(); optimizer.step()` with a
minimising optimizer descends on J (SURVEY q1) -- pass `maximize=True` to ascend.
"""
from __future__ import annotations

import copy
import os
from abc import ABC, abstractmethod

import torch

from . import _lib as L
from . import engine


class Algorithm(ABC):
    """algorithms/algorithm.py:3-36."""

    def __init__(self):
        pass

    @abstractmethod
    def learn(self):
        pass

    @abstractmethod
    def metadata(self):
        return {}

    @abstractmethod
    def save(self, path: str):
        pass

    @abstractmethod
    def load(self, path: str):
        pass


class _FlatOptimizer:
    """Applies a flat gradient to the policy's flat parameter vector.

    torch.optim.Adam with default flags (what every reference pipeline builds,
    pipelines/cartpole_pipeline_grpo.py:65) runs as ONE tg_adam_step launch whose
    moment buffers are aliased into `optimizer.state`, so `optimizer.state_dict()`
    checkpoints (grpo.py:150-160, ppo.py:207-225) keep working and
    `optimizer.load_state_dict()` (a resumed run) is picked up: state tensors that are
    not our aliases were put there by torch, so their moments are copied in and their
    step count is taken verbatim.  Any other optimizer gets `p.grad` views of the flat
    gradient and its own `step()`.
    """

    def __init__(self, optimizer, policy):
        self.opt, self.policy = optimizer, policy
        self.m = self.v = None
        self.step_count = 0
        self._steps = {}          # id(param) -> its own CPU step tensor (torch's Adam keeps one per parameter)
        self._ok_key = None
        self._ok = False
        self._comm = None         # engine.PeerComm: gradient allreduce + Adam over NVLink peer memory (world > 1)
        self._comm_tried = False

    def _fused_adam_ok(self, flat):
        groups = self.opt.param_groups
        g = groups[0] if groups else {}
        key = (type(self.opt), len(groups), id(g.get("params")), len(g.get("params", ())), flat.data_ptr(),
               flat.numel(), g.get("amsgrad"), g.get("maximize"), g.get("weight_decay"), g.get("capturable"),
               g.get("differentiable"))
        if key == self._ok_key:
            return self._ok
        ok = type(self.opt) is torch.optim.Adam and len(groups) == 1
        if ok:
            off, base = 0, flat.data_ptr()
            for p in g["params"]:                                     # parameters alias the flat vector, in order
                if p.data_ptr() != base + 4 * off:
                    ok = False
                    break
                off += p.numel()
            ok = ok and off == flat.numel()
        ok = ok and not g.get("amsgrad", False) and not g.get("maximize", False) and g.get("weight_decay", 0) == 0 \
            and not g.get("capturable", False) and not g.get("differentiable", False)
        self._ok_key, self._ok = key, ok
        return ok

    def _sync_adam_state(self, flat):
        if self.m is None or self.m.numel() != flat.numel() or self.m.device != flat.device:
            self.m, self.v = torch.zeros_like(flat), torch.zeros_like(flat)
            self._steps = {}
        off = 0
        loaded_step = None
        for p in self.opt.param_groups[0]["params"]:
            n = p.numel()
            st = self.opt.state[p]
            for key, buf in (("exp_avg", self.m), ("exp_avg_sq", self.v)):
                view = buf[off:off + n].view(p.shape)
                cur = st.get(key)
                if cur is not None and cur.data_ptr() != view.data_ptr():
                    view.copy_(cur.to(view.device, torch.float32))      # state came from load_state_dict()
                st[key] = view
            mine = self._steps.get(id(p))
            cur = st.get("step")
            if cur is not None and cur is not mine:                     # replaced by load_state_dict(): verbatim
                loaded_step = int(float(cur))
            if mine is None:
                mine = self._steps[id(p)] = torch.tensor(float(self.step_count))
            st["step"] = mine
            off += n
        if loaded_step is not None:
            self.step_count = loaded_step
            for t in self._steps.values():
                t.fill_(float(loaded_step))

    def peer_comm(self, flat):
        """The peer-memory gradient window of a sharded run (built on first use, collectively), or None: world
        size 1, an optimizer the fused Adam kernel does not cover, TG_PEER_ALLREDUCE=0, or the windows could
        not be mapped on every rank (the NCCL allreduce + tg_adam_step path is then used)."""
        if self._comm_tried:
            return self._comm if (self._comm is None or self._comm.n >= flat.numel()) else None
        self._comm_tried = True
        if _dist_world() > 1 and self._fused_adam_ok(flat) and os.environ.get("TG_PEER_ALLREDUCE", "1") != "0":
            self._comm = engine.PeerComm.try_create(flat.numel(), flat.device)
        return self._comm

    def step_allreduced(self, flat, comm):
        """Adam on the sum over ranks of the gradients the ranks wrote into their comm slots (one fused launch)."""
        self._sync_adam_state(flat)
        g = self.opt.param_groups[0]
        self.step_count += 1
        comm.allreduce_adam_step(flat, self.m, self.v, self.step_count, g["lr"], g["betas"][0], g["betas"][1], g["eps"])
        for t in self._steps.values():
            t.fill_(float(self.step_count))

    def step(self, flat, grad):
        if self._fused_adam_ok(flat):
            self._sync_adam_state(flat)
            g = self.opt.param_groups[0]
            self.step_count += 1
            engine.adam_step(flat, grad, self.m, self.v, self.step_count, g["lr"], g["betas"][0], g["betas"][1],
                             g["eps"])
            for t in self._steps.values():
                t.fill_(float(self.step_count))
            return
        off = 0
        params = [p for grp in self.opt.param_groups for p in grp["params"]]
        if sum(p.numel() for p in params) != grad.numel():
            raise L.EngineError("optimizer parameters do not match the policy's flat parameter vector")
        for p in params:
            p.grad = grad[off:off + p.numel()].view(p.shape)
            off += p.numel()
        self.opt.step()


_WORLD_OVERRIDE = None


class single_process:
    """with algorithms.single_process(): learn() treats the rollout as unsharded even though a process group is
    initialised (used to compute the single-GPU reference of a sharded run inside the same process)."""

    def __enter__(self):
        global _WORLD_OVERRIDE
        self._prev, _WORLD_OVERRIDE = _WORLD_OVERRIDE, 1
        return self

    def __exit__(self, *exc):
        global _WORLD_OVERRIDE
        _WORLD_OVERRIDE = self._prev
        return False


def _dist_world():
    if _WORLD_OVERRIDE is not None:
        return _WORLD_OVERRIDE
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size()
    return 1


def _rollout_of(buffer):
    r = getattr(buffer, "device_rollout", None)
    if r is None:
        if getattr(buffer, "group_observations", None) is None:
            raise L.EngineError("buffer holds no rollout: call buffer.sample() or buffer.store(...) first")
        from .buffers import Rollout_Buffer
        tmp = Rollout_Buffer.__new__(Rollout_Buffer)
        tmp.avg_reward = []
        Rollout_Buffer.store(tmp, buffer.group_observations, buffer.group_actions, buffer.group_rewards,
                             buffer.group_masks.sum(-1) if getattr(buffer, "group_lengths", None) is None
                             else buffer.group_lengths, buffer.group_masks)
        r = tmp.device_rollout
    return r


def _check_ref_model(ref, policy):
    """GRPO's reference policy: a Gaussian actor (or actor-critic, whose actor is used) of this package on the policy's
    device, with the policy's obs and action dims and storage of its own.  Its hidden dims, activation and covariance
    may differ from the policy's."""
    from .policies import GaussianActor_NeuralNetwork, GaussianActorCritic_NeuralNetwork
    if not isinstance(ref, (GaussianActor_NeuralNetwork, GaussianActorCritic_NeuralNetwork)):
        raise L.EngineError(f"ref_model must be a GaussianActor_NeuralNetwork or GaussianActorCritic_NeuralNetwork, "
                            f"got {type(ref).__name__}")
    if ref is policy:
        raise L.EngineError("ref_model is the policy itself: a reference that moves with the updates is no reference")
    pa, ra = policy.actor.dims, ref.actor.dims
    if (ra[0], ra[-1]) != (pa[0], pa[-1]):
        raise L.EngineError(f"ref_model maps {ra[0]} obs to {ra[-1]} actions, the policy {pa[0]} to {pa[-1]}")
    pflat, rflat = policy.flat_parameters(), ref.actor.flat_params()
    if rflat.device != pflat.device:
        raise L.EngineError(f"ref_model is on {rflat.device}, the policy on {pflat.device}")
    if rflat.untyped_storage().data_ptr() == pflat.untyped_storage().data_ptr():
        raise L.EngineError("ref_model shares its parameter storage with the policy: it would move with the updates")


class GRPO(Algorithm):
    """algorithms/grpo.py:12-168.  With a ref_model and beta != 0 the objective gains the k3 KL penalty
    -(beta / G) sum_valid (exp(u) - u - 1), u = log pi_ref(a|s) - log pi_theta(a|s) (INTEGRATION.md)."""

    def __init__(self, epsilon: float, beta: float, gamma: float, policy, optimizer, ref_model=None,
                 updates_per_iter: int = 10, *, maximize: bool = False):
        self.epsilon, self.policy, self.ref_model, self.beta = epsilon, policy, ref_model, beta
        self.gamma, self.updates_per_iter, self.optimizer = gamma, updates_per_iter, optimizer
        self.maximize = maximize
        if ref_model is not None:
            _check_ref_model(ref_model, policy)
        self.old_policy = copy.deepcopy(self.policy)                 # grpo.py:48
        self._synced_tag = policy.param_tag()                        # old_policy == policy at this tag ...
        self._old_tag = self.old_policy.param_tag()                  # ... while old_policy itself is untouched
        self._seen_loads = getattr(policy, "checkpoint_loads", 0)
        self._flat_opt = _FlatOptimizer(optimizer, policy)
        self.last_stats = None

    def _ref_actor(self):
        """(dims, activation, flat params, cov) of the reference actor, or None when the KL term is off
        (no ref_model, or beta == 0: then no reference forward runs at all)."""
        if self.ref_model is None or self.beta == 0:
            return None
        a = self.ref_model.actor
        return a.dims, a.activation_name, a.flat_params(), self.ref_model.cov_diag

    def learn(self, buffer) -> None:
        r = _rollout_of(buffer)
        pol = self.policy
        self._resync_after_checkpoint_load()
        flat = pol.flat_parameters()
        old_flat = self.old_policy.flat_parameters()
        dims, act_name, cov = pol.actor.dims, pol.actor.activation_name, pol.cov_diag
        world = _dist_world()
        G_global = r.G * world
        # grpo.py:66-74, 108-115
        adv, _ = engine.advantage(L.ADV_GRPO, r.G, r.E, r.T, self.gamma, 0.0, r.rew, r.len)
        # grpo.py:118-119: log-prob under the frozen old policy.  The rollout kernel already
        # evaluated it when the rollout was produced by weights identical to old_policy.
        cur_tag = pol.param_tag()
        if r.logp is not None and r.policy_tag == cur_tag and self._synced_tag == cur_tag \
                and self.old_policy.param_tag() == self._old_tag:
            old_logp = r.logp
        else:
            _, old_logp = engine.policy_forward_traj(dims, act_name, old_flat[:flat.numel()].contiguous(), r.obs, cov,
                                                     r.act, r.len)
        scale = (-1.0 if self.maximize else 1.0) / G_global         # grpo.py:140 (J /= group_size)
        comm = self._flat_opt.peer_comm(flat) if world > 1 else None
        ref = self._ref_actor()
        with engine.length_order(r.len, r.T):                       # lengths are fixed for all updates of this learn()
            # grpo.py:129: log pi_ref(a|s), once: the reference is frozen, so every update would see the same values
            ref_logp = None if ref is None else engine.policy_forward_traj(ref[0], ref[1], ref[2], r.obs, ref[3], r.act,
                                                                           r.len)[1]
            for _ in range(self.updates_per_iter):                  # grpo.py:106
                # the path's only collective: the gradient summed over ranks.  With the peer-memory window the kernel
                # writes its gradient into this rank's slot and ONE launch does allreduce + Adam (tg_comm.cu);
                # otherwise NCCL allreduce + tg_adam_step
                slot = comm.grad_slot()[:flat.numel()] if comm is not None else None
                grad, stats = engine.policy_grad(dims, act_name, flat, cov, r.obs, r.act, adv, old_logp, r.len,
                                                 self.epsilon, scale, out_grad=slot, ref_logp=ref_logp,
                                                 ref_scale=self.beta * scale)
                if comm is not None:
                    self._flat_opt.step_allreduced(flat, comm)      # grpo.py:143-145 on the summed gradient
                else:
                    if world > 1:
                        import torch.distributed as dist
                        dist.all_reduce(grad)
                    self._flat_opt.step(flat, grad)                 # grpo.py:143-145
                pol.bump_param_epoch()
                self.last_stats = stats
        self.old_policy.load_state_dict(self.policy.state_dict())   # grpo.py:148
        self._synced_tag = pol.param_tag()
        self._old_tag = self.old_policy.param_tag()

    def learn_streamed(self, manager, init_state=None, chunk_groups: int = 8192):
        """One whole epoch -- rollout AND learn (pipelines/pipeline.py:163-164) -- for more envs than trajectories fit
        in HBM (BASELINE configs[4]: up to 4M envs per GPU x 1000 steps x 104 B = 416 GB).

        The reference stores every trajectory (rollout_worker.py:64-68) because its GRPO.learn revisits them in
        every update (grpo.py:106-145).  Here only the initial states and the Philox seed are kept; the rollout is
        REMATERIALISED chunk by chunk (whole GRPO groups, so the group statistics of grpo.py:108-115 stay exact):

            for each update:  for each chunk of `chunk_groups` groups:
                K1 rollout of the chunk under the FROZEN old policy (deterministic: same seed, same global env
                   index -> the identical trajectories, log-probs included, in every update)
                K2 advantages of the chunk         K3 gradient of the chunk under the current weights, accumulated
            [gradient allreduce]  Adam

        One trajectory buffer of chunk size is reused.  With updates_per_iter == 1 no work is repeated.  With a
        reference policy (ref_model, beta != 0) each chunk also runs the reference forward into a chunk-sized
        log-prob buffer, once per chunk and update, because the buffer is reused.
        Equal to sample() + learn() on the same seed up to the fp32 summation order of the per-chunk gradients.
        Returns the number of valid env-steps of this rank's rollout as a 0-dim CUDA tensor (no host sync)."""
        pol = self.policy
        self._resync_after_checkpoint_load()
        flat = pol.flat_parameters()
        if self.old_policy.param_tag() != self._old_tag or self._synced_tag != pol.param_tag():
            self.old_policy.load_state_dict(pol.state_dict())      # start of an epoch: old == current (grpo.py:148)
        old_flat = self.old_policy.actor.flat_params()
        dims, act_name, cov = pol.actor.dims, pol.actor.activation_name, pol.cov_diag
        env, E = manager.env, manager.num_episodes_per_worker
        G_loc = manager.local_workers
        world = _dist_world()
        dev = flat.device
        init_state, seed = manager.next_epoch(init_state, dtype=torch.float32)
        scale = (-1.0 if self.maximize else 1.0) / (G_loc * world)
        n_valid = torch.zeros((), dtype=torch.int64, device=dev)
        ret_sum = torch.zeros((), dtype=torch.float64, device=dev)
        out = getattr(self, "_stream_out", None)
        grad_own, grad_part = torch.empty_like(flat), torch.empty_like(flat)
        comm = self._flat_opt.peer_comm(flat) if world > 1 else None
        ref = self._ref_actor()
        ref_store = None if ref is None else \
            torch.empty(env.max_steps * min(G_loc, chunk_groups) * E, dtype=torch.float32, device=dev)
        for u in range(self.updates_per_iter):
            grad_total = comm.grad_slot()[:flat.numel()] if comm is not None else grad_own
            grad_total.zero_()
            for g0 in range(0, G_loc, chunk_groups):
                g1 = min(G_loc, g0 + chunk_groups)
                n0, n1 = g0 * E, g1 * E
                s0 = init_state[:, n0:n1].contiguous()
                out = engine.rollout(env._tg_kind, env.max_steps, env.timestep, dims, act_name, old_flat, cov, s0,
                                     seed=seed, env_offset=manager.env_offset + n0, phys=getattr(env, "_tg_phys", None),
                                     out=out)
                adv, _ = engine.advantage(L.ADV_GRPO, g1 - g0, E, env.max_steps, self.gamma, 0.0, out["rew"], out["len"])
                ref_logp = None
                if ref is not None:
                    ref_logp = ref_store[:env.max_steps * (n1 - n0)].view(env.max_steps, n1 - n0)
                    engine.policy_forward_traj(ref[0], ref[1], ref[2], out["obs"], ref[3], out["act"], out["len"],
                                               out_logp=ref_logp)
                _, stats = engine.policy_grad(dims, act_name, flat, cov, out["obs"], out["act"], adv, out["logp"],
                                              out["len"], self.epsilon, scale, out_grad=grad_part, ref_logp=ref_logp,
                                              ref_scale=self.beta * scale)
                grad_total.add_(grad_part)
                if u == 0:
                    n_valid.add_(out["len"].sum())
                    ret_sum.add_(out["ret"].sum(dtype=torch.float64))
                self.last_stats = stats
            if comm is not None:
                self._flat_opt.step_allreduced(flat, comm)
            else:
                if world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(grad_total)
                self._flat_opt.step(flat, grad_total)
            pol.bump_param_epoch()
        self._stream_out = out
        self.old_policy.load_state_dict(self.policy.state_dict())   # grpo.py:148
        self._synced_tag = pol.param_tag()
        self._old_tag = self.old_policy.param_tag()
        self.last_mean_return = ret_sum / (G_loc * E)
        return n_valid

    def _resync_after_checkpoint_load(self):
        """policy.load(path) (an engine extension: the reference's GaussianActor has no load(), so its GRPO runs
        cannot resume at all) restores the weights a checkpoint holds -- the state right after a learn(), where
        old_policy had just been synchronised (grpo.py:148).  The resumed run continues like the uninterrupted one
        only if old_policy is restored with them.  Plain load_state_dict() calls keep the reference's semantics
        (old_policy untouched)."""
        loads = getattr(self.policy, "checkpoint_loads", 0)
        if loads != self._seen_loads:
            self._seen_loads = loads
            self.old_policy.load_state_dict(self.policy.state_dict())
            self._synced_tag = self.policy.param_tag()
            self._old_tag = self.old_policy.param_tag()

    def save(self, path: str) -> None:
        if L.is_checkpoint_writer():
            torch.save(self.optimizer.state_dict(), os.path.join(path, "optimizer.pth"))

    def load(self, path: str) -> None:
        """grpo.py:156-160."""
        self.optimizer.load_state_dict(torch.load(os.path.join(path, "optimizer.pth"), weights_only=True))

    def metadata(self):
        return {"algorithm": "GRPO", "epsilon": self.epsilon, "beta": self.beta,
                "updates_per_iter": self.updates_per_iter}


class PPO(Algorithm):
    """algorithms/ppo.py:8-225: full-batch updates (batch_size=None, the shipped pipelines' setting) and randperm
    minibatches (batch_size=k, the constructor's default).  Both shard over GPUs (RolloutManager(rank=, world_size=)):
    for minibatches, rank 0 draws the epoch's torch.randperm from its default CPU generator and broadcasts it, every
    rank computes the gradient of its own samples of each minibatch scaled by the global 1/len(batch), and the ranks
    sum their gradients before each Adam step -- the single-GPU minibatch step up to fp32 summation order."""

    def __init__(self, epsilon: float, policy, optimizer, ref_model, updates_per_iter: int, c1: float = 0.5,
                 kl_coeff: float = 0.5, gamma: float = 0.99, lam: float = 0.95, entropy: float = 0.01,
                 batch_size: int = 64, monte_carlo: bool = True):
        self.epsilon, self.c1, self.policy, self.ref_model = epsilon, c1, policy, ref_model
        self.updates_per_iter, self.optimizer, self.gamma, self.lam = updates_per_iter, optimizer, gamma, lam
        self.entropy, self.batch_size, self.kl_coeff, self.monte_carlo = entropy, batch_size, kl_coeff, monte_carlo
        if not hasattr(policy, "critic"):
            raise L.EngineError("PPO needs a GaussianActorCritic_NeuralNetwork policy")
        self.old_policy = copy.deepcopy(self.policy)                 # ppo.py:62
        self._flat_opt = _FlatOptimizer(optimizer, policy)
        self.last_stats = None

    def learn(self, buffer) -> None:
        world = _dist_world()
        r = _rollout_of(buffer)
        pol = self.policy
        flat = pol.flat_parameters()
        na = pol.actor.n_params()
        a_flat, c_flat = flat[:na], flat[na:]
        a_dims, c_dims, act_name, cov = pol.actor.dims, pol.critic.dims, pol.actor.activation_name, pol.cov_diag
        # ppo.py:93-94: critic values over the rollout
        values, _ = engine.policy_forward_traj(c_dims, act_name, c_flat, r.obs, None, None, r.len, want_mu=True,
                                               want_logp=False)
        values = values.view(r.T, r.N)
        mode = L.ADV_PPO_MC if self.monte_carlo else L.ADV_PPO_GAE
        # ppo.py:100-139.  The z-scores are over every valid step of the WHOLE rollout: a rank that holds
        # a shard (whole groups per GPU) computes its raw values and five additive sums, the sums are
        # allreduced (40 bytes), and every rank normalises with the global statistics (SURVEY 8e).
        adv, rtg, sums = engine.advantage_ppo_raw(mode, r.G, r.E, r.T, self.gamma, self.lam, r.rew, r.len, values)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(sums)
        engine.advantage_ppo_normalize(r.T, r.len, sums, adv, rtg)
        # ppo.py:142-143: old log-prob from self.policy at the start of learn()
        _, old_logp = engine.policy_forward_traj(a_dims, act_name, a_flat, r.obs, cov, r.act, r.len)
        n_valid = int(round(float(sums[4].item())))                 # global valid-step count (the .mean()s)
        grad = torch.empty_like(flat)
        comm = self._flat_opt.peer_comm(flat) if world > 1 else None
        if self.batch_size is not None:
            self._learn_minibatched(r, flat, grad, comm, world, na, a_dims, c_dims, act_name, cov, adv, rtg, old_logp,
                                    n_valid)
            self.old_policy.load_state_dict(self.policy.state_dict())   # ppo.py:186
            return
        with engine.length_order(r.len, r.T):
            for _ in range(self.updates_per_iter):                      # ppo.py:147 (full batch; the order of a
                # permutation does not change a mean)
                if comm is not None:
                    grad = comm.grad_slot()[:flat.numel()]               # this rank's slot of the peer-memory window
                _, stats = engine.policy_grad(a_dims, act_name, a_flat, cov, r.obs, r.act, adv, old_logp, r.len,
                                              self.epsilon, -1.0 / n_valid, self.kl_coeff / n_valid,
                                              out_grad=grad[:na])        # :160-166, 175-176
                engine.value_grad(c_dims, act_name, c_flat, r.obs, rtg, r.len, self.c1 / n_valid, out_grad=grad[na:])
                if comm is not None:
                    self._flat_opt.step_allreduced(flat, comm)          # actor + critic gradients, allreduce + Adam fused
                else:
                    if world > 1:
                        import torch.distributed as dist
                        dist.all_reduce(grad)                            # actor + critic gradients in one message
                    self._flat_opt.step(flat, grad)                     # :181-183 (entropy term has zero gradient)
                pol.bump_param_epoch()
                self.last_stats = stats
        self.old_policy.load_state_dict(self.policy.state_dict())   # ppo.py:186

    def _learn_minibatched(self, r, flat, grad, comm, world, na, a_dims, c_dims, act_name, cov, adv, rtg, old_logp,
                           n_valid):
        """ppo.py:147-183 with batch_size != None: one `torch.randperm(data_size)` per epoch from torch's
        default CPU generator (the reference's call, so a seeded run draws the same permutation), sliced
        into minibatches over the valid steps in the reference's flattening order (env-major, step-minor);
        one Adam step per minibatch.  tg_minibatch_plan turns the permutation into this rank's flat slot ids
        for the *_batch kernels, grouped by minibatch.

        Sharded, rank r owns the global valid steps [base_r, base_r + n_r) (whole groups, ranks in order).  Rank 0
        draws the permutation and broadcasts it; the other ranks leave their generators alone.  Each rank computes
        the gradient of its own samples of minibatch b with the global 1/m_b (a rank without samples contributes
        zeros) and the ranks sum their gradients, so every rank takes the same Adam step."""
        a_flat, c_flat = flat[:na], flat[na:]
        dev = flat.device
        bs = self.batch_size
        if world > 1:
            import torch.distributed as dist
            n_loc = r.len.sum(dtype=torch.int64).reshape(1)
            counts = [torch.empty_like(n_loc) for _ in range(world)]
            dist.all_gather(counts, n_loc)
            counts = [int(c.item()) for c in counts]
            if sum(counts) != n_valid:
                raise L.EngineError(f"ranks hold {counts} valid steps, {sum(counts)} in all; the advantage sums "
                                    f"counted {n_valid}")
            rank = dist.get_rank()
            base, n_local = sum(counts[:rank]), counts[rank]
        else:
            base, n_local = 0, n_valid
        for _ in range(self.updates_per_iter):
            if world > 1:
                perm = torch.randperm(n_valid).to(dev) if rank == 0 else \
                    torch.empty((n_valid,), dtype=torch.int64, device=dev)
                dist.broadcast(perm, 0)
            else:
                perm = torch.randperm(n_valid).to(dev)              # ppo.py:149
            ids, offsets = engine.minibatch_plan(perm, r.len, bs, base, n_local=n_local)
            del perm                                                # 8 bytes per valid step of the whole rollout
            offsets = offsets.tolist()
            for b in range(len(offsets) - 1):                       # ppo.py:152-153
                m = min(bs, n_valid - b * bs)                       # the reference's .mean() over the batch
                g = comm.grad_slot()[:flat.numel()] if comm is not None else grad
                if offsets[b + 1] > offsets[b]:
                    sid = ids[offsets[b]:offsets[b + 1]]
                    _, stats = engine.policy_grad_batch(a_dims, act_name, a_flat, cov, r.obs, r.act, adv, old_logp,
                                                        sid, self.epsilon, -1.0 / m, self.kl_coeff / m,
                                                        out_grad=g[:na])
                    engine.value_grad_batch(c_dims, act_name, c_flat, r.obs, rtg, sid, self.c1 / m, out_grad=g[na:])
                    self.last_stats = stats
                else:
                    g.zero_()                                       # no samples here: still part of the sum
                if comm is not None:
                    self._flat_opt.step_allreduced(flat, comm)
                else:
                    if world > 1:
                        dist.all_reduce(g)
                    self._flat_opt.step(flat, g)
                self.policy.bump_param_epoch()

    def learn_streamed(self, manager, init_state=None, chunk_groups: int = 8192):
        """One whole full-batch epoch -- rollout AND learn -- for more envs than the rollout fits in HBM, with the
        contract of GRPO.learn_streamed: only the initial states and the Philox seed are kept, the rollout is
        rematerialised chunk by chunk (`chunk_groups` whole groups) under the weights of the start of the epoch.

        PPO z-scores advantages and returns over the WHOLE rollout before the first gradient (ppo.py:127-139), so the
        epoch is one statistics pass followed by one pass per update:

            statistics:  per chunk: K1 -> critic values -> raw K2; the five float64 sums added up
                         [40-byte allreduce]; the global valid-step count read once
            each update: per chunk: K1 -> critic values -> raw K2 -> z-score with the global sums
                                    -> old log-probs -> actor + critic K3, accumulated into one gradient
                         [gradient exchange]  Adam

        The rematerialisations (rollout, values, old log-probs) use a copy of the flat parameters taken at the
        start; only the gradients see the live weights.  One chunk-sized set of buffers is reused throughout.  An
        epoch costs updates_per_iter + 1 rollouts and critic forwards, and updates_per_iter actor forwards and
        gradients.  With one chunk it trains bit-identically to sample() + learn(); with several, up to the fp32
        order in which the chunks' gradients are summed.  `last_stats` holds the actor statistics of the last update
        summed over the chunks.  The update passes z-score with the global sums of the statistics pass; the sums
        that K2 returns with each rematerialised chunk's raw advantages are a by-product and go unused.  Full batch
        only (batch_size=None): a randperm minibatch draws from every chunk.  `init_state`, when given, is this rank's
        [S, local envs] float32 / float64 tensor on the policy's device.
        Returns the number of valid env-steps of this rank's rollout as a 0-dim CUDA tensor (no host sync)."""
        if self.batch_size is not None:
            raise L.EngineError(f"PPO.learn_streamed needs batch_size=None (got {self.batch_size}): every minibatch "
                                "would need the whole rollout rematerialised")
        if chunk_groups < 1:
            raise L.EngineError(f"chunk_groups must be positive, got {chunk_groups}")
        import math
        world = _dist_world()
        pol = self.policy
        flat = pol.flat_parameters()
        na = pol.actor.n_params()
        a_flat, c_flat = flat[:na], flat[na:]
        a_dims, c_dims, act_name, cov = pol.actor.dims, pol.critic.dims, pol.actor.activation_name, pol.cov_diag
        env, E, G_loc = manager.env, manager.num_episodes_per_worker, manager.local_workers
        T, O, A = int(env.max_steps), a_dims[0], a_dims[-1]
        mode = L.ADV_PPO_MC if self.monte_carlo else L.ADV_PPO_GAE
        dev = flat.device
        kind = getattr(env, "_tg_kind", -1)
        if kind < 0:
            raise L.EngineError(f"{type(env).__name__} has no fused kernel (supported: CartPole, Pendulum, "
                                "QuadPole2D, QuadPole)")
        if init_state is not None:                                  # every chunk is a column slice of it
            want = (engine.OBS_DIM[kind], G_loc * E)
            if not (isinstance(init_state, torch.Tensor) and init_state.device == dev
                    and init_state.dtype in (torch.float32, torch.float64) and tuple(init_state.shape) == want):
                got = (f"{init_state.dtype} {tuple(init_state.shape)} on {init_state.device}"
                       if isinstance(init_state, torch.Tensor) else type(init_state).__name__)
                raise L.EngineError(f"init_state must be a float32 or float64 tensor of shape {want} (this rank's "
                                    f"envs) on {dev}, got {got}")
        init_state, seed = manager.next_epoch(init_state)
        frozen = flat.clone()                                       # the actor and critic of the start of learn()
        fa, fc = frozen[:na], frozen[na:]
        chunks = [(g0, min(G_loc, g0 + chunk_groups)) for g0 in range(0, G_loc, chunk_groups)]

        def shapes(n):
            return {"obs": (T, O, n), "act": (T, A, n), "rew": (T, n), "len": (n,), "ret": (n,), "val": (T, 1, n),
                    "adv": (T, n), "rtg": (T, n), "old_logp": (T, n)}

        n_max = (chunks[0][1] - chunks[0][0]) * E
        store = {k: torch.empty(math.prod(s), dtype=torch.int32 if k == "len" else torch.float32, device=dev)
                 for k, s in shapes(n_max).items()}

        def rematerialise(g0, g1):
            """K1, critic values and raw K2 of local groups [g0, g1) under the frozen weights -> (buffers, sums)."""
            n0, n = g0 * E, (g1 - g0) * E
            c = {k: store[k][:math.prod(s)].view(s) for k, s in shapes(n).items()}
            roll = {k: c[k] for k in ("obs", "act", "rew", "len", "ret")}
            s0 = init_state[:, n0:n0 + n].contiguous()
            out = engine.rollout(kind, T, env.timestep, a_dims, act_name, fa, cov, s0, seed=seed,
                                 env_offset=manager.env_offset + n0, phys=getattr(env, "_tg_phys", None), out=roll)
            if out is not roll:                                     # the kernels below read the chunk buffers
                raise L.EngineError("the rollout did not write the chunk buffers")
            engine.policy_forward_traj(c_dims, act_name, fc, c["obs"], None, None, c["len"], want_mu=True,
                                       want_logp=False, out_mu=c["val"])
            _, _, sums = engine.advantage_ppo_raw(mode, g1 - g0, E, T, self.gamma, self.lam, c["rew"], c["len"],
                                                  c["val"].view(T, n), out_adv=c["adv"], out_rtg=c["rtg"])
            return c, sums

        # statistics pass (ppo.py:127-139 over the whole rollout)
        n_valid = torch.zeros((), dtype=torch.int64, device=dev)
        ret_sum = torch.zeros((), dtype=torch.float64, device=dev)
        sums = None
        for g0, g1 in chunks:
            c, s = rematerialise(g0, g1)
            sums = s if sums is None else sums.add_(s)
            n_valid.add_(c["len"].sum())
            ret_sum.add_(c["ret"].sum(dtype=torch.float64))
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(sums)
        n = int(round(float(sums[4].item())))                       # global valid-step count (the .mean()s)

        grad_own = torch.empty_like(flat)
        grad_part = torch.empty_like(flat) if len(chunks) > 1 else None
        comm = self._flat_opt.peer_comm(flat) if world > 1 else None
        for _ in range(self.updates_per_iter):                      # ppo.py:147 (full batch)
            grad = comm.grad_slot()[:flat.numel()] if comm is not None else grad_own
            stats = None
            for g0, g1 in chunks:
                c, _ = rematerialise(g0, g1)
                engine.advantage_ppo_normalize(T, c["len"], sums, c["adv"], c["rtg"])
                g = grad if g0 == 0 else grad_part                  # the first chunk writes the sum's first term
                with engine.length_order(c["len"], T):              # one length order for the chunk's forward + K3s
                    engine.policy_forward_traj(a_dims, act_name, fa, c["obs"], cov, c["act"], c["len"],
                                               out_logp=c["old_logp"])
                    _, st = engine.policy_grad(a_dims, act_name, a_flat, cov, c["obs"], c["act"], c["adv"],
                                               c["old_logp"], c["len"], self.epsilon, -1.0 / n, self.kl_coeff / n,
                                               out_grad=g[:na])
                    engine.value_grad(c_dims, act_name, c_flat, c["obs"], c["rtg"], c["len"], self.c1 / n,
                                      out_grad=g[na:])
                if g0 != 0:
                    grad.add_(grad_part)
                stats = st if stats is None else stats.add_(st)
            if comm is not None:
                self._flat_opt.step_allreduced(flat, comm)
            else:
                if world > 1:
                    import torch.distributed as dist
                    dist.all_reduce(grad)
                self._flat_opt.step(flat, grad)
            pol.bump_param_epoch()
            self.last_stats = stats
        self.old_policy.load_state_dict(self.policy.state_dict())   # ppo.py:186
        self.last_mean_return = ret_sum / (G_loc * E)
        return n_valid

    def metadata(self) -> dict:
        return {"algorithm": "PPO", "epsilon": self.epsilon, "c1": self.c1, "kl_coeff": self.kl_coeff,
                "gamma": self.gamma, "lam": self.lam, "entropy": self.entropy, "batch_size": self.batch_size,
                "updates_per_iter": self.updates_per_iter}

    def save(self, path: str) -> None:
        if L.is_checkpoint_writer():
            torch.save(self.optimizer.state_dict(), os.path.join(path, "optimizer.pt"))

    def load(self, path: str) -> None:
        """ppo.py:217-225."""
        self.optimizer.load_state_dict(torch.load(os.path.join(path, "optimizer.pt"), weights_only=True))
        self.old_policy.load_state_dict(self.policy.state_dict())
