#!/usr/bin/env python
"""Benchmark of the rollout-and-update hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one training epoch of the reference's loop (pipelines/pipeline.py:163-164):
`buffer.sample()` (policy-in-the-loop rollout of every env for the full horizon) followed by
`algorithm.learn(buffer)` (RTG + group-relative advantages + `updates_per_iter` clipped-surrogate
updates with Adam).

Default workload = the per-GPU shard of BASELINE.json configs[3], the north-star configuration and the
largest one that fits a single GPU: 3-D quadrotor QuadPole GRPO, 524,288 envs x 1000 steps per GPU
(8 GPUs = the full 4,194,304 envs), group size 64, MLP 20-256-256-4, exploration covariance 0.3 and Adam
3e-4 as the reference's quadrotor pipeline sets them (pipelines/quadpole_pipeline_ppo.py:54-80),
`updates_per_iter` = 1 as the reference's only shipped GRPO pipeline (cartpole_pipeline_grpo.py:72).
Weak scaling: every rank runs the full per-GPU shape with whole groups; the only collective on the data
path is the gradient allreduce.  The policy starts from a stabilising linear feedback embedded in the ReLU
network (bench_assets/quadpole_lqr_gain.json, designed by oracle/make_start_policy.py) so that >= 99 % of
the envs stay alive for the horizon under the full exploration noise; `value` counts VALID steps only and
slot-steps/s and the valid fraction are printed beside it.

`value`  : valid env-steps/s of the whole job with the initial states already in HBM.
`e2e`    : the same through the reference-facing host API (`Rollout_Buffer.sample()` / `GRPO.learn()`) with
           HOST initial states copied H2D from pinned memory every step and the episode lengths + mean
           return read back D2H.
Extra keys: K1/K2/K3 times, rooflines, GRPO updates/s, `other_configs` (BASELINE configs[1], Pendulum),
`rank_weights_identical` (all ranks hold bit-identical weights after the timed epochs), the CPU baseline
measured on this box, clocks under load.

`--dump-outputs DIR` writes what the last timed epoch of the device-resident arm computed, as rank 0 holds it,
to DIR/<name>.npy (float32 / float64, under 64 MB): the policy parameters after the update, the mean return,
the episode length of every env and the full trajectories of a fixed, seeded sample of envs.  Initial states,
noise seeds and start weights are seeded, so two builds run with the same arguments can be compared array by
array.  With several GPUs everything but the weights (identical on every rank) covers rank 0's envs only: the mean
return, the valid env-step count, the lengths and the sample are those of its shard, so compare dumps taken with
the same --gpus.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE configs[3] per GPU (8 x 524,288 = 4,194,304 envs x 1000 steps, group 64); 57 GB of trajectory per GPU
    "quadpole_cfg4": dict(kind=3, cls="QuadPole", T=1000, E=64, G=8192, hidden=[256, 256], cov=0.3, gamma=0.999, eps=0.2,
                          lr=3e-4, updates=1, start="lqr",
                          desc="3D QuadPole GRPO, 524,288 envs per GPU x 1000 steps (BASELINE configs[3]: 4,194,304 envs on "
                               "8 GPUs), group 64, MLP 256x256, cov 0.3, stabilising start policy"),
    # BASELINE configs[1]
    "pendulum": dict(kind=1, cls="Pendulum", T=200, E=16, G=4096, hidden=[64, 64], cov=0.5, gamma=0.99, eps=0.2,
                     lr=5e-4, updates=5, desc="Pendulum GRPO, 65,536 envs x 200-step horizon, group size 16, MLP 64x64"),
    # BASELINE configs[0]
    "cartpole": dict(kind=0, cls="CartPole", T=500, E=10, G=10, hidden=[128, 128, 128, 128], cov=0.5, gamma=0.5,
                     eps=0.15, lr=3e-4, updates=1, restart=False, desc="CartPole GRPO (scripts/cartpole_nn_grpo.py defaults)"),
    # BASELINE configs[2] at FULL size on one GPU: 1,048,576 envs x 500 steps (29 GB of trajectory), MLP 128x128; cov 0.5, lr 2e-4,
    # gamma 0.99 as pipelines/quadpole2d_pipeline_ppo.py:54-80 sets them; stabilising start on the vehicle coordinates
    "quadpole2d_cfg3": dict(kind=2, cls="QuadPole2D", T=500, E=16, G=65536, hidden=[128, 128], cov=0.5, gamma=0.99,
                            eps=0.2, lr=2e-4, updates=1, start="lqr",
                            desc="QuadPole2D GRPO, 1,048,576 envs x 500 steps (BASELINE configs[2] at full size), group 16, "
                                 "MLP 128x128, cov 0.5, stabilising start policy"),
    # the same with PPO (actor + critic, full batch, Monte-Carlo returns, c1 0.5, kl 0.5: the shipped pipeline's setting; 2 of
    # its 24 updates per epoch to keep the run short) at a quarter of the size
    "quadpole2d_ppo": dict(kind=2, cls="QuadPole2D", T=500, E=16, G=16384, hidden=[128, 128], cov=0.5, gamma=0.99,
                           eps=0.2, lr=2e-4, updates=2, start="lqr", algo="ppo",
                           desc="QuadPole2D PPO (actor + critic 128x128, full batch), 262,144 envs x 500 steps, cov 0.5, "
                                "stabilising start policy"),
    # hover-biased start (output layer zeroed, cov 1e-4): ragged episodes (valid fraction 0.5) for kernel measurements
    "quadpole2d": dict(kind=2, cls="QuadPole2D", T=500, E=16, G=16384, hidden=[128, 128], cov=1e-4, gamma=0.99,
                       eps=0.2, lr=2e-7, updates=2, start="hover",
                       desc="QuadPole2D GRPO, 262,144 envs x 500 steps, group 16, MLP 128x128, hover-biased start (ragged)"),
    # one eighth of the cfg-4 shard (kernel profiling runs)
    "quadpole": dict(kind=3, cls="QuadPole", T=1000, E=64, G=1024, hidden=[256, 256], cov=0.3, gamma=0.999, eps=0.2,
                     lr=3e-4, updates=1, start="lqr",
                     desc="3D QuadPole GRPO, 65,536 envs x 1000 steps, group 64, MLP 256x256, cov 0.3, stabilising start"),
    # BASELINE configs[4]: 1M..32M envs over 1..8 GPUs -- more envs per GPU than trajectories fit in HBM, run as
    # a streamed epoch over chunks of whole groups (trajectories rematerialised per chunk, see GRPO.learn_streamed)
    "quadpole_sweep": dict(kind=3, cls="QuadPole", T=1000, E=64, G=16384, hidden=[256, 256], cov=0.3, gamma=0.999, eps=0.2,
                           lr=3e-4, updates=1, start="lqr", chunk_groups=8192,
                           desc="3D QuadPole GRPO sweep point: 1,048,576 envs per GPU x 1000 steps in 2 streamed chunks "
                                "(--sweep-envs-per-gpu to change), group 64, MLP 256x256"),
}
OBS = {0: 5, 1: 3, 2: 10, 3: 20}
ACT = {0: 1, 1: 1, 2: 2, 3: 4}


def mlp_macs(dims):
    return sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1))


def start_policy_arrays(w, seed=1234):
    """The start weights of a workload as numpy [W_l, b_l] lists (torch's default Linear init, seeded), plus
    * start == "lqr":   a = -K z embedded exactly in the 20-256-256-4 ReLU net (z = relu(z) - relu(-z)): hidden units
                        0..31 of both layers carry +-z, every other unit keeps its random init and feeds the output
                        layer with weight 0 (bench_assets/quadpole_lqr_gain.json; oracle/make_start_policy.py);
    * start == "hover": output layer zeroed (mean action = hover thrust)."""
    import torch
    kind = w["kind"]
    dims = [OBS[kind]] + w["hidden"] + [ACT[kind]]
    torch.manual_seed(seed)
    Ws, bs = [], []
    for i in range(len(dims) - 1):
        lin = torch.nn.Linear(dims[i], dims[i + 1])
        Ws.append(lin.weight.detach().numpy().copy()); bs.append(lin.bias.detach().numpy().copy())
    if w.get("start") == "hover":
        Ws[-1][:] = 0.0; bs[-1][:] = 0.0
    elif w.get("start") == "lqr":
        g = json.load(open(os.path.join(ROOT, "bench_assets", {3: "quadpole_lqr_gain.json", 2: "quadpole2d_lqr_gain.json"}[kind])))
        K, sel = np.asarray(g["K"], np.float32), g["sel"]
        nz = len(sel)
        assert len(w["hidden"]) == 2 and min(w["hidden"]) >= 2 * nz
        Ws[0][:2 * nz] = 0.0; bs[0][:2 * nz] = 0.0
        for i, s in enumerate(sel):
            Ws[0][i, s] = 1.0; Ws[0][nz + i, s] = -1.0
        Ws[1][:2 * nz] = 0.0; bs[1][:2 * nz] = 0.0
        Ws[1][:2 * nz, :2 * nz] = np.eye(2 * nz, dtype=np.float32)
        Ws[2][:] = 0.0; bs[2][:] = 0.0
        Ws[2][:, :nz] = -K; Ws[2][:, nz:2 * nz] = K
    return dims, Ws, bs


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region, in-process through NVML
    (a polling `nvidia-smi -lms` subprocess was measured to add ~5 ms of launch stalls per step)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.samples, self.stop_flag, self.thread = index, [], False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # torch's device index follows CUDA_VISIBLE_DEVICES; NVML's does not
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            try:
                self.power_limit_w = pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
            except Exception:
                self.power_limit_w = None
            self.power = []

            def loop():
                while not self.stop_flag:
                    try:
                        self.samples.append((pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM),
                                             pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)))
                        self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    except Exception:
                        pass
                    time.sleep(0.02)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)
            self.thread = None

    def stop(self):
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.thread.join(timeout=2)
        sm = [c for c, _ in self.samples]
        reasons = set()
        for _, mask in self.samples:
            for bit, name in self.REASONS.items():
                if mask & bit:
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(sm),
                "power_w": float(np.median(self.power)) if self.power else None, "power_limit_w": self.power_limit_w}


# --------------------------------------------------------------------------------------
# CPU arm: the reference's way (oracle/cpu_port.py), bounded sample of the same workload
# --------------------------------------------------------------------------------------
def cpu_leg(w, seed=0, budget_workers=None):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_port
    import restate as R
    import torch
    kind, T = w["kind"], w["T"]
    _, Ws, bs = start_policy_arrays(w)            # the same start policy as the GPU arm
    cores = os.cpu_count() or 1
    G = budget_workers or cores                  # one group per host core
    E = max(2, min(w["E"], int(3000 // T) or 2))  # ~3k env-steps per worker: a 10-30 s sample
    cov = [w["cov"]] * ACT[kind]
    (obs, act, rew, lens, mask), t_roll, procs = cpu_port.rollout_mp(kind, T, R.DEFAULT_DT[kind], Ws, bs, cov, G, E,
                                                                     w.get("restart", True), seed)
    torch.set_num_threads(cores)
    t_learn = cpu_port.grpo_learn(obs, act, rew, mask, Ws, bs, cov, w["gamma"], w["eps"], w["updates"], w["lr"])
    steps = int(lens.sum())
    return {
        "value": steps / (t_roll + t_learn), "unit": "env-steps/s", "cores": procs, "kind": "port",
        "sample": f"{G} groups x {E} episodes x <={T} steps ({steps} valid env-steps, valid fraction "
                  f"{steps / (G * E * T):.2f}) rollout on {procs} worker processes (OMP_NUM_THREADS=1) + GRPO.learn "
                  f"x{w['updates']} updates on torch-CPU ({cores} threads)",
        "rollout_env_steps_per_s": steps / t_roll, "rollout_s": t_roll, "learn_s": t_learn,
        "updates_per_s": w["updates"] / t_learn,
    }


def run_reference(args, w):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every host thread (torch reads
    # the variable when it is first imported, which happens inside cpu_leg)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(k, None)
    vals, ms, last = [], [], None
    for i in range(args.warmup + args.steps):
        last = cpu_leg(w, seed=i)
        if i >= args.warmup:
            vals.append(last["value"])
            ms.append(1e3 * (last["rollout_s"] + last["learn_s"]))      # one step = one bounded sample (config.cpu_sample)
    v = float(np.mean(vals))
    last["value"] = v
    line = {
        "impl": "reference", "metric": "policy-in-loop env-steps/sec (rollout + GRPO update epoch)", "value": v,
        "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean(ms)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": w["desc"], "cpu_sample": last["sample"]},
        "cpu_baseline": last, "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0,
                                      "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
class Dist:
    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, x, op="sum"):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


DUMP_SAMPLE_ENVS = 256      # trajectories of 256 envs: at most 27 MB (QuadPole, T = 1000); lengths of 1M envs: 8 MB


def dump_outputs(path, policy, rollout, mean_return, valid_env_steps):
    """What a caller of the timed epoch holds afterwards: the updated weights (`policy.flat_parameters()`) and,
    unless the epoch was streamed, the buffer's rollout (`Rollout_Buffer.device_rollout`)."""
    import torch
    arrays = {"policy_params": policy.flat_parameters(), "mean_return": mean_return,
              "valid_env_steps": valid_env_steps}
    if rollout is not None:
        r = rollout
        idx = np.sort(np.random.default_rng(0).choice(r.N, size=min(r.N, DUMP_SAMPLE_ENVS), replace=False))
        sel = torch.from_numpy(idx).to(r.len.device)
        arrays.update({
            "lengths": r.len, "sample_env_index": idx,
            "sample_observations": r.obs.index_select(2, sel).permute(2, 0, 1),     # [envs, T, O]
            "sample_actions": r.act.index_select(2, sel).permute(2, 0, 1),          # [envs, T, A]
            "sample_rewards": r.rew.index_select(1, sel).t(),                       # [envs, T]
            "sample_log_probs": r.logp.index_select(1, sel).t(),                    # [envs, T]
        })
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a.detach().cpu() if torch.is_tensor(a) else a)
        # integers (lengths, counts, indices) as float64: exact, where float32 is not above 2^24
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def measure(D, w, steps, warmup, full, args, dump=None):
    """One workload on this rank's GPU.  full=False: device-resident arm only (the `other_configs` lines).
    dump: directory for dump_outputs() of the last timed device-resident epoch."""
    import torch
    import trajopt_grpo_b200 as tg
    from trajopt_grpo_b200 import engine

    torch, dev, rank, world = D.torch, D.dev, D.rank, D.world
    kind, T, E, G = w["kind"], w["T"], w["E"], w["G"]
    N = G * E
    O, A = OBS[kind], ACT[kind]
    dims, Ws, bs = start_policy_arrays(w)          # identical initial weights on every rank
    P = mlp_macs(dims)
    ppo = w.get("algo") == "ppo"
    torch.manual_seed(1234)
    policy = (tg.GaussianActorCritic_NeuralNetwork if ppo else tg.GaussianActor_NeuralNetwork)(O, A, w["hidden"], "ReLU",
                                                                                              w["cov"])
    policy.actor.load_state_dict({f"network.{2 * i}.{nm}": torch.from_numpy(a) for i, (W_, b_) in enumerate(zip(Ws, bs))
                                  for nm, a in (("weight", W_), ("bias", b_))})
    policy.bump_param_epoch()
    opt = torch.optim.Adam(policy.parameters(), lr=w["lr"])
    if ppo:
        algo = tg.PPO(w["eps"], policy, opt, None, w["updates"], c1=0.5, kl_coeff=0.5, gamma=w["gamma"], lam=0.95,
                      entropy=0.01, batch_size=None, monte_carlo=True)
    else:
        # maximize=True: the reference's `J.backward(); optimizer.step()` DESCENDS on the surrogate (SURVEY q1; its own
        # comment says ascent was meant).  Measured here (profiles/README_r2.md): descent destroys the stabilising start
        # policy within 6 epochs (valid fraction 1.0 -> 0.06), so the work per epoch is not stationary.  The benchmark
        # therefore ascends -- the same kernels, the gradient scaled by -1 on the host; the class default stays the
        # reference's sign.
        algo = tg.GRPO(w["eps"], 0.01, w["gamma"], policy, opt, None, updates_per_iter=w["updates"],
                       maximize=w.get("start") == "lqr")
    env_cls = getattr(tg, w["cls"])
    mgr = tg.RolloutManager(lambda: env_cls(max_steps=T), policy, restart=w.get("restart", True), num_workers=G * world,
                            num_episodes_per_worker=E, use_multiprocessing=False, seed=7, rank=rank, world_size=world,
                            reuse_buffers=True, precision=args.precision)
    buf = tg.Rollout_Buffer(mgr)
    env = mgr.env
    rng = np.random.default_rng(100 + rank)
    total = warmup + steps
    restart = w.get("restart", True)

    def host_init():
        s0 = np.repeat(env.sample_initial_states(G, rng), E, axis=0) if restart else env.sample_initial_states(N, rng)
        return torch.from_numpy(np.ascontiguousarray(s0.T)).to(torch.float64 if args.precision == "f64"
                                                               else torch.float32).pin_memory()

    ev = lambda: torch.cuda.Event(enable_timing=True)
    chunked = w.get("chunk_groups") is not None

    # ---------------- device-resident arm: inputs already in HBM ----------------
    inits = [host_init().to(dev) for _ in range(total)]
    phase = {"rollout": [], "update": []}
    lens_sum = torch.zeros((), dtype=torch.int64, device=dev)
    last_valid = {}

    def one_step_device(i, timed):
        e = [ev() for _ in range(3)]
        e[0].record()
        if chunked:
            n_valid = algo.learn_streamed(mgr, init_state=inits[i], chunk_groups=w["chunk_groups"])
            e[1].record(); e[2].record()
        else:
            buf.sample(init_state=inits[i], sync_metrics=False)
            e[1].record()
            algo.learn(buf)
            e[2].record()
            n_valid = buf.device_rollout.len.sum()
        lens_sum.add_(n_valid)
        last_valid["n"] = n_valid
        if timed:
            phase["rollout"].append((e[0], e[1]))
            phase["update"].append((e[1], e[2]))

    for i in range(warmup):
        one_step_device(i, False)
    lens_sum.zero_()
    clocks = ClockSampler(D.local)
    if rank == 0 and full:
        clocks.start()          # NVML initialisation takes tens of ms on a cold driver: BEFORE the barrier, so that the
    D.barrier()                 # other ranks do not start their timed region (and wait in the first allreduce) meanwhile
    launches0 = engine.COUNTERS["launches"]
    t0, t1 = ev(), ev()
    t0.record()
    for i in range(warmup, total):
        one_step_device(i, True)
    t1.record()
    D.barrier()
    launches = engine.COUNTERS["launches"] - launches0
    ms_total = D.reduce(t0.elapsed_time(t1), "max")
    valid_rank = float(lens_sum.item())
    valid_steps = D.reduce(valid_rank)
    value = valid_steps / (ms_total * 1e-3)
    roll_ms = float(np.mean([a.elapsed_time(b) for a, b in phase["rollout"]]))
    upd_ms = float(np.mean([a.elapsed_time(b) for a, b in phase["update"]]))
    if dump and rank == 0:
        # before the per-kernel timing below: with reuse_buffers its rollouts overwrite the trajectory buffers
        dump_outputs(dump, policy, None if chunked else buf.device_rollout,
                     algo.last_mean_return if chunked else buf.avg_reward[-1], last_valid["n"])
    valid_per_step_rank = valid_rank / steps
    slots_per_step = float(N * T)

    # all ranks must hold bit-identical weights after the timed epochs (same allreduced gradient, same Adam)
    flat = policy.flat_parameters()
    chk = torch.stack([flat.double().sum(), flat.view(torch.int32).to(torch.int64).sum().double()])
    if world > 1:
        allc = [torch.empty_like(chk) for _ in range(world)]
        D.dist.all_gather(allc, chk)
        identical = all(bool(torch.equal(c, allc[0])) for c in allc)
    else:
        identical = True
    finite = bool(torch.isfinite(flat).all())
    # sharded == single GPU, visible to the driver at every N > 1: one small GRPO step (Pendulum, tensor-core kernels) and one
    # small PPO step (QuadPole2D, FP32-pipe kernels) run sharded over all ranks, and unsharded on rank 0 alone
    sharded_ok = None
    if world > 1 and full:
        sys.path.insert(0, os.path.join(ROOT, "tests", "helpers"))
        import mgpu_case
        from trajopt_grpo_b200 import algorithms as _alg
        got = mgpu_case.run_case(rank, world, groups=8 * world)
        got.pop("_peer", None)
        if rank == 0:
            with _alg.single_process():
                ref = mgpu_case.run_case(0, 1, groups=8 * world)
            sharded_ok = all(float(np.abs(got[k] - ref[k]).max()) <= 2e-5 * max(1.0, float(np.abs(ref[k]).max())) for k in got)

    out = {
        "workload": w["desc"], "value": value, "unit": "env-steps/s", "ms_per_step": ms_total / steps,
        "slot_steps_per_s": slots_per_step * world / (ms_total / steps * 1e-3),
        "valid_fraction": valid_per_step_rank / slots_per_step, "updates_per_iter": w["updates"],
        "phase_ms": {"rollout": roll_ms, "learn": upd_ms}, "gpu_launches": launches,
        "rank_weights_identical": identical, "weights_finite": finite, "sharded_equals_single_gpu": sharded_ok,
        "rollout_env_steps_per_s": valid_per_step_rank * world / (roll_ms * 1e-3) if not chunked else None,
        "grpo_updates_per_s": w["updates"] / (upd_ms * 1e-3) if not chunked else w["updates"] / (ms_total / steps * 1e-3),
    }
    if chunked:
        out["chunks_per_epoch"] = -(-G // w["chunk_groups"])
        return out, None, None

    # ---------------- per-kernel timing, each alone, CUDA events on its stream -------------
    aflat = policy.actor.flat_params()

    kernel_clocks = {}

    def timeit(fn, warm, reps, name=None):
        ts = []
        for i in range(warm):
            fn()
        torch.cuda.synchronize()
        sampler = ClockSampler(D.local) if (name and rank == 0) else None
        if sampler:
            sampler.start()
        for i in range(reps):
            a, b = ev(), ev()
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        if sampler:
            c = sampler.stop()
            kernel_clocks[name] = {k: c.get(k) for k in ("sm_mhz", "power_w", "reasons")}
        return float(np.mean(ts))

    big = slots_per_step > 5e7
    # K1 first: with reuse_buffers the rollout it leaves behind is the one K2 / K3 are then timed on
    k1_ms = timeit(lambda: mgr.rollout_device(init_state=inits[0]), 1 if big else 2, 2 if big else 3, "k1")
    r = mgr.last
    adv, _ = engine.advantage(0, r.G, r.E, r.T, w["gamma"], 0.0, r.rew, r.len)
    k3_ms = timeit(lambda: engine.policy_grad(dims, "ReLU", aflat, policy.cov_diag, r.obs, r.act, adv, r.logp, r.len,
                                              w["eps"], 1.0 / G), 1 if big else 3, 2 if big else 5, "k3")
    k2_ms = timeit(lambda: engine.advantage(0, r.G, r.E, r.T, w["gamma"], 0.0, r.rew, r.len), 2, 3)
    # env-steps a rollout tile actually executes: a tile of 128 consecutive envs runs until its longest episode ends
    ln_t = r.len.to(torch.int64)
    tile_max = torch.nn.functional.pad(ln_t, (0, (-ln_t.numel()) % 128)).view(-1, 128).max(dim=1).values
    k1_exec_steps = float(tile_max.sum().item()) * 128.0
    valid_k = float(ln_t.sum().item())            # valid steps of the rollout the kernels are timed on
    kern = {"k1_ms": k1_ms, "k2_ms": k2_ms, "k3_ms": k3_ms, "valid_k": valid_k, "k1_exec_steps": k1_exec_steps,
            "P": P, "dims": dims, "N": N, "T": T, "O": O, "A": A,
            "k3_traffic": engine.policy_grad_traffic_bytes(dims, int(valid_k), r.len)}
    out.update({"k1_ms": k1_ms, "k2_ms": k2_ms, "k3_ms": k3_ms, "kernel_clocks": kernel_clocks})
    if not full:
        return out, kern, None

    clock_info = clocks.stop() if rank == 0 else None
    # ---------------- end-to-end arm: host buffers in, host scalars out, through the reference-facing calls ------------
    host_inits = [host_init() for _ in range(total)]
    h2d = host_inits[0].numel() * 4
    d2h = N * 4 + 4
    lens_host = torch.empty(N, dtype=torch.int32).pin_memory()

    def one_step_e2e(i):
        x = host_inits[i].to(dev, non_blocking=True)                 # H2D of this step's inputs
        buf.sample(init_state=x)                                     # rollout + D2H of the mean return (avg_reward)
        algo.learn(buf)
        lens_host.copy_(buf.device_rollout.len, non_blocking=True)   # D2H of the episode lengths
        torch.cuda.current_stream().synchronize()
        return int(lens_host.sum())

    for i in range(warmup):
        one_step_e2e(i)
    D.barrier()
    a, b = ev(), ev()
    wall0 = time.perf_counter()
    a.record()
    n_e2e = 0
    for i in range(warmup, total):
        n_e2e += one_step_e2e(i)
    b.record()
    D.barrier()
    wall = time.perf_counter() - wall0
    e2e_ms = D.reduce(max(a.elapsed_time(b), wall * 1e3), "max")
    e2e_value = D.reduce(float(n_e2e)) / (e2e_ms * 1e-3)
    e2e = {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": e2e_ms / steps, "api": "Rollout_Buffer.sample(init_state=host tensor) + GRPO.learn(buffer)"}
    out["clocks"] = clock_info
    return out, kern, e2e


def rooflines(kern, w, fp32_peak, peaks):
    P, dims, N, T, O, A = (kern[k] for k in ("P", "dims", "N", "T", "O", "A"))
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    bf16_peak = peaks.get("bf16_tflops", 1590.0)
    valid = kern["valid_k"]
    k3_flops, k1_flops = 6.0 * P * valid, 2.0 * P * valid
    k3_tf = k3_flops / (kern["k3_ms"] * 1e-3) / 1e12
    k1_tf = k1_flops / (kern["k1_ms"] * 1e-3) / 1e12
    hid = w["hidden"]
    tc = hid in ([64, 64], [128, 128], [256, 256])     # shapes with a tcgen05 update path (fused 64, streamed 128/256)
    k3_name = ("update_tc_kernel (tg_policy_grad: fused fwd + clipped surrogate + MLP backward, tcgen05 3xTF32)"
               if hid == [64, 64] else
               "update_tcw_fwdbwd_kernel + update_tcw_wgrad_kernel (tg_policy_grad: streamed forward/backward + split-K "
               "weight gradients, tcgen05 3xTF32)")
    src = ("MEASURED_PEAKS.json bf16_tflops (burst; kernel timed alone)" if peaks else
           "fallback of /opt/skills/guides/B200_PROFILING.md (MEASURED_PEAKS.json absent)")
    tr = kern["k3_traffic"]
    if tc:
        # K3/K1 hidden GEMMs run on the tensor cores as 3xTF32: every algorithmic MAC costs 3 tf32 MMA-MACs and
        # tf32 peaks at half the bf16 rate, so an fp32-faithful kernel tops out at bf16_peak / 6.
        roof = {"kernel": k3_name, "bound": "tensor", "achieved": k3_tf, "peak": bf16_peak, "unit": "TFLOP/s",
                "frac": k3_tf / bf16_peak, "peak_source": src,
                "traffic": tr["total"], "traffic_detail": tr,
                "traffic_source": "computed on the host from this run's episode lengths: algorithmic trajectory reads "
                                  "(4*(O+A+2) B per valid step) + the HBM scratch between the two kernels of the wide path "
                                  "(bytes per 128-sample tile x live tiles, written once and read back by the weight-gradient "
                                  "kernel); the r2 ncu --set full capture under profiles/ holds the dram__bytes counters",
                "achieved_note": "algorithmic FLOPs (6*P per valid step, SURVEY 8d) / CUDA-event time of the launch",
                "frac_of_3xtf32_ceiling": k3_tf / (bf16_peak / 6.0),
                "frac_of_measured_fp32_fma_peak": k3_tf / fp32_peak, "fp32_fma_peak_tflops": fp32_peak,
                "ms_per_launch": kern["k3_ms"], "flops_per_launch": k3_flops}
    else:
        roof = {"kernel": "update_kernel (tg_policy_grad: fused fwd + clipped surrogate + MLP backward, FP32 pipe)",
                "bound": "fp32-fma", "achieved": k3_tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": k3_tf / fp32_peak,
                "traffic": tr["total"], "traffic_detail": tr,
                "peak_source": "tg_fp32_peak FFMA microbenchmark measured in this run (MEASURED_PEAKS.json has no FP32 figure)",
                "frac_of_measured_bf16_tensor_peak": k3_tf / bf16_peak,
                "ms_per_launch": kern["k3_ms"], "flops_per_launch": k3_flops}
    k1_tc = len(hid) >= 2 and len(set(hid)) == 1 and hid[0] in (64, 128) or hid == [256, 256]   # tg_rollout's routing
    k1_name = {64: "rollout_tc_kernel", 128: "rollout_tc2_kernel", 256: "rollout_tc256_kernel"}.get(hid[0]) if k1_tc \
        else "rollout_kernel"
    k1_exec_tf = 2.0 * P * kern["k1_exec_steps"] / (kern["k1_ms"] * 1e-3) / 1e12
    k2_gbs = 8.0 * N * T / (kern["k2_ms"] * 1e-3) / 1e9
    roof["others"] = {
        k1_name: {"bound": "tensor" if k1_tc else "fp32-fma", "ms": kern["k1_ms"], "achieved_tflops": k1_tf,
                  "executed_tflops": k1_exec_tf, "frac": k1_tf / (bf16_peak if k1_tc else fp32_peak),
                  "frac_of_3xtf32_ceiling": k1_exec_tf / (bf16_peak / 6.0) if k1_tc else None,
                  "frac_of_measured_fp32_fma_peak": k1_tf / fp32_peak,
                  "traj_write_gbs": 4.0 * (O + A + 2) * N * T / (kern["k1_ms"] * 1e-3) / 1e9},
        "adv_grpo_kernel": {"bound": "hbm", "ms": kern["k2_ms"], "achieved_gbs": k2_gbs, "peak_gbs": hbm_peak,
                            "frac": k2_gbs / hbm_peak, "algorithmic_bytes": "8 B per slot-step (rew read once, adv written once)"},
    }
    return roof


def run_ours(args, w):
    from trajopt_grpo_b200 import engine
    D = Dist()
    if args.sweep_envs_per_gpu:
        w = dict(w)
        w["G"] = args.sweep_envs_per_gpu // w["E"]
        w["desc"] = (f"3D QuadPole GRPO sweep point: {w['G'] * w['E']:,} envs per GPU x 1000 steps in "
                     f"{-(-w['G'] // w['chunk_groups'])} streamed chunks, group 64, MLP 256x256")
    full = not args.device_only
    out, kern, e2e = measure(D, w, args.steps, args.warmup, full, args, dump=args.dump_outputs)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if args.device_only:
        if D.rank == 0:
            line = {"device_only": True, **out}
            if kern is not None:
                line["roofline"] = rooflines(kern, w, engine.fp32_peak_tflops(D.dev), peaks)
            print(json.dumps(line))
        D.close()
        return
    fp32_peak = engine.fp32_peak_tflops(D.dev)
    roof = rooflines(kern, w, fp32_peak, peaks) if kern is not None else None
    # ---------------- the other BASELINE configuration with a published shape: configs[1] (Pendulum) ----------------
    others = {}
    if args.workload == "quadpole_cfg4" and not args.no_other:
        import gc
        import torch
        gc.collect(); torch.cuda.empty_cache()
        for key, name, st, wu in (("pendulum", "pendulum (BASELINE configs[1], device-resident arm)", 5, 3),
                                  ("quadpole2d_cfg3", "quadpole2d_cfg3 (BASELINE configs[2] at full size per GPU, device-resident arm)", 2, 2)):
            w2 = WORKLOADS[key]
            o2, k2, _ = measure(D, w2, st, wu, False, args)
            o2["roofline"] = rooflines(k2, w2, fp32_peak, peaks)
            others[name] = o2
            gc.collect(); torch.cuda.empty_cache()
    if D.rank != 0:
        D.close()
        return
    cpu = cpu_leg(w) if (D.world == 1 and not args.no_cpu) else None
    kind = w["kind"]
    O, A = OBS[kind], ACT[kind]
    N, T = w["G"] * w["E"], w["T"]
    tc = w["hidden"] in ([64, 64], [128, 128], [256, 256])
    line = {
        "metric": "policy-in-loop env-steps/sec (rollout + GRPO update epoch)", "value": out["value"], "unit": "env-steps/s",
        "n_gpus": D.world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": out["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": w["desc"], "envs_per_gpu": N, "horizon": T, "group_size": w["E"],
                   "mlp": [O] + w["hidden"] + [A], "updates_per_iter": w["updates"], "cov": w["cov"], "lr": w["lr"],
                   "objective_sign": ("ascent (GRPO(maximize=True)); the reference's literal sign descends on J and destroys "
                                      "the start policy within 6 epochs (measured), see bench.py") if w.get("start") == "lqr"
                   else "reference (descent on J, grpo.py:140-145)",
                   "start_policy": {"lqr": "stabilising linear feedback embedded in the ReLU net "
                                           "(bench_assets/quadpole_lqr_gain.json), other weights torch default init",
                                    "hover": "torch default init, output layer zeroed"}.get(w.get("start"), "torch default init"),
                   "precision": "fp32 state; hidden GEMMs 3xTF32 on tcgen05 (fp32-faithful), rest fp32" if tc else
                                "fp32 state + fp32 MLP (FP32 pipe)",
                   "l2": "per-step working set %.0f MB > 126 MB L2 (inputs larger than L2, no flush)" %
                         (4.0 * (O + A + 3) * N * T / 1e6),
                   "parallelism": f"dp{D.world} (whole GRPO groups per GPU, gradient allreduce)"},
        "e2e": e2e, "gpu_launches": out["gpu_launches"],
        "slot_steps_per_s": out["slot_steps_per_s"], "valid_fraction": out["valid_fraction"],
        "rollout_env_steps_per_s": out["rollout_env_steps_per_s"], "grpo_updates_per_s": out["grpo_updates_per_s"],
        "phase_ms": out["phase_ms"], "kernel_ms": {k: out.get(k) for k in ("k1_ms", "k2_ms", "k3_ms")}, "kernel_clocks": out.get("kernel_clocks"),
        "rank_weights_identical": out["rank_weights_identical"], "weights_finite": out["weights_finite"],
        "sharded_equals_single_gpu": out.get("sharded_equals_single_gpu"),
        "roofline": roof, "cpu_baseline": cpu, "clocks": out.get("clocks"), "other_configs": others,
    }
    print(json.dumps(line))
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="quadpole_cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-other", action="store_true", help="skip the other_configs (Pendulum) line")
    ap.add_argument("--device-only", action="store_true", help="device-resident arm only (profiling runs)")
    ap.add_argument("--sweep-envs-per-gpu", type=int, default=0, help="quadpole_sweep: envs per GPU (multiple of 64)")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"],
                    help="env-state arithmetic of the rollout kernel: f32 (throughput mode, default) or f64 (the reference's)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed epoch to DIR/<name>.npy (see the module docstring); "
                         "with several GPUs all but the weights cover rank 0's envs only")
    args = ap.parse_args()
    w = WORKLOADS[args.workload]
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
