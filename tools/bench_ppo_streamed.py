"""Full-batch PPO on a rollout streamed in chunks (PPO.learn_streamed) against sample() + learn().

    python tools/bench_ppo_streamed.py [--gpus 1,2,8] [--fit-envs 524288] [--big-envs 4194304] [--steps 1000]
                                       [--updates 24] [--chunk-groups 8192] [--group 64] [--out FILE]

Workload: the shipped 3-D QuadPole PPO settings -- 20-256-256-4 actor and 20-256-256-1 critic, cov 0.3, gamma 0.999,
lambda 0.95, eps 0.2, c1 0.5, kl 0.5, Monte-Carlo returns, full batch, Adam lr 3e-4 -- from the stabilising start of
bench.py (bench_assets/quadpole_lqr_gain.json), so episodes run the whole horizon as in a trained run.  Each rank draws
its own initial states (group `--group`, one reset per group).

For each GPU count (skipped when fewer GPUs are visible) the script starts itself under torch.distributed.run, one
process per GPU, and times one epoch with CUDA events at two points per rank:
  --fit-envs  (fits in HBM): sample() + learn(), then the streamed epoch on the same seed, initial states and weights
  --big-envs  (does not fit): the streamed epoch only
Every engine call of an epoch is bracketed by CUDA events and booked to a pass and a category.  Pass 0 is the
streamed epoch's statistics pass (its first `chunks` rollouts with their values and raw advantages), or sample() + the
critic values and raw advantages of learn() (the one-time z-score and old log-probs of learn() land in its first
update pass).  Every update pass ends with its Adam step.  Categories: k1 (rollout), forward (critic values, actor old
log-probs), k2 (raw advantages + z-score), k3_actor, k3_critic, exchange (the 40-byte sums allreduce, the gradient
allreduce + Adam, or the fused peer-memory allreduce + Adam).  Also reported: the peak memory of torch's allocator
over the epoch (the engine's own context scratch is allocated outside it), and whether the two arms at the fit point
end with bit-identical weights.  A small warm-up epoch of both arms runs first.  Card name and power limit are read in
the same run.  Prints one JSON line; writes nothing unless --out.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOAD = dict(kind=3, cls="QuadPole", hidden=[256, 256], cov=0.3, gamma=0.999, lam=0.95, eps=0.2, lr=3e-4,
                start="lqr")


def card_info(index):
    r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


class PassTimer:
    """Brackets the engine calls of learn() / learn_streamed() with CUDA events and books them to passes."""
    CATEGORY = {"rollout": "k1", "policy_forward_traj": "forward", "advantage_ppo_raw": "k2",
                "advantage_ppo_normalize": "k2", "policy_grad": "k3_actor", "value_grad": "k3_critic"}

    def __init__(self, torch, engine, algorithms, dist):
        self.torch = torch
        self.start()
        self._undo = []

        def wrap(owner, name, category):
            fn = getattr(owner, name)

            def timed(*a, **k):
                if self.pass_idx == 0:                      # does this call open the first update pass?
                    if self.chunks is None and name == "advantage_ppo_normalize":
                        self.pass_idx = 1
                    elif self.chunks is not None and name == "rollout":
                        self.rollouts += 1
                        self.pass_idx = int(self.rollouts > self.chunks)
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
                out = fn(*a, **k)
                e1.record()
                self.calls.append((self.pass_idx, category, e0, e1))
                if category == "exchange" and name != "all_reduce":
                    self.pass_idx += 1                      # an update pass ends with its Adam step
                return out

            setattr(owner, name, timed)
            self._undo.append((owner, name, fn))

        for name, cat in self.CATEGORY.items():
            wrap(engine, name, cat)
        wrap(algorithms._FlatOptimizer, "step", "exchange")
        wrap(algorithms._FlatOptimizer, "step_allreduced", "exchange")
        wrap(dist, "all_reduce", "exchange")

    def start(self, chunks=None):
        """chunks: the streamed epoch's chunk count (its statistics pass holds that many rollouts); None for
        sample() + learn()."""
        self.calls, self.pass_idx, self.chunks, self.rollouts = [], 0, chunks, 0

    def report(self):
        """[{category: ms, ..., "wall_ms": first start -> last end} for pass 0, 1, ...] (ms of device time)."""
        self.torch.cuda.synchronize()
        passes = {}
        for p, cat, e0, e1 in self.calls:
            d = passes.setdefault(p, {"cats": {}, "first": e0, "last": e1})
            d["cats"][cat] = d["cats"].get(cat, 0.0) + e0.elapsed_time(e1)
            d["last"] = e1
        return [dict(passes[p]["cats"], wall_ms=passes[p]["first"].elapsed_time(passes[p]["last"]))
                for p in sorted(passes)]

    def close(self):
        for owner, name, fn in reversed(self._undo):
            setattr(owner, name, fn)


def worker(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import bench
    import trajopt_grpo_b200 as tg
    from trajopt_grpo_b200 import algorithms, engine
    w = dict(WORKLOAD, T=args.steps)
    dims, Ws, bs = bench.start_policy_arrays(w)
    E = args.group

    def make(envs):
        torch.manual_seed(1234)
        pol = tg.GaussianActorCritic_NeuralNetwork(dims[0], dims[-1], w["hidden"], "ReLU", w["cov"])
        sd = {f"network.{2 * i}.{nm}": torch.from_numpy(a)
              for i, (W_, b_) in enumerate(zip(Ws, bs)) for nm, a in (("weight", W_), ("bias", b_))}
        pol.actor.load_state_dict(sd)
        ppo = tg.PPO(w["eps"], pol, torch.optim.Adam(pol.parameters(), lr=w["lr"]), None, args.updates, c1=0.5,
                     kl_coeff=0.5, gamma=w["gamma"], lam=w["lam"], entropy=0.01, batch_size=None, monte_carlo=True)
        mgr = tg.RolloutManager(lambda: tg.QuadPole(max_steps=args.steps), pol, restart=True,
                                num_workers=envs // E * world, num_episodes_per_worker=E, use_multiprocessing=False,
                                seed=7, rank=rank, world_size=world)
        rng = np.random.default_rng(100 + rank)
        s0 = np.repeat(mgr.env.sample_initial_states(envs // E, rng), E, axis=0)
        init = torch.from_numpy(np.ascontiguousarray(s0.T)).float().cuda()
        return pol, ppo, mgr, init

    timer = PassTimer(torch, engine, algorithms, dist)

    def epoch(envs, streamed):
        pol, ppo, mgr, init = make(envs)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        chunks = -(-(envs // E) // args.chunk_groups)
        timer.start(chunks if streamed else None)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if streamed:
            n_valid = ppo.learn_streamed(mgr, init_state=init, chunk_groups=args.chunk_groups)
        else:
            buf = tg.Rollout_Buffer(mgr)
            buf.sample(init_state=init, sync_metrics=False)
            n_valid = buf.device_rollout.len.sum(dtype=torch.int64)
            ppo.learn(buf)
        e1.record()
        torch.cuda.synchronize()
        res = {"arm": "streamed" if streamed else "sample_learn", "envs_per_rank": envs,
               "epoch_ms": e0.elapsed_time(e1), "n_valid_rank": int(n_valid),
               "peak_allocated_GB": (torch.cuda.max_memory_allocated() - base) / 1e9,
               "peer_memory_allreduce": ppo._flat_opt._comm is not None, "passes": timer.report()}
        if streamed:
            res["chunks"] = chunks
        weights = pol.flat_parameters().detach().clone()
        del pol, ppo, mgr, init
        if not streamed:
            del buf
        torch.cuda.empty_cache()
        return res, weights

    warm = 2 * E
    epoch(warm, False)
    epoch(warm, True)
    points = []
    a, wa = epoch(args.fit_envs, False)
    b, wb = epoch(args.fit_envs, True)
    b["weights_bit_identical_to_sample_learn"] = bool(torch.equal(wa, wb))
    del wa, wb
    points += [a, b]
    if args.big_envs:
        c, _ = epoch(args.big_envs, True)
        points.append(c)
    timer.close()
    mine = {"rank": rank, "points": points, "card": card_info(local)}
    every = [None] * world
    dist.all_gather_object(every, mine)
    if rank == 0:
        print("RESULT " + json.dumps({"gpus": world, "steps": args.steps, "group": E, "updates": args.updates,
                                      "chunk_groups": args.chunk_groups, "ranks": every}), flush=True)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--fit-envs", type=int, default=524288, help="envs per rank of the point that fits in HBM")
    ap.add_argument("--big-envs", type=int, default=4194304, help="envs per rank of the streamed-only point (0: skip)")
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--updates", type=int, default=24, help="updates_per_iter")
    ap.add_argument("--chunk-groups", type=int, default=8192)
    ap.add_argument("--group", type=int, default=64)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    for v in (args.fit_envs, args.big_envs):
        if v % args.group:
            raise SystemExit(f"envs per rank ({v}) must be a multiple of the group size {args.group}")
    if args.worker:
        return worker(args)
    import torch
    have = torch.cuda.device_count()
    if have == 0:
        raise SystemExit("no CUDA device: this script measures on the GPU only")
    runs, skipped = [], []
    for i, g in enumerate(int(x) for x in args.gpus.split(",")):
        if g > have:
            skipped.append(g)
            continue
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(g), "--master-addr",
               "127.0.0.1", "--master-port", str(29631 + i), os.path.abspath(__file__), "--worker", "--fit-envs",
               str(args.fit_envs), "--big-envs", str(args.big_envs), "--steps", str(args.steps), "--updates",
               str(args.updates), "--chunk-groups", str(args.chunk_groups), "--group", str(args.group)]
        p = subprocess.run(cmd, capture_output=True, text=True)
        line = next((l for l in p.stdout.splitlines() if l.startswith("RESULT ")), None)
        if p.returncode != 0 or line is None:
            raise SystemExit(f"{g} GPUs failed (exit {p.returncode}):\n{p.stdout[-3000:]}\n{p.stderr[-5000:]}")
        runs.append(json.loads(line[len("RESULT "):]))
    out = json.dumps({"tool": "bench_ppo_streamed", "runs": runs, "skipped_gpu_counts": skipped})
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
