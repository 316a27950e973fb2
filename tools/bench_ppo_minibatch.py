"""Minibatched PPO on a sharded rollout: epoch time, time per minibatch and the planner kernel.

    python tools/bench_ppo_minibatch.py [--gpus 1,2,8] [--envs 65536] [--steps 500] [--batch-sizes 65536,4096]

For each GPU count (skipped when fewer GPUs are visible) the script starts itself under torch.distributed.run, one
process per GPU.  Each rank rolls out `--envs` QuadPole2D envs x `--steps` steps (10-128-128-2 actor, 10-128-128-1
critic) and runs ONE PPO.learn (updates_per_iter=1) per batch size, timed with CUDA events:
  epoch_ms          learn() end to end: critic values, advantages (+ allreduce of the sums), old log-probs, the
                    permutation (drawn on rank 0's CPU, broadcast), the plan, and one Adam step per minibatch
  minibatch_loop_ms from the return of engine.minibatch_plan to the end of learn(): the minibatch steps alone
  per_minibatch_us  minibatch_loop_ms / number of minibatches
The planner (tg_minibatch_plan, four kernels) is then timed on its own over the same rollout, 20 launches between
events after 3 warm-up launches, against its algorithmic traffic: 8 n_total bytes read (the permutation) + 8 n_local +
8 (n_batches + 1) bytes written.  Its permutation is larger than the 126 MB L2 at the default sizes, so the reads come
from HBM.  Card name and power limit are read in the same run.  Prints one JSON line; writes nothing unless --out.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def card_info(index):
    r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


def worker(args):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import trajopt_grpo_b200 as tg
    from trajopt_grpo_b200 import _lib as L
    from trajopt_grpo_b200 import engine

    marks = []
    plan = engine.minibatch_plan

    def marked_plan(*a, **k):             # timestamps the start of the minibatch loop inside learn()
        out = plan(*a, **k)
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append(ev)
        return out

    engine.minibatch_plan = marked_plan
    group = 16

    def make(bs, envs):
        torch.manual_seed(0)
        pol = tg.GaussianActorCritic_NeuralNetwork(10, 2, [128, 128], "ReLU", 0.3)
        ppo = tg.PPO(0.2, pol, torch.optim.Adam(pol.parameters(), lr=3e-4), None, 1, batch_size=bs, monte_carlo=False)
        mgr = tg.RolloutManager(lambda: tg.QuadPole2D(max_steps=args.steps), pol, num_workers=envs * world // group,
                                num_episodes_per_worker=group, use_multiprocessing=False, seed=7, rank=rank,
                                world_size=world)
        buf = tg.Rollout_Buffer(mgr)
        buf.device_rollout = mgr.rollout_device()
        return ppo, buf

    results = []
    for bs in args.batch_sizes:
        ppo, buf = make(bs, 1024)                            # warm-up: every kernel and the exchange at this batch size
        ppo.learn(buf)
        ppo, buf = make(bs, args.envs)
        marks.clear()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ppo.learn(buf)
        e1.record()
        torch.cuda.synchronize()
        n_mb = ppo._flat_opt.step_count
        loop_ms = marks[-1].elapsed_time(e1)
        results.append({"batch_size": bs, "epoch_ms": e0.elapsed_time(e1), "minibatches": n_mb,
                        "minibatch_loop_ms": loop_ms, "per_minibatch_us": 1e3 * loop_ms / n_mb,
                        "peer_memory_allreduce": ppo._flat_opt._comm is not None})
    engine.minibatch_plan = plan

    # the planner alone, on this rank's shard of the last rollout
    r = buf.device_rollout
    n_loc = r.len.sum(dtype=torch.int64).reshape(1)
    counts = [torch.empty_like(n_loc) for _ in range(world)]
    dist.all_gather(counts, n_loc)
    counts = [int(c) for c in counts]
    n_total, n_local, base = sum(counts), counts[rank], sum(counts[:rank])
    perm = torch.randperm(n_total, generator=torch.Generator().manual_seed(1)).cuda()
    row0 = torch.cumsum(r.len.to(torch.int64), 0) - r.len
    lib = L.load()
    planner = []
    for bs in args.batch_sizes:
        nb = -(-n_total // bs)
        ids = torch.empty(n_local, dtype=torch.int64, device="cuda")
        offs = torch.empty(nb + 1, dtype=torch.int64, device="cuda")
        ws = torch.empty(max(1, lib.tg_minibatch_plan_workspace_bytes(n_total)), dtype=torch.uint8, device="cuda")

        def launch():
            L.check(lib.tg_minibatch_plan(L.ctx(), r.len.numel(), L.ptr(r.len), L.ptr(row0), L.ptr(perm), n_total, bs,
                                          base, n_local, n_local, L.ptr(ids), L.ptr(offs), L.ptr(ws), L.stream_ptr()),
                    "tg_minibatch_plan")

        for _ in range(3):
            launch()
        reps = 20
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            launch()
        e1.record()
        torch.cuda.synchronize()
        assert int(offs[-1]) == n_local
        us = 1e3 * e0.elapsed_time(e1) / reps
        nbytes = 8 * n_total + 8 * n_local + 8 * (nb + 1)
        planner.append({"batch_size": bs, "kernel_us": us, "bytes": nbytes, "GB_per_s": nbytes / us / 1e3,
                        "share_of_hbm_peak": nbytes / (us * 1e-6) / HBM_BYTES_PER_S})
    mine = {"rank": rank, "n_local": n_local, "learn": results, "planner": planner, "card": card_info(local)}
    every = [None] * world
    dist.all_gather_object(every, mine)
    if rank == 0:
        print("RESULT " + json.dumps({"gpus": world, "envs_per_rank": args.envs, "steps": args.steps,
                                      "n_valid": n_total, "ranks": every}), flush=True)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="1,2,8")
    ap.add_argument("--envs", type=int, default=65536, help="envs per rank")
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--batch-sizes", default="65536,4096")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    args.batch_sizes = [int(b) for b in args.batch_sizes.split(",")]
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
               "127.0.0.1", "--master-port", str(29611 + i), os.path.abspath(__file__), "--worker", "--envs",
               str(args.envs), "--steps", str(args.steps), "--batch-sizes", ",".join(map(str, args.batch_sizes))]
        p = subprocess.run(cmd, capture_output=True, text=True)
        line = next((l for l in p.stdout.splitlines() if l.startswith("RESULT ")), None)
        if p.returncode != 0 or line is None:
            raise SystemExit(f"{g} GPUs failed (exit {p.returncode}):\n{p.stdout[-3000:]}\n{p.stderr[-5000:]}")
        runs.append(json.loads(line[len("RESULT "):]))
    out = json.dumps({"tool": "bench_ppo_minibatch", "runs": runs, "skipped_gpu_counts": skipped})
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
