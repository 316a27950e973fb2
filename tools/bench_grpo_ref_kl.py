"""Cost of GRPO's KL penalty to a reference policy (GRPO(ref_model=..., beta=0.04)) on the bench.py default workload.

    python tools/bench_grpo_ref_kl.py [--reps 3] [--steps 1000] [--streamed-envs 1048576] [--chunk-groups 8192]
                                      [--out FILE]

Workload: bench.py's quadpole_cfg4 -- the cfg-4 shard of one GPU, 524,288 QuadPole envs (8,192 groups of 64) x 1000
steps, 20-256-256-4 ReLU policy, cov 0.3, maximize=True, one update, from the stabilising start policy.  The reference
policy is a copy of the start policy (so every u = log pi_ref - log pi_theta is 0 up to the rollout's own log-probs:
the term costs what it costs at any u).

Two arms alternate in the same process, `--reps` times each: sample() + learn() without a reference, and with one.
Every engine call of learn() is bracketed by CUDA events: K1 (the rollout of sample()), K2 (advantages), forward (the
reference forward; the old log-probs come from the rollout), K3 (tg_policy_grad / tg_policy_grad_ref).  The median
over the reps is reported with the min and max.  Then one GRPO.learn_streamed epoch with the reference at
`--streamed-envs` (more than sample() + learn() holds in HBM) is timed with the same brackets.  Card name and power
limit are read in the same run.  Prints one JSON line; writes nothing unless --out.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CATEGORY = {"rollout": "k1", "advantage": "k2", "policy_forward_traj": "forward", "policy_grad": "k3"}


def card_info():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else f"nvidia-smi failed: {r.stderr.strip()}"


class Timer:
    def __init__(self, torch, engine):
        self.torch, self.calls, self._undo = torch, [], []
        for name, cat in CATEGORY.items():
            self._wrap(engine, name, cat)

    def _wrap(self, owner, name, cat):
        fn, torch = getattr(owner, name), self.torch

        def timed(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            self.calls.append((cat, e0, e1))
            return out

        setattr(owner, name, timed)
        self._undo.append((owner, name, fn))

    def take(self):
        self.torch.cuda.synchronize()
        out = {}
        for cat, e0, e1 in self.calls:
            out[cat] = out.get(cat, 0.0) + e0.elapsed_time(e1)
        if self.calls:
            out["wall_ms"] = self.calls[0][1].elapsed_time(self.calls[-1][2])
        self.calls = []
        return out

    def close(self):
        for owner, name, fn in reversed(self._undo):
            setattr(owner, name, fn)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--streamed-envs", type=int, default=1048576)
    ap.add_argument("--chunk-groups", type=int, default=8192)
    ap.add_argument("--beta", type=float, default=0.04)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    import trajopt_grpo_b200 as tg
    from trajopt_grpo_b200 import engine
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the B200 kernels")
    w = dict(bench.WORKLOADS["quadpole_cfg4"], T=args.steps)
    dims, Ws, bs = bench.start_policy_arrays(w)
    E = w["E"]
    sd = {f"network.{2 * i}.{nm}": torch.from_numpy(a)
          for i, (W_, b_) in enumerate(zip(Ws, bs)) for nm, a in (("weight", W_), ("bias", b_))}

    def actor():
        p = tg.GaussianActor_NeuralNetwork(dims[0], dims[-1], w["hidden"], "ReLU", w["cov"])
        p.actor.load_state_dict(sd)
        return p

    def make(groups, with_ref):
        pol = actor()
        algo = tg.GRPO(w["eps"], args.beta, w["gamma"], pol, torch.optim.Adam(pol.parameters(), lr=w["lr"]),
                       actor() if with_ref else None, updates_per_iter=w["updates"], maximize=True)
        mgr = tg.RolloutManager(lambda: tg.QuadPole(max_steps=args.steps), pol, restart=True, num_workers=groups,
                                num_episodes_per_worker=E, use_multiprocessing=False, seed=7)
        s0 = np.repeat(mgr.env.sample_initial_states(groups, np.random.default_rng(100)), E, axis=0)
        return algo, mgr, torch.from_numpy(np.ascontiguousarray(s0.T)).float().cuda()

    timer = Timer(torch, engine)
    runs = {"no_ref": [], "ref": []}
    for rep in range(args.reps + 1):                          # rep 0 warms both arms up
        for arm in ("no_ref", "ref"):
            algo, mgr, init = make(w["G"], arm == "ref")
            buf = tg.Rollout_Buffer(mgr)
            timer.take()
            buf.sample(init_state=init)
            algo.learn(buf)
            t = timer.take()
            if rep:
                runs[arm].append(t)
            del algo, mgr, buf
            torch.cuda.empty_cache()
    summary = {}
    for arm, ts in runs.items():
        summary[arm] = {k: {"median_ms": float(np.median([t.get(k, 0.0) for t in ts])),
                            "min_ms": float(min(t.get(k, 0.0) for t in ts)),
                            "max_ms": float(max(t.get(k, 0.0) for t in ts))}
                        for k in ("k1", "k2", "forward", "k3", "wall_ms")}
    algo, mgr, init = make(args.streamed_envs // E, True)
    algo.learn_streamed(mgr, init_state=init, chunk_groups=args.chunk_groups)   # warm-up epoch
    timer.take()
    torch.cuda.reset_peak_memory_stats()
    algo.learn_streamed(mgr, init_state=init, chunk_groups=args.chunk_groups)
    streamed = timer.take()
    streamed["peak_alloc_gb"] = torch.cuda.max_memory_allocated() / 1e9
    timer.close()
    res = {"tool": "bench_grpo_ref_kl", "card": card_info(), "workload": w["desc"], "steps": args.steps,
           "beta": args.beta, "reps": args.reps, "learn": summary,
           "k3_ref_over_no_ref": summary["ref"]["k3"]["median_ms"] / summary["no_ref"]["k3"]["median_ms"],
           "streamed_with_ref": dict(envs=args.streamed_envs, chunk_groups=args.chunk_groups, **streamed)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
