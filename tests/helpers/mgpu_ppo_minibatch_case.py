"""Minibatched PPO.learn (batch_size=k) on a rollout sharded over `world` ranks, run under torch.distributed.run by
tests/test_gpu_ppo_minibatch_shard.py.

    pair REF.npz       2 ranks: QuadPole2D rollout through RolloutManager(rank=, world_size=), batch sizes 64 and 3,
                       two updates; against the single-GPU run of the same seeds stored in REF.npz (run_case(0, 1, bs))
    fixture GOLD.npz   3 ranks, one group each, of the reference's ppo_minibatch_quadpole2d fixture; against the
                       reference's post-Adam weights

Every rank other than 0 reseeds torch's CPU generator before learn(): only rank 0's draw may shape the minibatches."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH_SIZES = (64, 3)
LR = 1e-3
UPDATES = 2


def run_case(rank: int, world: int, batch_size: int) -> dict:
    import trajopt_grpo_b200 as tg
    torch.manual_seed(1)
    pol = tg.GaussianActorCritic_NeuralNetwork(10, 2, [32, 32], "ReLU", 0.05)
    opt = torch.optim.Adam(pol.parameters(), lr=LR)
    ppo = tg.PPO(0.2, pol, opt, None, UPDATES, c1=0.5, kl_coeff=0.5, gamma=0.99, lam=0.95, entropy=0.01,
                 batch_size=batch_size, monte_carlo=False)
    mgr = tg.RolloutManager(lambda: tg.QuadPole2D(max_steps=16), pol, restart=False, num_workers=4,
                            num_episodes_per_worker=4, use_multiprocessing=False, seed=5, rank=rank, world_size=world)
    buf = tg.Rollout_Buffer(mgr)
    buf.device_rollout = mgr.rollout_device()
    torch.manual_seed(77 if rank == 0 else 1000 + rank)
    ppo.learn(buf)
    return {"w": pol.flat_parameters().detach().cpu().numpy().copy(),
            "steps": np.int64(ppo._flat_opt.step_count), "_peer": ppo._flat_opt._comm is not None}


def run_fixture(rank: int, world: int, path: str) -> dict:
    import trajopt_grpo_b200 as tg
    g = dict(np.load(path, allow_pickle=False))
    G = int(g["G"])
    assert G == world, "one group per rank"
    hidden = [int(h) for h in g["hidden"]]
    pol = tg.GaussianActorCritic_NeuralNetwork(10, 2, hidden, "ReLU", float(g["cov"]))
    for net, pre in ((pol.actor, ""), (pol.critic, "c")):
        sd = {}
        i = 0
        while f"{pre}W{i}" in g:
            sd[f"network.{2 * i}.weight"] = torch.from_numpy(g[f"{pre}W{i}"])
            sd[f"network.{2 * i}.bias"] = torch.from_numpy(g[f"{pre}b{i}"])
            i += 1
        net.load_state_dict(sd)
    algo = tg.PPO(float(g["eps_clip"]), pol, torch.optim.Adam(pol.parameters(), lr=2e-4), None, int(g["updates"]),
                  c1=0.5, kl_coeff=0.5, gamma=float(g["gamma"]), lam=float(g["lam"]), entropy=0.01,
                  batch_size=int(g["batch_size"]), monte_carlo=bool(g["monte_carlo"]))
    buf = tg.Rollout_Buffer.__new__(tg.Rollout_Buffer)
    buf.avg_reward = []
    buf.device_rollout = None
    sl = slice(rank, rank + 1)
    tg.Rollout_Buffer.store(buf, g["obs"][sl], g["act"][sl], g["rew"][sl], g["len"][sl], g["mask"][sl])
    torch.manual_seed(int(g["torch_seed"]) if rank == 0 else 1000 + rank)
    algo.learn(buf)
    n_steps = int(g["updates"]) * -(-int(g["len"].sum()) // int(g["batch_size"]))
    assert algo._flat_opt.step_count == n_steps, (algo._flat_opt.step_count, n_steps)
    return {"w": pol.flat_parameters().detach().cpu().numpy().copy(), "params": [p.detach().cpu().numpy() for p in
                                                                              pol.parameters()], "g": g}


def _same_on_every_rank(w, world, what):
    import torch.distributed as dist
    t = torch.from_numpy(w).cuda()
    all_t = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(all_t, t)
    for o in all_t:
        assert torch.equal(o, all_t[0]), f"{what}: weights differ between ranks"


def main():
    import torch.distributed as dist
    mode, path = sys.argv[1], sys.argv[2]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if mode == "pair":
        ref = np.load(path)
        for bs in BATCH_SIZES:
            got = run_case(rank, world, bs)
            if rank == 0 and bs == BATCH_SIZES[0]:
                from trajopt_grpo_b200 import engine
                print("peer-memory allreduce:", got["_peer"], "(", engine.PeerComm.last_failure, ")")
            _same_on_every_rank(got["w"], world, f"batch {bs}")
            steps = int(ref[f"bs{bs}_steps"])
            assert int(got["steps"]) == steps, (bs, int(got["steps"]), steps)
            # Adam amplification of fp32 summation-order differences (as test_streamed_epoch_equals_sample_plus_learn):
            # no element moves by more than 2 lr per optimizer step, 99.9 % agree within 1e-6
            d = np.abs(got["w"] - ref[f"bs{bs}_w"])
            within = float((d <= 1e-6).mean())
            if rank == 0:
                print(f"batch {bs}: {steps} optimizer steps, max |sharded - single| = {d.max():.3e}, "
                      f"{100 * within:.3f} % within 1e-6")
            assert d.max() <= 2 * LR * steps, (bs, d.max())
            assert within >= 0.999, (bs, within)
    elif mode == "fixture":
        got = run_fixture(rank, world, path)
        _same_on_every_rank(got["w"], world, "fixture")
        g = got["g"]
        worst = 0.0
        for i, p in enumerate(got["params"]):
            ref = g[f"ppo_mb_adam_p{i}"]
            worst = max(worst, float(np.abs(p - ref).max()))
            np.testing.assert_allclose(p, ref, rtol=1e-3, atol=2e-5, err_msg=f"param {i}")
        if rank == 0:
            print(f"fixture: max |sharded - reference| = {worst:.3e}")
    else:
        raise SystemExit(f"unknown mode {mode}")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
