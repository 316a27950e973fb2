"""PPO.learn_streamed on a rollout sharded over `world` ranks, run under torch.distributed.run by
tests/test_gpu_ppo_streamed.py:

    python -m torch.distributed.run --nproc-per-node 2 mgpu_ppo_streamed_case.py REF.npz

Each rank draws its block of the global initial states through RolloutManager(rank=, world_size=) and runs one streamed
epoch (chunks of 4 groups, so the chunking differs from the single-GPU run's); the weights must be bit-identical on
every rank and match the single-GPU streamed run stored in REF.npz (run_case(0, 1)) up to fp32 summation order."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LR = 3e-4
UPDATES = 3


def run_case(rank: int, world: int) -> dict:
    import trajopt_grpo_b200 as tg
    torch.manual_seed(1)
    pol = tg.GaussianActorCritic_NeuralNetwork(10, 2, [128, 128], "ReLU", 0.3)
    with torch.no_grad():
        pol.actor.network[-1].bias.add_(torch.tensor([0.5, -0.5], device=pol.device))
    ppo = tg.PPO(0.2, pol, torch.optim.Adam(pol.parameters(), lr=LR), None, UPDATES, c1=0.5, kl_coeff=0.5, gamma=0.999,
                 lam=0.95, entropy=0.01, batch_size=None, monte_carlo=False)
    mgr = tg.RolloutManager(lambda: tg.QuadPole2D(max_steps=60), pol, restart=False, num_workers=12,
                            num_episodes_per_worker=16, use_multiprocessing=False, seed=5, rank=rank, world_size=world)
    n_valid = ppo.learn_streamed(mgr, chunk_groups=4)
    assert torch.equal(ppo.old_policy.flat_parameters(), pol.flat_parameters())
    return {"w": pol.flat_parameters().detach().cpu().numpy().copy(), "n_valid": np.int64(int(n_valid)),
            "_peer": ppo._flat_opt._comm is not None}


def main():
    import torch.distributed as dist
    path = sys.argv[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ref = np.load(path)
    got = run_case(rank, world)
    if rank == 0:
        from trajopt_grpo_b200 import engine
        print("peer-memory allreduce:", got["_peer"], "(", engine.PeerComm.last_failure, ")")
    t = torch.from_numpy(got["w"]).cuda()
    every = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(every, t)
    for o in every:
        assert torch.equal(o, every[0]), "weights differ between ranks"
    n = torch.tensor([int(got["n_valid"])], device="cuda")
    dist.all_reduce(n)
    assert int(n) == int(ref["n_valid"]), (int(n), int(ref["n_valid"]))
    # the bound of test_streamed_epoch_equals_sample_plus_learn: no element moves by more than 2 lr per update,
    # 99.9 % agree within 1e-6
    d = np.abs(got["w"] - ref["w"])
    within = float((d <= 1e-6).mean())
    if rank == 0:
        print(f"max |sharded - single| = {d.max():.3e}, {100 * within:.3f} % within 1e-6")
    assert d.max() <= 2 * LR * UPDATES + 1e-7, d.max()
    assert within >= 0.999, within
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
