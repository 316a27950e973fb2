"""GRPO with a KL penalty to a reference policy on `world` ranks (tests/test_gpu_grpo_ref_kl.py): GRPO.learn and
GRPO.learn_streamed.  Each rank evaluates the reference on its own groups; the term is inside the gradient the ranks
already sum, so sharding changes nothing but the fp32 summation order.  The single-process result is the reference."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _setup(tg, rank, world, seed):
    torch.manual_seed(seed)
    pol = tg.GaussianActor_NeuralNetwork(20, 4, [128, 128], "ReLU", 0.3)
    ref = tg.GaussianActor_NeuralNetwork(20, 4, [64, 64], "Tanh", 0.5)
    algo = tg.GRPO(0.2, 0.04, 0.99, pol, torch.optim.Adam(pol.parameters(), lr=1e-3), ref, updates_per_iter=2,
                   maximize=True)
    mgr = tg.RolloutManager(lambda: tg.QuadPole(max_steps=40), pol, restart=True, num_workers=8,
                            num_episodes_per_worker=16, use_multiprocessing=False, seed=3, rank=rank, world_size=world)
    return pol, algo, mgr


def run_case(rank: int, world: int) -> dict:
    import trajopt_grpo_b200 as tg
    out = {}
    pol, algo, mgr = _setup(tg, rank, world, 0)
    buf = tg.Rollout_Buffer(mgr)
    buf.device_rollout = mgr.rollout_device()
    algo.learn(buf)
    out["learn"] = pol.flat_parameters().detach().cpu().numpy().copy()
    out["_peer"] = algo._flat_opt._comm is not None
    pol, algo, mgr = _setup(tg, rank, world, 1)
    algo.learn_streamed(mgr, chunk_groups=3)
    out["streamed"] = pol.flat_parameters().detach().cpu().numpy().copy()
    return out


def main():
    import torch.distributed as dist
    from trajopt_grpo_b200 import engine
    ref_path = sys.argv[1]
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    got = run_case(rank, world)
    ref = np.load(ref_path)
    if rank == 0:
        print("peer-memory allreduce:", got.pop("_peer"), "(", engine.PeerComm.last_failure, ")")
    got.pop("_peer", None)
    for k, v in got.items():
        t = torch.from_numpy(v).cuda()
        all_t = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(all_t, t)
        for o in all_t:
            assert torch.equal(o, all_t[0]), f"{k}: weights differ between ranks"
        err = np.abs(v - ref[k]).max()
        if rank == 0:
            print(f"[grpo-kl] 2 GPUs {k}: max |sharded - single| = {err:.3e} (<= 2e-5)")
        assert err <= 2e-5 * max(1.0, np.abs(ref[k]).max()), (k, err)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
