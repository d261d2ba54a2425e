"""Two ranks under torchrun (tests/test_qr_gpu.py::test_two_ranks_under_nccl): a QR-DQN BrainDQNNature per rank on its own env
shard, trained through loss_backward + NCCL all_reduce + Adam; params, target and the Adam slots must end bit-identical on both
ranks, and asking for the in-step peer exchange with the QR head must raise."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402


def main():
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    torch.cuda.set_device(rank)
    from dqnflappybird_b200 import brains, game
    N = 64
    dev = f"cuda:{rank}"
    brain = brains.BrainDQNNature(2, "bird", num_envs=N, device=dev, replay_memory_per_env=12, observe=6., batch_size=32 * world, seed=1,
                                  first_env_id=rank * N, replace_target_iter=5, lr=1e-4, quantile=True)
    assert brain.net.exchange is None and brain.net.quantile
    gs = game.GameState(num_envs=N, device=dev, seed=2, first_env_id=rank * N, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device=dev))
    brain.setInitState(obs)
    p0 = brain.net.params.clone()
    for _ in range(30):
        a = brain.getAction()
        obs, r, t, s = gs.frame_step(a, out=brain.next_rows()[1:])
        brain.setPerception(obs, a, r, t, s)
    gs.check_errors()
    state = torch.cat([brain.net.params, brain.net.target, brain.net.adam_m, brain.net.adam_v])
    got = [torch.empty_like(state) for _ in range(world)]
    dist.all_gather(got, state)
    assert all(torch.equal(got[0], g) for g in got[1:]), "replicas diverged"
    assert brain.net.adam_steps == 30 - 7 and not torch.equal(brain.net.params, p0)
    try:
        brains.BrainDQNNature(2, "bird", num_envs=8, device=dev, replay_memory_per_env=4, quantile=True, peer_exchange=True)
        raise AssertionError("peer_exchange=True with quantile=True did not raise")
    except ValueError:
        pass
    dist.barrier()
    if rank == 0:
        print("QR_TWO_RANK_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
