#!/usr/bin/env python
"""Where the in-step gradient exchange's time goes (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/dist_probe.py

Times the minibatch-256 training step (CUDA events, max over ranks) with the exchange as shipped, and with parts of it switched
off through fb_dist_debug_mask (the results of those runs are WRONG by construction -- this is a timing experiment):
bucket 0 = W_fc1 beside the backward pass, bucket 1 = the other 79,522 parameters at the step's tail."""
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from dqnflappybird_b200 import _lib, dist as fdist, qnet  # noqa: E402
from dqnflappybird_b200.game import GameState  # noqa: E402


def main():
    rank, world, local = fdist.init("nccl")
    dev = torch.device("cuda", local)
    B, K = 256, 300
    gs = GameState(num_envs=B, device=dev, seed=50 + rank, history=5)
    gs.step_random(45, 0.3, 11 + rank)
    order = [(gs.slot - 4 + k) % 5 for k in range(5)]
    frames = gs.ring[:, order].contiguous()
    a = (torch.rand(B, device=dev) < 0.5).to(torch.uint8)
    r = torch.full((B,), 0.1, device=dev)
    term = torch.zeros(B, dtype=torch.uint8, device=dev)
    net = qnet.QNetwork(device=dev, max_batch=B, seed=5, precision="fp16")
    x = net.enable_peer_exchange()
    assert net.exchange_in_step
    L = _lib.lib()
    out = {}
    cases = [("as shipped", 0), ("bucket 0 sums its own gradient only (no NVLink reads)", 1), ("bucket 1 sums its own gradient only", 2),
             ("both local sums, handshakes kept", 3), ("bucket 0 without handshake or reads", 5), ("bucket 1 without handshake or reads", 10),
             ("no exchange work at all", 15)]
    for name, mask in cases:
        _lib.check(L.fb_dist_debug_mask(x._h, mask), "fb_dist_debug_mask")
        for on in (0, 1):                                                           # drop the graphs: re-capture with the new mask
            _lib.check(L.fb_qnet_use_graphs(net._h, on), "fb_qnet_use_graphs")
        dist.barrier()
        for _ in range(20):
            net.train_step("nature", frames, a, r, term, global_batch=B * world)
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            net.train_step("nature", frames, a, r, term, global_batch=B * world)
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / K * 1000.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out[name] = round(t.item(), 2)
        dist.barrier()
    if rank == 0:
        print(json.dumps({"world": world, "minibatch_per_rank": B, "us_per_update": out}, indent=1))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
