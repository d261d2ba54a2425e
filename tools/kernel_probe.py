#!/usr/bin/env python
"""Time the GEMM kernels of the tensor-core Q-network path in isolation (CUDA events), or run them under ncu.

    python tools/kernel_probe.py [--batch 2048] [--reps 20] [--which 1 2 3 4 5 6]

--which takes fb_debug_tc_kernel's ids 1..11 (NAMES below; id 0, conv1 as a kernel of its own, is retired).
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch  # noqa: E402

from dqnflappybird_b200 import _lib, qnet  # noqa: E402
from dqnflappybird_b200.game import GameState  # noqa: E402

NAMES = ["conv1_fwd_retired", "conv2_fwd", "conv3_fwd", "fc1_fwd", "conv1_wgrad", "conv3_dgrad", "fc1_dgrad", "conv1_fused_act", "conv1_fused_train", "conv1_pooled_act", "conv1_pooled_train", "conv1_pooled_nopool"]
# algorithmic FLOP per sample (SURVEY 2.2): 2 * M * N * K of the reference's own GEMM view
FLOP = [6553600, 1638400, 1843200, 1638400, 6553600, 1843200, 1638400, 6553600, 6553600, 6553600, 6553600, 6553600]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--which", type=int, nargs="*", default=list(range(1, 7)))
    a = ap.parse_args()
    B = a.batch
    gs = GameState(num_envs=B, seed=3, history=5)
    gs.step_random(60, 0.3, 7)
    order = [(gs.slot - 4 + k) % 5 for k in range(5)]
    frames = gs.ring[:, order].contiguous()
    net = qnet.QNetwork(max_batch=B, precision="bf16")
    net.params.mul_(3.0)
    act = torch.randint(0, 2, (B,), dtype=torch.uint8, device="cuda")
    rew = torch.full((B,), 0.1, device="cuda"); term = torch.zeros(B, dtype=torch.uint8, device="cuda")
    net.loss_backward("nature", frames, act, rew, term)          # fills every workspace tensor the kernels read
    torch.cuda.synchronize()
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    out = {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for w in a.which:
        _lib.check(L.fb_debug_tc_kernel(net._h, w, B, 3, net.params.data_ptr(), st), "probe")
        torch.cuda.synchronize()
        e0.record()
        _lib.check(L.fb_debug_tc_kernel(net._h, w, B, a.reps, net.params.data_ptr(), st), "probe")
        e1.record(); torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / a.reps
        out[NAMES[w]] = {"us": us, "tflops": FLOP[w] * B / (us * 1e-6) / 1e12}
    print(json.dumps({"batch": B, "reps": a.reps, "kernels": out}))


if __name__ == "__main__":
    main()
