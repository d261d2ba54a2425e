#!/usr/bin/env python
"""Cost of n-step returns: the fused update (BrainDQNNature, fp16, minibatch 256, 16,384 envs) at n = 1, 3 and 5 in the same
process, alternating, timed with CUDA events; and the configs[2] closed loop (getAction -> frame_step -> setPerception with one
update per step) at n = 1 and n = 3.

    python tools/nstep_probe.py [--updates 1000] [--rounds 5] [--out profiles/nstep_probe.json]

The replay ring of each brain is u8[16384][C + n + 3][80][80] (3.7 GB at C = 28), far larger than L2, so the drawn frames
come from HBM.  The card's name and power limit are recorded with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch  # noqa: E402

from dqnflappybird_b200.brains import BrainDQNNature  # noqa: E402
from dqnflappybird_b200.game import GameState  # noqa: E402


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        out["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return out


def filled_brain(n, N, C, B, dev):
    brain = BrainDQNNature(2, "bird", num_envs=N, device=dev, replay_memory_per_env=C, batch_size=B, observe=1e18, seed=0,
                           max_act_batch=2048, precision="fp16", n_step=n)
    gs = GameState(num_envs=N, device=dev, seed=42, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device=dev))
    brain.setInitState(obs)
    for k in range(1, C + n + 8):
        a_row, r_row, t_row = brain.replayMemory.rows(k)
        gs.step_random(1, 0.5, 1234, a_row, r_row, t_row, None)
        brain._k = k
        brain.replayMemory.appended(k)
    brain.timeStep = 1
    return brain


def time_updates(brain, count):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(count):
        brain._trainQNetwork()
        brain.timeStep += 1
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / count


def closed_loop(n, N, B, C, steps, dev, observe_steps=4):
    brain = BrainDQNNature(2, "bird", num_envs=N, device=dev, seed=0, replay_memory_per_env=C, batch_size=B, observe=observe_steps,
                           max_act_batch=4096, n_step=n)
    gs = GameState(num_envs=N, device=dev, seed=17, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device=dev))
    brain.setInitState(obs)

    def one():
        action = brain.getAction()
        nxt, reward, terminal, score = gs.frame_step(action, out=brain.next_rows()[1:])
        brain.setPerception(nxt, action, reward, terminal, score)
    for _ in range(observe_steps + n + 8):
        one()
    torch.cuda.synchronize()
    upd0 = brain.net.adam_steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    gs.check_errors()
    res = {"n_step": n, "envs": N, "minibatch": B, "replay_per_env": C, "steps": steps, "env_frames_per_s": N * steps / (ms * 1e-3),
           "updates_per_s": (brain.net.adam_steps - upd0) / (ms * 1e-3), "ms_per_loop_step": ms / steps,
           "params_finite": bool(torch.isfinite(brain.net.params).all())}
    del brain, gs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--updates", type=int, default=1000, help="timed updates per n, split over --rounds alternating rounds")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--replay-per-env", type=int, default=28)
    ap.add_argument("--loop-steps", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nstep_probe needs a CUDA device")
    dev = "cuda:0"
    ns = (1, 3, 5)
    brains = {n: filled_brain(n, a.envs, a.replay_per_env, a.batch, dev) for n in ns}
    for n in ns:
        time_updates(brains[n], a.warmup)
    per_round = max(1, a.updates // a.rounds)
    samples = {n: [] for n in ns}
    for _ in range(a.rounds):
        for n in ns:
            samples[n].append(time_updates(brains[n], per_round))
    update = {}
    for n in ns:
        s = sorted(samples[n])
        update[f"n{n}"] = {"us_per_update_median": s[len(s) // 2], "us_per_update_min": s[0], "us_per_update_max": s[-1],
                           "rounds_us": samples[n], "updates_timed": per_round * a.rounds}
    for n in ns:
        update[f"n{n}"]["delta_vs_n1_us"] = update[f"n{n}"]["us_per_update_median"] - update["n1"]["us_per_update_median"]
    del brains
    torch.cuda.empty_cache()
    loops = {f"configs2_dqnnature_n{n}": closed_loop(n, a.envs, a.batch, a.replay_per_env, a.loop_steps, dev) for n in (1, 3)}
    res = {"card": card(), "fused_update": {"model": "BrainDQNNature", "precision": "fp16", "envs": a.envs, "minibatch": a.batch,
                                             "replay_per_env": a.replay_per_env, "timing": "CUDA events, alternating rounds", **update},
           "closed_loop": loops}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
