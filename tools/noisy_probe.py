#!/usr/bin/env python
"""Cost of noisy networks: the fused-sampling update (BrainDQNNature, fp16, minibatch 256, 16,384 envs) plain vs noisy in the
same process, alternating rounds timed with CUDA events; acting (getAction's QNetwork.act) at 16,384 and 131,072 envs plain vs
noisy; and the configs[2] closed loop (getAction -> frame_step -> setPerception with one update per step) plain vs noisy.

    python tools/noisy_probe.py [--updates 1000] [--rounds 5] [--out profiles/noisy_probe.json]

The noisy update is two effective-weight builds (online and target draw), the gradient-only update graph, and the Adam over
(mu, sigma); the plain one is a single graph with Adam inside.  The card's name and power limit are recorded with the numbers.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch  # noqa: E402

from dqnflappybird_b200.brains import BrainDQNNature  # noqa: E402
from dqnflappybird_b200.game import GameState  # noqa: E402
from dqnflappybird_b200.qnet import FrameBatch, QNetwork  # noqa: E402
from nstep_probe import card, time_updates  # noqa: E402

KINDS = ("plain", "noisy")


def filled_brain(noisy, N, C, B, dev):
    brain = BrainDQNNature(2, "bird", num_envs=N, device=dev, replay_memory_per_env=C, batch_size=B, observe=1e18, seed=0,
                           max_act_batch=2048, precision="fp16", noisy=noisy)
    gs = GameState(num_envs=N, device=dev, seed=42, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device=dev))
    brain.setInitState(obs)
    for k in range(1, C + 8):
        a_row, r_row, t_row = brain.replayMemory.rows(k)
        gs.step_random(1, 0.5, 1234, a_row, r_row, t_row, None)
        brain._k = k
        brain.replayMemory.appended(k)
    brain.timeStep = 1
    return brain


def stats(samples):
    s = sorted(samples)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1], "rounds": samples}


def acting(N, rounds, calls, dev, chunk=4096):
    """envs/s of QNetwork.act on a frame ring of N envs (the getAction of the Brains), plain vs noisy, alternating rounds"""
    gs = GameState(num_envs=N, device=dev, seed=5, history=4)
    gs.step_random(6, 0.4, 3)
    fb = FrameBatch.from_ring(gs.ring, gs.slot)
    nets = {k: QNetwork(dev, max_batch=chunk, seed=0, precision="fp16", noisy=k == "noisy") for k in KINDS}
    rng = torch.zeros(N, dtype=torch.int32, device=dev)
    acts = torch.zeros(N, dtype=torch.uint8, device=dev)
    q = torch.zeros((N, 2), dtype=torch.float32, device=dev)
    samples = {k: [] for k in KINDS}
    for r in range(rounds + 1):
        for k in KINDS:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(calls):
                nets[k].act(fb, 0.0, 1, 0, rng, acts, q)
            e1.record()
            torch.cuda.synchronize()
            if r:                                               # round 0 is the warm-up
                samples[k].append(N * calls / (e0.elapsed_time(e1) * 1e-3))
    res = {k: {"envs_per_s": stats(samples[k])} for k in KINDS}
    res["noisy_over_plain"] = res["noisy"]["envs_per_s"]["median"] / res["plain"]["envs_per_s"]["median"]
    del nets, gs
    torch.cuda.empty_cache()
    return res


def closed_loop(noisy, N, B, C, steps, dev, observe_steps=4):
    brain = BrainDQNNature(2, "bird", num_envs=N, device=dev, seed=0, replay_memory_per_env=C, batch_size=B, observe=observe_steps,
                           max_act_batch=4096, noisy=noisy)
    gs = GameState(num_envs=N, device=dev, seed=17, history=brain.ring.shape[1], ring=brain.ring)
    obs, *_ = gs.frame_step(torch.zeros(N, dtype=torch.uint8, device=dev))
    brain.setInitState(obs)

    def one():
        action = brain.getAction()
        nxt, reward, terminal, score = gs.frame_step(action, out=brain.next_rows()[1:])
        brain.setPerception(nxt, action, reward, terminal, score)
    for _ in range(observe_steps + 8):
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
    res = {"noisy": noisy, "envs": N, "minibatch": B, "replay_per_env": C, "steps": steps, "env_frames_per_s": N * steps / (ms * 1e-3),
           "updates_per_s": (brain.net.adam_steps - upd0) / (ms * 1e-3), "ms_per_loop_step": ms / steps,
           "params_finite": bool(torch.isfinite(brain.net.params).all())}
    del brain, gs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--updates", type=int, default=1000, help="timed updates per kind, split over --rounds alternating rounds")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--replay-per-env", type=int, default=28)
    ap.add_argument("--act-calls", type=int, default=20)
    ap.add_argument("--loop-steps", type=int, default=40)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("noisy_probe needs a CUDA device")
    dev = "cuda:0"
    brains = {k: filled_brain(k == "noisy", a.envs, a.replay_per_env, a.batch, dev) for k in KINDS}
    for k in KINDS:
        time_updates(brains[k], a.warmup)
    per_round = max(1, a.updates // a.rounds)
    samples = {k: [] for k in KINDS}
    for _ in range(a.rounds):
        for k in KINDS:
            samples[k].append(time_updates(brains[k], per_round))
    update = {k: {"us_per_update": stats(samples[k]), "updates_timed": per_round * a.rounds} for k in KINDS}
    update["noisy_minus_plain_us"] = update["noisy"]["us_per_update"]["median"] - update["plain"]["us_per_update"]["median"]
    finite = bool(torch.isfinite(brains["noisy"].net.params).all() and torch.isfinite(brains["noisy"].net.sigma).all())
    del brains
    torch.cuda.empty_cache()
    act = {f"envs_{N}": acting(N, a.rounds, a.act_calls, dev) for N in (16384, 131072)}
    loops = {f"configs2_dqnnature_{k}": closed_loop(k == "noisy", a.envs, a.batch, a.replay_per_env, a.loop_steps, dev) for k in KINDS}
    res = {"card": card(), "fused_update": {"model": "BrainDQNNature", "precision": "fp16", "envs": a.envs, "minibatch": a.batch,
                                             "replay_per_env": a.replay_per_env, "timing": "CUDA events, alternating rounds",
                                             "noisy_params_finite": finite, **update},
           "acting": act, "closed_loop": loops}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
