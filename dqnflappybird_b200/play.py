"""The reference's driver loop (FlappyBirdDQN.py:36-79), batched: ``python -m dqnflappybird_b200.play --model dqn``.

Same five steps -- build the Brain the ``--model`` flag names (FlappyBirdDQN.py:41-50), build the game, take one no-op
step for the initial state (:63-69), then ``getAction -> frame_step -> setPerception`` forever (:72-76) -- with two
differences that come from running on the device: ``num_envs`` games advance per call, and ``preprocess`` (:31-34) is
gone because ``frame_step`` already returns the 80x80 thresholded observation, drawn straight into the Brain's frame ring.
``actorcritic`` / ``policygradient`` are outside the DQN hot path (SURVEY 8f N4) and rejected like an unknown model.

Under ``torchrun`` every rank plays its own shard of the envs and the learner is replicated (dist.py).
"""
from __future__ import annotations

import argparse
import json
import time

import torch

from . import dist as fdist
from .brains import MODELS
from .game import GameState


def playFlappyBird(model: str, num_envs: int = 1, steps: int | None = None, device=None, seed: int = 0, replay_memory_per_env: int | None = None,
                   report_every: int = 0, **brain_kw):
    """Runs the loop for ``steps`` env steps (forever when None, like the reference) and returns ``(brain, game, stats)``."""
    if model not in MODELS:
        print("invalid model!")                    # FlappyBirdDQN.py:51-54
        raise SystemExit(1)
    rank, world, local_rank = fdist.init()
    if device is None:
        device = f"cuda:{local_rank}"
    first_env, n_local = fdist.shard_envs(num_envs, rank, world)
    # Step 1: init the Brain (the env draws into its ring, so no frame is ever copied)
    actionNum, gameName = 2, "bird"
    brain = MODELS[model](actionNum, gameName, num_envs=n_local, device=device, seed=seed, first_env_id=first_env,
                          replay_memory_per_env=replay_memory_per_env, **brain_kw)
    # Step 2: init Flappy Bird Game
    flappyBird = GameState(num_envs=n_local, device=device, seed=seed + 17, first_env_id=first_env, history=brain.ring.shape[1], ring=brain.ring)
    # Step 3.1: obtain init state -- one "do nothing" step
    action0 = torch.zeros(n_local, dtype=torch.uint8, device=device) if n_local > 1 else [1, 0]
    observation0, reward0, terminal, curScore = flappyBird.frame_step(action0)
    brain.setInitState(observation0)
    # Step 3.2: run the game
    t0, done, last = time.perf_counter(), 0, 0
    while steps is None or done < steps:
        action = brain.getAction()
        out = brain.next_rows()[1:] if n_local > 1 else None          # reward / terminal land in the replay rows: nothing is copied
        nextObserv, reward, terminal, curScore = flappyBird.frame_step(action, out=out)
        brain.setPerception(nextObserv, action, reward, terminal, curScore)
        done += 1
        if report_every and done % report_every == 0 and rank == 0:
            torch.cuda.synchronize(device)
            dt = time.perf_counter() - t0
            print(f"TIMESTEP {brain.timeStep} / EPSILON {brain.epsilon:.6f} / GAME_TIMES {brain.gameTimes} / "
                  f"{(done - last) * n_local * world / max(dt, 1e-9):.3e} env frames/s", flush=True)
            t0, last = time.perf_counter(), done
    flappyBird.check_errors()
    torch.cuda.synchronize(device)
    return brain, flappyBird, {"steps": done, "envs": n_local * world, "updates": brain.net.adam_steps}


def main(argv=None):
    parser = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    parser.add_argument("--model")                                   # FlappyBirdDQN.py:25-27
    parser.add_argument("--envs", type=int, default=1, help="games advanced per frame_step (the reference plays 1)")
    parser.add_argument("--steps", type=int, default=None, help="stop after this many steps (default: run forever, like the reference)")
    parser.add_argument("--root-dir", default=None, help="where saved_parameters/ and logs_bird/ go (default: nothing is written)")
    parser.add_argument("--batch", type=int, default=32)
    parser.add_argument("--replay-per-env", type=int, default=None)
    parser.add_argument("--report-every", type=int, default=1000)
    parser.add_argument("--seed", type=int, default=0)
    parser.add_argument("--n-step", type=int, default=1, help="horizon of the TD target (1: the reference's one-step target)")
    parser.add_argument("--noisy", action="store_true", help="NoisyNet exploration: factorised-Gaussian noisy fc1 and head layers")
    parser.add_argument("--noisy-sigma0", type=float, default=0.5, help="initial noise scale: sigma = sigma0 / sqrt(fan-in)")
    parser.add_argument("--distributional", action="store_true", help="C51 head: a distribution over --atoms atoms per action")
    parser.add_argument("--atoms", type=int, default=51, help="atoms of the C51 support")
    parser.add_argument("--v-min", type=float, default=-10.0, help="lowest atom of the C51 support")
    parser.add_argument("--v-max", type=float, default=20.0, help="highest atom of the C51 support")
    parser.add_argument("--quantile", action="store_true", help="QR-DQN head: --quantiles learned quantiles per action")
    parser.add_argument("--quantiles", type=int, default=32, help="quantiles per action of the QR-DQN head (1..64)")
    parser.add_argument("--kappa", type=float, default=1.0, help="threshold of the quantile-Huber loss (0: pure quantile regression)")
    parser.add_argument("--initial-epsilon", type=float, default=None,
                        help="start of the epsilon-greedy schedule (default: the reference's 0.03; 0 explores by noise alone)")
    a = parser.parse_args(argv)
    brain, _, stats = playFlappyBird(a.model, a.envs, a.steps, seed=a.seed, replay_memory_per_env=a.replay_per_env, report_every=a.report_every,
                                     batch_size=a.batch, root_dir=a.root_dir, record=a.root_dir is not None, n_step=a.n_step,
                                     noisy=a.noisy, noisy_sigma0=a.noisy_sigma0, distributional=a.distributional, atoms=a.atoms,
                                     v_min=a.v_min, v_max=a.v_max, quantile=a.quantile, quantiles=a.quantiles, kappa=a.kappa,
                                     **({} if a.initial_epsilon is None else {"initial_epsilon": a.initial_epsilon}))
    if a.root_dir is not None:
        brain.save()
    if fdist.dist.is_initialized() and fdist.dist.get_rank() != 0:
        return
    print(json.dumps(stats))


if __name__ == "__main__":
    main()
