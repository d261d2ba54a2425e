#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ from the REAL reference.

Needs a checkout of the reference project: $FLAPPY_REFERENCE, default
/root/reference (as oracle/ref_verbatim.stage).  Nothing here is imported by the
tests; the tests read the committed .npz files.

  ref_env_trajectories.npz
      The reference's own game/wrapped_flappy_bird.py + game/flappy_bird_utils.py,
      imported UNMODIFIED on the pygame shim (oracle/pygame_shim), driven with
      scripted gap draws (game.random replaced by a scripted object -- a module
      attribute, wrapped_flappy_bird.py:3,212 -- no source edit) and scripted
      actions.  Each trajectory is a fresh import, i.e. a fresh reference
      process (PLAYER_INDEX_GEN is a module global).  Stored per step: action,
      reward, terminal, score, post-step state, the 80x80 observation computed
      by REAL cv2 exactly as FlappyBirdDQN.py:31-34 (bit-packed), and a sample
      of full 288x512x3 frames.
  ref_logs.npz
      (ACTION, REWARD, SCORE, episode ends) parsed from the five run logs the
      reference ships (dqn.log, ddqn.log, dqnnature.log, duelingdqn.log,
      prioritydqn.log) plus the two logged epsilon values of SURVEY section 4.
  ref_per.npz
      The reference's SumTree / Memory classes (BrainPrioritizedReplyDQN.py:32-151)
      AST-extracted and executed verbatim on a scripted store/sample/update
      sequence with a seeded np.random.
  cv2_preprocess.npz
      random 288x512x3 frames -> real cv2 preprocess, pre-threshold gray kept.
"""
import ast
import importlib
import os
import re
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("FLAPPY_REFERENCE", "/root/reference")


class ScriptedRandom:
    """Stands in for the `random` module inside wrapped_flappy_bird."""

    def __init__(self, gaps):
        self.gaps = list(gaps)
        self.used = 0

    def randint(self, a, b):
        assert (a, b) == (0, 7)
        g = self.gaps[self.used % len(self.gaps)]
        self.used += 1
        return int(g)


def fresh_reference_game(gaps):
    """Import the reference env as a fresh process would."""
    for m in [m for m in sys.modules if m.split(".")[0] in ("pygame", "wrapped_flappy_bird", "flappy_bird_utils")]:
        del sys.modules[m]
    sys.path.insert(0, os.path.join(ROOT, "oracle", "pygame_shim"))
    sys.path.insert(0, os.path.join(REF, "game"))
    cwd = os.getcwd()
    os.chdir(REF)                      # sprites load by relative path, flappy_bird_utils.py:19-32
    try:
        game = importlib.import_module("wrapped_flappy_bird")
    finally:
        os.chdir(cwd)
        sys.path.pop(0); sys.path.pop(0)
    game.random = ScriptedRandom(gaps)
    return game


def preprocess(observ):
    # FlappyBirdDQN.py:31-34, verbatim calls
    observ = cv2.cvtColor(cv2.resize(observ, (80, 80)), cv2.COLOR_BGR2GRAY)
    ret, observ = cv2.threshold(observ, 1, 255, cv2.THRESH_BINARY)
    return np.reshape(observ, (80, 80, 1))


def state_of(game, gs):
    """post-step state in the shared 16-int export order (see oracle fo_env_export_state)."""
    out = np.zeros(16, np.int32)
    out[0] = int(gs.playery); out[1] = gs.playerVelY; out[2] = gs.playerIndex; out[3] = gs.loopIter
    out[5] = gs.basex; out[6] = gs.score; out[7] = len(gs.upperPipes)
    for k, (u, l) in enumerate(zip(gs.upperPipes, gs.lowerPipes)):
        out[8 + k] = int(u["x"])
        gapY = u["y"] + game.PIPE_HEIGHT          # :218
        out[11 + k] = (gapY - 80 - 20) // 10
        assert l["y"] == gapY + game.PIPEGAPSIZE
    out[14] = game.random.used
    return out


def policy_actions(kind, T, rng):
    if kind == "noop":
        return lambda t, gs, game: 0
    if kind == "flap":
        return lambda t, gs, game: 1
    if kind == "random":
        a = rng.integers(0, 2, T)
        return lambda t, gs, game: int(a[t])
    if kind == "sparse":
        a = (rng.random(T) < 0.08).astype(int)
        return lambda t, gs, game: int(a[t])
    if kind == "controller":            # SURVEY 8(d) coverage mix
        u = rng.random(T)

        def f(t, gs, game):
            nxt = None
            for up in gs.upperPipes:
                if up["x"] + game.PIPE_WIDTH > gs.playerx:
                    nxt = up; break
            centre = (nxt["y"] + game.PIPE_HEIGHT + game.PIPEGAPSIZE / 2) if nxt else 256
            below = (gs.playery + 12) - centre > 8
            return int(u[t] < (0.9 if below else 0.02))
        return f
    raise ValueError(kind)


def gen_env_trajectories():
    rng = np.random.default_rng(20261018)
    specs = [("controller", 3000), ("controller", 3000), ("controller", 3000), ("random", 1500),
             ("sparse", 1500), ("noop", 60), ("flap", 160), ("controller", 3000)]
    out = {}
    n_frames_kept = 0
    for ti, (kind, T) in enumerate(specs):
        gaps = rng.integers(0, 8, 509).astype(np.uint8)       # prime length: wraps out of phase
        game = fresh_reference_game(gaps)
        gs = game.GameState()
        pol = policy_actions(kind, T, rng)
        acts = np.zeros(T, np.uint8); rew = np.zeros(T, np.float32); term = np.zeros(T, np.uint8)
        score = np.zeros(T, np.int32); st = np.zeros((T, 16), np.int32)
        obs = np.zeros((T, 800), np.uint8)
        keep_idx, keep_frames = [], []
        for t in range(T):
            a = 0 if t == 0 else pol(t, gs, game)             # first step is the driver's no-op, FlappyBirdDQN.py:65-66
            onehot = np.array([1, 0]) if a == 0 else np.array([0, 1])
            image, r, done, sc = gs.frame_step(onehot)
            assert image.shape == (288, 512, 3) and image.dtype == np.uint8
            o = preprocess(image)[:, :, 0]
            assert set(np.unique(o)) <= {0, 255}
            acts[t] = a; rew[t] = r; term[t] = done; score[t] = sc; st[t] = state_of(game, gs)
            obs[t] = np.packbits(o > 0)
            if t % 97 == 0 or done or r == 3:
                if len(keep_idx) < 24:
                    keep_idx.append(t); keep_frames.append(image.copy())
        out[f"t{ti}_kind"] = np.array(kind)
        out[f"t{ti}_gaps"] = gaps
        out[f"t{ti}_actions"] = acts; out[f"t{ti}_reward"] = rew; out[f"t{ti}_terminal"] = term
        out[f"t{ti}_score"] = score; out[f"t{ti}_state"] = st; out[f"t{ti}_obsbits"] = obs
        # every other kept frame: full 288x512x3 frames dominate the file, which stays under 1 MB this way
        out[f"t{ti}_frame_idx"] = np.array(keep_idx[::2], np.int32)
        out[f"t{ti}_frames"] = np.stack(keep_frames[::2])
        n_frames_kept += len(keep_idx[::2])
        print(f"traj {ti} {kind:10s} T={T} crashes={int(term.sum())} scores={int((rew == 3).sum())} "
              f"max_pipes={int(st[:, 7].max())} gaps_used={game.random.used}")
    out["n_traj"] = np.array(len(specs))
    out["cv2_version"] = np.array(cv2.__version__)
    np.savez_compressed(os.path.join(HERE, "ref_env_trajectories.npz"), **out)
    print("frames kept:", n_frames_kept)


def gen_env_long():
    """ONE long reference trajectory with a competent (and occasionally lapsing) controller: >= 1,000 scoring events, pipes
    spawned / popped hundreds of times, crashes into LOWER pipes, upper pipes and the ground -- the reference's own
    game/wrapped_flappy_bird.py on the shim, real cv2 preprocess.  Stored per step: action, reward, terminal, score, state;
    the 80x80 observation (bit-packed) for every 5th step and every step with a score or a crash."""
    rng = np.random.default_rng(20261019)
    T = 42000
    gaps = rng.integers(0, 8, 1021).astype(np.uint8)          # prime length
    game = fresh_reference_game(gaps)
    gs = game.GameState()
    acts = np.zeros(T, np.uint8); rew = np.zeros(T, np.float32); term = np.zeros(T, np.uint8)
    score = np.zeros(T, np.int32); st = np.zeros((T, 16), np.int32)
    obs_idx, obs_bits, crash_kind = [], [], []
    lapse, lapse_p = 0, 0.0
    for t in range(T):
        if t == 0:
            a = 0
        else:
            nxt = None
            for up in gs.upperPipes:
                if up["x"] + game.PIPE_WIDTH > gs.playerx:
                    nxt = up; break
            centre = (nxt["y"] + game.PIPE_HEIGHT + game.PIPEGAPSIZE / 2) if nxt else 256
            if lapse > 0:
                lapse -= 1
                a = int(rng.random() < lapse_p)                         # a lapse either stops flapping (falls into a lower pipe
                                                                         # or the ground) or flaps wildly (climbs into an upper pipe)
            else:
                a = int((gs.playery + 12) - centre > 14)
                if rng.random() < 0.0016:
                    lapse = int(rng.integers(12, 40))
                    lapse_p = 0.0 if rng.random() < 0.6 else 0.6
        y_before = gs.playery
        onehot = np.array([1, 0]) if a == 0 else np.array([0, 1])
        image, r, done, sc = gs.frame_step(onehot)
        o = preprocess(image)[:, :, 0]
        acts[t] = a; rew[t] = r; term[t] = done; score[t] = sc; st[t] = state_of(game, gs)
        if t % 5 == 0 or done or r == 3:
            obs_idx.append(t); obs_bits.append(np.packbits(o > 0))
        if done:
            crash_kind.append(int(y_before))
    out = {"gaps": gaps, "actions": acts, "reward": rew, "terminal": term, "score": score, "state": st,
           "obs_idx": np.array(obs_idx, np.int32), "obsbits": np.stack(obs_bits), "crash_y_before": np.array(crash_kind, np.int32),
           "cv2_version": np.array(cv2.__version__)}
    np.savez_compressed(os.path.join(HERE, "ref_env_long.npz"), **out)
    print(f"long trajectory: T={T} scores={int((rew == 3).sum())} crashes={int(term.sum())} max_score={int(score.max())} "
          f"frames kept={len(obs_idx)} gaps_used={game.random.used}")


def gen_logs():
    out = {}
    pat = re.compile(r"TIMESTEP (\d+) / STATE (\w+) / ACTION ([\d.]+) / EPSILON (\S+) / REWARD (\S+)(?: / SCORE (\d+))?")
    for name in ["dqn", "ddqn", "dqnnature", "duelingdqn", "prioritydqn"]:
        acts, rews, scores, ends, eps, ts = [], [], [], [], [], []
        with open(os.path.join(REF, name + ".log")) as f:
            for line in f:
                m = pat.match(line)
                if m:
                    ts.append(int(m.group(1))); acts.append(int(float(m.group(3)))); eps.append(float(m.group(4)))
                    rews.append(float(m.group(5))); scores.append(int(m.group(6)) if m.group(6) else -1)
                elif line.startswith("GAME_TIMES"):
                    ends.append(len(acts) - 1)
        out[name + "_timestep"] = np.array(ts, np.int64)
        out[name + "_action"] = np.array(acts, np.uint8)
        out[name + "_reward"] = np.array(rews, np.float32)
        out[name + "_score"] = np.array(scores, np.int32)
        out[name + "_episode_end"] = np.array(ends, np.int32)
        out[name + "_epsilon"] = np.array(eps, np.float64)
        print(name, len(acts), "steps", len(ends), "episodes")
    np.savez_compressed(os.path.join(HERE, "ref_logs.npz"), **out)


def load_reference_per_classes():
    src = open(os.path.join(REF, "BrainPrioritizedReplyDQN.py")).read()
    tree = ast.parse(src)
    keep = [n for n in tree.body if isinstance(n, ast.ClassDef) and n.name in ("SumTree", "Memory")]
    ns = {"np": np}
    exec(compile(ast.Module(body=keep, type_ignores=[]), "BrainPrioritizedReplyDQN.py", "exec"), ns)
    return ns["SumTree"], ns["Memory"]


def gen_per():
    SumTree, Memory = load_reference_per_classes()
    out = {}
    for case, (cap, n_store, batch, rounds) in enumerate([(8, 5, 4, 6), (50, 120, 8, 40), (1000, 1500, 32, 60), (50000, 3000, 32, 30)]):
        np.random.seed(1000 + case)
        rng = np.random.default_rng(77 + case)
        mem = Memory(cap)
        for k in range(n_store):
            mem.store(k)
        u_all, idx_all, w_all, err_all, tot_all, data_all = [], [], [], [], [], []
        for r in range(rounds):
            # record the uniforms np.random.uniform will produce: replay the legacy state
            st = np.random.get_state()
            total = mem.sum_tree.total_p
            seg = total / batch
            us = np.array([np.random.uniform(seg * i, seg * (i + 1)) for i in range(batch)])
            np.random.set_state(st)
            idx, data, w = mem.sample(batch)
            errs = rng.random(batch) * rng.choice([0.01, 0.5, 3.0])
            mem.batch_update(idx, errs.copy())
            u_all.append(us); idx_all.append(idx.copy()); w_all.append(w[:, 0].copy()); err_all.append(errs)
            tot_all.append(total); data_all.append(np.array([int(d) for d in data]))
            for k in range(3):                       # interleave stores like setPerception does
                mem.store(n_store + r * 3 + k)
        out[f"c{case}_cap"] = np.array(cap); out[f"c{case}_nstore"] = np.array(n_store); out[f"c{case}_batch"] = np.array(batch)
        out[f"c{case}_v"] = np.stack(u_all); out[f"c{case}_idx"] = np.stack(idx_all); out[f"c{case}_w"] = np.stack(w_all)
        out[f"c{case}_abs_err"] = np.stack(err_all); out[f"c{case}_total"] = np.array(tot_all); out[f"c{case}_data"] = np.stack(data_all)
        out[f"c{case}_final_tree"] = mem.sum_tree.tree.copy()
        out[f"c{case}_final_beta"] = np.array(mem.beta)
        print("per case", case, "cap", cap, "final total", mem.sum_tree.total_p)
    out["n_cases"] = np.array(4)
    np.savez_compressed(os.path.join(HERE, "ref_per.npz"), **out)


def gen_cv2():
    rng = np.random.default_rng(5)
    frames = rng.integers(0, 256, (4, 288, 512, 3), dtype=np.uint8)
    # low-intensity frames exercise the `> 1` threshold boundary
    frames[2] = rng.integers(0, 6, (288, 512, 3), dtype=np.uint8)
    frames[3] = (rng.random((288, 512, 3)) < 0.02) * rng.integers(0, 256, (288, 512, 3), dtype=np.uint8)
    frames = frames[[0, 2, 3]]        # one frame of each kind (full range, low intensity, sparse): the file stays under 1 MB
    gray = np.stack([cv2.cvtColor(cv2.resize(f, (80, 80)), cv2.COLOR_BGR2GRAY) for f in frames])
    obs = np.stack([preprocess(f)[:, :, 0] for f in frames])
    np.savez_compressed(os.path.join(HERE, "cv2_preprocess.npz"), frames=frames, gray=gray, obs=obs,
                        cv2_version=np.array(cv2.__version__))


def gen_graphs():
    """The reference's own TensorFlow graphs: MetaGraphDef files of its checkpoints (weights are absent, the graphs are not),
    parsed by oracle/tf_graph.py into JSON: vanilla DQN (BrainDQN.py:119-172, reduce_sum loss) and Nature DQN
    (BrainDQNNature.py:35-123, eval_net + target_net, reduce_mean loss; --model ddqn saved the same graph, SURVEY Q1)."""
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from oracle import tf_graph
    for out, rel in (("ref_graph_dqn.json", "train_history/dqn/4/bird-2500000.meta"),
                     ("ref_graph_dqn_nature.json", "train_history/dqn_nature/bird-2000000.meta"),
                     ("ref_graph_double_dqn.json", "train_history/double_dqn/bird-1500000.meta")):
        g = tf_graph.parse_meta(os.path.join(REF, rel))
        g["source"] = rel
        # initialisers, Saver and summary nodes are not on the path: keep what the forward / loss / gradient / Adam ops reach
        tf_graph.dump_json(g, os.path.join(HERE, out))
        print(out, len(g["nodes"]), "nodes, TensorFlow", g["tf_version"])


if __name__ == "__main__":
    which = sys.argv[1:] or ["env", "logs", "per", "cv2", "graphs"]
    if "graphs" in which: gen_graphs()
    if "envlong" in which: gen_env_long()
    if "env" in which: gen_env_trajectories()
    if "logs" in which: gen_logs()
    if "per" in which: gen_per()
    if "cv2" in which: gen_cv2()
