"""TEST / BENCH INFRASTRUCTURE ONLY -- the reference's own Python, executed verbatim, as the CPU baseline.

The reference (angela000/DQNFlappyBird) is a Python program without packaging metadata; its env needs pygame and its Brains
need TensorFlow 1.12, neither of which exists in this image.  What CAN run unmodified is

  * ``game/wrapped_flappy_bird.py`` + ``game/flappy_bird_utils.py`` on the ~120-line pygame shim of ``oracle/pygame_shim``
    (the same arrangement that generated ``tests/golden/ref_env_trajectories.npz``), followed by the three cv2 calls of
    ``FlappyBirdDQN.py:31-34``;
  * the ``SumTree`` / ``Memory`` classes of ``BrainPrioritizedReplyDQN.py:32-151`` (AST-extracted, numpy only).

``stage()`` copies exactly those files (plus the sprites they load and the five run logs) from the reference checkout
(``$FLAPPY_REFERENCE``, default ``/root/reference``, the ``reference_path`` of BASELINE.json) into the git-ignored
``oracle/_ref/``; the reference is not part of this repository, and a copied tree that keeps ``oracle/_ref/`` can run the
verbatim baseline where there is no checkout.  ``__graft_entry__.build()`` calls it; it does nothing when there is no
checkout.  Nothing under ``dqnflappybird_b200/`` imports this module.

Three env figures are reported by ``bench.py`` (SURVEY 8d), each labelled:
  1. as shipped: 30 frames/s/process -- ``FPSCLOCK.tick(FPS)`` sleeps every frame (wrapped_flappy_bird.py:14,179);
  2. verbatim on the shim with the clock neutralised (``game.FPSCLOCK`` replaced by a no-op object, no source edit), one
     process per host core because ``SCREEN`` / ``FPSCLOCK`` / ``PLAYER_INDEX_GEN`` are module globals (one env per process);
     NumPy blits are slower than SDL's C blits, so this flatters the GPU;
  3. the fair CPU figure: the C port ``oracle/flappy_oracle.c`` (what SDL + cv2 do natively), all host threads.
"""
from __future__ import annotations

import ast
import glob
import os
import shutil
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")
SHIM = os.path.join(ROOT, "oracle", "pygame_shim")


def stage(ref_root: str | None = None, dst: str = DST) -> bool:
    """Copy the files named above from the reference checkout (default: $FLAPPY_REFERENCE, else /root/reference) into
    oracle/_ref (idempotent).  False if there is no checkout."""
    ref_root = ref_root or os.environ.get("FLAPPY_REFERENCE", "/root/reference")
    if not os.path.isdir(os.path.join(ref_root, "game")):
        return False
    os.makedirs(os.path.join(dst, "game"), exist_ok=True)
    os.makedirs(os.path.join(dst, "assets", "sprites"), exist_ok=True)
    for f in glob.glob(os.path.join(ref_root, "game", "*.py")):
        shutil.copy2(f, os.path.join(dst, "game"))
    for f in glob.glob(os.path.join(ref_root, "assets", "sprites", "*.png")):
        shutil.copy2(f, os.path.join(dst, "assets", "sprites"))
    shutil.copy2(os.path.join(ref_root, "BrainPrioritizedReplyDQN.py"), dst)
    for f in glob.glob(os.path.join(ref_root, "*.log")):
        shutil.copy2(f, dst)
    return True


def available(dst: str = DST) -> bool:
    return os.path.exists(os.path.join(dst, "game", "wrapped_flappy_bird.py")) and os.path.isdir(os.path.join(dst, "assets", "sprites"))


class _NoTick:
    """stands in for pygame.time.Clock(): FPSCLOCK.tick(FPS) would sleep to 30 frames/s (wrapped_flappy_bird.py:179)"""

    def tick(self, *a, **k):
        return 0


def _import_game(dst: str):
    for m in [m for m in sys.modules if m.split(".")[0] in ("pygame", "wrapped_flappy_bird", "flappy_bird_utils")]:
        del sys.modules[m]
    sys.path.insert(0, SHIM)
    sys.path.insert(0, os.path.join(dst, "game"))
    cwd = os.getcwd()
    os.chdir(dst)                                  # sprites load by relative path (flappy_bird_utils.py:19-32)
    try:
        import importlib
        game = importlib.import_module("wrapped_flappy_bird")
    finally:
        os.chdir(cwd)
    game.FPSCLOCK = _NoTick()
    return game


def _env_worker(args):
    """one reference process: GameState() + frame_step(random one-hot action) + preprocess; `segments` timed loops of `n_steps`"""
    dst, n_steps, seed, p_flap, segments = args
    import cv2
    import numpy as np
    cv2.setNumThreads(1)
    game = _import_game(dst)
    rng = np.random.default_rng(seed)
    gs = game.GameState()

    def step(flap):
        a = np.zeros(2); a[1 if flap else 0] = 1
        image, reward, terminal, score = gs.frame_step(a)
        obs = cv2.cvtColor(cv2.resize(image, (80, 80)), cv2.COLOR_BGR2GRAY)           # FlappyBirdDQN.py:32
        _, obs = cv2.threshold(obs, 1, 255, cv2.THRESH_BINARY)                        # FlappyBirdDQN.py:33
        return obs, reward, terminal
    for k in range(8):
        step(k & 1)
    times, acc = [], 0
    for _ in range(segments):
        flaps = rng.random(n_steps) < p_flap
        t0 = time.perf_counter()
        for k in range(n_steps):
            obs, r, t = step(flaps[k])
            acc += int(obs[40, 10]) + int(t)
        times.append(time.perf_counter() - t0)
    return times, acc


def env_segments(processes: int, n_steps: int, segments: int, p_flap: float = 0.5, dst: str = DST):
    """`segments` timed loops of `n_steps` frame_steps in each of `processes` reference processes (one env per OS process, as
    the reference's module globals require: each is `python -m oracle.ref_verbatim --worker ...`).  Returns, per segment, the
    slowest process' seconds (the processes run side by side; imports and sprite loading are outside the timed loops)."""
    import subprocess
    procs = [subprocess.Popen([sys.executable, "-m", "oracle.ref_verbatim", "--worker", dst, str(n_steps), str(1234 + i), str(p_flap), str(segments)],
                              cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for i in range(processes)]
    per_proc = []
    for pr in procs:
        out, err = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError("reference worker failed:\n" + err[-2000:])
        per_proc.append([float(x) for x in out.strip().splitlines()[-1].split()[:segments]])
    return [max(t[k] for t in per_proc) for k in range(segments)]


def env_frames_per_s(processes: int, n_steps: int, p_flap: float = 0.5, dst: str = DST):
    """(frames/s over all processes, seconds of the slowest process)"""
    slowest = env_segments(processes, n_steps, 1, p_flap, dst)[0]
    return processes * n_steps / slowest, slowest


def load_per_classes(dst: str = DST):
    """SumTree and Memory of BrainPrioritizedReplyDQN.py:32-151, executed verbatim (the module's top imports TensorFlow)"""
    import numpy as np
    src = open(os.path.join(dst, "BrainPrioritizedReplyDQN.py")).read()
    import warnings
    with warnings.catch_warnings():          # the reference's docstrings hold '\\ ' escapes: its text, not ours to edit
        warnings.simplefilter("ignore", SyntaxWarning)
        tree = ast.parse(src)
    ns = {"np": np}
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name in ("SumTree", "Memory"):
            exec(compile(ast.Module([node], []), "BrainPrioritizedReplyDQN.py", "exec"), ns)
    return ns["SumTree"], ns["Memory"]


def per_sample_ms(capacity: int = 50000, batch: int = 32, calls: int = 3, dst: str = DST):
    """ms per reference Memory.sample(32) on a full 50,000-leaf tree (REPLAY_MEMORY, BrainDQN.py:26) and ms per Memory.store"""
    import numpy as np
    _, Memory = load_per_classes(dst)
    mem = Memory(capacity)
    t0 = time.perf_counter()
    for i in range(capacity):
        mem.store((i,))
    store_ms = (time.perf_counter() - t0) * 1e3 / capacity
    rng = np.random.default_rng(0)
    idx, _, _ = mem.sample(batch)
    mem.batch_update(idx, rng.random(batch) * 2)
    t0 = time.perf_counter()
    for _ in range(calls):
        idx, _, w = mem.sample(batch)
    sample_ms = (time.perf_counter() - t0) * 1e3 / calls
    return sample_ms, store_ms


if __name__ == "__main__":
    if len(sys.argv) >= 7 and sys.argv[1] == "--worker":
        times, acc = _env_worker((sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), float(sys.argv[5]), int(sys.argv[6])))
        print(" ".join(repr(t) for t in times), acc)
    else:
        print("staged" if stage() else "no reference checkout", "| available:", available())
