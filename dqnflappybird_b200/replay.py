"""Device-resident replay memory (host mirror of csrc/fb_replay.cu).

Reference: the ``deque`` + ``random.sample`` of BrainDQN.py:35,69-72,197-201 and the ``SumTree`` /
``Memory`` classes of BrainPrioritizedReplyDQN.py:32-151.  Frames are never copied on append: the
memory indexes the env's own frame ring; per-step action / reward / terminal rows are written by the
act / step kernels straight into the ``[L][N]`` tensors owned here.

``n_step`` > 1 turns every transition into its n-step form (csrc/fb_replay.cu, include/flappy_b200.h fb_step_sampling):
(s_{k-1}, a_k, R_k, s_{k+n-1}, disc_k) with the return R_k and the discount disc_k computed by the gather in float64.  A
transition is live once its horizon is complete, i.e. the memory at time t holds what a 1-step memory holds at
t_eff = t - n + 1, and the ring needs C + n + 3 frames.  n-step minibatches are drawn inside the training step only
(``step_sampling``).
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib


def cpython_setsize(k: int) -> int:
    """Lib/random.py ``sample``: the population size below which CPython shuffles a pool instead of keeping a set."""
    setsize = 21
    if k > 5:
        setsize += 4 ** math.ceil(math.log(k * 3, 4))
    return setsize


MAX_N_STEP = 16


def frames_per_sample(n_step: int) -> int:
    """F of a minibatch row u8[F][80][80]: s = frames 0..3, s' = frames min(n,4)..min(n,4)+3 (5 for 1-step)"""
    return 4 + min(n_step, 4)


class Minibatch:
    __slots__ = ("frames", "actions", "rewards", "terminals", "idx", "tree_idx", "is_weights", "is_weights_f32", "env", "k",
                 "returns", "disc")


class ReplayMemory:
    """Uniform replay over ``ring`` u8[N][L][80][80] with ``capacity_per_env`` transitions per env
    (REPLAY_MEMORY = N * capacity_per_env; the reference's 50,000 is for its single env, BrainDQN.py:26).
    ``n_step``: horizon of the TD target (1 = the reference's transitions); the ring must hold C + n_step + 3 frames."""

    prioritized = False

    def __init__(self, ring: torch.Tensor, capacity_per_env: int | None = None, seed: int = 0, max_batch: int = 256, n_step: int = 1):
        assert ring.dim() == 4 and ring.dtype == torch.uint8 and ring.is_cuda and ring.is_contiguous()
        n_step = int(n_step)
        if not 1 <= n_step <= MAX_N_STEP:
            raise ValueError(f"n_step must be in 1..{MAX_N_STEP}, got {n_step}")
        self.ring = ring
        self.device = ring.device
        self.N, self.L = ring.shape[0], ring.shape[1]
        self.n_step = n_step
        self.C = capacity_per_env if capacity_per_env is not None else self.L - n_step - 3
        if self.L < self.C + n_step + 3:
            raise ValueError(f"a ring of {self.L} frames holds at most {self.L - n_step - 3} {n_step}-step transitions per env "
                             f"(capacity {self.C} needs {self.C + n_step + 3})")
        # the n_step handed to the library: 0 selects the original 1-step path for n = 1; 1 would run the n-step path at n = 1,
        # which computes the same bits (the tests hold the two against each other)
        self.lib_n_step = 0 if n_step == 1 else n_step
        self.seed = seed
        self.max_batch = max_batch
        self._L = _lib.lib()
        h = C.c_void_p()
        _lib.check(self._L.fb_replay_create(self.N, self.L, self.C, int(self.prioritized), max_batch, C.byref(h)), "fb_replay_create")
        self._h = h
        dev = self.device
        self.act = torch.zeros((self.L, self.N), dtype=torch.uint8, device=dev)
        self.rew = torch.zeros((self.L, self.N), dtype=torch.float32, device=dev)
        self.term = torch.zeros((self.L, self.N), dtype=torch.uint8, device=dev)
        self.t = 0                                  # time of the newest stored transition (0 = only the initial frame)
        B = max_batch
        self._frames = torch.empty((B, frames_per_sample(n_step), 80, 80), dtype=torch.uint8, device=dev)
        self._a = torch.empty(B, dtype=torch.uint8, device=dev)
        self._r = torch.empty(B, dtype=torch.float32, device=dev)
        self._t = torch.empty(B, dtype=torch.uint8, device=dev)
        self._idx = torch.empty(B, dtype=torch.int32, device=dev)
        self._env = torch.empty(B, dtype=torch.int32, device=dev)
        self._k = torch.empty(B, dtype=torch.int32, device=dev)
        self._ret = torch.zeros(B, dtype=torch.float64, device=dev)      # R_k and disc_k of an n-step minibatch
        self._disc = torch.zeros(B, dtype=torch.float64, device=dev)

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._L.fb_replay_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def __len__(self):
        """len(replayMemory): number of live transitions (n-step: those whose horizon is complete)"""
        return self.N * self.count_per_env()

    @property
    def t_eff(self) -> int:
        """newest transition with a complete n-step horizon: t - n_step + 1 (t for 1-step)"""
        return self.t - self.n_step + 1

    def count_per_env(self) -> int:
        t = self.t_eff
        return max(0, t - max(1, t - self.C + 1) + 1) if t >= 1 else 0

    def rows(self, k: int):
        """(actions, rewards, terminals) rows of step k, for the act / step kernels to write into"""
        s = k % self.L
        return self.act[s], self.rew[s], self.term[s]

    def appended(self, k: int):
        """replayMemory.append(transition) (BrainDQN.py:70-72): step k of every env is now stored"""
        self.t = k

    def _gather(self, idx: torch.Tensor, batch: int, per: bool) -> Minibatch:
        if self.n_step != 1:
            raise ValueError("n-step minibatches are drawn inside the training step only (step_sampling)")
        _lib.check(self._L.fb_replay_gather(self._h, self.ring.data_ptr(), self.act.data_ptr(), self.rew.data_ptr(),
                                            self.term.data_ptr(), self.t, int(per), idx.data_ptr(), batch,
                                            self._frames.data_ptr(), self._a.data_ptr(), self._r.data_ptr(), self._t.data_ptr(),
                                            self._env.data_ptr(), self._k.data_ptr(), self._stream()), "fb_replay_gather")
        return self._minibatch(idx, batch)

    def _minibatch(self, idx: torch.Tensor, batch: int) -> Minibatch:
        mb = Minibatch()
        mb.frames, mb.actions, mb.rewards, mb.terminals = self._frames[:batch], self._a[:batch], self._r[:batch], self._t[:batch]
        mb.idx, mb.env, mb.k = idx[:batch], self._env[:batch], self._k[:batch]
        mb.tree_idx = mb.is_weights = mb.is_weights_f32 = None
        mb.returns, mb.disc = (self._ret[:batch], self._disc[:batch]) if self.lib_n_step else (None, None)
        return mb

    def _nstep_fields(self):
        return self.lib_n_step, self._ret.data_ptr(), self._disc.data_ptr()

    def step_sampling(self, batch: int):
        """``sample(batch)`` as a descriptor instead of two launches: (fb_step_sampling, Minibatch of the buffers it fills).
        ``QNetwork.train_step(..., sampling=...)`` runs the draw and the gather as the first two kernels of the update."""
        if self.t_eff < 1 or len(self) < batch:
            raise ValueError("Sample larger than population or is negative")
        sp = _lib.StepSampling(self._h.value, self.ring.data_ptr(), self.act.data_ptr(), self.rew.data_ptr(), self.term.data_ptr(), self.t,
                               batch, cpython_setsize(batch), self.seed, self._idx.data_ptr(), self._frames.data_ptr(), self._a.data_ptr(),
                               self._r.data_ptr(), self._t.data_ptr(), self._env.data_ptr(), self._k.data_ptr(),
                               0, 0, 0.0, None, None, None, None, *self._nstep_fields())
        return sp, self._minibatch(self._idx, batch)

    def sample(self, batch: int) -> Minibatch:
        """random.sample(self.replayMemory, BATCH_SIZE) (BrainDQN.py:197) + the four list comprehensions (:198-201)"""
        if self.n_step != 1:
            raise ValueError("n-step minibatches are drawn inside the training step only (step_sampling)")
        rc = self._L.fb_replay_sample_uniform(self._h, self.t, batch, cpython_setsize(batch), self.seed, self._idx.data_ptr(),
                                              self._stream())
        if rc == -1 and b"Sample larger" in self._L.fb_last_error():
            raise ValueError("Sample larger than population or is negative")
        _lib.check(rc, "fb_replay_sample_uniform")
        return self._gather(self._idx, batch, per=False)

    def rng_positions(self):
        pos = (C.c_uint64 * 2)()
        _lib.check(self._L.fb_replay_rng_pos(self._h, pos, 0, self._stream()), "fb_replay_rng_pos")
        return int(pos[0]), int(pos[1])

    def set_rng_positions(self, pos):
        """restore the (uniform, prioritized) word-stream positions ``rng_positions()`` returned (resume / replay of a draw)"""
        arr = (C.c_uint64 * 2)(int(pos[0]), int(pos[1]))
        _lib.check(self._L.fb_replay_rng_pos(self._h, arr, 1, self._stream()), "fb_replay_rng_pos")


class PrioritizedMemory(ReplayMemory):
    """``Memory`` (BrainPrioritizedReplyDQN.py:107-151) on a device SumTree.

    mode "reference": every update is the reference's ``ancestor += change`` in item order (bit-identical
    float64 tree for one env); mode "rebuild": ancestors recomputed as left+right (parallel; default for N > 1).
    """

    prioritized = True
    epsilon, alpha, beta_increment_per_sampling, abs_err_upper = 0.01, 0.6, 0.001, 1.0

    def __init__(self, ring, capacity_per_env=None, seed=0, max_batch=256, mode: str | None = None, n_step: int = 1):
        super().__init__(ring, capacity_per_env, seed, max_batch, n_step)
        self.mode = mode or ("reference" if self.N == 1 else "rebuild")
        self._mode = {"reference": 0, "rebuild": 1}[self.mode]
        self.beta = 0.4
        dev = self.device
        self._tree_idx = torch.empty(max_batch, dtype=torch.int32, device=dev)
        self._isw = torch.empty(max_batch, dtype=torch.float64, device=dev)
        self._isw32 = torch.empty(max_batch, dtype=torch.float32, device=dev)     # what the tf.float32 placeholder receives (:243)
        self._prio = torch.empty(max_batch, dtype=torch.float64, device=dev)
        self._gmin = None

    def use_global_min(self, on: bool = True):
        """Several ranks, one memory sharded over them: ``min_prob`` of Memory.sample (:131) is the minimum over EVERY leaf, so the
        shards agree on it with one MIN all-reduce of a scalar before each sample (ISWeights = (p_i / min_p)^-beta needs nothing
        else that is global).  Needs an initialised process group; off: each shard normalises by its own minimum."""
        if on:
            if self._gmin is None:
                self._gmin = torch.empty(1, dtype=torch.float64, device=self.device)
            _lib.check(self._L.fb_per_set_global_min(self._h, self._gmin.data_ptr()), "fb_per_set_global_min")
        else:
            _lib.check(self._L.fb_per_set_global_min(self._h, None), "fb_per_set_global_min")
            self._gmin = None

    def _reduce_min(self):
        if self._gmin is not None:
            _lib.check(self._L.fb_per_min_root(self._h, self._gmin.data_ptr(), self._stream()), "fb_per_min_root")
            torch.distributed.all_reduce(self._gmin, op=torch.distributed.ReduceOp.MIN)

    def appended(self, k: int):
        """Memory.store(transition) for step k of every env (:121-125): new leaves get the max priority.  n-step: the
        transition stored is k - n_step + 1, the one whose horizon step k completes (none while that is below 1)"""
        super().appended(k)
        if k - self.n_step + 1 >= 1:
            _lib.check(self._L.fb_per_store(self._h, k - self.n_step + 1, self._mode, self._stream()), "fb_per_store")

    def sample(self, batch: int) -> Minibatch:
        """Memory.sample(n) (:127-144) -> tree_idx, minibatch, ISWeights"""
        if self.n_step != 1:
            raise ValueError("n-step minibatches are drawn inside the training step only (step_sampling)")
        self.beta = min(1.0, self.beta + self.beta_increment_per_sampling)
        self._reduce_min()
        _lib.check(self._L.fb_per_sample(self._h, batch, self.beta, self.seed, self._tree_idx.data_ptr(), self._idx.data_ptr(),
                                         self._isw.data_ptr(), self._prio.data_ptr(), self._isw32.data_ptr(), self._stream()),
                   "fb_per_sample")
        mb = self._gather(self._idx, batch, per=True)
        mb.tree_idx = self._tree_idx[:batch]
        mb.is_weights = self._isw[:batch]
        mb.is_weights_f32 = self._isw32[:batch]
        return mb

    def step_sampling(self, batch: int):
        """``sample(batch)`` (and the ``batch_update`` that follows the update) as a descriptor: Memory.sample rides at the head
        of ``QNetwork.train_step(..., sampling=...)``'s graph, Memory.batch_update at its tail"""
        if self.lib_n_step and self.t_eff < 1:
            raise ValueError("Sample larger than population or is negative")      # no transition has a complete horizon yet
        self.beta = min(1.0, self.beta + self.beta_increment_per_sampling)
        self._reduce_min()                       # enqueued ahead of the step's graph on the same stream
        sp = _lib.StepSampling(self._h.value, self.ring.data_ptr(), self.act.data_ptr(), self.rew.data_ptr(), self.term.data_ptr(), self.t,
                               batch, 0, self.seed, self._idx.data_ptr(), self._frames.data_ptr(), self._a.data_ptr(),
                               self._r.data_ptr(), self._t.data_ptr(), self._env.data_ptr(), self._k.data_ptr(),
                               1, self._mode, self.beta, self._tree_idx.data_ptr(), self._isw.data_ptr(), self._prio.data_ptr(),
                               self._isw32.data_ptr(), *self._nstep_fields())
        mb = self._minibatch(self._idx, batch)
        mb.tree_idx, mb.is_weights, mb.is_weights_f32 = self._tree_idx[:batch], self._isw[:batch], self._isw32[:batch]
        return sp, mb

    def batch_update(self, tree_idx: torch.Tensor, abs_errors: torch.Tensor | None = None, priorities: torch.Tensor | None = None):
        """Memory.batch_update(tree_idx, abs_errors) (:146-151)"""
        n = tree_idx.shape[0]
        ae = abs_errors.data_ptr() if abs_errors is not None else None
        pr = priorities.data_ptr() if priorities is not None else None
        _lib.check(self._L.fb_per_update(self._h, tree_idx.data_ptr(), ae, pr, n, self._mode, self._stream()), "fb_per_update")

    def tree(self) -> torch.Tensor:
        """copy of the SumTree array, f64[2*capacity-1]"""
        n = 2 * self.N * self.C - 1
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        _lib.check(self._L.fb_per_tree_copy(self._h, out.data_ptr(), n, self._stream()), "fb_per_tree_copy")
        return out

    def aux_tree(self, which: str) -> torch.Tensor:
        """copy of the min-positive-leaf ("min") or max-leaf ("max") tree kept beside the SumTree (same shape): the device
        reads Memory.sample's min_prob and Memory.store's max priority from their roots instead of scanning the leaves"""
        n = 2 * self.N * self.C - 1
        out = torch.empty(n, dtype=torch.float64, device=self.device)
        _lib.check(self._L.fb_per_aux_tree_copy(self._h, {"min": 1, "max": 2}[which], out.data_ptr(), n, self._stream()), "fb_per_aux_tree_copy")
        return out

    @property
    def total_p(self) -> float:
        return float(self.tree()[0].item())
