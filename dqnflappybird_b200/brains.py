"""The reference's ``Brain*`` agents, batched over N envs and resident on the device.

Same surface as the reference (BrainDQN.py:32-239): ``Brain(actionNum, gameName)``, ``setInitState``,
``getAction``, ``setPerception(nextObserv, action, reward, terminal, curScore)``, ``_trainQNetwork`` /
``trainQNetwork``, and the attributes callers and logs read (``timeStep``, ``onlineTimeStep``, ``epsilon``,
``gameTimes``, ``replayMemory``, ``currentState``).  The module-level hyper-parameters of the reference
(BrainDQN.py:19-28) are constructor keywords with the reference's values as defaults.

    class                      reference file                      target            head     loss
    BrainDQN                   BrainDQN.py                         online net        plain    sum  (:162)
    BrainDQNNature             BrainDQNNature.py                   target net        plain    mean (:119)
    BrainDoubleDQN             BrainDoubleDQN.py:51-61             double            plain    mean
    BrainDuelingDQN            BrainDuelingDQN_CC.py:68-77         target net        dueling  mean
    BrainPrioritizedReplyDQN   BrainPrioritizedReplyDQN.py         target net        plain    mean of w*err^2, SumTree

Reference quirks (SURVEY 2.3) are switchable: ``reference_quirks=True`` reproduces what the shipped code
really executes (Q1: ``--model ddqn`` runs the Nature update; Q2: ``--model duelingdqn`` builds the plain
head; Q3: the PER brain never syncs its target net; and the PER cost as TensorFlow evaluates
``ISWeights[B,1] * squared_difference[B]`` -- broadcast to [B,B], i.e. mean(w) * mean(err^2),
BrainPrioritizedReplyDQN.py:243-251); the default runs the intended algorithm (mean of w_i * err_i^2).

``n_step`` (default 1, the reference's target) trains on n-step TD targets: y = R_k + gamma^n X(s_{k+n-1}), cut at the
first terminal inside the window (replay.py, csrc/fb_replay.cu).  It needs the minibatch drawn inside the update
(``fuse_sampling``), and for prioritized replay on several ranks the in-step gradient exchange.

``noisy=True`` explores with NoisyNet layers (Fortunato et al. 2018): fc1 and the head run on mu + sigma * eps with factorised
Gaussian noise drawn afresh for every update and every getAction (qnet.py, csrc/fb_noisy.cu).  The epsilon-greedy schedule is
left as it is; pass ``initial_epsilon=0`` to explore by the noise alone.  On several ranks it takes the NCCL all-reduce path.

All math runs in libflappy_b200.so; with torch.distributed initialised every rank trains on its own env /
replay shard and the replicated learner sums the ranks' gradients inside the update's CUDA graph over NVLink
peer memory (fb_dist.cu), or with an NCCL all-reduce before the Adam step when ``peer_exchange=False``.
"""
from __future__ import annotations

import os
import pickle

import numpy as np
import torch

from . import _lib
from .qnet import FrameBatch, QNetwork
from .replay import PrioritizedMemory, ReplayMemory

# Hyper Parameters (BrainDQN.py:19-28)
FRAME_PER_ACTION = 1
BATCH_SIZE = 32
OBSERVE = 1000.
EXPLORE = 1000000.
GAMMA = 0.99
FINAL_EPSILON = 0
INITIAL_EPSILON = 0.03
REPLAY_MEMORY = 50000
REPLACE_TARGET_ITER = 500
SAVE_EVERY = 100000                 # BrainDQN.py:227: weights, (gameTimes, timeStep, epsilon) and the logs every 100,000 steps


class BrainDQN:
    variant = "vanilla"
    dueling = False
    loss_sum = True                 # BrainDQN.py:162 reduce_sum; every subclass uses reduce_mean
    prioritized = False
    uses_target = False
    dir_name = "/dqn/"              # BrainDQN.py:62-63 _setDirName

    def __init__(self, actionNum: int = 2, gameName: str = "bird", num_envs: int = 1, device="cuda:0", ring: torch.Tensor | None = None,
                 batch_size: int = BATCH_SIZE, observe: float = OBSERVE, explore: float = EXPLORE, gamma: float = GAMMA,
                 final_epsilon: float = FINAL_EPSILON, initial_epsilon: float = INITIAL_EPSILON,
                 replay_memory_per_env: int | None = None, replace_target_iter: int | None = REPLACE_TARGET_ITER,
                 hidden: int = 512, lr: float = 1e-6, seed: int = 0, first_env_id: int = 0, updates_per_step: int = 1,
                 reference_quirks: bool = False, copy_target_at_init: bool = False, record: bool = False, max_act_batch: int = 4096,
                 precision: str = "fp16", peer_exchange: bool | None = None, root_dir: str | None = None, save_every: int = SAVE_EVERY,
                 log_capacity: int = 1 << 20, n_step: int = 1, noisy: bool = False, noisy_sigma0: float = 0.5):
        if actionNum != 2:
            raise ValueError("the Flappy Bird hot path has two actions (FlappyBirdDQN.py:38)")
        self.actionNum, self.gameName = actionNum, gameName
        self.device = torch.device(device)
        self.num_envs = N = int(num_envs)
        self.batch_size, self.observe, self.explore, self.gamma = batch_size, observe, explore, gamma
        self.final_epsilon, self.initial_epsilon = final_epsilon, initial_epsilon
        self.replace_target_iter = replace_target_iter
        self.updates_per_step = updates_per_step
        self.reference_quirks = reference_quirks
        self.record = record
        self.fuse_sampling = True                  # uniform replay on one GPU: draw the minibatch inside the update's graph
        self.seed, self.first_env_id = seed, first_env_id
        self.n_step = int(n_step)
        self.noisy = bool(noisy)
        # distributed: one process per GPU, replicated learner (SURVEY 8e)
        self.world = torch.distributed.get_world_size() if torch.distributed.is_available() and torch.distributed.is_initialized() else 1
        from .dist import local_batch as _local_batch
        self.local_batch = _local_batch(batch_size, self.world)     # raises unless the minibatch divides evenly over the ranks
        self.rank = torch.distributed.get_rank() if self.world > 1 else 0
        # init replay memory (BrainDQN.py:35): REPLAY_MEMORY transitions per env, frames shared with the env's ring
        C = replay_memory_per_env if replay_memory_per_env is not None else (REPLAY_MEMORY if N == 1 else 60)
        L = C + self.n_step + 3                      # s_{k-1} .. s_{k+n-1} of the oldest live transition (C + 4 for 1-step)
        if ring is None:
            ring = torch.zeros((N, L, 80, 80), dtype=torch.uint8, device=self.device)
        assert ring.shape == (N, L, 80, 80), f"ring must be u8[{N}][{L}][80][80] (capacity {C} + {self.n_step + 3} frames)"
        self.ring = ring
        mem_cls = PrioritizedMemory if self.prioritized else ReplayMemory
        self.replayMemory = mem_cls(ring, C, seed=seed + 1, max_batch=max(self.local_batch, 8), n_step=self.n_step)
        # init other parameters (BrainDQN.py:37-41)
        self.onlineTimeStep = 0
        self.timeStep = 0
        self.epsilon = initial_epsilon
        # init Q network (BrainDQN.py:60)
        dueling = self.dueling and not (reference_quirks and type(self).__name__ == "BrainDuelingDQN")
        self.net = QNetwork(self.device, hidden=hidden, dueling=dueling, max_batch=max(self.local_batch, min(N, max_act_batch)),
                            seed=seed, lr=lr, copy_target_at_init=copy_target_at_init, precision=precision, noisy=self.noisy,
                            sigma0=noisy_sigma0)
        if self.prioritized and reference_quirks:
            # what the shipped graph really minimises: ISWeights [B,1] x square(...) [B] broadcasts to [B,B], so every sample is
            # weighted by mean(ISWeights) (BrainPrioritizedReplyDQN.py:243-251); the default is the intended per-sample weight
            self.net.set_per_broadcast(True)
        # one process per GPU under NCCL: sum the gradients from NVLink peer memory inside the Adam kernel (fb_dist.cu)
        if self.noisy and peer_exchange:
            raise ValueError("noisy=True trains through loss_backward + all_reduce + the noisy Adam; the in-step peer exchange "
                             "applies plain Adam and is not available with it")
        if peer_exchange is None:
            peer_exchange = not self.noisy and self.world > 1 and torch.distributed.get_backend() == "nccl"
        if peer_exchange and self.world > 1:
            self.net.enable_peer_exchange()
        if self.n_step > 1 and self.prioritized and self.world > 1 and not self.net.exchange_in_step:
            raise ValueError("n_step > 1 with prioritized replay on several ranks needs the in-step gradient exchange")
        if self.prioritized and self.world > 1:
            self.replayMemory.use_global_min()     # min_prob of Memory.sample over every shard's leaves (one scalar, MIN all-reduce)
        self._k = 0                               # time index of the newest frame in the ring
        self._rng_pos = torch.zeros(N, dtype=torch.int32, device=self.device)
        self._actions = torch.zeros(N, dtype=torch.uint8, device=self.device)
        self._q = torch.zeros((N, 2), dtype=torch.float32, device=self.device)
        self._abs_err = torch.zeros(max(self.local_batch, 8), dtype=torch.float32, device=self.device)
        self._q_target = torch.zeros(max(self.local_batch, 8), dtype=torch.float32, device=self.device)
        self._game_times = torch.zeros((), dtype=torch.int64, device=self.device)
        # logs (BrainDQN.py:44-58).  With record=True they are fed from device-side accumulators (no host sync on the
        # step path) and reach these lists / the reference's five text files when flushed.
        self.gameName = gameName
        self.lost_hist, self.q_target_list = [], []
        self.score_every_episode, self.time_steps_when_episode_end, self.reward_every_time_step = [], [], []
        self.episode_envs = []                     # which env ended each logged episode (no reference equivalent: one env there)
        self.save_every = int(save_every)
        self.save_path = self.logs_path = self.saved_parameters_file_path = None
        if root_dir is not None:
            self.save_path = os.path.join(root_dir, "saved_parameters" + self.dir_name)
            self.saved_parameters_file_path = self.save_path + self.gameName + "-saved-parameters.txt"
            self.logs_path = os.path.join(root_dir, "logs_" + self.gameName + self.dir_name)      # "logs_bird/dqn/"
            os.makedirs(self.save_path, exist_ok=True)
            os.makedirs(self.logs_path, exist_ok=True)
        if record:
            cap = int(log_capacity)
            self._log_cap = cap
            self._ep_log = torch.zeros((cap, 3), dtype=torch.int32, device=self.device)
            self._ep_count = torch.zeros((), dtype=torch.int32, device=self.device)
            self._rew_log = torch.zeros(cap, dtype=torch.float32, device=self.device)
            self._rew_n = 0
            self._upd_cap = ucap = max(1, min(cap, (1 << 24) // max(1, self.local_batch)))
            self._loss_log = torch.zeros(ucap, dtype=torch.float32, device=self.device)
            self._qt_log = torch.zeros((ucap, self.local_batch), dtype=torch.float32, device=self.device)
            self._upd_n = 0
        if self.save_path is not None:
            self._load_saved_parameters()

    # ------------------------------------------------------------------ state
    @property
    def slot(self) -> int:
        return self._k % self.ring.shape[1]

    @property
    def currentState(self) -> torch.Tensor:
        """u8[N,80,80,4] copy of the last four frames, newest last (BrainDQN.py:68,239)"""
        L = self.ring.shape[1]
        idx = [max(self._k - 3 + c, 0) % L for c in range(4)]
        return self.ring[:, idx].permute(0, 2, 3, 1).contiguous()

    def _to_ring(self, observ, slot):
        dst = self.ring[:, slot]
        if torch.is_tensor(observ) and observ.is_cuda and observ.data_ptr() == dst.data_ptr():
            return                                 # the env drew straight into our ring
        o = torch.as_tensor(np.asarray(observ) if not torch.is_tensor(observ) else observ)
        dst.copy_(o.reshape(self.num_envs, 80, 80).to(self.device, torch.uint8))

    def setInitState(self, observ):
        """currentState = np.stack((observ,)*4, axis=2) (BrainDQN.py:238-239): frame 0; earlier times clamp to it"""
        self._k = 0
        self._to_ring(observ, 0)
        self.replayMemory.t = 0

    def _act_view(self) -> FrameBatch:
        L = self.ring.shape[1]
        off = [(max(self._k - 3 + c, 0) % L) * 6400 for c in range(4)]
        return FrameBatch(self.ring, L * 6400, off, self.num_envs)

    def next_rows(self):
        """(actions u8[N], rewards f32[N], terminals u8[N]): the replay rows of the transition the next setPerception will
        store.  getAction already writes its actions there; hand the other two to ``GameState.frame_step(..., out=...)`` and
        pass everything back to setPerception, which then has nothing to copy (the observation is in the shared ring too)."""
        return self.replayMemory.rows(self._k + 1)

    # ------------------------------------------------------------------ acting
    def getAction(self):
        """BrainDQN.py:99-116.  Returns u8[N] action indices on the device (0 = [1,0] no-op, 1 = [0,1] flap), written
        straight into the replay row of the coming transition; for a single env the reference's one-hot float array."""
        if self.num_envs > 1:
            self._actions = self.replayMemory.rows(self._k + 1)[0]
        self.net.act(self._act_view(), self.epsilon, self.seed + 2, self.first_env_id, self._rng_pos, self._actions, self._q)
        # change epsilon (BrainDQN.py:112-114), float64 like the reference
        if self.epsilon > self.final_epsilon and self.onlineTimeStep > self.observe:
            self.epsilon -= (self.initial_epsilon - self.final_epsilon) / self.explore
        if self.num_envs == 1:
            action = np.zeros(self.actionNum)
            action[int(self._actions[0].item())] = 1
            return action
        return self._actions

    # ------------------------------------------------------------------ perception
    def setPerception(self, nextObserv, action, reward, terminal, curScore=None):
        """BrainDQN.py:66-96 for all envs: append the transition, train once past OBSERVE, advance the counters."""
        k = self._k + 1
        L = self.ring.shape[1]
        self._to_ring(nextObserv, k % L)
        a_row, r_row, t_row = self.replayMemory.rows(k)
        dev = self.device
        same = lambda x, row: torch.is_tensor(x) and x.is_cuda and x.data_ptr() == row.data_ptr() and x.dtype == row.dtype
        if not same(action, a_row):                  # (rows handed out by next_rows() / getAction are already in place)
            a = torch.as_tensor(np.asarray(action) if not torch.is_tensor(action) else action)
            if a.dim() >= 1 and a.shape[-1] == 2 and (a.dim() == 2 or self.num_envs == 1):
                a = a.reshape(-1, 2)[:, 1]           # one-hot -> index
            a_row.copy_(a.reshape(-1).to(dev).to(torch.uint8))
        if not same(reward, r_row):
            r_row.copy_(torch.as_tensor(reward, dtype=torch.float32).reshape(-1).to(dev))
        if not same(terminal, t_row):
            t_row.copy_(torch.as_tensor(terminal).reshape(-1).to(dev).to(torch.uint8))
        self._k = k
        self.replayMemory.appended(k)               # deque.append / Memory.store
        if self.onlineTimeStep > self.observe:
            for _ in range(self.updates_per_step):
                self._trainQNetwork()
        self._game_times += t_row.sum()              # gameTimes += 1 per terminal (BrainDQN.py:88-90), kept on the device
        if self.record:
            self._log_step(r_row, t_row, curScore)
        self.timeStep += 1
        self.onlineTimeStep += 1

    @property
    def gameTimes(self) -> int:
        """episodes finished so far over all envs (BrainDQN.py:88-90); counted on the device, reading it synchronises"""
        return int(self._game_times.item())

    gameTimesTotal = gameTimes

    # ------------------------------------------------------------------ training
    def _maybe_sync_target(self):
        if self.uses_target and self.replace_target_iter and self.timeStep % self.replace_target_iter == 0:
            self.net.sync_target()                   # BrainDQNNature.py:151-152

    def _update(self, variant: str):
        mem = self.replayMemory
        sampling = None
        if self.fuse_sampling and (self.world == 1 or not self.prioritized or self.net.exchange_in_step):
            sampling, mb = mem.step_sampling(self.local_batch)    # random.sample + gather ride at the head of the step's graph
        elif self.n_step > 1:
            raise ValueError("n_step > 1 draws its minibatch inside the update: fuse_sampling must stay on (and prioritized replay "
                             "on several ranks needs the in-step gradient exchange)")
        else:
            mb = mem.sample(self.local_batch)
        isw = mb.is_weights_f32 if mb.is_weights is not None else None   # the placeholder is tf.float32 (BrainPrioritizedReplyDQN.py:243)
        args = (variant, mb.frames, mb.actions, mb.rewards, mb.terminals, isw, self.gamma, self.loss_sum, self.local_batch * self.world,
                self._abs_err[:self.local_batch], self._q_target[:self.local_batch])
        if self.world == 1 or self.net.exchange_in_step:
            # one call: on the tensor-core path one CUDA graph, Adam included -- and, on several GPUs, the gradient exchange too
            # (W_fc1's 91 % of the vector beside the convolution gradients, the rest at the tail: csrc/fb_dist.cu)
            self.net.train_step(*args, sampling=sampling)
        else:
            self.net.loss_backward(*args, sampling=sampling)
            if self.net.exchange is None:
                torch.distributed.all_reduce(self.net.grads)      # sum of per-shard gradients of the global loss
            self.net.adam_step()                                  # with a peer exchange the sum happens inside the Adam kernel
        if mb.tree_idx is not None and sampling is None:
            mem.batch_update(mb.tree_idx, abs_errors=self._abs_err[:self.local_batch])   # :316 (else: the last kernel of the step's graph)
        if self.record:                                              # BrainDQN.py:222-225, kept on the device until flushed
            if self._upd_n == self._upd_cap:
                self.flush_logs()
            self._loss_log[self._upd_n].copy_(self.net.loss.reshape(()))
            self._qt_log[self._upd_n].copy_(self._q_target[:self.local_batch])
            self._upd_n += 1
        # save network and other data every 100,000 iterations (BrainDQN.py:226-233)
        if self.save_path is not None and self.save_every and self.timeStep % self.save_every == 0:
            self.save()

    def _trainQNetwork(self):
        """BrainDQN.py:195-223"""
        self._update("vanilla")

    # ------------------------------------------------------------------ logging surface (row N3)
    def _log_step(self, r_row, t_row, curScore):
        """reward_every_time_step / score_every_episode / time_steps_when_episode_end (BrainDQN.py:87-93) without a host sync:
        the step's mean reward (the reward itself for one env) and one (timeStep, env, score) record per finished episode"""
        if self._rew_n == self._log_cap:
            self.flush_logs()
        self._rew_log[self._rew_n].copy_(r_row.mean() if self.num_envs > 1 else r_row[0])
        self._rew_n += 1
        if curScore is None:
            return
        sc = torch.as_tensor(curScore).reshape(-1).to(self.device, torch.int32)
        _lib.check(_lib.lib().fb_log_episodes(t_row.data_ptr(), sc.data_ptr(), self.num_envs, self.first_env_id, int(self.timeStep),
                                              self._ep_log.data_ptr(), self._ep_count.data_ptr(), self._log_cap,
                                              torch.cuda.current_stream(self.device).cuda_stream), "fb_log_episodes")

    def flush_logs(self):
        """move the device-side accumulators into the reference's lists (one host sync); episodes sorted by (timeStep, env)"""
        if not self.record:
            return
        n = int(self._ep_count.item())
        if n > self._log_cap:
            raise RuntimeError(f"episode log overflow: {n} episodes since the last flush, capacity {self._log_cap} (raise log_capacity)")
        if n:
            ep = self._ep_log[:n].cpu().numpy()
            ep = ep[np.lexsort((ep[:, 1], ep[:, 0]))]
            self.time_steps_when_episode_end += ep[:, 0].tolist()
            self.episode_envs += ep[:, 1].tolist()
            self.score_every_episode += ep[:, 2].tolist()
            self._ep_count.zero_()
        if self._rew_n:
            self.reward_every_time_step += [float(np.float32(x)) for x in self._rew_log[:self._rew_n].cpu().numpy()]
            self._rew_n = 0
        if self._upd_n:
            self.lost_hist += [float(x) for x in self._loss_log[:self._upd_n].cpu().numpy()]
            self.q_target_list += self._qt_log[:self._upd_n].cpu().numpy().tolist()
            self._upd_n = 0

    def _save_loss_score_timestep_reward_qtarget_to_file(self):
        """BrainDQN.py:270-294: append every list to its text file as ``str(x) + ' '`` and clear it"""
        self.flush_logs()
        if self.logs_path is None:
            raise RuntimeError("no root_dir: the brain was built without a place to put logs_<game>/<model>/")
        for name, values in (("lost_hist.txt", self.lost_hist), ("score_every_episode.txt", self.score_every_episode),
                             ("time_steps_when_episode_end.txt", self.time_steps_when_episode_end),
                             ("reward_every_time_step.txt", self.reward_every_time_step), ("q_targets.txt", self.q_target_list)):
            with open(self.logs_path + name, "a") as f:
                for v in values:
                    f.write(str(v) + " ")
            del values[:]
        del self.episode_envs[:]

    def _get_loss_score_timestep_reward_qtarget_from_file(self):
        """BrainDQN.py:297-330: the five files back as lists of floats (q_targets is a list of per-update lists there too:
        the reference parses it with the same whitespace split, which only works for its other four files -- here it is
        parsed properly)"""
        def floats(name):
            with open(self.logs_path + name) as f:
                return [float(t) for t in f.readline().split(" ")[:-1]]
        with open(self.logs_path + "q_targets.txt") as f:
            txt = f.readline()
        q = [float(t) for t in txt.replace("[", " ").replace("]", " ").replace(",", " ").split()]
        return (floats("lost_hist.txt"), floats("score_every_episode.txt"), floats("time_steps_when_episode_end.txt"),
                floats("reward_every_time_step.txt"), q)

    # ------------------------------------------------------------------ checkpoint (row N2)
    def save(self):
        """BrainDQN.py:226-233: the network (weights, target, Adam slots) under save_path + gameName + '-' + timeStep, a
        ``checkpoint`` file naming the newest one, (gameTimes, timeStep, epsilon) as three pickles in
        <game>-saved-parameters.txt exactly like the reference writes them, then the logs"""
        if self.save_path is None:
            raise RuntimeError("no root_dir: the brain was built without a place to put saved_parameters/<model>/")
        if self.world > 1:
            # replicas are bit-identical: rank 0 alone writes (concurrent writers would corrupt the files); the others
            # only flush their device-side logs and meet rank 0 at the barrier
            if self.rank != 0:
                self.flush_logs()
                for lst in (self.lost_hist, self.q_target_list, self.score_every_episode, self.time_steps_when_episode_end,
                            self.reward_every_time_step, self.episode_envs):
                    del lst[:]
                torch.distributed.barrier()
                return
        name = f"{self.gameName}-{self.timeStep}"
        torch.save(self.net.state_dict(), self.save_path + name + ".pt")
        with open(self.save_path + "checkpoint", "w") as f:
            f.write(f'model_checkpoint_path: "{name}"\n')
        with open(self.saved_parameters_file_path, "wb") as f:
            pickle.dump(self.gameTimesTotal, f)
            pickle.dump(self.timeStep, f)
            pickle.dump(self.epsilon, f)
        if self.record:
            self._save_loss_score_timestep_reward_qtarget_to_file()
        if self.world > 1:
            torch.distributed.barrier()

    def _load_saved_parameters(self) -> bool:
        """BrainDQN.py:176-192: restore the newest checkpoint if there is one; timeStep and epsilon come back,
        onlineTimeStep does not (so a resumed run observes for OBSERVE steps again, as in the reference)"""
        ck = self.save_path + "checkpoint"
        if not os.path.exists(ck):
            return False                            # "Could not find old network weights"
        with open(ck) as f:
            name = f.readline().split('"')[1]
        self.net.load_state_dict(torch.load(self.save_path + name + ".pt", map_location=self.device))
        if os.path.exists(self.saved_parameters_file_path) and os.path.getsize(self.saved_parameters_file_path) > 0:
            with open(self.saved_parameters_file_path, "rb") as f:
                self._game_times.fill_(int(pickle.load(f)))
                self.timeStep = int(pickle.load(f))
                self.epsilon = float(pickle.load(f))
        return True

    def state_dict(self):
        return {"net": self.net.state_dict(), "gameTimes": self.gameTimesTotal, "timeStep": self.timeStep, "epsilon": self.epsilon}

    def load_state_dict(self, sd):
        """_load_saved_parameters (BrainDQN.py:176-192): timeStep and epsilon are restored, onlineTimeStep is not (Q12)"""
        self.net.load_state_dict(sd["net"])
        self._game_times.fill_(int(sd["gameTimes"]))
        self.timeStep, self.epsilon = int(sd["timeStep"]), float(sd["epsilon"])


class BrainDQNNature(BrainDQN):
    variant = "nature"
    dir_name = '/dqn_nature/'              # BrainDQNNature.py:126
    loss_sum = False
    uses_target = True

    def _trainQNetwork(self):
        """BrainDQNNature.py:149-183"""
        self._maybe_sync_target()
        self._update("nature")


class BrainDoubleDQN(BrainDQNNature):
    variant = "double"
    dir_name = '/double_dqn/'              # BrainDoubleDQN.py:35

    def trainQNetwork(self):
        """BrainDoubleDQN.py:37-69 -- the Double target the file defines but the shipped loop never calls (Q1)"""
        self._maybe_sync_target()
        self._update("double")

    def _trainQNetwork(self):
        if self.reference_quirks:
            return BrainDQNNature._trainQNetwork(self)
        return self.trainQNetwork()


class BrainDuelingDQN(BrainDQNNature):
    dueling = True
    dir_name = '/dueling_dqn/'             # BrainDuelingDQN_CC.py:35

    def trainQNetwork(self):
        """BrainDuelingDQN_CC.py:171-202 (Nature target on the dueling net)"""
        return BrainDQNNature._trainQNetwork(self)


class BrainPrioritizedReplyDQN(BrainDQNNature):
    prioritized = True
    dir_name = '/prioritized_reply_dqn/'   # BrainPrioritizedReplyDQN.py:162

    def _trainQNetwork(self):
        """BrainPrioritizedReplyDQN.py:277-315; the reference never runs target_replace_op here (Q3)"""
        if not self.reference_quirks:
            self._maybe_sync_target()
        self._update("nature")


MODELS = {"dqn": BrainDQN, "ddqn": BrainDoubleDQN, "dqnnature": BrainDQNNature, "duelingdqn": BrainDuelingDQN,
          "prioritydqn": BrainPrioritizedReplyDQN}       # FlappyBirdDQN.py:41-50
