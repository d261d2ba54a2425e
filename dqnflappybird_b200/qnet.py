"""Host-side owner of the Q-network tensors; all math runs in libflappy_b200.so (csrc/fb_qnet*.cu).

Reference: the TensorFlow graph every Brain builds (BrainDQN.py:119-163; target copy
BrainDQNNature.py:75-111; dueling head BrainDuelingDQN_CC.py:68-77) and
``tf.train.AdamOptimizer(1e-6)`` (BrainDQN.py:163).  PyTorch owns the flat fp32 vectors
(parameters, target parameters, gradients, Adam slots); nothing here computes.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

VARIANTS = {"vanilla": 0, "nature": 1, "double": 2}
PRECISIONS = {"fp32": 0, "bf16": 1, "fp16": 2}


def truncated_normal_(t: torch.Tensor, std: float, generator=None):
    """tf.truncated_normal: N(0, std) resampled beyond two standard deviations (BrainDQN.py:122)."""
    torch.nn.init.trunc_normal_(t, mean=0.0, std=std, a=-2 * std, b=2 * std, generator=generator)
    return t


class FrameBatch:
    """A view of u8 frames as network inputs: sample b, channel c = base + b*stride + chan_off[c]."""

    def __init__(self, tensor: torch.Tensor, sample_stride: int, chan_off, batch: int, base_offset: int = 0):
        self.tensor = tensor                      # keeps the storage alive
        self.ptr = tensor.data_ptr() + base_offset
        self.sample_stride = int(sample_stride)
        self.chan_off = (C.c_int32 * 4)(*[int(o) for o in chan_off])
        self.batch = int(batch)

    @staticmethod
    def from_ring(ring: torch.Tensor, newest_slot: int) -> "FrameBatch":
        """Acting input: the last four frames of every env in a ring u8[N][L][80][80], newest last."""
        N, L = ring.shape[0], ring.shape[1]
        off = [((newest_slot - 3 + k) % L) * 6400 for k in range(4)]
        return FrameBatch(ring, L * 6400, off, N)

    @staticmethod
    def from_stack(frames: torch.Tensor, first: int = 0) -> "FrameBatch":
        """frames u8[B][F][80][80] with F >= first+4: channels = frames first..first+3."""
        B, Fr = frames.shape[0], frames.shape[1]
        assert frames.is_contiguous() and frames.dtype == torch.uint8 and Fr >= first + 4
        return FrameBatch(frames, Fr * 6400, [(first + k) * 6400 for k in range(4)], B)


class QNetwork:
    def __init__(self, device="cuda:0", hidden: int = 512, dueling: bool = False, max_batch: int = 256, seed: int = 0,
                 lr: float = 1e-6, beta1: float = 0.9, beta2: float = 0.999, adam_eps: float = 1e-8,
                 copy_target_at_init: bool = False, precision: str = "fp16", noisy: bool = False, sigma0: float = 0.5,
                 distributional: bool = False, atoms: int = 51, v_min: float = -10.0, v_max: float = 20.0,
                 quantile: bool = False, quantiles: int = 32, kappa: float = 1.0):
        """``quantile``: the QR-DQN head (Dabney et al. 2018, csrc/fb_qr.cu) -- per action ``quantiles`` N (1..64) learned quantile
        locations at the fractions (2i + 1) / (2N); Q is their mean, so acting is unchanged, and the update minimises the
        quantile-Huber loss with threshold ``kappa`` (0: the paper's QR-DQN-0, pure quantile regression).  ``abs_err`` receives the
        per-sample loss.  N defaults to 32, not the paper's 200: the head kernels take at most 64 outputs per action.  There is no
        support to choose.  Not together with ``distributional``.

        ``distributional``: the C51 head (Bellemare et al. 2017, csrc/fb_c51.cu) -- per action a categorical distribution over
        ``atoms`` atoms spread evenly over [v_min, v_max]; Q is its expectation, so acting is unchanged, and the update minimises the
        cross-entropy against the projected target distribution (``abs_err`` then receives that cross-entropy, Rainbow's priority).
        The support defaults to [-10, 20], not the paper's [-10, 10]: with this game's rewards (0.1 per step, +3 per pipe, -3 for a
        crash) a bird that keeps flying reaches a discounted return near 20 at gamma = 0.99, and a crash gives about -3.

        ``noisy``: NoisyNet (Fortunato et al. 2018) with factorised Gaussian noise on fc1 and the head (csrc/fb_noisy.cu).
        ``params`` / ``target`` are then mu (initialised exactly as without noise), ``sigma`` / ``target_sigma`` start at
        sigma0 / sqrt(fan-in) on the noisy layers and 0 elsewhere, and training and acting run on the effective weights
        mu + sigma * eps of a fresh draw; the noise stream is (``seed``, draw id), the same on every rank."""
        if not torch.cuda.is_available():
            raise _lib.FlappyError("QNetwork needs a CUDA device (B200); there is no CPU path")
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        self._L = _lib.lib()
        h = C.c_void_p()
        if quantile and distributional:
            raise ValueError("quantile=True and distributional=True are two different heads; choose one")
        self.quantile = bool(quantile)
        self.quantiles, self.kappa = (int(quantiles), float(kappa)) if self.quantile else (0, 0.0)
        self.distributional = bool(distributional)
        self.atoms, self.v_min, self.v_max = (int(atoms), float(v_min), float(v_max)) if self.distributional else (0, 0.0, 0.0)
        if self.distributional:
            _lib.check(self._L.fb_qnet_create_c51(hidden, int(dueling), max_batch, self.atoms, self.v_min, self.v_max, C.byref(h)),
                       "fb_qnet_create_c51")
        elif self.quantile:
            _lib.check(self._L.fb_qnet_create_qr(hidden, int(dueling), max_batch, self.quantiles, self.kappa, C.byref(h)), "fb_qnet_create_qr")
        else:
            _lib.check(self._L.fb_qnet_create(hidden, int(dueling), max_batch, C.byref(h)), "fb_qnet_create")
        self._h = h
        self.hidden, self.dueling, self.max_batch = hidden, bool(dueling), max_batch
        # "bf16" / "fp16": tcgen05 tensor cores (16-bit operands, fp32 accumulation; fp16 has TF32's significand); "fp32": strict CUDA-core FMA
        self.precision = precision
        _lib.check(self._L.fb_qnet_set_precision(self._h, PRECISIONS[precision]), "fb_qnet_set_precision")
        self._seen_versions = None
        self.compute_path = {"bf16": "TMA + tcgen05 implicit GEMM (bf16 operands, fp32 accumulate in TMEM)",
                             "fp16": "TMA + tcgen05 implicit GEMM (fp16 operands = TF32's 11-bit significand, fp32 accumulate in TMEM, "
                                     "power-of-two gradient scaling)",
                             "fp32": "fp32 CUDA-core implicit GEMM"}[precision]
        lay = (C.c_int32 * 16)()
        _lib.check(self._L.fb_qnet_layout(self._h, lay), "fb_qnet_layout")
        names = ["w1", "b1", "w2", "b2", "w3", "b3", "wf1", "bf1", "wf2", "bf2", "wv", "bv", "wa", "ba"]
        self.offsets = {n: int(lay[i]) for i, n in enumerate(names) if lay[i] >= 0}
        self.n_params = int(lay[14])
        z = lambda: torch.zeros(self.n_params, dtype=torch.float32, device=self.device)
        self.params, self.target, self.grads, self.adam_m, self.adam_v = z(), z(), z(), z(), z()
        self.loss = torch.zeros(1, dtype=torch.float32, device=self.device)
        # TF variable initialisers: truncated_normal(0.01) weights, constant 0.01 biases (BrainDQN.py:122-123);
        # the target net is initialised INDEPENDENTLY (BrainDQNNature.py:75-102, SURVEY Q4) unless asked otherwise
        g = torch.Generator(device="cpu").manual_seed(seed)
        self.params.copy_(self._init_flat(g))
        self.target.copy_(self.params if copy_target_at_init else self._init_flat(g))
        self.lr, self.beta1, self.beta2, self.adam_eps = np.float32(lr), np.float32(beta1), np.float32(beta2), np.float32(adam_eps)
        self.beta1_power, self.beta2_power = np.float32(beta1), np.float32(beta2)      # TF keeps these as fp32 variables
        self.adam_steps = 0
        self.exchange = None                    # dist.PeerGradExchange once enable_peer_exchange() was called
        self.exchange_in_step = False
        self.noisy = bool(noisy)
        if self.noisy:
            self._init_noise(seed, float(sigma0))

    # ---------------------------------------------------------------- noisy networks
    def _init_noise(self, seed: int, sigma0: float):
        lay = (C.c_int32 * 20)()
        _lib.check(self._L.fb_noisy_layout(self._h, lay), "fb_noisy_layout")
        # per noisy layer: parameter offsets of weight [p][q] and bias [q], and where f(eps_in) [p] / f(eps_out) [q] sit in a draw
        self.noise_layout = [dict(w=lay[2 + 6 * k], b=lay[3 + 6 * k], p=lay[4 + 6 * k], q=lay[5 + 6 * k], f_in=lay[6 + 6 * k],
                                  f_out=lay[7 + 6 * k]) for k in range(int(lay[0]))]
        self.n_factors = int(lay[1])
        self.noise_seed, self.sigma0 = int(seed), sigma0
        z = lambda n: torch.zeros(n, dtype=torch.float32, device=self.device)
        self.sigma, self.target_sigma, self.sigma_m, self.sigma_v = z(self.n_params), z(self.n_params), z(self.n_params), z(self.n_params)
        # effective weights of the update's online / target draw and of the last acting draw, and the factor vectors they came from
        self.weff, self.weff_target, self.weff_act = z(self.n_params), z(self.n_params), z(self.n_params)
        self.noise_online, self.noise_target, self.noise_act = z(self.n_factors), z(self.n_factors), z(self.n_factors)
        sig = torch.zeros(self.n_params, dtype=torch.float32)
        for ly in self.noise_layout:                  # Fortunato's factorised rule: sigma0 / sqrt(fan-in), weights and bias alike
            s0 = np.float32(sigma0 / np.sqrt(ly["p"]))
            sig[ly["w"]:ly["w"] + ly["p"] * ly["q"]] = float(s0)
            sig[ly["b"]:ly["b"] + ly["q"]] = float(s0)
        self.sigma.copy_(sig); self.target_sigma.copy_(sig)
        self.update_draws = 0                         # draw counters: update u (online and target role), acting call a
        self.act_draws = 0

    def draw_noise(self, role: str, counter: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """the factor vector of draw (role, counter), role in online / target / act (include/flappy_b200.h fb_noisy_draw)"""
        out = out if out is not None else torch.empty(self.n_factors, dtype=torch.float32, device=self.device)
        _lib.check(self._L.fb_noisy_draw(self._h, self.noise_seed, {"online": 0, "target": 1, "act": 2}[role], int(counter),
                                         out.data_ptr(), self._stream()), "fb_noisy_draw")
        return out

    def noisy_weights(self, mu: torch.Tensor, sigma: torch.Tensor, factors: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
        """out = mu + sigma * eps on the noisy layers, mu elsewhere (fb_noisy_weights)"""
        _lib.check(self._L.fb_noisy_weights(self._h, mu.data_ptr(), sigma.data_ptr(), factors.data_ptr(), out.data_ptr(), self._stream()),
                   "fb_noisy_weights")
        return out

    def _act_weights(self, target: bool = False) -> torch.Tensor:
        """effective weights of the next acting draw (consumes it)"""
        self.draw_noise("act", self.act_draws, self.noise_act)
        self.act_draws += 1
        mu, sigma = (self.target, self.target_sigma) if target else (self.params, self.sigma)
        return self.noisy_weights(mu, sigma, self.noise_act, self.weff_act)

    def _train_weights(self, variant: str):
        """(online, target) vectors the update runs on: the parameters, or for a noisy net the effective weights of update u's
        online draw and -- for the Nature and Double targets -- its target draw (vanilla and Double evaluate Q(s') with the
        online draw, no extra draw)"""
        if not self.noisy:
            return self.params, self.target
        u = self.update_draws
        self.noisy_weights(self.params, self.sigma, self.draw_noise("online", u, self.noise_online), self.weff)
        if VARIANTS[variant] != 0:
            self.noisy_weights(self.target, self.target_sigma, self.draw_noise("target", u, self.noise_target), self.weff_target)
        return self.weff, self.weff_target

    def set_per_broadcast(self, on: bool):
        """PER loss exactly as the reference's graph evaluates it (BrainPrioritizedReplyDQN.py:243-251): the [B,1] ISWeights
        placeholder times the [B] squared error broadcasts to [B,B], i.e. every sample is weighted by mean(ISWeights)."""
        _lib.check(self._L.fb_qnet_set_per_broadcast(self._h, int(bool(on))), "fb_qnet_set_per_broadcast")

    def enable_peer_exchange(self, exchange=None):
        """Multi-GPU: keep the gradient vector in an NVLink-mapped exchange buffer and let adam_step() sum every rank's
        gradients from peer memory inside the Adam kernel (csrc/fb_dist.cu) instead of a separate all-reduce."""
        from .dist import PeerGradExchange
        if self.quantile:
            raise ValueError("a QR net takes the all-reduce path (loss_backward, all_reduce(grads), adam_step): the in-step peer exchange "
                             "is not available with it")
        if self.distributional:
            raise ValueError("a C51 net takes the all-reduce path (loss_backward, all_reduce(grads), adam_step): the in-step peer exchange "
                             "is not available with it")
        if self.noisy:
            raise ValueError("a noisy net takes the all-reduce path (loss_backward, all_reduce(grads), adam_step): the peer exchange "
                             "applies plain Adam inside its own kernels")
        self.exchange =exchange if exchange is not None else PeerGradExchange(self.n_params, self.device)
        self.grads = self.exchange.grads
        # tensor-core path: the exchange rides INSIDE the training step's graph (fb_dist.cu buckets) instead of after it
        self.exchange_in_step = self.precision != "fp32" and self.exchange.world > 1 and not getattr(self.exchange, "no_wait", False)
        _lib.check(self._L.fb_qnet_attach_exchange(self._h, self.exchange._h if self.exchange_in_step else None), "fb_qnet_attach_exchange")
        return self.exchange

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._L.fb_qnet_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def _sizes(self):
        order = sorted(self.offsets.items(), key=lambda kv: kv[1])
        ends = [o for _, o in order[1:]] + [self.n_params]
        return [(n, o, e - o) for (n, o), e in zip(order, ends)]

    def _init_flat(self, gen) -> torch.Tensor:
        flat = torch.empty(self.n_params, dtype=torch.float32)
        for n, o, sz in self._sizes():
            if n.startswith("b"):
                flat[o:o + sz] = 0.01
            else:
                truncated_normal_(flat[o:o + sz], 0.01, gen)
        return flat

    def view(self, name: str, which: str = "params") -> torch.Tensor:
        """Named slice of a flat vector (which in params/target/grads/adam_m/adam_v), TF shapes."""
        n = self.atoms or self.quantiles                                             # C51 / QR: column a N + i of the A / plain head
        nv, na = (n, 2 * n) if n else (1, 2)
        shapes = {"w1": (8, 8, 4, 32), "b1": (32,), "w2": (4, 4, 32, 64), "b2": (64,), "w3": (3, 3, 64, 64), "b3": (64,),
                  "wf1": (1600, self.hidden), "bf1": (self.hidden,), "wf2": (self.hidden, na), "bf2": (na,),
                  "wv": (self.hidden, nv), "bv": (nv,), "wa": (self.hidden, na), "ba": (na,)}
        o = self.offsets[name]
        shp = shapes[name]
        return getattr(self, which)[o:o + int(np.prod(shp))].view(shp)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _sync_versions(self):
        """The library refreshes its bf16 operand copies after its own Adam / target-sync; in-place writes made
        through torch (tests, load_state_dict, an all-reduce of the parameters) are noticed here."""
        v = (self.params._version, self.target._version)
        if v != self._seen_versions:
            _lib.check(self._L.fb_qnet_invalidate(self._h), "fb_qnet_invalidate")
            self._seen_versions = v

    # ---------------------------------------------------------------- forward / act
    def forward(self, fb: FrameBatch, target: bool = False, out: torch.Tensor | None = None, noise: bool | None = None) -> torch.Tensor:
        """QValue.eval(feed_dict={stateInput: ...}) (BrainDQN.py:100): f32[B][2].  A noisy net evaluates the effective weights
        of the next acting draw (noise=False: mu)."""
        q = out if out is not None else torch.empty((fb.batch, 2), dtype=torch.float32, device=self.device)
        p = self.target if target else self.params
        self._sync_versions()
        if self.noisy and noise is not False:
            p = self._act_weights(target)
        _lib.check(self._L.fb_qnet_forward(self._h, p.data_ptr(), fb.ptr, fb.sample_stride, fb.chan_off, fb.batch,
                                           q.data_ptr(), self._stream()), "fb_qnet_forward")
        return q

    def forward_dist(self, fb: FrameBatch, target: bool = False, noise: bool | None = None):
        """C51 net: (probs f32[B][2][atoms], q f32[B][2]) -- the per-action distributions and their expectations
        (fb_qnet_forward_dist); a noisy net evaluates the next acting draw as forward() does"""
        if not self.distributional:
            raise ValueError("forward_dist needs distributional=True")
        probs = torch.empty((fb.batch, 2, self.atoms), dtype=torch.float32, device=self.device)
        q = torch.empty((fb.batch, 2), dtype=torch.float32, device=self.device)
        p = self.target if target else self.params
        self._sync_versions()
        if self.noisy and noise is not False:
            p = self._act_weights(target)
        _lib.check(self._L.fb_qnet_forward_dist(self._h, p.data_ptr(), fb.ptr, fb.sample_stride, fb.chan_off, fb.batch, probs.data_ptr(),
                                                q.data_ptr(), self._stream()), "fb_qnet_forward_dist")
        return probs, q

    def forward_quantiles(self, fb: FrameBatch, target: bool = False, noise: bool | None = None):
        """QR net: (theta f32[B][2][quantiles], q f32[B][2]) -- the per-action quantile locations and their means
        (fb_qnet_forward_quantiles); a noisy net evaluates the next acting draw as forward() does"""
        if not self.quantile:
            raise ValueError("forward_quantiles needs quantile=True")
        theta = torch.empty((fb.batch, 2, self.quantiles), dtype=torch.float32, device=self.device)
        q = torch.empty((fb.batch, 2), dtype=torch.float32, device=self.device)
        p = self.target if target else self.params
        self._sync_versions()
        if self.noisy and noise is not False:
            p = self._act_weights(target)
        _lib.check(self._L.fb_qnet_forward_quantiles(self._h, p.data_ptr(), fb.ptr, fb.sample_stride, fb.chan_off, fb.batch, theta.data_ptr(),
                                                     q.data_ptr(), self._stream()), "fb_qnet_forward_quantiles")
        return theta, q

    def act(self, fb: FrameBatch, epsilon: float, seed: int, first_env_id: int, rng_pos: torch.Tensor,
            actions_out: torch.Tensor, q_out: torch.Tensor, noise: bool | None = None):
        """getAction (BrainDQN.py:99-108) for every env of the batch.  A noisy net acts on the effective weights of the next
        acting draw; the epsilon-greedy draws are unchanged.  noise=False acts on mu (evaluation)."""
        self._sync_versions()
        p = self._act_weights() if self.noisy and noise is not False else self.params
        _lib.check(self._L.fb_qnet_act(self._h, p.data_ptr(), fb.ptr, fb.sample_stride, fb.chan_off, fb.batch,
                                       float(epsilon), seed, first_env_id, rng_pos.data_ptr(), q_out.data_ptr(),
                                       actions_out.data_ptr(), self._stream()), "fb_qnet_act")
        return actions_out

    # ---------------------------------------------------------------- training
    def _step(self, variant, params, target, frames, actions, rewards, terminals, is_weights, gamma, loss_sum, global_batch, abs_err,
              q_target, sampling, adam=False, grad_scale=1.0):
        """fb_qnet_step on (params, target): loss and gradients of the caller's minibatch, or of the one ``sampling`` draws inside
        the step; with ``adam`` the Adam update of self.params too"""
        ptr = lambda t: t.data_ptr() if t is not None else None
        a = _lib.QnetStepArgs(VARIANTS[variant], int(loss_sum), 0, global_batch or 0, float(gamma), params.data_ptr(), target.data_ptr())
        if sampling is not None:
            a.sampling = C.addressof(sampling)
        else:                                   # u8[B][5][80][80]: s = frames 0..3, s' = frames 1..4 of each sample
            assert frames.shape[1:] == (5, 80, 80) and frames.dtype == torch.uint8 and frames.is_contiguous()
            a.batch, a.frames_dev, a.sample_stride = frames.shape[0], frames.data_ptr(), 5 * 6400
            a.chan_off_s[:] = (0, 6400, 12800, 19200)
            a.chan_off_next[:] = (6400, 12800, 19200, 25600)
            a.actions_dev, a.rewards_dev, a.terminals_dev = actions.data_ptr(), rewards.data_ptr(), terminals.data_ptr()
            a.is_weights_dev = ptr(is_weights)
        a.grads_dev, a.loss_out_dev = self.grads.data_ptr(), self.loss.data_ptr()
        a.abs_err_out_dev, a.q_target_out_dev = ptr(abs_err), ptr(q_target)
        if adam:
            a.m_dev, a.v_dev = self.adam_m.data_ptr(), self.adam_v.data_ptr()
            a.lr, a.beta1, a.beta2, a.eps, a.grad_scale = self.lr, self.beta1, self.beta2, self.adam_eps, grad_scale
            a.beta1_power, a.beta2_power = self.beta1_power, self.beta2_power
        _lib.check(self._L.fb_qnet_step(self._h, C.byref(a), self._stream()), "fb_qnet_step")
        return self.loss

    def loss_backward(self, variant: str, frames: torch.Tensor, actions: torch.Tensor, rewards: torch.Tensor,
                      terminals: torch.Tensor, is_weights: torch.Tensor | None = None, gamma: float = 0.99,
                      loss_sum: bool = False, global_batch: int | None = None, abs_err: torch.Tensor | None = None,
                      q_target: torch.Tensor | None = None, sampling=None) -> torch.Tensor:
        """frames u8[B][5][80][80]: s = frames 0..3, s' = frames 1..4 of each sample.  Fills self.grads, self.loss.
        ``sampling``: as in train_step -- the minibatch is drawn by the first two kernels of the same graph (u8[B][F][80][80]
        rows for n-step returns, whose targets then come from the replay's R / disc)."""
        self._sync_versions()
        p, tg = self._train_weights(variant)        # mu, or the effective weights of update u's draws
        return self._step(variant, p, tg, frames, actions, rewards, terminals, is_weights, gamma, loss_sum, global_batch, abs_err,
                          q_target, sampling)

    def train_step(self, variant: str, frames: torch.Tensor, actions: torch.Tensor, rewards: torch.Tensor, terminals: torch.Tensor,
                   is_weights: torch.Tensor | None = None, gamma: float = 0.99, loss_sum: bool = False, global_batch: int | None = None,
                   abs_err: torch.Tensor | None = None, q_target: torch.Tensor | None = None, grad_scale: float = 1.0,
                   sampling=None) -> torch.Tensor:
        """session.run(trainStep) (BrainDQN.py:204-207): loss_backward + adam_step as one library call, bit-identical to the
        two; on the tensor-core path one CUDA graph launch with Adam inside the step's last kernel.  With a peer exchange
        (several GPUs) that is not carried inside the step the sum over ranks lives in the Adam kernel, so the two calls are
        made separately.

        ``sampling`` (``ReplayMemory.step_sampling(batch)[0]``): the minibatch is drawn and gathered by the step's first two
        kernels -- ``random.sample`` and the list comprehensions of BrainDQN.py:197-201 ride in the same graph; ``frames`` /
        ``actions`` / ``rewards`` / ``terminals`` must then be the replay's own minibatch buffers.  A memory with ``n_step`` > 1
        hands out u8[B][F][80][80] rows and the step forms the n-step target from its R / disc.

        A noisy net: the gradient-only step on the effective weights of update u's draws, then the Adam over (mu, sigma)."""
        if self.noisy or (self.exchange is not None and not self.exchange_in_step):
            self.loss_backward(variant, frames, actions, rewards, terminals, is_weights, gamma, loss_sum, global_batch, abs_err, q_target,
                               sampling=sampling)
            self.adam_step(grad_scale)
            return self.loss
        self._sync_versions()
        self._step(variant, self.params, self.target, frames, actions, rewards, terminals, is_weights, gamma, loss_sum, global_batch,
                   abs_err, q_target, sampling, adam=True, grad_scale=grad_scale)
        self._after_fused_step()
        return self.loss

    def _after_fused_step(self):
        self._advance_powers()
        if self.exchange_in_step:                # the step's graph carried the exchange: switch to the other exchange buffer
            _lib.check(self._L.fb_dist_advance(self.exchange._h), "fb_dist_advance")
            self.grads = self.exchange.grads

    def _advance_powers(self):
        """beta1_power *= beta1, beta2_power *= beta2 in fp32, like the update ops TF-1's Adam runs after every step"""
        self.beta1_power = np.float32(self.beta1_power * self.beta1)
        self.beta2_power = np.float32(self.beta2_power * self.beta2)
        self.adam_steps += 1

    def adam_step(self, grad_scale: float = 1.0):
        """One tf.train.AdamOptimizer step on self.params with self.grads (TF-1 ApplyAdam)."""
        one = np.float32(1)
        alpha = np.float32(self.lr * np.sqrt(one - self.beta2_power) / (one - self.beta1_power))
        if self.noisy:                          # mu with g, sigma with g * eps of update u's online draw; then draw u + 1
            _lib.check(self._L.fb_qnet_noisy_adam(self._h, self.params.data_ptr(), self.sigma.data_ptr(), self.grads.data_ptr(),
                                                  self.noise_online.data_ptr(), self.adam_m.data_ptr(), self.adam_v.data_ptr(),
                                                  self.sigma_m.data_ptr(), self.sigma_v.data_ptr(), float(alpha), float(self.beta1),
                                                  float(self.beta2), float(self.adam_eps), float(grad_scale), self._stream()),
                       "fb_qnet_noisy_adam")
            self.update_draws += 1
        elif self.exchange is not None:         # sum over ranks + Adam in one kernel; then switch to the other buffer
            self.exchange.adam(self, alpha, grad_scale, wait=self.exchange.world > 1 and not getattr(self.exchange, "no_wait", False))
            self.grads = self.exchange.grads
        else:
            _lib.check(self._L.fb_qnet_adam(self._h, self.params.data_ptr(), self.grads.data_ptr(), self.adam_m.data_ptr(),
                                            self.adam_v.data_ptr(), float(alpha), float(self.beta1), float(self.beta2),
                                            float(self.adam_eps), float(grad_scale), self._stream()), "fb_qnet_adam")
        self._advance_powers()

    def sync_target(self):
        """sess.run(target_replace_op) (BrainDQNNature.py:107-111,151-152)."""
        _lib.check(self._L.fb_qnet_sync_target(self._h, self.target.data_ptr(), self.params.data_ptr(), self._stream()),
                   "fb_qnet_sync_target")
        if self.noisy:
            _lib.check(self._L.fb_qnet_sync_target(self._h, self.target_sigma.data_ptr(), self.sigma.data_ptr(), self._stream()),
                       "fb_qnet_sync_target")

    # ---------------------------------------------------------------- checkpoint (row N2, weights + Adam slots + powers)
    def state_dict(self):
        return {"params": self.params.clone(), "target": self.target.clone(), "adam_m": self.adam_m.clone(),
                "adam_v": self.adam_v.clone(), "beta1_power": float(self.beta1_power), "beta2_power": float(self.beta2_power),
                "adam_steps": self.adam_steps, "hidden": self.hidden, "dueling": self.dueling, **self._noise_state(), **self._dist_state()}

    def _dist_state(self):
        if self.quantile:
            return {"quantiles": self.quantiles, "kappa": self.kappa}
        return {"atoms": self.atoms, "v_min": self.v_min, "v_max": self.v_max} if self.distributional else {}

    _NOISE_TENSORS = ("sigma", "target_sigma", "sigma_m", "sigma_v")

    def _noise_state(self):
        if not self.noisy:
            return {}
        return {"noisy": True, **{k: getattr(self, k).clone() for k in self._NOISE_TENSORS}, "update_draws": self.update_draws,
                "act_draws": self.act_draws, "noise_seed": self.noise_seed, "sigma0": self.sigma0}

    def load_state_dict(self, sd):
        assert sd["hidden"] == self.hidden and sd["dueling"] == self.dueling
        assert bool(sd.get("noisy", False)) == self.noisy, "plain and noisy checkpoints are not interchangeable"
        assert (sd.get("atoms", 0), sd.get("v_min", 0.0), sd.get("v_max", 0.0)) == (self.atoms, self.v_min, self.v_max), \
            "expected-value and C51 checkpoints (or C51 ones with another support) are not interchangeable"
        assert (sd.get("quantiles", 0), sd.get("kappa", 0.0)) == (self.quantiles, self.kappa), \
            "QR checkpoints are not interchangeable with other heads, nor with QR ones of another quantile count or kappa"
        for k in ("params", "target", "adam_m", "adam_v") + (self._NOISE_TENSORS if self.noisy else ()):
            getattr(self, k).copy_(sd[k])
        self.beta1_power, self.beta2_power = np.float32(sd["beta1_power"]), np.float32(sd["beta2_power"])
        self.adam_steps = int(sd["adam_steps"])
        if self.noisy:
            self.update_draws, self.act_draws = int(sd["update_draws"]), int(sd["act_draws"])
            self.noise_seed, self.sigma0 = int(sd["noise_seed"]), float(sd["sigma0"])
