/*
 * flappy_b200.h -- C ABI of libflappy_b200.so, the B200 (sm_100a) implementation of
 * the data-parallel hot path of angela000/DQNFlappyBird.
 *
 * The reference has no FFI of its own: its boundary is two duck-typed Python
 * objects used by a five-line loop (FlappyBirdDQN.py:60-76).  The entry points
 * below are what a ctypes binding of that boundary calls; the reference symbol
 * each one replaces is cited next to it.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every function returns 0 on success, a negative fb_status otherwise;
 *     fb_last_error() returns a thread-local message for the last failure;
 *   - pointers named *_dev are CUDA device pointers owned by the caller (the
 *     Python host code lets PyTorch own them); *_host are host pointers;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *     all device work is asynchronous on it, no hidden synchronisation, no
 *     allocation after the *_create call;
 *   - a handle is used from one host thread at a time;
 *   - no C++ exception crosses this boundary.
 */
#ifndef FLAPPY_B200_H
#define FLAPPY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FB_OBS 80                 /* preprocess output is 80x80, FlappyBirdDQN.py:32 */
#define FB_FRAME_BYTES 6400
#define FB_SCREEN_W 288           /* wrapped_flappy_bird.py:16 */
#define FB_SCREEN_H 512           /* wrapped_flappy_bird.py:17 */
#define FB_STATE_INTS 16          /* ints per env in fb_env_export_state */

typedef enum {
    FB_OK = 0,
    FB_ERR_INVALID = -1,          /* bad argument */
    FB_ERR_CUDA = -2,             /* CUDA runtime error, see fb_last_error() */
    FB_ERR_ASSETS = -3,           /* assets missing or not supported by the fast path */
    FB_ERR_ACTION = -4,           /* an action was not 0/1 (reference: ValueError, wrapped_flappy_bird.py:99-100) */
    FB_ERR_STATE = -5
} fb_status;

const char *fb_last_error(void);
int fb_version(void);

/* ---- assets: flappy_bird_utils.load() + getHitmask (game/flappy_bird_utils.py:16-124)
 * `packed` is the FBPK blob of dqnflappybird_b200/assets.py.  Derives the hitmask
 * bit rows, the cv2 coefficient tables and the observation tables and uploads
 * them to the current device.  Must be called once per process and device
 * before fb_env_create. */
int fb_assets_load(const uint8_t *packed_host, size_t n);

/* ---- environment: game.GameState (game/wrapped_flappy_bird.py:58-183), batched */
typedef struct fb_env fb_env;

/* GameState() x n_envs (wrapped_flappy_bird.py:59-85).  Env k of this handle is
 * global env `first_env_id + k`: its gap draws come from the Philox4x32-10 stream
 * (seed, purpose 0, env id) with CPython's randint(0,7) rule (top 4 bits of a
 * 32-bit word, rejected while >= 8; wrapped_flappy_bird.py:212). */
int fb_env_create(int n_envs, uint64_t seed, uint64_t first_env_id, fb_env **out);
int fb_env_destroy(fb_env *env);
int fb_env_num_envs(const fb_env *env);

/* Replay mode: gap draws are consumed from a logged script instead of Philox.
 * gaps_dev: u8[n_envs][per_env_len], values 0..7, read modulo per_env_len.
 * The buffer must stay alive while the handle uses it.  NULL switches back. */
int fb_env_set_gap_replay(fb_env *env, const uint8_t *gaps_dev, int per_env_len);

/* (Re)run GameState.__init__ for every env: fresh state, cycle phase 0, RNG
 * position 0, two gap draws each. */
int fb_env_reset(fb_env *env, void *stream);

/* n_steps x frame_step (wrapped_flappy_bird.py:87-183) + preprocess
 * (FlappyBirdDQN.py:31-34) for every env.
 *   actions_dev  u8[n_steps][n_envs]   0 = [1,0] no-op, 1 = [0,1] flap.  Any other
 *                                      value sets the handle's error flag
 *                                      (fb_env_check) and is treated as no-op.
 *   obs_ring_dev u8[n_envs][ring_len][80][80]  frame of step s is written to slot
 *                                      (ring_slot + s) % ring_len; obs[i][j]: i ~ game x,
 *                                      j ~ game y (cv2 rows/cols of array3d)
 *   reward_dev   f32[n_steps][n_envs]  0.1 / 3 / -3  (wrapped_flappy_bird.py:95,148,162)
 *   terminal_dev u8 [n_steps][n_envs]
 *   score_dev    i32[n_steps][n_envs]  score before the reset (:155)
 * Any output pointer may be NULL. */
int fb_env_step(fb_env *env, int n_steps, const uint8_t *actions_dev, uint8_t *obs_ring_dev, int ring_len,
                int ring_slot, float *reward_dev, uint8_t *terminal_dev, int32_t *score_dev, void *stream);

/* Draw the CURRENT state of every env into slot ring_slot without stepping (the fast table
 * path of fb_env_step; used after fb_env_reset / fb_env_import_state). */
int fb_env_draw(fb_env *env, uint8_t *obs_ring_dev, int ring_len, int ring_slot, void *stream);

/* Same, with actions drawn on the device: step s of env e flaps iff word
 * (first_step + s) of Philox stream (action_seed, purpose 1, env id) is below
 * flap_threshold (2^31 = p 0.5).  actions_out_dev (u8[n_steps][n_envs]) may be NULL. */
int fb_env_step_random(fb_env *env, int n_steps, uint64_t action_seed, uint32_t first_step, uint32_t flap_threshold,
                       uint8_t *actions_out_dev, uint8_t *obs_ring_dev, int ring_len, int ring_slot,
                       float *reward_dev, uint8_t *terminal_dev, int32_t *score_dev, void *stream);

/* The reference-facing call with HOST buffers (one frame_step for every env):
 * copies actions_host (u8[n]) to the device, steps, and copies reward / terminal /
 * score back; the observation stays in the device ring.  Synchronises `stream`. */
int fb_env_step_host(fb_env *env, const uint8_t *actions_host, uint8_t *obs_ring_dev, int ring_len, int ring_slot,
                     float *reward_host, uint8_t *terminal_host, int32_t *score_host, void *stream);
/* The same call split in two so that two steps can be in flight (copies of step t overlap the kernel of step t+1):
 * submit returns once everything is queued; wait blocks until the OLDEST submitted step has filled its host buffers.
 * At most two submits may be outstanding.  fb_env_step_host == submit + wait. */
int fb_env_step_host_submit(fb_env *env, const uint8_t *actions_host, uint8_t *obs_ring_dev, int ring_len, int ring_slot,
                            float *reward_host, uint8_t *terminal_host, int32_t *score_host, void *stream);
int fb_env_step_host_wait(fb_env *env);

/* Reads and clears the device error flag (synchronises `stream`): FB_OK or FB_ERR_ACTION. */
int fb_env_check(fb_env *env, void *stream);

/* Parity-test access to the packed state.  out/in: i32[n_envs][16]:
 * [0] playery [1] playerVelY [2] playerIndex [3] loopIter [4] cycle phase of PLAYER_INDEX_GEN
 * [5] basex [6] score [7] number of pipes [8..10] pipe x [11..13] gap index (0..7)
 * [14] RNG draws consumed [15] reserved */
int fb_env_export_state(fb_env *env, int32_t *out_dev, void *stream);
int fb_env_import_state(fb_env *env, const int32_t *in_dev, void *stream);

/* Observation of the CURRENT state computed with per-pixel fixed-point arithmetic
 * only (no tables): the in-library cross-check of the fast path.  obs_dev u8[n_envs][80][80]. */
int fb_env_obs_exact(fb_env *env, uint8_t *obs_dev, void *stream);

/* image_data of frame_step (wrapped_flappy_bird.py:165-177): u8[n][288][512][3] for envs
 * [first, first+n) of the handle. */
int fb_render_full(fb_env *env, int first, int n, uint8_t *rgb_dev, void *stream);

/* The cv2 coefficient tables the library derived: i32[6][80] = sx,a0,a1,sy,b0,b1. */
int fb_resize_tables(int32_t *out_host);

/* ---- Q-network: the TensorFlow graph of every Brain (BrainDQN.py:119-163; dueling head
 * BrainDuelingDQN_CC.py:68-77), getAction (BrainDQN.py:99-116), _trainQNetwork (BrainDQN.py:195-223,
 * BrainDQNNature.py:149-183, BrainDoubleDQN.py:37-69, BrainPrioritizedReplyDQN.py:277-315) and
 * tf.train.AdamOptimizer (BrainDQN.py:163).
 *
 * Parameters, target parameters, gradients and the Adam slots are flat fp32 vectors owned by the
 * caller, laid out in TF variable-creation order: W_conv1[8,8,4,32] b_conv1[32] W_conv2[4,4,32,64]
 * b_conv2[64] W_conv3[3,3,64,64] b_conv3[64] W_fc1[1600,H] b_fc1[H] then W_fc2[H,2] b_fc2[2], or for
 * the dueling net W_fc2_v[H,1] b_fc2_v[1] W_fc2_a[H,2] b_fc2_a[2].  fb_qnet_layout returns the
 * offsets: {w1,b1,w2,b2,w3,b3,wf1,bf1,wf2,bf2,wv,bv,wa,ba,total,H} (-1 where absent).
 *
 * The input of sample b is never materialised as [80,80,4]: channel c (oldest frame first, newest
 * last, BrainDQN.py:68) is the u8 frame at frames_dev + b*sample_stride + chan_off[c] -- a view of
 * the frame ring (acting) or of a gathered replay batch (training). */
typedef struct fb_qnet fb_qnet;
int fb_qnet_create(int hidden, int dueling, int max_batch, fb_qnet **out);
/* The distributional (C51) head (Bellemare et al. 2017; csrc/fb_c51.cu) on the same trunk: per action a categorical
 * distribution over `atoms` N (2..64) atoms z_i = (float)(v_min + i dz), dz = (v_max - v_min) / (N - 1) in float64.  The head
 * variables keep their slots in fb_qnet_layout with N outputs per action: W_fc2[H,2N] b_fc2[2N] (column a N + i), or dueling
 * W_fc2_v[H,N] b_fc2_v[N] W_fc2_a[H,2N] b_fc2_a[2N] with logits v_i + (a_{a,i} - (a_{0,i} + a_{1,i}) / 2).  p = softmax over the
 * atoms (fp32), Q[a] = sum_i z_i p[a][i]: fb_qnet_forward / fb_qnet_act return Q and act on it unchanged.  In fb_qnet_step the
 * TD loss becomes the cross-entropy of p[a](s) against the float64 projection m of R + disc z under p[a*](s') (a* the variant's
 * first argmax of Q(s')): loss = sum_b w_b CE_b (mean losses: / global batch), abs_err_out = CE_b (the Rainbow priority, unweighted
 * and unscaled), q_target_out = sum_i z_i m_i.  hidden must be a multiple of 32 and at most 2048.  FB_ERR_INVALID for atoms
 * outside 2..64 or a support that is not finite with v_min < v_max.  A C51 net refuses a step with fb_qnet_set_per_broadcast on and
 * a non-NULL fb_qnet_attach_exchange (it takes the all-reduce path on several GPUs). */
int fb_qnet_create_c51(int hidden, int dueling, int max_batch, int atoms, double v_min, double v_max, fb_qnet **out);
/* The quantile-regression (QR-DQN) head (Dabney, Rowland, Bellemare and Munos 2018; csrc/fb_qr.cu) on the same trunk: per action
 * `quantiles` N (1..64) quantile locations theta[a][i] at the fractions tau_i = (2i + 1) / (2N).  The head variables keep the C51
 * head's slots and column routing with N outputs per action (theta takes the place of the logits; dueling: v_i + (a_{a,i} -
 * (a_{0,i} + a_{1,i}) / 2)).  Q[a] = (1/N) sum_i theta[a][i] (fp32, ascending i): fb_qnet_forward / fb_qnet_act return Q and act
 * on it unchanged.  In fb_qnet_step the TD loss becomes the quantile-Huber loss: a* the variant's first argmax of Q(s') (Double:
 * online argmax, target theta), T_j = the expected-value head's TD target of theta[a*][j](s') (1-step or n-step, same rounding),
 * u_ij = T_j - theta[a_b][i](s), L_b = sum_i (1/N) sum_j |tau_i - 1{u_ij < 0}| H(u_ij) with H(u) = u^2 / (2 kappa) for |u| <= kappa,
 * else |u| - kappa / 2 (kappa = 0: H(u) = |u|); loss = sum_b w_b L_b (mean losses: / global batch), abs_err_out = L_b (the priority,
 * unweighted and unscaled), q_target_out = (1/N) sum_j T_j.  hidden must be a multiple of 32 and at most 2048.  FB_ERR_INVALID for
 * quantiles outside 1..64 or a kappa that is negative or not finite.  A QR net refuses what a C51 net refuses (fb_qnet_set_per_broadcast
 * in a step, a non-NULL fb_qnet_attach_exchange) and fb_qnet_forward_dist. */
int fb_qnet_create_qr(int hidden, int dueling, int max_batch, int quantiles, double kappa, fb_qnet **out);
int fb_qnet_destroy(fb_qnet *net);

/* Arithmetic of the contractions (the TF ops of BrainDQN.py:123-154 and their gradients):
 *   FB_PRECISION_FP32  CUDA-core FMA, fp32 everywhere (strict; the tolerance anchor)
 *   FB_PRECISION_BF16  tcgen05 tensor cores fed by TMA: bf16 operands (the {0,255} inputs are exact), fp32
 *                      accumulation in TMEM, bf16 activations between layers; head, TD loss and Adam stay fp32.
 * fb_qnet_invalidate tells the net that the caller rewrote a parameter vector itself (the bf16 operand copies
 * are otherwise refreshed after fb_qnet_adam / fb_qnet_sync_target). */
#define FB_PRECISION_FP32 0
#define FB_PRECISION_BF16 1
/* FB_PRECISION_FP16: the same tensor-core kernels with IEEE fp16 operands -- an 11-bit significand, exactly TF32's, at the
 * bf16 tensor rate and byte count.  fp16's narrow exponent range is handled like mixed-precision training does: the gradient
 * tensors (dh1 and everything downstream) carry a power-of-two factor (8 for the sum loss, 8 x minibatch rounded up to a power
 * of two for the mean losses) that is removed exactly where weight / bias gradients are finalised.  The precision north_star
 * names ("fp32/TF32 tolerance"); the default of the Brain classes. */
#define FB_PRECISION_FP16 2
int fb_qnet_set_precision(fb_qnet *net, int precision);
int fb_qnet_get_precision(const fb_qnet *net);
int fb_qnet_invalidate(fb_qnet *net);
/* PER loss exactly as the reference's graph evaluates it (BrainPrioritizedReplyDQN.py:243-251): the [B,1] ISWeights
 * placeholder times the [B] squared error is broadcast to [B,B], so the cost is mean(w) * mean(err^2) and every sample's
 * gradient is scaled by mean(w).  on = 0 (default): the intended mean(w_i * err_i^2). */
int fb_qnet_set_per_broadcast(fb_qnet *net, int on);
/* test hook: overwrite the bf16 operand copies of slot 0 (online) / 1 (target) with NaNs WITHOUT marking them stale --
 * whoever reads them before the next pack kernel has finished shows up as NaN Q-values */
int fb_debug_poison_packed(fb_qnet *net, int slot, void *stream);
/* measurement hook (tools/write_bw_probe.py): n_chunks chunks of 6,400 bytes at dst + k * stride_bytes, written by one warp each
 * with 16-byte streaming stores (mode 0) or through shared memory + cp.async.bulk (mode 1); no computation */
int fb_debug_write_probe(uint8_t *dst_dev, int n_chunks, long long stride_bytes, int mode, int ctas, void *stream);
/* Tensor-core precisions (FB_PRECISION_BF16 / _FP16) only: replay fb_qnet_step as a CUDA graph once the same arguments were seen twice
 * (default on; the eager two-stream path is identical work).  Every call drops the graphs captured so far. */
int fb_qnet_use_graphs(fb_qnet *net, int enable);
int fb_qnet_param_count(const fb_qnet *net);
int fb_qnet_layout(const fb_qnet *net, int32_t *out16_host);

/* QValue.eval (BrainDQN.py:100): q_out_dev f32[batch][2] */
int fb_qnet_forward(fb_qnet *net, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                    const int32_t *chan_off_host4, int batch, float *q_out_dev, void *stream);

/* C51 net only (FB_ERR_INVALID otherwise): the distributions probs_out_dev f32[batch][2][atoms] beside q_out_dev f32[batch][2];
 * chunked above max_batch like fb_qnet_forward */
int fb_qnet_forward_dist(fb_qnet *net, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                         const int32_t *chan_off_host4, int batch, float *probs_out_dev, float *q_out_dev, void *stream);

/* QR net only (FB_ERR_INVALID otherwise): the quantile locations theta_out_dev f32[batch][2][quantiles] beside their means
 * q_out_dev f32[batch][2]; chunked above max_batch like fb_qnet_forward */
int fb_qnet_forward_quantiles(fb_qnet *net, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                              const int32_t *chan_off_host4, int batch, float *theta_out_dev, float *q_out_dev, void *stream);

/* getAction (BrainDQN.py:99-108) for `batch` envs: forward, then random.random() <= epsilon ?
 * randrange(2) : argmax.  Env e draws from Philox stream (seed, purpose 2, first_env_id + e) at
 * word position rng_pos_dev[e] (updated).  actions_out_dev u8[batch] (0 no-op / 1 flap). */
int fb_qnet_act(fb_qnet *net, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                const int32_t *chan_off_host4, int batch, double epsilon, uint64_t seed, uint64_t first_env_id,
                uint32_t *rng_pos_dev, float *q_out_dev, uint8_t *actions_out_dev, void *stream);

/* One TF-1 ApplyAdam step over the flat vector; alpha = lr*sqrt(1-beta2^t)/(1-beta1^t) from the caller. */
int fb_qnet_adam(fb_qnet *net, float *params_dev, const float *grads_dev, float *m_dev, float *v_dev, float alpha,
                 float beta1, float beta2, float eps, float grad_scale, void *stream);

/* target_replace_op (BrainDQNNature.py:107-111) */
int fb_qnet_sync_target(fb_qnet *net, float *target_dev, const float *params_dev, void *stream);

/* ---- noisy networks (Fortunato et al. 2018, factorised Gaussian noise; csrc/fb_noisy.cu).  The noisy layers are fc1 and the
 * head (plain: W_fc2 / b_fc2; dueling: the V head and the A head, each its own layer); the convolutions stay deterministic.  A
 * noisy net keeps mu (the usual parameter vector) and sigma (same layout, zero outside the noisy layers).  A draw fills the
 * factor vector: per noisy layer, in layer order, f(eps_in)[p] then f(eps_out)[q], f(x) = sgn(x) sqrt|x| in fp32.  The layer
 * runs on W[i][j] = mu[i][j] + sigma[i][j] * (f(eps_in[i]) * f(eps_out[j])), b[j] = mu_b[j] + sigma_b[j] * f(eps_out[j]) (fp32,
 * each operation rounded once): the effective-weight vector has the parameter layout, and every forward / training call above
 * takes it in place of the parameters.  The gradient they return is dL/dmu; dL/dsigma = dL/dW * eps.
 *
 * fb_noisy_layout: out20_host = {number of noisy layers (2 or 3), factor-vector length, then per layer (3 slots, -1 / 0 where
 * absent): weight offset, bias offset, fan-in p, fan-out q, offset of f(eps_in), offset of f(eps_out)}. */
int fb_noisy_layout(const fb_qnet *net, int32_t *out20_host);
/* One draw into factors_dev.  Normal k comes from words 2k, 2k+1 (w0, w1) of Philox stream (seed, purpose 5,
 * (counter << 2) | role) by Box-Muller in float64: u1 = (w0 + 1) 2^-32, u2 = w1 2^-32, z = sqrt(-2 ln u1) cos(2 pi u2), rounded
 * to fp32.  role 0: online net of update `counter`; 1: target net of that update; 2: acting call `counter`.  The stream does
 * not depend on the rank, so replicas draw the same noise without communicating. */
int fb_noisy_draw(fb_qnet *net, uint64_t seed, int role, uint64_t counter, float *factors_dev, void *stream);
/* weff_dev = mu + sigma * eps on the noisy layers, mu elsewhere; the operand copies made from weff_dev are marked stale */
int fb_noisy_weights(fb_qnet *net, const float *mu_dev, const float *sigma_dev, const float *factors_dev, float *weff_dev, void *stream);
/* One TF-1 Adam step over (mu, sigma) with one alpha: mu with grads_dev (dL/dW at W_eff) over every parameter, sigma with
 * grads_dev * eps (eps recomputed from the draw's factors) over the noisy layers; the rule and operation order of fb_qnet_adam */
int fb_qnet_noisy_adam(fb_qnet *net, float *mu_dev, float *sigma_dev, const float *grads_dev, const float *factors_dev, float *m_dev,
                       float *v_dev, float *sigma_m_dev, float *sigma_v_dev, float alpha, float beta1, float beta2, float eps,
                       float grad_scale, void *stream);

/* ---- multi-GPU gradient exchange fused with Adam (the one exchange step of the path: the sum of the per-shard
 * gradients of the replicated learner, SURVEY 8e).  One process per GPU; each rank's gradient vector lives in an exchange
 * buffer the peers map through CUDA IPC; fb_dist_adam publishes this rank's step, waits for every rank's, sums the
 * gradients of ranks 0..G-1 in rank order straight from peer memory over NVLink and applies TF-1 Adam in the same kernel
 * (bitwise identical parameters on every rank).  Buffers alternate by step parity: write the gradients of the next step to
 * fb_dist_grads(d, fb_dist_parity(d)). */
typedef struct fb_dist fb_dist;
int fb_dist_create(int rank, int world, long long n_floats, fb_dist **out);
int fb_dist_destroy(fb_dist *d);
int fb_dist_handle_bytes(void);
int fb_dist_set_two_shot(fb_dist *d, int on);                       /* default: two-shot (reduce own slice, then gather) from 4 ranks up */
int fb_dist_handles(fb_dist *d, uint8_t *out_host);                 /* this rank's IPC handles */
int fb_dist_connect(fb_dist *d, const uint8_t *all_handles_host);   /* world x fb_dist_handle_bytes(), rank-major */
int fb_dist_connect_local(fb_dist *d, int q, fb_dist *peer);        /* test hook: "ranks" inside one process */
int fb_dist_grads(fb_dist *d, int parity, float **out_dev_ptr);
int fb_dist_parity(const fb_dist *d);
/* With an exchange attached to a net on the tensor-core path (fb_qnet_attach_exchange) the training step carries the exchange
 * inside its own CUDA graph: W_fc1's 91 % of the gradient vector is summed over NVLink peer memory and Adam-updated beside the
 * convolution gradients, the remaining 79,522 parameters at the tail; step number and alpha live in device memory.
 * fb_dist_advance: that step has been enqueued, the next one writes the other exchange buffer. */
int fb_dist_advance(fb_dist *d);
/* timing experiments only (tools/dist_probe.py): bit b: bucket b of the in-step exchange sums its own gradient alone, bit 2+b: it skips
 * the publish / wait handshake.  Results are WRONG while a bit is set. */
int fb_dist_debug_mask(fb_dist *d, int mask);
int fb_qnet_attach_exchange(fb_qnet *net, fb_dist *d);
int fb_dist_adam(fb_dist *d, fb_qnet *net, float *params_dev, float *m_dev, float *v_dev, float alpha, float beta1, float beta2,
                 float eps, float grad_scale, float *reduced_out_dev /* may be NULL */, int wait, void *stream);
/* debug: %globaltimer (ns) of the last exchange's phase boundaries on this rank: start, all gradients published, own slice
 * reduced, all slices published, Adam done.  The first call switches the stamping on. */
int fb_dist_debug_stamps(fb_dist *d, unsigned long long *out_host5);

/* ---- replay memory: the deque + random.sample of BrainDQN.py:69-72,197-201 and the SumTree / Memory of
 * BrainPrioritizedReplyDQN.py:32-151, over the env's own frame ring (no frame is copied on append).
 * Transition k >= 1 of env e is (s_{k-1}, a_k, r_k, s_k, term_k), s_k = frames k-3..k of the ring
 * u8[N][ring_len][80][80]; a/r/term of step k live in [ring_len][N] arrays at row k % ring_len (the step /
 * act kernels write them there).  capacity_per_env C <= ring_len-4 transitions are live per env; the
 * population of random.sample at time t is j = e*cnt + (k-k_lo), k_lo = max(1,t-C+1), cnt = t-k_lo+1, and
 * the SumTree data index is e*C + (k-1)%C -- for one env exactly the reference's deque / data_pointer order. */
typedef struct fb_replay fb_replay;
int fb_replay_create(int n_envs, int ring_len, int capacity_per_env, int prioritized, int max_batch, fb_replay **out);
int fb_replay_destroy(fb_replay *r);

/* random.sample(replayMemory, batch) (BrainDQN.py:197) with CPython's algorithm over the word stream
 * Philox(seed, purpose 3).  setsize is CPython's threshold 21 + 4**ceil(log(3*batch, 4)) (computed by the
 * caller with the same float expression).  idx_out_dev i32[batch] population indices.  FB_ERR_INVALID with
 * "Sample larger than population or is negative" when batch exceeds the population (ValueError). */
int fb_replay_sample_uniform(fb_replay *r, long long t, int batch, uint32_t setsize, uint64_t seed, int32_t *idx_out_dev, void *stream);

/* minibatch assembly: frames_out_dev u8[batch][5][80][80] (s = frames 0..3, s' = frames 1..4), action / reward /
 * terminal per sample; idx are population indices (prioritized_index 0) or SumTree data indices (1). */
int fb_replay_gather(fb_replay *r, const uint8_t *ring_dev, const uint8_t *act_dev, const float *rew_dev, const uint8_t *term_dev,
                     long long t, int prioritized_index, const int32_t *idx_dev, int batch, uint8_t *frames_out_dev,
                     uint8_t *act_out_dev, float *rew_out_dev, uint8_t *term_out_dev, int32_t *env_out_dev, int32_t *k_out_dev,
                     void *stream);

/* Logging surface (BrainDQN.py:88-93: score_every_episode.append(curScore), time_steps_when_episode_end.append(timeStep)):
 * every env whose terminal flag is set appends (time_step, first_env_id + env, score) to log_dev i32[capacity][3] and
 * bumps *count_dev (which keeps counting past capacity so the host can see an overflow).  Entries of one step arrive in
 * no fixed order; the host sorts by (time_step, env) when it flushes. */
int fb_log_episodes(const uint8_t *terminal_dev, const int32_t *score_dev, int n_envs, int first_env_id, int time_step,
                    int32_t *log_dev, int *count_dev, int capacity, void *stream);

/* Memory.store (:121-125) of transition k for every env, in env order.  mode 0 = the reference's
 * "every ancestor += change" arithmetic in item order (bit-exact rounding history); mode 1 = set leaves
 * and recompute touched ancestors as left+right (parallel, deterministic). */
int fb_per_store(fb_replay *r, long long k, int mode, void *stream);
/* Memory.sample (:127-144); beta is the already-incremented value.  Word stream Philox(seed, purpose 4).
 * is_weights_f32_dev (optional): the same weights rounded to fp32, what the tf.float32 ISWeights placeholder receives (:243). */
int fb_per_sample(fb_replay *r, int batch, double beta, uint64_t seed, int32_t *tree_idx_dev, int32_t *data_idx_dev,
                  double *is_weights_dev, double *prio_out_dev, float *is_weights_f32_dev, void *stream);
/* Memory.batch_update (:146-151): priorities from |TD error| (abs_err_dev, fp32 like the reference's arrays)
 * or given directly (prio_dev f64). */
int fb_per_update(fb_replay *r, const int32_t *tree_idx_dev, const float *abs_err_dev, const double *prio_dev, int batch, int mode, void *stream);
/* copy of the SumTree array (f64[2*N*C-1]) for inspection / checkpoints */
int fb_per_tree_copy(fb_replay *r, double *out_dev, int n_nodes, void *stream);
/* test hook: the min-positive-leaf tree (which = 1) or the max-leaf tree (2) kept beside the SumTree, same shape */
int fb_per_aux_tree_copy(fb_replay *r, int which, double *out_dev, int n_nodes, void *stream);
/* Several GPUs, one memory sharded over the ranks: Memory.sample's min_prob (BrainPrioritizedReplyDQN.py:131, the min over every leaf)
 * is global, and ISWeights = (p_i / min_p)^-beta needs nothing else that is.  fb_per_min_root: this shard's smallest positive leaf
 * (+inf if none) into a device scalar; reduce it over the ranks (MIN) and register the scalar with fb_per_set_global_min: every
 * later fb_per_sample / sampled training step reads it instead of the local root (NULL: local again). */
int fb_per_min_root(fb_replay *r, double *out_dev, void *stream);
int fb_per_set_global_min(fb_replay *r, const double *global_min_dev);
int fb_replay_rng_pos(fb_replay *r, uint64_t *pos_host2, int set, void *stream);

/* The minibatch of fb_qnet_step drawn INSIDE the step: random.sample + the list comprehensions of BrainDQN.py:197-201
 * (fb_replay_sample_uniform + fb_replay_gather with these arguments) run as the first two kernels of the step, so that on
 * the tensor-core path sampling, gather, forward, backward and Adam are ONE CUDA graph launch; `t` is the only field that
 * changes from step to step and is patched into the two kernel nodes (a captured step is matched on the descriptor's bytes,
 * padding included: zero-fill it before setting the fields).  frames_out_dev etc. are the minibatch buffers the gather fills
 * (u8[batch][5][80][80]: s = frames 0..3, s' = frames 1..4). */
typedef struct fb_step_sampling {
    fb_replay *replay;
    const uint8_t *ring_dev, *act_dev; const float *rew_dev; const uint8_t *term_dev;
    long long t;                        /* time of the newest stored transition */
    int batch; uint32_t setsize; uint64_t seed;
    int32_t *idx_out_dev;
    uint8_t *frames_out_dev, *act_out_dev; float *rew_out_dev; uint8_t *term_out_dev;
    int32_t *env_out_dev, *k_out_dev;   /* optional */
    /* prioritized != 0: Memory.sample (fb_per_sample with `beta`, which like `t` is patched per step) instead of
     * random.sample, the loss weighted by is_weights_f32_out_dev, and Memory.batch_update (fb_per_update from the step's
     * |TD errors|, abs_err_out_dev of the call is then required) as the graph's last kernel */
    int prioritized, per_mode;
    double beta;
    int32_t *tree_idx_out_dev;
    double *is_weights_out_dev, *prio_out_dev;
    float *is_weights_f32_out_dev;
    /* n-step returns.  n_step = 0 (a zero-initialised tail): the 1-step transitions above, unchanged.  1 <= n_step <= 16:
     * transition k is (s_{k-1}, a_k, R_k, s_{k+n-1}, disc_k) with m the first i in 1..n whose term_{k+i-1} is set (else n),
     * R_k = sum_{i<m} gamma^i r_{k+i} (float64, accumulated forward: R += g r; g *= gamma) and disc_k = 0 after a terminal,
     * else gamma^n (that same product); the TD target is y = disc == 0 ? R : R + disc X, gamma being the step's `gamma`.
     * A transition is drawn once its horizon is complete: the population / SumTree is that of t_eff = t - n_step + 1 (so
     * the caller stores transition t - n + 1 into a prioritized memory at time t).  The frame ring must hold
     * ring_len >= capacity_per_env + n_step + 3 frames (FB_ERR_INVALID otherwise).  frames_out_dev is then
     * u8[batch][F][80][80], F = 4 + min(n, 4): s = frames 0..3, s' = frames F-4..F-1; ret_out_dev / disc_out_dev f64[batch]
     * receive R_k and disc_k (required). */
    int n_step;
    double *ret_out_dev, *disc_out_dev;
} fb_step_sampling;

/* ---- one training step of the Q-network: _trainQNetwork (BrainDQN.py:195-223 and the variants' versions) up to and including
 * session.run(trainStep) (:204-207).  TD target + loss + backward into grads_dev, then, when m_dev / v_dev are set, one TF-1
 * Adam step bit-identical to fb_qnet_adam with alpha = lr*sqrt(1-beta2_power)/(1-beta1_power) in fp32; beta1_power /
 * beta2_power are the caller's beta^t (TF's beta1_power / beta2_power variables, before this step).
 *   variant       0 vanilla / 1 Nature target net / 2 Double (target_params_dev required for 1 and 2); the dueling head is a
 *                 property of the net
 *   loss_sum      != 0: sum of squares (BrainDQN.py:162), else the mean over global_batch (BrainDQNNature.py:119; <= 0: batch),
 *                 so that a sum-allreduce of the gradients of `batch`-sized shards is the gradient of the global mean loss
 *   sampling      NULL: the caller's minibatch -- `batch` samples, s = channels chan_off_s, s' = channels chan_off_next of the
 *                 per-sample block at frames_dev + b*sample_stride, is_weights_dev != NULL selects the PER loss.
 *                 Non-NULL: the step draws its minibatch first (fb_step_sampling; uniform or prioritized replay), batch is
 *                 sampling->batch (`batch` 0 or equal), s = frames 0..3 and s' = frames F-4..F-1 of each drawn row, and the
 *                 caller-minibatch fields (frames_dev .. is_weights_dev) must be 0 / NULL.  FB_ERR_INVALID with "Sample larger
 *                 than population or is negative" when the replay holds fewer than `batch` transitions (random.sample's
 *                 ValueError).
 *   outputs       loss f32[1], abs_err f32[batch] (PER, :247; required with prioritized sampling), q_target f32[batch]; may
 *                 be NULL otherwise
 * On the tensor-core precisions Adam runs inside the step's last kernel from powers kept in device memory (re-seeded only when
 * they differ from the caller's), so the whole step replays as one CUDA graph launch (fb_qnet_use_graphs); params_dev is
 * updated in place, grads_dev / loss_out_dev are still written.  With an exchange attached (fb_qnet_attach_exchange) Adam
 * applies the sum of every rank's gradients. */
typedef struct fb_qnet_step_args {
    int variant, loss_sum, batch, global_batch;
    double gamma;
    float *params_dev; const float *target_params_dev;
    const fb_step_sampling *sampling;
    const uint8_t *frames_dev; long long sample_stride; int32_t chan_off_s[4], chan_off_next[4];
    const uint8_t *actions_dev; const float *rewards_dev; const uint8_t *terminals_dev; const float *is_weights_dev;
    float *grads_dev, *loss_out_dev, *abs_err_out_dev, *q_target_out_dev;
    float *m_dev, *v_dev;                           /* both NULL: gradients only; both set: Adam as well */
    float lr, beta1, beta2, eps, grad_scale, beta1_power, beta2_power;
} fb_qnet_step_args;
int fb_qnet_step(fb_qnet *net, const fb_qnet_step_args *args, void *stream);


/* ---- test hooks (host only, no device needed): the library's own physics / table / exact-pixel
 * code compiled for the host, so the CPU test-suite can pin it against the oracle. */
int fb_debug_assets_load_host(const uint8_t *packed_host, size_t n);
/* sizeof(S) followed by the byte offset of each field of S, in declaration order, for S = fb_step_sampling (which 0) or
 * fb_qnet_step_args (which 1); returns the count written */
int fb_debug_struct_layout(int which, int32_t *out, int capacity);
int fb_debug_step_sampling_layout(int32_t *out, int capacity);     /* fb_debug_struct_layout(0, out, capacity) */
int fb_debug_host_reset(int32_t *state16, const uint8_t *gaps, int gaps_len, uint64_t seed, uint64_t env_id);
int fb_debug_host_step(int32_t *state16, int action, const uint8_t *gaps, int gaps_len, uint64_t seed,
                       uint64_t env_id, float *reward, uint8_t *terminal, int32_t *score);
int fb_debug_host_obs(const int32_t *state16, int mode /* 0 tables, 1 per-pixel */, uint8_t *out6400);
int fb_debug_host_mixed(const int32_t *state16);
/* device test hook, C51 net: m_out_dev f32[batch][atoms] = the target projection of the training step's loss kernel (the same
 * device function) of p_next_dev f32[batch][atoms] under the 1-step target (ret_dev / disc_dev NULL: R = r, disc = terminal ? 0 :
 * gamma) or the n-step one (f64[batch] R and disc) */
int fb_debug_c51_project(fb_qnet *net, const float *p_next_dev, const float *rewards_dev, const uint8_t *terminals_dev, const double *ret_dev,
                         const double *disc_dev, double gamma, int batch, float *m_out_dev, void *stream);
/* device test hook, QR net: the training step's quantile-Huber loss (the same device function) on given theta.  theta_s_dev
 * f32[batch][2][quantiles] (theta of s), theta_next_astar_dev f32[batch][quantiles] (theta[a*] of s'), actions u8[batch]; the 1-step
 * target (ret_dev / disc_dev NULL: rewards and terminals) or the n-step one (f64[batch] R and disc).  dtheta_out_dev
 * f32[batch][quantiles] = dL_b/dtheta[a_b][i] and loss_b_out_dev f32[batch] = L_b, unweighted and unscaled */
int fb_debug_qr_loss(fb_qnet *net, const float *theta_s_dev, const float *theta_next_astar_dev, const uint8_t *actions_dev, const float *rewards_dev,
                     const uint8_t *terminals_dev, const double *ret_dev, const double *disc_dev, double gamma, int batch, float *dtheta_out_dev,
                     float *loss_b_out_dev, void *stream);
/* device test hook: one raw bf16 GEMM through the tcgen05 kernel of the Q-network path (descriptor self-test).
 * mode 0: D[M][N] = A[M][K] Bt[N][K]^T;  mode 1: D[M][N] = A[K][M]^T B[K][N];  bn = N tile (32/64/128). */
int fb_debug_tc_gemm(int mode, int bn, int M, int N, int K, const void *a_bf16_dev, const void *b_bf16_dev, float *d_dev,
                     const uint32_t *strides6_host, void *stream);
/* measurement hook: SM cycles for `iters` back-to-back tcgen05.mma (M 128, K 16, bf16) of width n from one thread */
int fb_debug_tc_mma_rate(int n, int mn_major, int naccs, int iters, int same_operands, long long *cycles_dev, void *stream);
/* measurement hook: re-launch one GEMM kernel of the tensor-core path `reps` times on the current workspace contents
 * (which: 1 conv2 fwd, 2 conv3 fwd, 3 fc1 fwd, 4 conv1 wgrad, 5 conv3 dgrad, 6 fc1 dgrad; 7..11 the fused conv1 on the frames of the
 * net's last forward: from the u8 frames without / with Z1 (7 / 8), from X2 without / with Z1 (9 / 10), from X2 without pooling (11).
 * 0, conv1 as a kernel of its own, is retired: FB_ERR_INVALID) */
int fb_debug_tc_kernel(fb_qnet *net, int which, int batch, int reps, const float *params_dev, void *stream);
/* test hook, tensor-core precisions only: on != 0 runs the separate conv2 / conv3 forward kernels and the separate conv3 data
 * gradient / conv2 data gradient / un-pool kernels at every minibatch (at minibatch <= 512 the fused kernels run otherwise; the
 * results are bit-identical).  Drops the net's captured graphs. */
int fb_debug_tc_separate_kernels(fb_qnet *net, int on);
/* device test hook: D[128][64] = A[shift..shift+128)[64] Bt[64][64]^T with A [256][64] loaded once as a swizzled slab and
 * the MMA descriptor started shift rows into it (the property the one-slab-many-taps convolution relies on). */
int fb_debug_tc_slab(int shift, int base_offset, const void *a_bf16_dev, const void *b_bf16_dev, float *d_dev, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FLAPPY_B200_H */
