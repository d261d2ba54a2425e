// Q-network geometry shared by the fp32 and tensor-core paths.
//
// Reference graph: BrainDQN.py:119-163 (identical in every Brain; dueling head
// BrainDuelingDQN_CC.py:68-77).  TensorFlow NHWC activations, HWIO weights, SAME padding:
//   x [B,80,80,4] -> conv 8x8 s4 (pad 2) +b relu [B,20,20,32] -> maxpool 2x2 s2 [B,10,10,32]
//     -> conv 4x4 s2 (pad 1) +b relu [B,5,5,64] -> conv 3x3 s1 (pad 1) +b relu [B,5,5,64]
//     -> flatten (h,w,c) 1600 -> fc H (512) relu -> fc A (2)   [dueling: V (1) and A (2) heads]
// Here x is never materialised: channel c of sample b is the 80x80 u8 frame at
// frames + b * sample_stride + chan_off[c] (a view of the frame ring or of a gathered batch),
// H = obs axis 0 (game x), W = obs axis 1 (game y), exactly the array the reference feeds.
#pragma once
#include <cuda_bf16.h>

#include "fb_common.cuh"

constexpr int kC1 = 32, kC2 = 64, kC3 = 64, kFlat = 1600, kActions = 2;
constexpr int kK1 = 8 * 8 * 4, kK2 = 4 * 4 * 32, kK3 = 3 * 3 * 64;

struct QnetLayout {             // offsets (in floats) into the flat parameter vector, TF variable creation order
    int hidden, dueling;
    int w1, b1, w2, b2, w3, b3, wf1, bf1;
    int wf2, bf2;               // plain head [H,2], [2]             (C51: [H,2N], [2N], column a N + i)
    int wv, bv, wa, ba;         // dueling heads [H,1],[1],[H,2],[2]  (C51: [H,N],[N],[H,2N],[2N])
    int total;
};
// The net's layout with its head: atoms 0 is the expected-value head; atoms N > 0 outputs per action are either the
// distributional (C51) head over N = 2..64 atoms (fb_c51.cu) with the support z_i = (float)(v_min + i dz), dz = (v_max - v_min) /
// (N - 1) in float64, or -- quantile set -- the quantile-regression (QR-DQN) head with N = 1..64 quantiles and the quantile-Huber
// threshold kappa (fb_qr.cu).  Kept apart from QnetLayout, which the trunk and expected-value head kernels take by value, so that
// their parameters and code stay as they are.
struct NetLayout : QnetLayout {
    int atoms;
    double v_min, v_max;
    int quantile;
    double kappa;
};

// the offsets; atoms > 0 sizes the C51 head
inline QnetLayout qnet_layout(int hidden, int dueling, int atoms = 0) {
    QnetLayout L{};
    L.hidden = hidden; L.dueling = dueling;
    const int nv = atoms ? atoms : 1, na = atoms ? kActions * atoms : kActions;     // outputs of the V head, of the A (or plain) head
    int o = 0;
    L.w1 = o; o += kK1 * kC1; L.b1 = o; o += kC1;
    L.w2 = o; o += kK2 * kC2; L.b2 = o; o += kC2;
    L.w3 = o; o += kK3 * kC3; L.b3 = o; o += kC3;
    L.wf1 = o; o += kFlat * hidden; L.bf1 = o; o += hidden;
    if (!dueling) { L.wf2 = o; o += hidden * na; L.bf2 = o; o += na; L.wv = L.bv = L.wa = L.ba = -1; }
    else { L.wv = o; o += hidden * nv; L.bv = o; o += nv; L.wa = o; o += hidden * na; L.ba = o; o += na; L.wf2 = L.bf2 = -1; }
    L.total = o;
    return L;
}

struct FrameView {              // where the 4 input channels of each sample live
    const uint8_t *base;
    long long sample_stride;    // bytes between consecutive samples
    int chan_off[4];            // byte offset of channel c (oldest frame first, newest last: BrainDQN.py:68)
    const long long *tab;       // nullptr, or [sample][tab_stride] byte offsets from `base` (replay samples read in place from the frame
                                // ring: the sampler wrote them); chan_off[c] is then the FRAME (0..tab_stride-1) channel c is, sample_stride unused
    int tab_stride;             // frames per sample in `tab`: 5 (1-step), 4 + min(n, 4) (n-step)
    __host__ __device__ const uint8_t *chan(int b, int c) const {
        return tab ? base + tab[b * tab_stride + chan_off[c]] : base + (size_t)b * sample_stride + chan_off[c];
    }
};

// The TD target of one sample, as the Python loop builds it in float64 and feeds it as fp32 (BrainDQN.py:208-214).  X is the
// variant's bootstrap value on s' (fp32).  ret == nullptr: the 1-step target y = r if terminal else r + gamma X, with the env's
// Python float 0.1.  ret != nullptr: the n-step target of fb_step_sampling.n_step, y = disc == 0 ? R : R + disc X; at n = 1
// R == r and disc == (terminal ? 0 : gamma) exactly, so both forms give the same bits.
__device__ __forceinline__ float td_target(float x, float rf, uint8_t terminal, const double *ret, const double *disc, int b, double gamma) {
    if (ret != nullptr) {
        const double R = ret[b], d = disc[b];
        return (float)(d == 0.0 ? R : R + d * (double)x);
    }
    const double r = rf == 0.1f ? 0.1 : (double)rf;          // the env returns the Python float 0.1
    return (float)(terminal ? r : r + gamma * (double)x);
}

// One tf.train.AdamOptimizer element (TF 1.12 ApplyAdam functor, as adam_kernel in fb_qnet.cu), alpha = lr sqrt(1 - beta2^t) /
// (1 - beta1^t): m += (g - m) (1 - beta1); v += (g^2 - v) (1 - beta2); var -= (m alpha) / (sqrt(v) + eps).  Returns the new var.
__device__ __forceinline__ float adam_math(float g, float pi, float &mi, float &vi, float alpha, float beta1, float beta2, float eps,
                                           float grad_scale) {
    float gi = g * grad_scale;
    mi += (gi - mi) * (1.f - beta1);
    vi += (gi * gi - vi) * (1.f - beta2);
    return pi - (mi * alpha) / (sqrtf(vi) + eps);
}

// Fused Adam (fb_qnet_step with m_dev / v_dev): one thread of the step's head kernel -- early on the step's critical path, exactly
// once per step -- turns the beta powers kept in device memory into this step's alpha = lr sqrt(1 - beta2^t) / (1 - beta1^t)
// (fp32, the host formula) and advances them; the step's last kernel reads alpha.  Nothing about a step is a launch argument.
struct AdamPow { int on; float *pow /* beta1^t, beta2^t */, *alpha; float lr, beta1, beta2; };
__device__ __forceinline__ void adam_pow_advance(const AdamPow &ap) {
    const float b1p = ap.pow[0], b2p = ap.pow[1];
    *ap.alpha = ap.lr * sqrtf(1.f - b2p) / (1.f - b1p);
    ap.pow[0] = b1p * ap.beta1; ap.pow[1] = b2p * ap.beta2;
}

// ---- distributional heads, L.atoms > 0: C51 (fb_c51.cu) and QR (fb_qr.cu).  Column space of the head's outputs: plain c = a N + i (W_fc2 /
// b_fc2); dueling c < N the V head's atom c, c = N + a N + i the A head's (a, i).  Per-sample loss gradients are kept in that
// space ([B][c51_cols]); the backward pass writes per row group partials [G][(H + 1) cols + H]: weight (j, c) at j cols + c,
// head bias c at H cols + c, fc1 bias j at (H + 1) cols + j.
constexpr int kC51MaxAtoms = 64;
constexpr int kC51Rows = 16;                // minibatch rows per head-backward row group (tensor-core path)
__host__ __device__ inline int c51_cols(const NetLayout &L) { return (L.dueling ? 3 : 2) * L.atoms; }
__host__ __device__ inline size_t c51_partial_stride(const NetLayout &L) { return (size_t)(L.hidden + 1) * c51_cols(L) + L.hidden; }
// flat parameter index of head weight (j, c), or of head bias c for j == hidden
__host__ __device__ inline int c51_flat(const NetLayout &L, int j, int c) {
    const int N = L.atoms, H = L.hidden;
    if (!L.dueling) return j < H ? L.wf2 + j * 2 * N + c : L.bf2 + c;
    if (c < N) return j < H ? L.wv + j * N + c : L.bv + c;
    return j < H ? L.wa + j * 2 * N + (c - N) : L.ba + (c - N);
}
// the inverse for a flat index inside the head
__host__ __device__ inline void c51_column(const NetLayout &L, int i, int *j, int *c) {
    const int N = L.atoms, H = L.hidden;
    if (!L.dueling) {
        if (i < L.bf2) { const int e = i - L.wf2; *j = e / (2 * N); *c = e % (2 * N); } else { *j = H; *c = i - L.bf2; }
    } else if (i < L.bv) { const int e = i - L.wv; *j = e / N; *c = e % N; }
    else if (i < L.wa) { *j = H; *c = i - L.bv; }
    else if (i < L.ba) { const int e = i - L.wa; *j = e / (2 * N); *c = N + e % (2 * N); }
    else { *j = H; *c = N + i - L.ba; }
}
// The loss kernels' shared steps.  a* of sample b: the first argmax of the variant's Q(s') (Double: qn is the online net's)
__device__ __forceinline__ int dist_astar(const float *qn, int b) { return qn[b * 2 + 1] > qn[b * 2] ? 1 : 0; }
// dLoss/d(head output c) when g = dLoss/d(output (act, c mod N)) and the other action's outputs get 0: plain, the column of the
// taken action; dueling, dv_i = sum_a d[a][i] for V columns, dalpha[a][i] = d[a][i] - sum_a d[.][i] / 2 for A columns
__device__ __forceinline__ float dist_route(const NetLayout &L, int c, int act, float g) {
    const int N = L.atoms, col = L.dueling ? c - N : c;         // col: a N + i of the output (dueling A columns), < 0 for V
    const float d0 = act == 0 ? g : 0.f, d1 = act == 1 ? g : 0.f;
    if (!L.dueling) return col / N == act ? g : 0.f;
    if (col < 0) return d0 + d1;
    return (col / N == 0 ? d0 : d1) - 0.5f * (d0 + d1);
}
int c51_prepare();              // kernel attributes (once per process, at create)
// head forward, one warp per sample: h1 from fc1's split-K partials (part != nullptr: sum in order + bias + ReLU, kept in h1_out
// when that is set) or read from h1_in; probs / logp [B][2][N] when set; q [B][2].  A QR net (L.quantile): probs receives the
// quantile locations theta, logp is not written, q = the mean of theta
int c51_launch_head_forward(const float *part, int splits, size_t split_stride, const float *h1_in, const float *params, const NetLayout &L,
                            int B, float *h1_out, float *probs, float *logp, float *q, cudaStream_t st);
// target projection, cross-entropy, dLoss/dlogits (column space) and the per-sample outputs.  pn: p of the Q(s') forward
// whose argmax (or, for Double, q_next_online's) picks a*
int c51_launch_loss(const NetLayout &L, int B, int variant, int loss_sum, int global_batch, double gamma, const float *ps, const float *logps,
                    const float *pn, const float *q_next, const float *q_next_online, const uint8_t *actions, const float *rewards,
                    const uint8_t *terminals, const float *isw, const double *ret, const double *disc, float *dl, float *terms, float *abs_err,
                    float *q_target, cudaStream_t st);
// QR net: quantile-Huber loss, dLoss/dtheta (column space) and the per-sample outputs (fb_qr.cu).  ths: theta of the training
// forward on s, thn: theta of the Q(s') forward whose argmax (or, for Double, q_next_online's) picks a*, both [B][2][N]
int qr_launch_loss(const NetLayout &L, int B, int variant, int loss_sum, int global_batch, double gamma, const float *ths, const float *thn,
                   const float *q_next, const float *q_next_online, const uint8_t *actions, const float *rewards, const uint8_t *terminals,
                   const float *isw, const double *ret, const double *disc, float *dl, float *terms, float *abs_err, float *q_target,
                   cudaStream_t st);
// head backward.  grads != nullptr (fp32 path): one row group, head weights / biases written into grads, dh1 fp32 into dh1_f32, the
// loss (terms in order) into loss_out.  Else: row groups of kC51Rows, partials into hp and the loss partial into hb[g * 4 + 2], dh1
// times gscale rounded to the 16-bit format (f16) into dh1_16, the fc1 bias partial from the rounded values; ap: the fused Adam's alpha
int c51_launch_head_backward(const NetLayout &L, int B, const float *h1, const float *dl, const float *params, const float *terms, float *grads,
                             float *loss_out, float *dh1_f32, float *hp, float *hb, void *dh1_16, int f16, float gscale, const AdamPow &ap,
                             cudaStream_t st);

// ---- handle shared by the strict-fp32 path (fb_qnet.cu) and the tcgen05 path (fb_qnet_tc.cu) ------------
struct fb_dist;                 // multi-GPU gradient exchange (fb_dist.cu)
struct TcState;                 // bf16 workspace, packed weights and TMA plans (fb_qnet_tc.cu)
struct fb_qnet {
    NetLayout L;
    int max_batch;
    int precision;              // FB_PRECISION_FP32 (CUDA-core FMA), FB_PRECISION_BF16 or FB_PRECISION_FP16 (tcgen05, fp32 accumulate)
    // fp32 activations of the online net on s (kept for backward) and scratch for the other forwards
    float *z1, *p1, *a2, *a3, *h1, *q;          // [max_batch] x {12800, 3200, 1600, 1600, H, 2}
    float *q_next, *q_next_online;
    float *dq, *dh1, *dz3, *dz2, *dp1, *dz1;
    float *partial; size_t partial_floats;
    float *loss_dev;
    TcState *tc;
    fb_dist *xch;                 // attached exchange: the training step sums every rank's gradients inside its own graph (or NULL)
    int per_broadcast;            // PER loss as the reference's graph really computes it: every sample weighted by mean(ISWeights)
    const float *packed_src[2];   // parameter vectors the bf16 operand copies (slot 0 online, 1 target) were made from
    // C51 head (L.atoms > 0), allocated at create for max_batch: p and log p of the training forward on s, p of the Q(s')
    // forward [B][2][N]; dLoss/dlogits [B][c51_cols]; loss terms [B]; head-backward partials [G][c51_partial_stride], [G][4].
    // A QR net keeps theta of s in c51_ps and theta of s' in c51_pn, and has no c51_logps
    float *c51_ps, *c51_logps, *c51_pn, *c51_dl, *c51_terms, *c51_hp, *c51_hb;
};

// small CUDA-core stages both paths share (defined in fb_qnet.cu)
void qnet_launch_head_forward(const float *h1, const float *params, const QnetLayout &L, int B, float *q, cudaStream_t st);
// ret / disc (f64[B], both or neither): n-step return and discount per sample (td_target); nullptr: the 1-step target
void qnet_launch_td_loss(const float *q_s, const float *q_next, const float *q_next_online, const uint8_t *actions,
                         const float *rewards, const uint8_t *terminals, const float *isw, int B, int global_batch, int variant,
                         double gamma, int loss_sum, float *dq, float *loss_out, float *abs_err, float *q_target, cudaStream_t st,
                         const double *ret = nullptr, const double *disc = nullptr);
void qnet_launch_head_backward(const float *h1, const float *dq, const float *params, const QnetLayout &L, int B, float *grads,
                               float *dh1_f32, __nv_bfloat16 *dh1_bf16, cudaStream_t st);

// One training step as fb_qnet_step validated it (fb_qnet.cu); both precisions run from it.  fb_qnet_step zero-fills it
// before setting any field: a captured tensor-core step is keyed on its bytes, padding included (tc_step).
// Adam: on the tensor-core path fused into the last kernel of the step, alpha from the beta powers kept in device memory, so a
// captured step replays without any per-step argument
struct AdamFuse { int on; float *m, *v; float lr, beta1, beta2, eps, grad_scale; };
struct QnetStep {
    int variant;
    const float *params, *target;
    FrameView fs, fn;                       // s and s' views of the minibatch frames
    const uint8_t *actions; const float *rewards; const uint8_t *terminals; const float *isw;
    int B, global_batch; double gamma; int loss_sum;
    float *grads, *loss_out, *abs_err, *q_target;
    AdamFuse ad;                            // ad.on: params is updated in place at the end of the step
    fb_dist *xch;                           // with ad.on: Adam over the SUM of all ranks' gradients (buckets of fb_dist.cu inside the graph)
    fb_step_sampling pro;                   // pro.replay != nullptr: the minibatch is drawn by the step's first two kernels
    const double *ret, *disc;               // n-step return / discount per sample (pro.n_step >= 1), else nullptr: 1-step target
};
// tcgen05 path entry points (fb_qnet_tc.cu); all return FB_OK or an error code with fb_set_error set
// fb_replay.cu: the two kernels of fb_replay_sample_uniform + fb_replay_gather on `st`; and the per-step patch of their
// nodes in an instantiated graph (`t` -- and through it the n-step horizon t - n + 1 -- is the only argument that changes).
// gamma: the step's discount, which the n-step gather folds into R and disc.
int replay_launch_sample_gather(const fb_step_sampling &p, double gamma, cudaStream_t st);
int replay_launch_sample(const fb_step_sampling &p, bool with_tab, cudaStream_t st);   // with_tab: ring offsets of the drawn frames -> replay_frame_tab
int replay_launch_gather(const fb_step_sampling &p, double gamma, cudaStream_t st);
const long long *replay_frame_tab(const fb_replay *r);                                   // [batch][F] byte offsets into the frame ring
int replay_frames_per_sample(const fb_step_sampling &p);                                 // F: 5 (1-step), 4 + min(n, 4) (n-step)
int replay_launch_per_update(const fb_step_sampling &p, const float *abs_err_dev, cudaStream_t st);     // Memory.batch_update, prioritized only
bool replay_is_sampler(const void *func);        // sample_uniform_kernel or per_sample_kernel
bool replay_is_gather(const void *func);
int replay_patch_nodes(cudaGraphExec_t exec, cudaGraphNode_t sampler, cudaGraphNode_t gather, const fb_step_sampling &p, double gamma);
inline bool tc_precision(int precision) { return precision == FB_PRECISION_BF16 || precision == FB_PRECISION_FP16; }
// fb_dist.cu: one bucket of the exchange + Adam as a kernel on `st` (bucket 0 = W_fc1, 1 = the rest), for the exchange buffer of
// the current parity; the buffer the step's gradients must have been written to
int dist_launch_bucket(fb_dist *d, fb_qnet *net, int bucket, float *params_dev, float *m_dev, float *v_dev, const float *alpha_dev, float beta1,
                       float beta2, float eps, float grad_scale, cudaStream_t st);
const float *dist_current_grads(const fb_dist *d);
int tc_state_create(fb_qnet *n);
int tc_set_format(fb_qnet *n, int f16);          // operand format of the tensor-core path: 0 bf16, 1 fp16
int tc_drop_graphs(fb_qnet *n);                 // captured steps embed the net's settings: drop them when one changes
void tc_state_destroy(fb_qnet *n);
int tc_pack_weights(fb_qnet *n, const float *params_dev, int slot /* 0 online, 1 target */, cudaStream_t st);
int tc_slot_for(fb_qnet *n, const float *params_dev, int want_slot, cudaStream_t st, int *slot_out);
// probs (C51 / QR net, may be nullptr): p (QR: theta) [B][2][N] beside Q
int tc_forward(fb_qnet *n, int slot, int ws, const float *params_dev, FrameView fv, int B, float *q_out, cudaStream_t st, float *probs = nullptr);
int tc_forward_chunks(fb_qnet *n, int slot, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                      const int32_t *chan_off, int batch, float *q_out_dev, cudaStream_t st, float *probs_dev = nullptr);
int tc_step(fb_qnet *n, const QnetStep &a, float beta1_power, float beta2_power, cudaStream_t st);
int tc_adam(fb_qnet *n, float *params_dev, const float *grads_dev, float *m_dev, float *v_dev, float alpha, float beta1, float beta2,
            float eps, float grad_scale, cudaStream_t st);
