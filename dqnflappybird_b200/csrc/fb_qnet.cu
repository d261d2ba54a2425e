// DQN-family Q-network: forward, epsilon-greedy acting, TD target + loss + backward, TF-1 Adam.
//
// Reference: BrainDQN.py:119-163 (graph), :99-116 (getAction), :195-223 (_trainQNetwork);
// BrainDQNNature.py:107-119,149-183 (target net, mean loss); BrainDoubleDQN.py:51-61 (Double
// target); BrainDuelingDQN_CC.py:68-77 (dueling head); BrainPrioritizedReplyDQN.py:245-253
// (IS-weighted loss, abs_errors).
//
// This file is the strict-fp32 path: every contraction is an implicit GEMM (im2col index
// arithmetic inside the tile loader, nothing materialised) on a generic shared-memory tiled
// kernel with fp32 FMA accumulation; weight gradients use deterministic split-K (partials +
// ordered reduction) and fold the bias gradient in as an extra all-ones row of the A operand.
// The tensor-core path (fb_qnet_tc.cu) replaces the big GEMMs and is checked against this one.
#include <math.h>
#include <string.h>

#include <new>

#include "fb_qnet.cuh"

// ---------------------------------------------------------------------------------- generic GEMM
// C[m][n] = sum_k A(m,k) * B(k,n) for k in this CTA's split; EP(m, n, acc, split) stores.
template <int BM, int BN, int BK, int TM, int TN, bool A_M_FAST, bool B_K_FAST, class AL, class BL, class EP>
__global__ void __launch_bounds__((BM / TM) * (BN / TN)) gemm_f32(int M, int N, int K, int klen, AL al, BL bl, EP ep) {
    constexpr int NT = (BM / TM) * (BN / TN);
    __shared__ float As[BM][BK + 1];
    __shared__ float Bs[BK][BN + 1];
    const int tid = threadIdx.x, tx = tid % (BN / TN), ty = tid / (BN / TN);
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int kbeg = blockIdx.z * klen, kend = min(K, kbeg + klen);
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
        for (int j = 0; j < TN; j++) acc[i][j] = 0.f;
    for (int k0 = kbeg; k0 < kend; k0 += BK) {
#pragma unroll
        for (int e = tid; e < BM * BK; e += NT) {
            int mm = A_M_FAST ? e % BM : e / BK, kk = A_M_FAST ? e / BM : e % BK;
            int m = m0 + mm, k = k0 + kk;
            As[mm][kk] = (m < M && k < kend) ? al(m, k) : 0.f;
        }
#pragma unroll
        for (int e = tid; e < BK * BN; e += NT) {
            int kk = B_K_FAST ? e % BK : e / BN, nn = B_K_FAST ? e / BK : e % BN;
            int k = k0 + kk, n = n0 + nn;
            Bs[kk][nn] = (k < kend && n < N) ? bl(k, n) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; kk++) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; i++) a[i] = As[ty * TM + i][kk];
#pragma unroll
            for (int j = 0; j < TN; j++) b[j] = Bs[kk][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; i++)
#pragma unroll
                for (int j = 0; j < TN; j++) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < TM; i++)
#pragma unroll
        for (int j = 0; j < TN; j++) {
            int m = m0 + ty * TM + i, n = n0 + tx * TN + j;
            if (m < M && n < N) ep(m, n, acc[i][j], (int)blockIdx.z);
        }
}

template <int BN, bool A_M_FAST, bool B_K_FAST, class AL, class BL, class EP>
static void launch_gemm(int M, int N, int K, int splits, AL al, BL bl, EP ep, cudaStream_t st) {
    int klen = (K + splits - 1) / splits;
    klen = (klen + 15) / 16 * 16;
    if (BN == 64) {
        dim3 grid((N + 63) / 64, (M + 63) / 64, splits);
        gemm_f32<64, 64, 16, 4, 4, A_M_FAST, B_K_FAST><<<grid, 256, 0, st>>>(M, N, K, klen, al, bl, ep);
    } else {
        dim3 grid((N + 31) / 32, (M + 63) / 64, splits);
        gemm_f32<64, 32, 16, 4, 2, A_M_FAST, B_K_FAST><<<grid, 256, 0, st>>>(M, N, K, klen, al, bl, ep);
    }
}

// ---------------------------------------------------------------------------------- loaders / epilogues
struct LoadPlain { const float *p; int ld; __device__ float operator()(int r, int c) const { return __ldg(p + (size_t)r * ld + c); } };
struct LoadTrans { const float *p; int ld; __device__ float operator()(int r, int c) const { return __ldg(p + (size_t)c * ld + r); } };

struct LoadConv1 {              // A(m = (b,oh,ow), k = (kh,kw,c)) of conv 8x8 s4 pad 2 on the u8 frames
    FrameView fv;
    __device__ float operator()(int m, int k) const {
        int b = m / 400, r = m - b * 400, oh = r / 20, ow = r - oh * 20;
        int kh = k >> 5, kw = (k >> 2) & 7, c = k & 3;
        int ih = oh * 4 + kh - 2, iw = ow * 4 + kw - 2;
        if ((unsigned)ih >= 80u || (unsigned)iw >= 80u) return 0.f;
        return (float)__ldg(fv.base + (size_t)b * fv.sample_stride + fv.chan_off[c] + ih * 80 + iw);
    }
};
struct LoadConv1T {             // wgrad: A(m = (kh,kw,c) | bias row 256, k = (b,oh,ow))
    FrameView fv;
    __device__ float operator()(int m, int k) const {
        if (m == kK1) return 1.f;
        return LoadConv1{fv}(k, m);
    }
};
struct LoadConv2 {              // A(m = (b,oh,ow) 5x5, k = (kh,kw,c) 4x4x32) on pooled [B,10,10,32], s2 pad 1
    const float *p1;
    __device__ float operator()(int m, int k) const {
        int b = m / 25, r = m - b * 25, oh = r / 5, ow = r - oh * 5;
        int kh = k >> 7, kw = (k >> 5) & 3, c = k & 31;
        int ih = oh * 2 + kh - 1, iw = ow * 2 + kw - 1;
        if ((unsigned)ih >= 10u || (unsigned)iw >= 10u) return 0.f;
        return __ldg(p1 + ((size_t)(b * 10 + ih) * 10 + iw) * 32 + c);
    }
};
struct LoadConv2T { const float *p1; __device__ float operator()(int m, int k) const { return m == kK2 ? 1.f : LoadConv2{p1}(k, m); } };
struct LoadConv3 {              // A(m = (b,oh,ow) 5x5, k = (kh,kw,c) 3x3x64) on [B,5,5,64], s1 pad 1
    const float *a2;
    __device__ float operator()(int m, int k) const {
        int b = m / 25, r = m - b * 25, oh = r / 5, ow = r - oh * 5;
        int kh = k / 192, r2 = k - kh * 192, kw = r2 >> 6, c = r2 & 63;
        int ih = oh + kh - 1, iw = ow + kw - 1;
        if ((unsigned)ih >= 5u || (unsigned)iw >= 5u) return 0.f;
        return __ldg(a2 + ((size_t)(b * 5 + ih) * 5 + iw) * 64 + c);
    }
};
struct LoadConv3T { const float *a2; __device__ float operator()(int m, int k) const { return m == kK3 ? 1.f : LoadConv3{a2}(k, m); } };
struct LoadFc1T {               // wgrad fc1: A(m = flat index | bias row, k = b)
    const float *a3;
    __device__ float operator()(int m, int k) const { return m == kFlat ? 1.f : __ldg(a3 + (size_t)k * kFlat + m); }
};
struct LoadDgrad3 {             // dgrad conv3: A(m = (b,ih,iw), k = (kh,kw,o)) = dz3[b][ih-kh+1][iw-kw+1][o]
    const float *dz3;
    __device__ float operator()(int m, int k) const {
        int b = m / 25, r = m - b * 25, ih = r / 5, iw = r - ih * 5;
        int kh = k / 192, r2 = k - kh * 192, kw = r2 >> 6, o = r2 & 63;
        int oh = ih - kh + 1, ow = iw - kw + 1;
        if ((unsigned)oh >= 5u || (unsigned)ow >= 5u) return 0.f;
        return __ldg(dz3 + ((size_t)(b * 5 + oh) * 5 + ow) * 64 + o);
    }
};
struct LoadW3T {                // B(k = (kh,kw,o), n = c) = W3[kh][kw][c][o]
    const float *w3;
    __device__ float operator()(int k, int n) const {
        int khkw = k >> 6, o = k & 63;
        return __ldg(w3 + ((size_t)khkw * 64 + n) * 64 + o);
    }
};
struct LoadDgrad2 {             // dgrad conv2 (s2 pad 1): A(m = (b,ih,iw) 10x10, k = (kh,kw,o) 4x4x64)
    const float *dz2;
    __device__ float operator()(int m, int k) const {
        int b = m / 100, r = m - b * 100, ih = r / 10, iw = r - ih * 10;
        int kh = k >> 8, kw = (k >> 6) & 3, o = k & 63;
        int oh2 = ih + 1 - kh, ow2 = iw + 1 - kw;
        if (oh2 < 0 || ow2 < 0 || (oh2 & 1) || (ow2 & 1) || oh2 >= 10 || ow2 >= 10) return 0.f;
        return __ldg(dz2 + ((size_t)(b * 5 + (oh2 >> 1)) * 5 + (ow2 >> 1)) * 64 + o);
    }
};
struct LoadW2T {                // B(k = (kh,kw,o), n = c) = W2[kh][kw][c][o]
    const float *w2;
    __device__ float operator()(int k, int n) const {
        int khkw = k >> 6, o = k & 63;
        return __ldg(w2 + ((size_t)khkw * 32 + n) * 64 + o);
    }
};

struct EpiBiasRelu { float *out; const float *bias; int ld; __device__ void operator()(int m, int n, float v, int) const { out[(size_t)m * ld + n] = fmaxf(v + __ldg(bias + n), 0.f); } };
struct EpiStore { float *out; int ld; __device__ void operator()(int m, int n, float v, int) const { out[(size_t)m * ld + n] = v; } };
struct EpiMaskPos { float *out; const float *act; int ld; __device__ void operator()(int m, int n, float v, int) const { size_t i = (size_t)m * ld + n; out[i] = __ldg(act + i) > 0.f ? v : 0.f; } };
struct EpiPartial { float *part; int ld; size_t split_stride; __device__ void operator()(int m, int n, float v, int s) const { part[(size_t)s * split_stride + (size_t)m * ld + n] = v; } };

// ---------------------------------------------------------------------------------- small kernels
__global__ void maxpool_kernel(const float *z1, float *p1, int B) {        // [B,20,20,32] -> [B,10,10,32], BrainDQN.py:128
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * 3200) return;
    int c = i & 31; size_t r = i >> 5; int pw = r % 10; r /= 10; int ph = r % 10; int b = (int)(r / 10);
    const float *s = z1 + (((size_t)b * 20 + ph * 2) * 20 + pw * 2) * 32 + c;
    p1[i] = fmaxf(fmaxf(s[0], s[32]), fmaxf(s[640], s[672]));
}

// dz1 = unpool(dp1) * relu'(z1): gradient goes to the first maximum of each 2x2 window (TF MaxPoolGrad)
__global__ void unpool_relu_kernel(const float *z1, const float *p1, const float *dp1, float *dz1, int B) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * 3200) return;
    int c = i & 31; size_t r = i >> 5; int pw = r % 10; r /= 10; int ph = r % 10; int b = (int)(r / 10);
    size_t base = (((size_t)b * 20 + ph * 2) * 20 + pw * 2) * 32 + c;
    float p = p1[i], g = dp1[i];
    const int off[4] = {0, 32, 640, 672};
    bool done = false;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        float z = z1[base + off[q]];
        bool hit = !done && z == p;
        dz1[base + off[q]] = (hit && z > 0.f) ? g : 0.f;
        done |= hit;
    }
}

// Q head.  plain: Q = h1 W + b (BrainDQN.py:151-154).  dueling: Q = V + (A - mean_a A) (BrainDuelingDQN_CC.py:68-77)
__global__ void head_forward_kernel(const float *h1, const float *params, QnetLayout L, int B, float *q) {
    int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    const float *h = h1 + (size_t)b * L.hidden;
    float s0 = 0.f, s1 = 0.f, sv = 0.f;
    for (int j = lane; j < L.hidden; j += 32) {
        float x = h[j];
        if (!L.dueling) { s0 = fmaf(x, params[L.wf2 + j * 2], s0); s1 = fmaf(x, params[L.wf2 + j * 2 + 1], s1); }
        else { s0 = fmaf(x, params[L.wa + j * 2], s0); s1 = fmaf(x, params[L.wa + j * 2 + 1], s1); sv = fmaf(x, params[L.wv + j], sv); }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) { s0 += __shfl_xor_sync(~0u, s0, o); s1 += __shfl_xor_sync(~0u, s1, o); sv += __shfl_xor_sync(~0u, sv, o); }
    if (lane == 0) {
        if (!L.dueling) { q[b * 2] = s0 + params[L.bf2]; q[b * 2 + 1] = s1 + params[L.bf2 + 1]; }
        else {
            float a0 = s0 + params[L.ba], a1 = s1 + params[L.ba + 1], v = sv + params[L.bv];
            float mean = (a0 + a1) * 0.5f;
            q[b * 2] = v + (a0 - mean); q[b * 2 + 1] = v + (a1 - mean);
        }
    }
}

// TD target, loss and dLoss/dQ.
//   variant 0 vanilla: X = max_a Q_online(s')          (BrainDQN.py:204-214)
//   variant 1 nature : X = max_a Q_target(s')          (BrainDQNNature.py:163-175)
//   variant 2 double : X = Q_target(s', argmax_a Q_online(s'))   (BrainDoubleDQN.py:51-61)
//   y = r if terminal else r + gamma * X, built in float64 like the Python loop, fed as fp32 (td_target in fb_qnet.cuh; with
//   ret / disc the n-step target disc == 0 ? R : R + disc * X).
//   loss = sum (y-q)^2 (loss_sum, BrainDQN.py:162) | mean (BrainDQNNature.py:119) | mean w (y-q)^2 (PER :251)
__global__ void td_loss_kernel(const float *q_s, const float *q_next, const float *q_next_online, const uint8_t *actions,
                               const float *rewards, const uint8_t *terminals, const float *isw, int B, int global_batch,
                               int variant, double gamma, int loss_sum, float *dq, float *loss_out, float *abs_err,
                               float *q_target, int isw_mean, const double *ret, const double *disc) {
    __shared__ float red[32];
    __shared__ float wmean_s;
    float local = 0.f;
    // isw_mean: ISWeights is a [B,1] placeholder multiplied with a [B] vector (BrainPrioritizedReplyDQN.py:243-251): TensorFlow
    // broadcasts to [B,B], so the cost the reference minimises is mean(w) * mean(err^2) -- every sample weighted by mean(w)
    if (isw && isw_mean) {
        if (threadIdx.x == 0) { float s = 0.f; for (int b = 0; b < B; b++) s += isw[b]; wmean_s = s / (float)B; }
        __syncthreads();
    }
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        float x;
        if (variant == 2) { int am = q_next_online[b * 2 + 1] > q_next_online[b * 2] ? 1 : 0; x = q_next[b * 2 + am]; }
        else x = fmaxf(q_next[b * 2], q_next[b * 2 + 1]);
        float y = td_target(x, rewards[b], terminals[b], ret, disc, b, gamma);
        int a = actions[b] ? 1 : 0;
        float qa = q_s[b * 2 + a];
        float err = y - qa;
        float w = isw ? (isw_mean ? wmean_s : isw[b]) : 1.f;
        float scale = loss_sum ? 1.f : 1.f / (float)global_batch;
        local += w * err * err * scale;
        float g = -2.f * w * err * scale;
        dq[b * 2 + a] = g; dq[b * 2 + (1 - a)] = 0.f;
        if (abs_err) abs_err[b] = fabsf(err);
        if (q_target) q_target[b] = y;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) local += __shfl_xor_sync(~0u, local, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int k = 0; k < (int)(blockDim.x >> 5); k++) s += red[k];
        if (loss_out) *loss_out = s;
    }
}

// head backward: grads of the head weights/biases (sum over b in order) and dh1 (masked by relu)
__global__ void head_backward_w_kernel(const float *h1, const float *dq, QnetLayout L, int B, float *grads) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;         // j in [0, hidden] ; hidden = bias row
    if (j > L.hidden) return;
    float g0 = 0.f, g1 = 0.f, gv = 0.f;
    for (int b = 0; b < B; b++) {
        float x = j == L.hidden ? 1.f : h1[(size_t)b * L.hidden + j];
        float d0 = dq[b * 2], d1 = dq[b * 2 + 1];
        if (!L.dueling) { g0 = fmaf(x, d0, g0); g1 = fmaf(x, d1, g1); }
        else { float m = (d0 + d1) * 0.5f; g0 = fmaf(x, d0 - m, g0); g1 = fmaf(x, d1 - m, g1); gv = fmaf(x, d0 + d1, gv); }
    }
    if (!L.dueling) {
        if (j < L.hidden) { grads[L.wf2 + j * 2] = g0; grads[L.wf2 + j * 2 + 1] = g1; }
        else { grads[L.bf2] = g0; grads[L.bf2 + 1] = g1; }
    } else {
        if (j < L.hidden) { grads[L.wa + j * 2] = g0; grads[L.wa + j * 2 + 1] = g1; grads[L.wv + j] = gv; }
        else { grads[L.ba] = g0; grads[L.ba + 1] = g1; grads[L.bv] = gv; }
    }
}

__global__ void head_backward_h_kernel(const float *h1, const float *dq, const float *params, QnetLayout L, int B, float *dh1,
                                       __nv_bfloat16 *dh1_bf16) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * L.hidden) return;
    int b = (int)(i / L.hidden), j = (int)(i - (size_t)b * L.hidden);
    float d0 = dq[b * 2], d1 = dq[b * 2 + 1], g;
    if (!L.dueling) g = d0 * params[L.wf2 + j * 2] + d1 * params[L.wf2 + j * 2 + 1];
    else { float m = (d0 + d1) * 0.5f; g = (d0 - m) * params[L.wa + j * 2] + (d1 - m) * params[L.wa + j * 2 + 1] + (d0 + d1) * params[L.wv + j]; }
    g = h1[i] > 0.f ? g : 0.f;
    if (dh1) dh1[i] = g;
    if (dh1_bf16) dh1_bf16[i] = __float2bfloat16(g);
}

void qnet_launch_head_forward(const float *h1, const float *params, const QnetLayout &L, int B, float *q, cudaStream_t st) {
    head_forward_kernel<<<(B + 3) / 4, 128, 0, st>>>(h1, params, L, B, q);
}
void qnet_launch_td_loss(const float *q_s, const float *q_next, const float *q_next_online, const uint8_t *actions,
                         const float *rewards, const uint8_t *terminals, const float *isw, int B, int global_batch, int variant,
                         double gamma, int loss_sum, float *dq, float *loss_out, float *abs_err, float *q_target, cudaStream_t st,
                         const double *ret, const double *disc) {
    td_loss_kernel<<<1, 256, 0, st>>>(q_s, q_next, q_next_online, actions, rewards, terminals, isw, B, global_batch, variant, gamma,
                                       loss_sum, dq, loss_out, abs_err, q_target, 0, ret, disc);
}
void qnet_launch_head_backward(const float *h1, const float *dq, const float *params, const QnetLayout &L, int B, float *grads,
                               float *dh1_f32, __nv_bfloat16 *dh1_bf16, cudaStream_t st) {
    head_backward_w_kernel<<<(L.hidden + 1 + 127) / 128, 128, 0, st>>>(h1, dq, L, B, grads);
    head_backward_h_kernel<<<(B * L.hidden + 255) / 256, 256, 0, st>>>(h1, dq, params, L, B, dh1_f32, dh1_bf16);
}

__global__ void splitk_reduce_kernel(const float *part, int splits, size_t n, float *out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = 0.f;
    for (int k = 0; k < splits; k++) s += part[(size_t)k * n + i];
    out[i] = s;
}

// tf.train.AdamOptimizer (TF 1.12 ApplyAdam functor), alpha = lr * sqrt(1 - beta2^t) / (1 - beta1^t):
//   m += (g - m) (1 - beta1);  v += (g^2 - v) (1 - beta2);  var -= (m alpha) / (sqrt(v) + eps)
__global__ void adam_kernel(float *p, const float *g, float *m, float *v, size_t n, float alpha, float beta1, float beta2,
                            float eps, float grad_scale) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float gi = g[i] * grad_scale;
    float mi = m[i], vi = v[i];
    mi += (gi - mi) * (1.f - beta1);
    vi += (gi * gi - vi) * (1.f - beta2);
    m[i] = mi; v[i] = vi;
    p[i] -= (mi * alpha) / (sqrtf(vi) + eps);
}

// epsilon-greedy (BrainDQN.py:102-108): random.random() <= epsilon ? randrange(2) : argmax(Q) (first max on ties).
// Each env owns Philox stream (seed, purpose 2, env id); random() consumes two words (a>>5, b>>6 -> 53 bits),
// randrange(2) = getrandbits(2) = word >> 30 with rejection while >= 2.
__global__ void egreedy_kernel(const float *q, int n, double epsilon, uint64_t seed, uint64_t first_env_id, uint32_t *rng_pos,
                               uint8_t *actions) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    uint32_t pos = rng_pos[e];
    uint64_t id = first_env_id + (uint64_t)e;
    uint32_t a = stream_word(seed, 2u, id, pos) >> 5, b = stream_word(seed, 2u, id, pos + 1) >> 6;
    pos += 2;
    double u = ((double)a * 67108864.0 + (double)b) * (1.0 / 9007199254740992.0);
    int act;
    if (u <= epsilon) {
        for (;;) { uint32_t r = stream_word(seed, 2u, id, pos++) >> 30; if (r < 2u) { act = (int)r; break; } }
    } else act = q[e * 2 + 1] > q[e * 2] ? 1 : 0;
    rng_pos[e] = pos;
    actions[e] = (uint8_t)act;
}

// ---------------------------------------------------------------------------------- handle (struct fb_qnet: fb_qnet.cuh)

// weight (+ bias, as the extra all-ones row M) gradient: (M+1) x N = A^T dz over K, deterministic split-K
template <bool A_M_FAST, class AL>
static void wgrad(fb_qnet *n, int M, int N, int K, int kchunk, AL al, const float *dz, float *gout, cudaStream_t st) {
    int splits = (K + kchunk - 1) / kchunk;
    size_t mn = (size_t)(M + 1) * N;
    if (N == 32) launch_gemm<32, A_M_FAST, false>(M + 1, N, K, splits, al, LoadPlain{dz, N}, EpiPartial{n->partial, N, mn}, st);
    else launch_gemm<64, A_M_FAST, false>(M + 1, N, K, splits, al, LoadPlain{dz, N}, EpiPartial{n->partial, N, mn}, st);
    splitk_reduce_kernel<<<(unsigned)((mn + 255) / 256), 256, 0, st>>>(n->partial, splits, mn, gout);
}

static int forward_chunk(fb_qnet *n, const float *params, FrameView fv, int B, float *q_out, cudaStream_t st) {
    const QnetLayout &L = n->L;
    launch_gemm<32, false, false>(B * 400, kC1, kK1, 1, LoadConv1{fv}, LoadPlain{params + L.w1, kC1},
                                  EpiBiasRelu{n->z1, params + L.b1, kC1}, st);
    maxpool_kernel<<<(B * 3200 + 255) / 256, 256, 0, st>>>(n->z1, n->p1, B);
    launch_gemm<64, false, false>(B * 25, kC2, kK2, 1, LoadConv2{n->p1}, LoadPlain{params + L.w2, kC2},
                                  EpiBiasRelu{n->a2, params + L.b2, kC2}, st);
    launch_gemm<64, false, false>(B * 25, kC3, kK3, 1, LoadConv3{n->a2}, LoadPlain{params + L.w3, kC3},
                                  EpiBiasRelu{n->a3, params + L.b3, kC3}, st);
    launch_gemm<64, false, false>(B, L.hidden, kFlat, 1, LoadPlain{n->a3, kFlat}, LoadPlain{params + L.wf1, L.hidden},
                                  EpiBiasRelu{n->h1, params + L.bf1, L.hidden}, st);
    head_forward_kernel<<<(B + 3) / 4, 128, 0, st>>>(n->h1, params, L, B, q_out);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

extern "C" int fb_qnet_create(int hidden, int dueling, int max_batch, fb_qnet **out) {
    FB_REQUIRE(out != nullptr && hidden > 0 && hidden % 4 == 0 && max_batch > 0, "fb_qnet_create: bad argument");
    fb_qnet *n = new (std::nothrow) fb_qnet();
    FB_REQUIRE(n != nullptr, "fb_qnet_create: out of host memory");
    n->L = qnet_layout(hidden, dueling ? 1 : 0);
    n->max_batch = max_batch;
    n->precision = FB_PRECISION_FP32;
    n->tc = nullptr;
    n->per_broadcast = 0;
    n->xch = nullptr;
    size_t B = (size_t)max_batch;
    auto alloc = [](float **p, size_t floats) { return cudaMalloc(p, floats * sizeof(float)); };
    FB_CUDA_OK(alloc(&n->z1, B * 12800)); FB_CUDA_OK(alloc(&n->p1, B * 3200)); FB_CUDA_OK(alloc(&n->a2, B * 1600));
    FB_CUDA_OK(alloc(&n->a3, B * 1600)); FB_CUDA_OK(alloc(&n->h1, B * hidden)); FB_CUDA_OK(alloc(&n->q, B * 2));
    FB_CUDA_OK(alloc(&n->q_next, B * 2)); FB_CUDA_OK(alloc(&n->q_next_online, B * 2));
    FB_CUDA_OK(alloc(&n->dq, B * 2)); FB_CUDA_OK(alloc(&n->dh1, B * hidden)); FB_CUDA_OK(alloc(&n->dz3, B * 1600));
    FB_CUDA_OK(alloc(&n->dz2, B * 1600)); FB_CUDA_OK(alloc(&n->dp1, B * 3200)); FB_CUDA_OK(alloc(&n->dz1, B * 12800));
    // split-K partials: the largest user is fc1 ((1600+1) x H per split) and conv1 (K = B*400)
    size_t s1 = (B * 400 + 2047) / 2048, s23 = (B * 25 + 511) / 512, sf = (B + 63) / 64;
    size_t need = s1 * (size_t)(kK1 + 1) * kC1;
    size_t c = s23 * (size_t)(kK3 + 1) * kC3; if (c > need) need = c;
    c = sf * (size_t)(kFlat + 1) * hidden; if (c > need) need = c;
    n->partial_floats = need;
    FB_CUDA_OK(alloc(&n->partial, need));
    FB_CUDA_OK(alloc(&n->loss_dev, 4));
    *out = n;
    return FB_OK;
}

extern "C" int fb_qnet_destroy(fb_qnet *n) {
    if (!n) return FB_OK;
    tc_state_destroy(n);
    float *ps[] = {n->z1, n->p1, n->a2, n->a3, n->h1, n->q, n->q_next, n->q_next_online, n->dq, n->dh1, n->dz3, n->dz2, n->dp1, n->dz1, n->partial, n->loss_dev};
    for (float *p : ps) cudaFree(p);
    delete n;
    return FB_OK;
}

extern "C" int fb_qnet_set_precision(fb_qnet *n, int precision) {
    FB_REQUIRE(n != nullptr && (precision == FB_PRECISION_FP32 || precision == FB_PRECISION_BF16 || precision == FB_PRECISION_FP16),
               "fb_qnet_set_precision: bad argument");
    if (precision != FB_PRECISION_FP32) { int rc = tc_state_create(n); if (rc) return rc; rc = tc_set_format(n, precision == FB_PRECISION_FP16); if (rc) return rc; }
    n->precision = precision;
    n->packed_src[0] = n->packed_src[1] = nullptr;
    return FB_OK;
}

extern "C" int fb_qnet_get_precision(const fb_qnet *n) { return n ? n->precision : -1; }

// Several GPUs, tensor-core path: fb_qnet_step with Adam then sums every rank's gradients inside its own graph (the
// exchange's two buckets are kernels of the step, fb_dist.cu) and applies Adam to the sum; `grads_dev` must be the exchange's
// current buffer (fb_dist_grads / fb_dist_parity) and the caller calls fb_dist_advance after each step.  NULL detaches.
extern "C" int fb_qnet_attach_exchange(fb_qnet *n, fb_dist *d) {
    FB_REQUIRE(n != nullptr, "fb_qnet_attach_exchange: NULL argument");
    n->xch = d;
    return tc_drop_graphs(n);
}

// PER loss as the reference's graph computes it (BrainPrioritizedReplyDQN.py:243-251): ISWeights [B,1] * square(...) [B] is
// broadcast to [B,B] by TensorFlow, so reduce_mean gives mean(w) * mean(err^2) and every sample's gradient is scaled by
// mean(w) instead of its own w.  Off (default): the intended mean(w_i err_i^2).
extern "C" int fb_qnet_set_per_broadcast(fb_qnet *n, int on) {
    FB_REQUIRE(n != nullptr, "fb_qnet_set_per_broadcast: NULL argument");
    n->per_broadcast = on ? 1 : 0;
    return tc_drop_graphs(n);
}

// The bf16 operand copies of a parameter vector are remade when the vector may have changed: after fb_qnet_adam /
// fb_qnet_sync_target on it, or when the caller says so (it wrote the tensor itself).
extern "C" int fb_qnet_invalidate(fb_qnet *n) {
    FB_REQUIRE(n != nullptr, "fb_qnet_invalidate: NULL argument");
    n->packed_src[0] = n->packed_src[1] = nullptr;
    return FB_OK;
}

extern "C" int fb_qnet_param_count(const fb_qnet *n) { return n ? n->L.total : 0; }

extern "C" int fb_qnet_layout(const fb_qnet *n, int32_t *o) {
    FB_REQUIRE(n != nullptr && o != nullptr, "fb_qnet_layout: NULL argument");
    const QnetLayout &L = n->L;
    int v[16] = {L.w1, L.b1, L.w2, L.b2, L.w3, L.b3, L.wf1, L.bf1, L.wf2, L.bf2, L.wv, L.bv, L.wa, L.ba, L.total, L.hidden};
    for (int k = 0; k < 16; k++) o[k] = v[k];
    return FB_OK;
}

// field by field: a view inside a zero-filled QnetStep keeps its padding bytes zero
static void set_view(FrameView &fv, const uint8_t *frames, long long stride, const int32_t *chan_off, const long long *tab = nullptr,
                     int tab_stride = 0) {
    fv.base = frames; fv.sample_stride = stride; fv.tab = tab; fv.tab_stride = tab_stride;
    for (int c = 0; c < 4; c++) fv.chan_off[c] = chan_off[c];
}

extern "C" int fb_qnet_forward(fb_qnet *n, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                               const int32_t *chan_off, int batch, float *q_out_dev, void *stream) {
    FB_REQUIRE(n && params_dev && frames_dev && chan_off && q_out_dev && batch > 0, "fb_qnet_forward: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    int slot = 0;
    if (tc_precision(n->precision)) {
        int rc = tc_slot_for(n, params_dev, -1, st, &slot); if (rc) return rc;
        return tc_forward_chunks(n, slot, params_dev, frames_dev, sample_stride, chan_off, batch, q_out_dev, st);
    }
    for (int b0 = 0; b0 < batch; b0 += n->max_batch) {
        int B = min(n->max_batch, batch - b0);
        FrameView fv;
        set_view(fv, frames_dev + (size_t)b0 * sample_stride, sample_stride, chan_off);
        int rc = tc_precision(n->precision) ? tc_forward(n, slot, 0, params_dev, fv, B, q_out_dev + (size_t)b0 * 2, st)
                                                   : forward_chunk(n, params_dev, fv, B, q_out_dev + (size_t)b0 * 2, st);
        if (rc) return rc;
    }
    return FB_OK;
}

extern "C" int fb_qnet_act(fb_qnet *n, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                           const int32_t *chan_off, int batch, double epsilon, uint64_t seed, uint64_t first_env_id,
                           uint32_t *rng_pos_dev, float *q_out_dev, uint8_t *actions_out_dev, void *stream) {
    FB_REQUIRE(rng_pos_dev && actions_out_dev, "fb_qnet_act: bad argument");
    int rc = fb_qnet_forward(n, params_dev, frames_dev, sample_stride, chan_off, batch, q_out_dev, stream);
    if (rc) return rc;
    egreedy_kernel<<<(batch + 255) / 256, 256, 0, (cudaStream_t)stream>>>(q_out_dev, batch, epsilon, seed, first_env_id, rng_pos_dev, actions_out_dev);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

// TD target, loss and backward of the strict-fp32 path into a.grads
static int loss_backward_impl(fb_qnet *n, const QnetStep &a, cudaStream_t st) {
    const QnetLayout &L = n->L;
    const int B = a.B;
    int rc;
    // Q(s') with the net the variant names (and the online net too for Double), then Q(s) last so that its
    // activations are the ones left in the workspace for the backward pass.
    if (a.variant == 2) { rc = forward_chunk(n, a.params, a.fn, B, n->q_next_online, st); if (rc) return rc; }
    rc = forward_chunk(n, a.variant == 0 ? a.params : a.target, a.fn, B, n->q_next, st); if (rc) return rc;
    rc = forward_chunk(n, a.params, a.fs, B, n->q, st); if (rc) return rc;
    td_loss_kernel<<<1, 256, 0, st>>>(n->q, n->q_next, n->q_next_online, a.actions, a.rewards, a.terminals, a.isw, B, a.global_batch,
                                       a.variant, a.gamma, a.loss_sum, n->dq, a.loss_out, a.abs_err, a.q_target, n->per_broadcast, a.ret,
                                       a.disc);
    // ---- backward
    head_backward_w_kernel<<<(L.hidden + 1 + 127) / 128, 128, 0, st>>>(n->h1, n->dq, L, B, a.grads);
    head_backward_h_kernel<<<(B * L.hidden + 255) / 256, 256, 0, st>>>(n->h1, n->dq, a.params, L, B, n->dh1, nullptr);
    // fc1: dW = a3^T dh1 (+ bias row), da3 = dh1 Wf1^T masked by relu(a3)
    wgrad<true>(n, kFlat, L.hidden, B, 64, LoadFc1T{n->a3}, n->dh1, a.grads + L.wf1, st);
    launch_gemm<64, false, true>(B, kFlat, L.hidden, 1, LoadPlain{n->dh1, L.hidden}, LoadTrans{a.params + L.wf1, L.hidden},
                                 EpiMaskPos{n->dz3, n->a3, kFlat}, st);
    // conv3
    wgrad<true>(n, kK3, kC3, B * 25, 512, LoadConv3T{n->a2}, n->dz3, a.grads + L.w3, st);
    launch_gemm<64, false, true>(B * 25, kC2, kK3, 1, LoadDgrad3{n->dz3}, LoadW3T{a.params + L.w3}, EpiMaskPos{n->dz2, n->a2, kC2}, st);
    // conv2
    wgrad<true>(n, kK2, kC2, B * 25, 512, LoadConv2T{n->p1}, n->dz2, a.grads + L.w2, st);
    launch_gemm<32, false, true>(B * 100, kC1, 4 * 4 * kC2, 1, LoadDgrad2{n->dz2}, LoadW2T{a.params + L.w2}, EpiStore{n->dp1, kC1}, st);
    unpool_relu_kernel<<<(B * 3200 + 255) / 256, 256, 0, st>>>(n->z1, n->p1, n->dp1, n->dz1, B);
    // conv1 (no input gradient)
    wgrad<false>(n, kK1, kC1, B * 400, 2048, LoadConv1T{a.fs}, n->dz1, a.grads + L.w1, st);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

extern "C" int fb_qnet_adam(fb_qnet *n, float *params_dev, const float *grads_dev, float *m_dev, float *v_dev, float alpha,
                            float beta1, float beta2, float eps, float grad_scale, void *stream) {
    FB_REQUIRE(n && params_dev && grads_dev && m_dev && v_dev, "fb_qnet_adam: NULL argument");
    if (tc_precision(n->precision))    // the same update, plus the bf16 operand copies of what it writes
        return tc_adam(n, params_dev, grads_dev, m_dev, v_dev, alpha, beta1, beta2, eps, grad_scale, (cudaStream_t)stream);
    size_t cnt = (size_t)n->L.total;
    adam_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, (cudaStream_t)stream>>>(params_dev, grads_dev, m_dev, v_dev, cnt, alpha, beta1, beta2, eps, grad_scale);
    FB_CUDA_OK(cudaGetLastError());
    for (int s = 0; s < 2; s++) if (n->packed_src[s] == params_dev) n->packed_src[s] = nullptr;
    return FB_OK;
}

// _trainQNetwork up to session.run(trainStep) (BrainDQN.py:195-223): sampling, loss, backward and Adam as the arguments ask.
// On the tensor-core path it is one CUDA graph launch (tc_step); here the same stages run one after the other.
extern "C" int fb_qnet_step(fb_qnet *n, const fb_qnet_step_args *a, void *stream) {
    FB_REQUIRE(n && a && a->params_dev && a->grads_dev, "fb_qnet_step: NULL argument");
    FB_REQUIRE(a->variant >= 0 && a->variant <= 2, "fb_qnet_step: variant must be 0 (vanilla), 1 (nature) or 2 (double)");
    FB_REQUIRE(a->variant == 0 || a->target_params_dev != nullptr, "fb_qnet_step: target parameters required");
    FB_REQUIRE((a->m_dev != nullptr) == (a->v_dev != nullptr), "fb_qnet_step: m_dev and v_dev must both be set (Adam) or both be NULL");
    const fb_step_sampling *sp = a->sampling;
    if (sp) {
        bool caller_minibatch = a->frames_dev || a->sample_stride || a->actions_dev || a->rewards_dev || a->terminals_dev || a->is_weights_dev;
        for (int c = 0; c < 4; c++) caller_minibatch = caller_minibatch || a->chan_off_s[c] || a->chan_off_next[c];
        FB_REQUIRE(!caller_minibatch, "fb_qnet_step: with `sampling` the step draws its minibatch: frames_dev .. is_weights_dev must be 0 / NULL");
        FB_REQUIRE(sp->replay && (a->batch == 0 || a->batch == sp->batch), "fb_qnet_step: bad sampling descriptor or batch");
        FB_REQUIRE(!sp->prioritized || a->abs_err_out_dev, "fb_qnet_step: prioritized replay needs abs_err_out_dev");
    } else {
        FB_REQUIRE(a->frames_dev && a->actions_dev && a->rewards_dev && a->terminals_dev, "fb_qnet_step: NULL argument");
    }
    const int batch = sp ? sp->batch : a->batch;
    FB_REQUIRE(batch > 0 && batch <= n->max_batch, "fb_qnet_step: batch outside 1..max_batch");
    const bool tc = tc_precision(n->precision);
    cudaStream_t st = (cudaStream_t)stream;

    QnetStep s;
    memset(&s, 0, sizeof(s));
    s.variant = a->variant; s.params = a->params_dev; s.target = a->target_params_dev;
    s.B = batch; s.global_batch = a->global_batch > 0 ? a->global_batch : batch; s.gamma = a->gamma; s.loss_sum = a->loss_sum;
    s.grads = a->grads_dev; s.loss_out = a->loss_out_dev ? a->loss_out_dev : n->loss_dev; s.abs_err = a->abs_err_out_dev;
    s.q_target = a->q_target_out_dev;
    if (a->m_dev) {
        s.ad.on = 1; s.ad.m = a->m_dev; s.ad.v = a->v_dev; s.ad.lr = a->lr; s.ad.beta1 = a->beta1; s.ad.beta2 = a->beta2;
        s.ad.eps = a->eps; s.ad.grad_scale = a->grad_scale;
        s.xch = n->xch;
    }
    if (sp) {
        s.pro = *sp;
        s.actions = sp->act_out_dev; s.rewards = sp->rew_out_dev; s.terminals = sp->term_out_dev;
        s.isw = sp->prioritized ? sp->is_weights_f32_out_dev : nullptr;
        if (sp->n_step > 0) { s.ret = sp->ret_out_dev; s.disc = sp->disc_out_dev; }
        // s = frames 0..3, s' = frames F-4..F-1 of each drawn row.  The tensor cores read them in place from the ring through the
        // offsets the sampler leaves behind (frame numbers into that table; the gather runs beside the forward passes); the
        // fp32 path reads the gathered rows (byte offsets)
        const int F = replay_frames_per_sample(*sp), unit = tc ? 1 : FB_FRAME_BYTES;
        int32_t off_s[4], off_n[4];
        for (int c = 0; c < 4; c++) { off_s[c] = c * unit; off_n[c] = (F - 4 + c) * unit; }
        if (tc) {
            set_view(s.fs, sp->ring_dev, 0, off_s, replay_frame_tab(sp->replay), F);
            set_view(s.fn, sp->ring_dev, 0, off_n, replay_frame_tab(sp->replay), F);
        } else {
            set_view(s.fs, sp->frames_out_dev, (long long)F * FB_FRAME_BYTES, off_s);
            set_view(s.fn, sp->frames_out_dev, (long long)F * FB_FRAME_BYTES, off_n);
        }
    } else {
        s.actions = a->actions_dev; s.rewards = a->rewards_dev; s.terminals = a->terminals_dev; s.isw = a->is_weights_dev;
        set_view(s.fs, a->frames_dev, a->sample_stride, a->chan_off_s);
        set_view(s.fn, a->frames_dev, a->sample_stride, a->chan_off_next);
    }
    if (tc) return tc_step(n, s, a->beta1_power, a->beta2_power, st);

    int rc = sp ? replay_launch_sample_gather(*sp, s.gamma, st) : FB_OK;
    if (rc == FB_OK) rc = loss_backward_impl(n, s, st);
    if (rc == FB_OK && s.ad.on) {
        const float alpha = a->lr * sqrtf(1.f - a->beta2_power) / (1.f - a->beta1_power);
        rc = fb_qnet_adam(n, a->params_dev, a->grads_dev, a->m_dev, a->v_dev, alpha, a->beta1, a->beta2, a->eps, a->grad_scale, stream);
    }
    if (rc == FB_OK && sp && sp->prioritized) rc = replay_launch_per_update(*sp, s.abs_err, st);
    return rc;
}

// target_replace_op (BrainDQNNature.py:107-111): hard copy of all variables
extern "C" int fb_qnet_sync_target(fb_qnet *n, float *target_dev, const float *params_dev, void *stream) {
    FB_REQUIRE(n && target_dev && params_dev, "fb_qnet_sync_target: NULL argument");
    FB_CUDA_OK(cudaMemcpyAsync(target_dev, params_dev, sizeof(float) * (size_t)n->L.total, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    for (int s = 0; s < 2; s++) if (n->packed_src[s] == target_dev) n->packed_src[s] = nullptr;
    return FB_OK;
}
