// Noisy networks (Fortunato et al., 2018, factorised Gaussian noise) on the fully connected layers of the Q-network.
//
// A noisy layer with p inputs and q outputs keeps mu (the usual parameters) and sigma of the same shape; one draw gives
// eps_in[p] and eps_out[q], and the layer runs on the effective weights
//     W[i][j] = mu[i][j] + sigma[i][j] * (f(eps_in[i]) * f(eps_out[j])),   b[j] = mu_b[j] + sigma_b[j] * f(eps_out[j]),
// f(x) = sgn(x) sqrt|x|.  The noisy layers are fc1 and the head (plain: W_fc2 / b_fc2; dueling: the V and the A head, each its
// own layer); the convolutions stay deterministic.  W_eff has the parameter vector's layout, so every existing forward /
// training kernel runs on it unchanged; the gradient they return is dL/dW at W_eff, which is dL/dmu, and dL/dsigma = dL/dW * eps.
//
// Gaussian source: Philox stream (seed, purpose 5, d), d = (counter << 2) | role (role 0 online net of update `counter`,
// 1 target net of that update, 2 acting call `counter`).  Normal k of a draw is Box-Muller in float64 on words 2k, 2k+1:
// u1 = (w0 + 1) 2^-32, u2 = w1 2^-32, z = sqrt(-2 ln u1) cos(2 pi u2), rounded to fp32; then f in fp32.  The factor vector of
// a draw is, per noisy layer in layer order, f(eps_in) then f(eps_out) -- normal k is factor k (fb_noisy_layout).
#include <math.h>

#include "fb_qnet.cuh"

namespace {

constexpr uint32_t kNoisePurpose = 5;     // Philox purposes 0..4: env gaps, random actions, epsilon-greedy, uniform sample, PER

struct NoisyLayers {
    int n;                                // 2 (plain head) or 3 (dueling: V and A heads)
    int w[3], b[3], p[3], q[3];           // parameter offsets of weight [p][q] and bias [q], fan-in p, fan-out q
    int fin[3], fout[3];                  // offsets of f(eps_in) [p] and f(eps_out) [q] in the factor vector
    int factors;                          // length of the factor vector
};

NoisyLayers noisy_layers(const NetLayout &L) {
    NoisyLayers N{};
    const int H = L.hidden;
    auto add = [&](int w, int b, int p, int q) {
        int k = N.n++;
        N.w[k] = w; N.b[k] = b; N.p[k] = p; N.q[k] = q;
        N.fin[k] = N.factors; N.fout[k] = N.factors + p;
        N.factors += p + q;
    };
    add(L.wf1, L.bf1, kFlat, H);
    const int nv = L.atoms ? L.atoms : 1, na = L.atoms ? kActions * L.atoms : kActions;      // C51: fan-out N and 2N
    if (!L.dueling) add(L.wf2, L.bf2, H, na);
    else { add(L.wv, L.bv, H, nv); add(L.wa, L.ba, H, na); }
    return N;
}

// f(z) = sgn(z) sqrt|z| in fp32 (sqrtf is correctly rounded); f(0) = +0
__device__ __forceinline__ float noise_f(float z) {
    const float s = sqrtf(fabsf(z));
    return z < 0.f ? -s : s;
}

__global__ void noise_draw_kernel(uint64_t seed, uint64_t d, int n, float *factors) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t w0 = stream_word(seed, kNoisePurpose, d, 2u * (uint32_t)k), w1 = stream_word(seed, kNoisePurpose, d, 2u * (uint32_t)k + 1u);
    const double u1 = ((double)w0 + 1.0) * (1.0 / 4294967296.0), u2 = (double)w1 * (1.0 / 4294967296.0);
    const double z = sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
    factors[k] = noise_f((float)z);
}

// eps of parameter i (the product of its layer's two factors, one fp32 rounding; the bias takes f(eps_out) alone), or false
// when i lies outside every noisy layer
__device__ __forceinline__ bool noise_of(const NoisyLayers &N, const float *__restrict__ fac, int i, float *eps) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
        if (k >= N.n) break;
        const int r = i - N.w[k];
        if (r >= 0 && r < N.p[k] * N.q[k]) {
            const int row = r / N.q[k], col = r - row * N.q[k];
            *eps = __fmul_rn(__ldg(fac + N.fin[k] + row), __ldg(fac + N.fout[k] + col));
            return true;
        }
        const int c = i - N.b[k];
        if (c >= 0 && c < N.q[k]) { *eps = __ldg(fac + N.fout[k] + c); return true; }
    }
    return false;
}

// W_eff = mu + sigma * eps on the noisy layers (product, times sigma, plus mu: each rounded once, no FMA contraction), mu elsewhere
__global__ void noisy_weights_kernel(const float *__restrict__ mu, const float *__restrict__ sigma, const float *__restrict__ fac,
                                     NoisyLayers N, int total, float *__restrict__ weff) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        float eps, m = mu[i];
        weff[i] = noise_of(N, fac, i, &eps) ? __fadd_rn(m, __fmul_rn(sigma[i], eps)) : m;
    }
}

// TF-1 Adam on mu with g over every index, and on sigma with g * eps over the noisy indices: one optimizer over (mu, sigma), one
// alpha.  Elsewhere sigma and its slots are left as they are (a zero gradient would leave them unchanged too).
__global__ void noisy_adam_kernel(float *__restrict__ mu, float *__restrict__ sigma, const float *__restrict__ g, const float *__restrict__ fac,
                                  float *__restrict__ m, float *__restrict__ v, float *__restrict__ sm, float *__restrict__ sv, NoisyLayers N,
                                  int total, float alpha, float beta1, float beta2, float eps_adam, float grad_scale) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const float gi = g[i];
        float mi = m[i], vi = v[i];
        mu[i] = adam_math(gi, mu[i], mi, vi, alpha, beta1, beta2, eps_adam, grad_scale);
        m[i] = mi; v[i] = vi;
        float e;
        if (noise_of(N, fac, i, &e)) {
            float smi = sm[i], svi = sv[i];
            sigma[i] = adam_math(__fmul_rn(gi, e), sigma[i], smi, svi, alpha, beta1, beta2, eps_adam, grad_scale);
            sm[i] = smi; sv[i] = svi;
        }
    }
}

int grid_for(int total) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return min((total + 255) / 256, sms * 8);
}

}  // namespace

extern "C" int fb_noisy_layout(const fb_qnet *n, int32_t *o) {
    FB_REQUIRE(n != nullptr && o != nullptr, "fb_noisy_layout: NULL argument");
    const NoisyLayers N = noisy_layers(n->L);
    o[0] = N.n; o[1] = N.factors;
    for (int k = 0; k < 3; k++) {
        const bool on = k < N.n;
        int v[6] = {on ? N.w[k] : -1, on ? N.b[k] : -1, on ? N.p[k] : 0, on ? N.q[k] : 0, on ? N.fin[k] : -1, on ? N.fout[k] : -1};
        for (int j = 0; j < 6; j++) o[2 + 6 * k + j] = v[j];
    }
    return FB_OK;
}

extern "C" int fb_noisy_draw(fb_qnet *n, uint64_t seed, int role, uint64_t counter, float *factors_dev, void *stream) {
    FB_REQUIRE(n && factors_dev && role >= 0 && role <= 2, "fb_noisy_draw: bad argument (role 0 online, 1 target, 2 acting)");
    const NoisyLayers N = noisy_layers(n->L);
    const uint64_t d = (counter << 2) | (uint64_t)role;
    noise_draw_kernel<<<(N.factors + 255) / 256, 256, 0, (cudaStream_t)stream>>>(seed, d, N.factors, factors_dev);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

extern "C" int fb_noisy_weights(fb_qnet *n, const float *mu_dev, const float *sigma_dev, const float *factors_dev, float *weff_dev,
                                void *stream) {
    FB_REQUIRE(n && mu_dev && sigma_dev && factors_dev && weff_dev, "fb_noisy_weights: NULL argument");
    FB_REQUIRE(weff_dev != mu_dev && weff_dev != sigma_dev, "fb_noisy_weights: W_eff must be its own buffer");
    const int total = n->L.total;
    noisy_weights_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(mu_dev, sigma_dev, factors_dev, noisy_layers(n->L), total, weff_dev);
    FB_CUDA_OK(cudaGetLastError());
    // the 16-bit operand copies made from this buffer are stale now
    for (int s = 0; s < 2; s++) if (n->packed_src[s] == weff_dev) n->packed_src[s] = nullptr;
    return FB_OK;
}

extern "C" int fb_qnet_noisy_adam(fb_qnet *n, float *mu_dev, float *sigma_dev, const float *grads_dev, const float *factors_dev, float *m_dev,
                                  float *v_dev, float *sigma_m_dev, float *sigma_v_dev, float alpha, float beta1, float beta2, float eps,
                                  float grad_scale, void *stream) {
    FB_REQUIRE(n && mu_dev && sigma_dev && grads_dev && factors_dev && m_dev && v_dev && sigma_m_dev && sigma_v_dev,
               "fb_qnet_noisy_adam: NULL argument");
    const int total = n->L.total;
    noisy_adam_kernel<<<grid_for(total), 256, 0, (cudaStream_t)stream>>>(mu_dev, sigma_dev, grads_dev, factors_dev, m_dev, v_dev, sigma_m_dev,
                                                                       sigma_v_dev, noisy_layers(n->L), total, alpha, beta1, beta2, eps,
                                                                       grad_scale);
    FB_CUDA_OK(cudaGetLastError());
    // nothing is repacked here: the noisy net runs on W_eff, never on mu, so no operand copy is left mirroring mu or sigma
    for (int s = 0; s < 2; s++) if (n->packed_src[s] == mu_dev || n->packed_src[s] == sigma_dev) n->packed_src[s] = nullptr;
    return FB_OK;
}
