// Quantile-regression (QR-DQN) value head (Dabney, Rowland, Bellemare and Munos, 2018): the Q-network's head outputs, per action,
// N learned quantile locations theta[a][i] of the return distribution at the fixed fractions tau_i = (2 i + 1) / (2 N), trained by
// quantile-Huber regression.  No support, no projection, no softmax.  The head shares everything but its loss with the C51 head
// (fb_c51.cu): the layout with N outputs per action, the head forward (its QR per-sample stage: theta, Q = mean theta), the head
// backward and the finalize of the tensor-core path.  This file is the loss, shared by the fp32 and the tensor-core path.
//
//   target   a* = the first argmax of the variant's Q(s') (vanilla: online; Nature: target; Double: online argmax, target theta);
//            T_j = td_target(theta[a*][j](s'), ...) (fb_qnet.cuh): the expected-value head's rounding rule, per quantile
//   loss     u_ij = T_j - theta[a_b][i](s),  L_b = sum_i (1/N) sum_j |tau_i - 1{u_ij < 0}| H(u_ij),
//            H(u) = u^2 / (2 kappa) if |u| <= kappa else |u| - kappa / 2 (kappa > 0), H(u) = |u| (kappa = 0);
//            loss = sum_b w_b L_b scale (scale 1 for the sum loss, else 1 / global batch)
//   gradient dL_b/dtheta[a_b][i] = -(1/N) sum_j |tau_i - 1{u_ij < 0}| H'(u_ij) (H'(0) = 0 at kappa = 0), 0 for the other action;
//            dLoss/dtheta = w scale dL_b/dtheta, routed into the head's column space (dist_route)
// Fixed orders, all fp32: lane i sums over j in ascending order (l_i and g_i); L_b = (sum_i l_i, ascending i) / N, dL_b/dtheta_i =
// -g_i / N, q_target = (sum_j T_j, ascending j) / N.  So eager runs, graph replays and repeated runs give the same bits.
#include <math.h>

#include "fb_qnet.cuh"

namespace {

struct QrScratch { float T[kC51MaxAtoms], l[kC51MaxAtoms], g[kC51MaxAtoms]; };

// One sample, one warp.  th: theta[a_b](s) [N]; tn: theta[a*](s') [N].  Leaves the targets in sc.T and dL_b/dtheta_i in sc.g; lane
// 0 returns L_b in *loss_b and mean T in *qt.  The loss kernel and fb_debug_qr_loss both run this function.
__device__ void qr_sample_warp(const float *th, const float *tn, const float *rewards, const uint8_t *terminals, const double *ret,
                               const double *disc, int b, double gamma, const NetLayout &L, QrScratch &sc, float *loss_b, float *qt) {
    const int N = L.atoms, lane = threadIdx.x & 31;
    const float kappa = (float)L.kappa;
    for (int j = lane; j < N; j += 32)
        sc.T[j] = td_target(tn[j], ret ? 0.f : rewards[b], ret ? (uint8_t)0 : terminals[b], ret, disc, b, gamma);
    __syncwarp();
    for (int i = lane; i < N; i += 32) {
        const float tau = (float)(2 * i + 1) / (float)(2 * N), t_i = th[i];
        float l = 0.f, g = 0.f;
        for (int j = 0; j < N; j++) {
            const float u = sc.T[j] - t_i, au = fabsf(u), wt = u < 0.f ? 1.f - tau : tau;
            float h, dh;
            if (kappa > 0.f && au <= kappa) { h = 0.5f * u * u / kappa; dh = u / kappa; }
            else { h = kappa > 0.f ? au - 0.5f * kappa : au; dh = u > 0.f ? 1.f : u < 0.f ? -1.f : 0.f; }
            l += wt * h;
            g += wt * dh;
        }
        sc.l[i] = l;
        sc.g[i] = -g / (float)N;
    }
    __syncwarp();
    if (lane == 0) {
        float s = 0.f, t = 0.f;
        for (int i = 0; i < N; i++) s += sc.l[i];
        for (int j = 0; j < N; j++) t += sc.T[j];
        *loss_b = s / (float)N;
        *qt = t / (float)N;
    }
}

struct QrLossArgs {
    int variant, loss_sum, global_batch;
    double gamma;
    const float *ths, *thn, *q_next, *q_next_online;
    const uint8_t *actions; const float *rewards; const uint8_t *terminals; const float *isw;
    const double *ret, *disc;
    float *dl, *terms, *abs_err, *q_target;
};

// One warp per sample: qr_sample_warp, then the lanes write dLoss/dtheta in column space and lane 0 the loss term, abs_err = L_b
// (unweighted, unscaled: the PER priority) and q_target.
__global__ void __launch_bounds__(128) qr_loss_kernel(const QrLossArgs a, NetLayout L, int B) {
    __shared__ QrScratch scr[4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, N = L.atoms, nc = c51_cols(L);
    const int b = blockIdx.x * 4 + warp;
    if (b >= B) return;
    const int astar = dist_astar(a.variant == 2 ? a.q_next_online : a.q_next, b);
    const int act = a.actions[b] ? 1 : 0;
    float lb, qt;
    qr_sample_warp(a.ths + ((size_t)b * 2 + act) * N, a.thn + ((size_t)b * 2 + astar) * N, a.rewards, a.terminals, a.ret, a.disc, b, a.gamma,
                   L, scr[warp], &lb, &qt);
    const float w = a.isw ? a.isw[b] : 1.f, scale = a.loss_sum ? 1.f : 1.f / (float)a.global_batch;
    for (int c = lane; c < nc; c += 32) a.dl[(size_t)b * nc + c] = dist_route(L, c, act, w * scale * scr[warp].g[c % N]);
    if (lane == 0) {
        a.terms[b] = w * lb * scale;
        if (a.abs_err) a.abs_err[b] = lb;
        if (a.q_target) a.q_target[b] = qt;
    }
}

// fb_debug_qr_loss: one warp per sample, the loss kernel's qr_sample_warp on given theta
__global__ void __launch_bounds__(128) qr_debug_kernel(const float *theta_s, const float *theta_na, const uint8_t *actions, const float *rewards,
                                                       const uint8_t *terminals, const double *ret, const double *disc, double gamma, int B,
                                                       NetLayout L, float *dtheta, float *loss_b) {
    __shared__ QrScratch scr[4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, N = L.atoms, b = blockIdx.x * 4 + warp;
    if (b >= B) return;
    const int act = actions[b] ? 1 : 0;
    float lb, qt;
    qr_sample_warp(theta_s + ((size_t)b * 2 + act) * N, theta_na + (size_t)b * N, rewards, terminals, ret, disc, b, gamma, L, scr[warp], &lb, &qt);
    for (int i = lane; i < N; i += 32) dtheta[(size_t)b * N + i] = scr[warp].g[i];
    if (lane == 0) loss_b[b] = lb;
}

}  // namespace

int qr_launch_loss(const NetLayout &L, int B, int variant, int loss_sum, int global_batch, double gamma, const float *ths, const float *thn,
                   const float *q_next, const float *q_next_online, const uint8_t *actions, const float *rewards, const uint8_t *terminals,
                   const float *isw, const double *ret, const double *disc, float *dl, float *terms, float *abs_err, float *q_target,
                   cudaStream_t st) {
    const QrLossArgs a{variant, loss_sum, global_batch, gamma, ths, thn, q_next, q_next_online, actions, rewards, terminals, isw, ret, disc,
                       dl, terms, abs_err, q_target};
    qr_loss_kernel<<<(B + 3) / 4, 128, 0, st>>>(a, L, B);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

// test hook (include/flappy_b200.h): dtheta_out[B][N] = dL_b/dtheta[a_b][i], loss_b_out[B] = L_b, for theta_s [B][2][N] and
// theta_next_astar [B][N] under the 1-step (ret == NULL) or n-step target
extern "C" int fb_debug_qr_loss(fb_qnet *n, const float *theta_s_dev, const float *theta_next_astar_dev, const uint8_t *actions_dev,
                                const float *rewards_dev, const uint8_t *terminals_dev, const double *ret_dev, const double *disc_dev, double gamma,
                                int batch, float *dtheta_out_dev, float *loss_b_out_dev, void *stream) {
    FB_REQUIRE(n && n->L.quantile, "fb_debug_qr_loss: needs a QR net (fb_qnet_create_qr)");
    FB_REQUIRE(theta_s_dev && theta_next_astar_dev && actions_dev && dtheta_out_dev && loss_b_out_dev && batch > 0, "fb_debug_qr_loss: bad argument");
    FB_REQUIRE((ret_dev != nullptr) == (disc_dev != nullptr), "fb_debug_qr_loss: ret and disc go together");
    FB_REQUIRE(ret_dev != nullptr || (rewards_dev && terminals_dev), "fb_debug_qr_loss: rewards and terminals required without ret / disc");
    qr_debug_kernel<<<(batch + 3) / 4, 128, 0, (cudaStream_t)stream>>>(theta_s_dev, theta_next_astar_dev, actions_dev, rewards_dev, terminals_dev,
                                                                       ret_dev, disc_dev, gamma, batch, n->L, dtheta_out_dev, loss_b_out_dev);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}
