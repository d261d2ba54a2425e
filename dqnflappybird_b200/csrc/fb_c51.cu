// Distributional (C51) value head (Bellemare, Dabney and Munos, 2017): the Q-network's head outputs, per action, a categorical
// distribution over N atoms z_i of a fixed support instead of one expected value.  The trunk (conv1..conv3, fc1) is unchanged;
// these are the three CUDA-core stages that replace the head's forward, TD loss and backward on a net with L.atoms > 0, shared
// by the fp32 path (fb_qnet.cu) and the tensor-core path (fb_qnet_tc.cu).
//
//   logits   l[a][i] = h1 . W[:, a N + i] + b[a N + i]; dueling: l[a][i] = v[i] + (alpha[a][i] - (alpha[0][i] + alpha[1][i]) / 2)
//   p[a]     = softmax_i l[a] in fp32 (max subtracted);  Q[a] = sum_i z_i p[a][i] in fp32, ascending i -- what acting and
//            egreedy_kernel see, so the epsilon-greedy rule is unchanged
//   target   a* = the first argmax of the variant's Q(s') (vanilla: online; Nature: target; Double: online argmax, target p);
//            m = the projection of (R + disc z) under p[a*](s') onto the support (c51_project), float64, rounded to fp32 once
//   loss     CE_b = -sum_i m_i log p[a_b][i](s), loss = sum_b w_b CE_b scale (scale 1 for the sum loss, else 1 / global batch);
//            dLoss/dl[a_b] = w scale (p - m), 0 for the other action
// Every sum runs in a fixed order, so eager runs, graph replays and repeated runs give the same bits.
#include <math.h>

#include "fb_qnet.cuh"
#include "fb_tc.cuh"

namespace {

constexpr int kMaxCols = 3 * kC51MaxAtoms;          // the dueling head's V and A columns at the largest N

__device__ __forceinline__ double c51_dz(const NetLayout &L) { return (L.v_max - L.v_min) / (double)(L.atoms - 1); }
// atom i of the support: v_min + i dz in float64 (each operation rounded once), then rounded to fp32
__device__ __forceinline__ float c51_z(const NetLayout &L, int i) { return __double2float_rn(__dadd_rn(L.v_min, __dmul_rn((double)i, c51_dz(L)))); }

// R and disc of sample b: the n-step return and discount of the replay (ret / disc), or the 1-step r (the env's Python float 0.1)
// and disc = terminal ? 0 : gamma, as td_target (fb_qnet.cuh) has them
__device__ __forceinline__ void c51_return(const float *rewards, const uint8_t *terminals, const double *ret, const double *disc, int b,
                                           double gamma, double *R, double *d) {
    if (ret != nullptr) { *R = ret[b]; *d = disc[b]; return; }
    const float rf = rewards[b];
    *R = rf == 0.1f ? 0.1 : (double)rf;
    *d = terminals[b] ? 0.0 : gamma;
}

// dst[e] <- src(e) for e = threadIdx.x + k T < n, eight loads in flight per thread (put(e, v) stores)
template <int T, class Src, class Put>
__device__ __forceinline__ void stage(int n, Src src, Put put) {
    for (int e0 = threadIdx.x; e0 < n; e0 += 8 * T) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { const int e = e0 + u * T; v[u] = e < n ? src(e) : 0.f; }
#pragma unroll
        for (int u = 0; u < 8; u++) { const int e = e0 + u * T; if (e < n) put(e, v[u]); }
    }
}

// The projected target distribution m[N] of one sample (Bellemare et al. 2017, Algorithm 1), float64: for each atom j,
// Tz = clamp(disc == 0 ? R : R + disc z_j, v_min, v_max), b = (Tz - v_min) / dz, l = floor(b), u = ceil(b); p_j goes whole to atom l
// when l == u, else p_j (u - b) to l and p_j (b - l) to u, the contributions to each atom added in ascending j.  p_j is the fp32
// target probability widened.  Every operation is rounded once (no FMA contraction), as the NumPy restatement in
// oracle/c51_oracle.py does; b is capped at N - 1, which (v_max - v_min) / dz may exceed by an ulp.  One warp per sample: lane j
// forms atom j's split (the float64 division is the long part), then lane i adds what atoms 0, 1, .. N - 1 sent to atom i, in that
// order -- the serial rule's sums exactly.  The loss kernel and fb_debug_c51_project both run this function.
struct ProjScratch { int l[kC51MaxAtoms], u[kC51MaxAtoms]; double cl[kC51MaxAtoms], cu[kC51MaxAtoms]; };
__device__ void c51_project_warp(const float *p, double R, double disc, const NetLayout &L, ProjScratch &ps, double *m) {
    const int N = L.atoms, lane = threadIdx.x & 31;
    const double dz = c51_dz(L);
    for (int j = lane; j < N; j += 32) {
        const double zj = (double)c51_z(L, j);
        double tz = disc == 0.0 ? R : __dadd_rn(R, __dmul_rn(disc, zj));
        tz = fmin(fmax(tz, L.v_min), L.v_max);
        const double b = fmin(__ddiv_rn(__dsub_rn(tz, L.v_min), dz), (double)(N - 1));
        const double l = floor(b), u = ceil(b), pj = (double)p[j];
        ps.l[j] = (int)l;
        if (l == u) { ps.cl[j] = pj; ps.u[j] = -1; ps.cu[j] = 0.0; }
        else { ps.cl[j] = __dmul_rn(pj, __dsub_rn(u, b)); ps.u[j] = (int)u; ps.cu[j] = __dmul_rn(pj, __dsub_rn(b, l)); }
    }
    __syncwarp();
    for (int i = lane; i < N; i += 32) {
        double s = 0.0;
        for (int j = 0; j < N; j++) {
            if (ps.l[j] == i) s = __dadd_rn(s, ps.cl[j]);
            if (ps.u[j] == i) s = __dadd_rn(s, ps.cu[j]);
        }
        m[i] = s;
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------------ head forward
// A CTA takes kFwdSamples samples, so that every head weight it reads from L2 serves that many samples.  Its kFwdWarps warps split
// the hidden units in ranges (warp w: h1 terms [w H / kFwdWarps, (w + 1) H / kFwdWarps) in ascending order), lane owns the output
// columns c = lane + 32 k, k < KC (2N, or 3N with the dueling head: KC = 2, 4 or 6 slots), each column's weight row read
// coalesced, 8 .. 16 rows in flight; the warps' partial sums are added in warp order.  Then one warp per sample: logits, softmax (max subtracted),
// Q = sum z p in ascending i.  Shared memory: h1 [S][H], partials [kFwdWarps][S][cols], head biases [cols], z [N], per warp
// logits / exp / p [3][2N].
constexpr int kFwdSamples = 8, kFwdWarps = 8, kFwdThreads = 32 * kFwdWarps;
constexpr int kMaxSplits = 5;                        // fc1's K-splits on the tensor-core path (fb_qnet_tc.cu, kFc1Splits)
size_t fwd_smem(int H, int nc, int N) {
    return sizeof(float) * ((size_t)kFwdSamples * H + (size_t)kFwdWarps * kFwdSamples * nc + nc + N + kFwdWarps * 6 * N);
}
// kQR: the QR head's per-sample stage instead (fb_qr.cu) -- theta[a][i] = the logit formula, written to probs when set, and
// Q[a] = (sum_i theta[a][i] in ascending i, fp32 adds) / N; no softmax, logp unused.  The h1 finish and the weight walk are shared.
template <int KC, bool kQR>
__global__ void __launch_bounds__(kFwdThreads) c51_head_forward_kernel(const float *__restrict__ part, int splits, size_t split_stride,
                                                                      const float *__restrict__ h1_in, const float *__restrict__ params,
                                                                      NetLayout L, int B, float *__restrict__ h1_out,
                                                                      float *__restrict__ probs, float *__restrict__ logp, float *__restrict__ q) {
    extern __shared__ float c51_fwd_smem[];
    constexpr int S = kFwdSamples, W = kFwdWarps, T = kFwdThreads;
    const int t = threadIdx.x, warp = t >> 5, lane = t & 31, H = L.hidden, N = L.atoms, N2 = 2 * N, nc = c51_cols(L);
    const int b0 = blockIdx.x * S, ns = min(S, B - b0);
    float *hs = c51_fwd_smem, *pt = hs + S * H, *bs = pt + W * S * nc, *zs = bs + nc, *wsc = zs + N + warp * 6 * N;
    float *ls = wsc, *es = ls + N2, *ps = es + N2;
    for (int i = t; i < N; i += T) zs[i] = c51_z(L, i);
    for (int c = t; c < nc; c += T) bs[c] = params[c51_flat(L, H, c)];
    // h1 of the CTA's samples: fc1's split-K partials summed in order + bias, ReLU (all split loads of eight elements in flight)
    for (int e0 = t; e0 < S * H; e0 += 8 * T) {
        float x[8], pz[kMaxSplits][8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int e = e0 + u * T, s_ = e / H, j = e - s_ * H;
            const bool on = e < S * H && s_ < ns;
            x[u] = 0.f;
            if (on) x[u] = part != nullptr ? params[L.bf1 + j] : h1_in[(size_t)(b0 + s_) * H + j];
#pragma unroll
            for (int z = 0; z < kMaxSplits; z++)
                pz[z][u] = on && part != nullptr && z < splits ? part[(size_t)z * split_stride + (size_t)(b0 + s_) * H + j] : 0.f;
        }
        if (part != nullptr) {
#pragma unroll
            for (int z = 0; z < kMaxSplits; z++)
                if (z < splits)
#pragma unroll
                    for (int u = 0; u < 8; u++) x[u] += pz[z][u];
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int e = e0 + u * T, s_ = e / H, j = e - s_ * H;
            if (e >= S * H) break;
            if (part != nullptr) {
                x[u] = fmaxf(x[u], 0.f);
                if (h1_out != nullptr && s_ < ns) h1_out[(size_t)(b0 + s_) * H + j] = x[u];
            }
            hs[e] = x[u];
        }
    }
    __syncthreads();
    {
        constexpr int R = KC >= 6 ? 8 : 16;                   // weight rows in flight per warp (within the register file)
        const float *wcol[KC];
        int wstride[KC];
#pragma unroll
        for (int k = 0; k < KC; k++) {
            const int c = lane + 32 * k;
            wcol[k] = params; wstride[k] = 0;
            if (c < nc) { wcol[k] = params + c51_flat(L, 0, c); wstride[k] = (!L.dueling || c >= N) ? N2 : N; }
        }
        float acc[KC][S];
#pragma unroll
        for (int k = 0; k < KC; k++)
#pragma unroll
            for (int s_ = 0; s_ < S; s_++) acc[k][s_] = 0.f;
        const int j0 = warp * (H / W), j1 = j0 + H / W;          // H is a multiple of 32
        for (int jb = j0; jb < j1; jb += R) {
            float w[R][KC];
#pragma unroll
            for (int u = 0; u < R; u++)
#pragma unroll
                for (int k = 0; k < KC; k++) w[u][k] = jb + u < j1 && lane + 32 * k < nc ? wcol[k][(size_t)(jb + u) * wstride[k]] : 0.f;
#pragma unroll
            for (int u = 0; u < R; u++) {
                if (jb + u >= j1) break;
#pragma unroll
                for (int s_ = 0; s_ < S; s_++) {
                    const float x = hs[s_ * H + jb + u];
#pragma unroll
                    for (int k = 0; k < KC; k++) acc[k][s_] = fmaf(x, w[u][k], acc[k][s_]);
                }
            }
        }
#pragma unroll
        for (int k = 0; k < KC; k++)
            if (lane + 32 * k < nc)
#pragma unroll
                for (int s_ = 0; s_ < S; s_++) pt[(warp * S + s_) * nc + lane + 32 * k] = acc[k][s_];
    }
    __syncthreads();
    for (int s_ = warp; s_ < ns; s_ += W) {
        const int b = b0 + s_;
        auto out = [&](int c) {                              // head output c: the warps' partials in order, then the bias
            float v = pt[s_ * nc + c];
            for (int w_ = 1; w_ < W; w_++) v += pt[(w_ * S + s_) * nc + c];
            return v + bs[c];
        };
        for (int e = lane; e < N2; e += 32) {                 // logits (dueling: v + (alpha - mean_a alpha))
            const int i = e % N;
            ls[e] = L.dueling ? out(i) + (out(N + e) - 0.5f * (out(N + i) + out(N2 + i))) : out(e);
            if (kQR && probs != nullptr) probs[(size_t)b * N2 + e] = ls[e];
        }
        if constexpr (kQR) {
            __syncwarp();
            if (lane < 2) {
                float acc = 0.f;
                for (int i = 0; i < N; i++) acc += ls[lane * N + i];
                q[b * 2 + lane] = acc / (float)N;
            }
            __syncwarp();
            continue;
        }
        // max and sum of exp per action: each lane over its own logits, then a butterfly (a fixed order)
        float mx[2] = {-INFINITY, -INFINITY}, sum[2] = {0.f, 0.f};
        for (int e = lane; e < N2; e += 32) { const int a = e / N; mx[a] = fmaxf(mx[a], ls[e]); }
#pragma unroll
        for (int o = 16; o; o >>= 1) { mx[0] = fmaxf(mx[0], __shfl_xor_sync(~0u, mx[0], o)); mx[1] = fmaxf(mx[1], __shfl_xor_sync(~0u, mx[1], o)); }
        for (int e = lane; e < N2; e += 32) { const int a = e / N; es[e] = expf(ls[e] - mx[a]); sum[a] += es[e]; }
#pragma unroll
        for (int o = 16; o; o >>= 1) { sum[0] += __shfl_xor_sync(~0u, sum[0], o); sum[1] += __shfl_xor_sync(~0u, sum[1], o); }
        for (int e = lane; e < N2; e += 32) {
            const int a = e / N;
            const float p = es[e] / sum[a];
            ps[e] = p;
            if (probs != nullptr) probs[(size_t)b * N2 + e] = p;
            if (logp != nullptr) logp[(size_t)b * N2 + e] = (ls[e] - mx[a]) - logf(sum[a]);
        }
        __syncwarp();
        if (lane < 2) {
            float acc = 0.f;
            for (int i = 0; i < N; i++) acc = fmaf(zs[i], ps[lane * N + i], acc);
            q[b * 2 + lane] = acc;
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------------ loss
// One warp per sample: the target projection (c51_project_warp), then lane 0 forms CE and sum z m in ascending order while the
// lanes write dLoss/dlogits routed into the head's column space (dueling: dv_i = sum_a dl[a][i], dalpha[a][i] = dl[a][i] -
// sum_a dl[.][i] / 2).
struct LossArgs {
    int variant, loss_sum, global_batch;
    double gamma;
    const float *ps, *logps, *pn, *q_next, *q_next_online;
    const uint8_t *actions; const float *rewards; const uint8_t *terminals; const float *isw;
    const double *ret, *disc;
    float *dl, *terms, *abs_err, *q_target;
};
__global__ void __launch_bounds__(128) c51_loss_kernel(const LossArgs a, NetLayout L, int B) {
    __shared__ ProjScratch scr[4];
    __shared__ double ms[4][kC51MaxAtoms];
    __shared__ float m32[4][kC51MaxAtoms];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, N = L.atoms, nc = c51_cols(L);
    const int b = blockIdx.x * 4 + warp;
    if (b >= B) return;
    const int astar = dist_astar(a.variant == 2 ? a.q_next_online : a.q_next, b);
    double R, d;
    c51_return(a.rewards, a.terminals, a.ret, a.disc, b, a.gamma, &R, &d);
    c51_project_warp(a.pn + ((size_t)b * 2 + astar) * N, R, d, L, scr[warp], ms[warp]);
    for (int i = lane; i < N; i += 32) m32[warp][i] = __double2float_rn(ms[warp][i]);
    __syncwarp();
    const int act = a.actions[b] ? 1 : 0;
    const float w = a.isw ? a.isw[b] : 1.f, scale = a.loss_sum ? 1.f : 1.f / (float)a.global_batch;
    const float *p = a.ps + ((size_t)b * 2 + act) * N;
    for (int c = lane; c < nc; c += 32) {
        const int i = c % N;
        a.dl[(size_t)b * nc + c] = dist_route(L, c, act, w * scale * (p[i] - m32[warp][i]));
    }
    if (lane == 0) {
        const float *lp = a.logps + ((size_t)b * 2 + act) * N;
        float ce = 0.f, qt = 0.f;
        for (int i = 0; i < N; i++) { ce = fmaf(-m32[warp][i], lp[i], ce); qt = fmaf(c51_z(L, i), m32[warp][i], qt); }
        a.terms[b] = w * ce * scale;
        if (a.abs_err) a.abs_err[b] = ce;
        if (a.q_target) a.q_target[b] = qt;
    }
}

// ------------------------------------------------------------------------------------------------ head backward
// Grid (H / 32 + 1, G), 256 threads.  Block x < H / 32 owns hidden units j0 .. j0 + 31 and walks its row group in chunks of
// kC51Rows rows: the chunk's dLoss/dlogits and h1 tile are staged in shared memory, then (1) dh1 = sum_c dl[c] W[j][c] (ascending c)
// masked by ReLU -- thread (row lane rl, unit jl) does rows rl and rl + 8 --, and (2) the weight gradients sum_b h1[b][j] dl[b][c]
// (ascending b) -- thread (warp w, lane) owns the pairs (j0 + lane, w + 8 k).  The last block does the head biases sum_b dl[b][c] and
// the loss.  Shared memory: W tile [32][cols | 1], dl [kC51Rows][cols], h1 [kC51Rows][32], [8][32] for the fc1 bias partials.
static_assert(kC51Rows == 16, "the dh1 stage gives each of the 8 row lanes two rows of a chunk");
struct BwdArgs {
    const float *h1, *dl, *params, *terms;
    int B, rows;                    // rows per row group
    float *grads, *loss_out, *dh1_f32;
    float *hp, *hb;
    unsigned short *dh1_16; int f16; float gscale;
    AdamPow ap;
};
size_t bwd_smem(int nc) { return sizeof(float) * ((size_t)32 * (nc + 1) + (size_t)kC51Rows * nc + kC51Rows * 32 + 8 * 32); }

__global__ void __launch_bounds__(256) c51_head_backward_kernel(const BwdArgs a, NetLayout L) {
    extern __shared__ float c51_bwd_smem[];
    const int H = L.hidden, nc = c51_cols(L), grp = blockIdx.y, t = threadIdx.x;
    const int r_beg = grp * a.rows, r_end = min(a.B, r_beg + a.rows);
    const bool direct = a.grads != nullptr;
    const size_t S = c51_partial_stride(L);
    if ((int)blockIdx.x == H / 32) {                 // head biases and the loss of this row group
        if (a.ap.on && grp == 0 && t == 0) adam_pow_advance(a.ap);
        if (t < nc) {
            float s = 0.f;
#pragma unroll 8
            for (int r = r_beg; r < r_end; r++) s += a.dl[(size_t)r * nc + t];
            if (direct) a.grads[c51_flat(L, H, t)] = s;
            else a.hp[grp * S + (size_t)H * nc + t] = s;
        } else if (t == 255) {
            float s = 0.f;
#pragma unroll 8
            for (int r = r_beg; r < r_end; r++) s += a.terms[r];
            if (direct) { if (a.loss_out) *a.loss_out = s; }
            else a.hb[grp * 4 + 2] = s;
        }
        return;
    }
    const int ws = nc | 1;                           // odd row stride: the 32 lanes read 32 different W rows without conflicts
    float *Ws = c51_bwd_smem, *dls = Ws + 32 * ws, *h1s = dls + kC51Rows * nc, *red = h1s + kC51Rows * 32;
    const int j0 = blockIdx.x * 32, lane = t & 31, warp = t >> 5;
    stage<256>(32 * nc, [&](int e) { const int jj = e / nc; return a.params[c51_flat(L, j0 + jj, e - jj * nc)]; },
               [&](int e, float v) { const int jj = e / nc; Ws[jj * ws + e - jj * nc] = v; });
    constexpr int kPerThread = kMaxCols / 8;         // columns w + 8 k of the pairs (j0 + lane, .)
    float acc[kPerThread];
#pragma unroll
    for (int k = 0; k < kPerThread; k++) acc[k] = 0.f;
    float gb = 0.f;
    for (int r0 = r_beg; r0 < r_end; r0 += kC51Rows) {
        const int nr = min(kC51Rows, r_end - r0);
        __syncthreads();                             // the previous chunk's readers are done (and the W tile is in place)
        stage<256>(nr * nc, [&](int e) { return a.dl[(size_t)r0 * nc + e]; }, [&](int e, float v) { dls[e] = v; });
        stage<256>(nr * 32, [&](int e) { return a.h1[(size_t)(r0 + (e >> 5)) * H + j0 + (e & 31)]; }, [&](int e, float v) { h1s[e] = v; });
        __syncthreads();
        {
            const int r_a = warp, r_b = warp + 8;
            float g0 = 0.f, g1 = 0.f;
            const float *wrow = Ws + lane * ws;
            for (int c = 0; c < nc; c++) {
                const float w = wrow[c];
                g0 = fmaf(dls[r_a * nc + c], w, g0);
                if (r_b < nr) g1 = fmaf(dls[r_b * nc + c], w, g1);
            }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int r = u ? r_b : r_a;
                if (r >= nr) break;
                float g = u ? g1 : g0;
                const size_t o = (size_t)(r0 + r) * H + j0 + lane;
                if (direct) a.dh1_f32[o] = h1s[r * 32 + lane] > 0.f ? g : 0.f;
                else {
                    g = h1s[r * 32 + lane] > 0.f ? g * a.gscale : 0.f;
                    a.dh1_16[o] = tc::pack1(g, a.f16);
                    gb += tc::round1(g, a.f16);      // the fc1 bias gradient sums what the weight-gradient GEMM sees (scaled)
                }
            }
        }
        for (int r = 0; r < nr; r++) {
            const float x = h1s[r * 32 + lane];
            const float *drow = dls + r * nc;
#pragma unroll
            for (int k = 0; k < kPerThread; k++)
                if (warp + 8 * k < nc) acc[k] = fmaf(x, drow[warp + 8 * k], acc[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < kPerThread; k++) {
        const int c = warp + 8 * k;
        if (c < nc) {
            if (direct) a.grads[c51_flat(L, j0 + lane, c)] = acc[k];
            else a.hp[grp * S + (size_t)(j0 + lane) * nc + c] = acc[k];
        }
    }
    if (!direct) {                                   // fc1 bias partial: the eight row lanes added in order
        red[warp * 32 + lane] = gb;
        __syncthreads();
        if (warp == 0) {
            float s = 0.f;
            for (int k = 0; k < 8; k++) s += red[k * 32 + lane];
            a.hp[grp * S + (size_t)(H + 1) * nc + j0 + lane] = s;
        }
    }
}

// fb_debug_c51_project: one warp per sample, the loss kernel's projection
__global__ void __launch_bounds__(128) c51_project_kernel(const float *p_next, const float *rewards, const uint8_t *terminals, const double *ret,
                                                          const double *disc, double gamma, int B, NetLayout L, float *m_out) {
    __shared__ ProjScratch scr[4];
    __shared__ double ms[4][kC51MaxAtoms];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, b = blockIdx.x * 4 + warp;
    if (b >= B) return;
    double R, d;
    c51_return(rewards, terminals, ret, disc, b, gamma, &R, &d);
    c51_project_warp(p_next + (size_t)b * L.atoms, R, d, L, scr[warp], ms[warp]);
    for (int i = lane; i < L.atoms; i += 32) m_out[(size_t)b * L.atoms + i] = __double2float_rn(ms[warp][i]);
}

}  // namespace

int c51_prepare() {
    FB_CUDA_OK(cudaFuncSetAttribute(c51_head_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_smem(kMaxCols)));
    const int fs = (int)fwd_smem(2048, kMaxCols, kC51MaxAtoms);
    for (const void *k : {(const void *)c51_head_forward_kernel<2, false>, (const void *)c51_head_forward_kernel<4, false>,
                          (const void *)c51_head_forward_kernel<6, false>, (const void *)c51_head_forward_kernel<2, true>,
                          (const void *)c51_head_forward_kernel<4, true>, (const void *)c51_head_forward_kernel<6, true>})
        FB_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, fs));
    return FB_OK;
}

int c51_launch_head_forward(const float *part, int splits, size_t split_stride, const float *h1_in, const float *params, const NetLayout &L,
                            int B, float *h1_out, float *probs, float *logp, float *q, cudaStream_t st) {
    FB_REQUIRE(part == nullptr || splits <= kMaxSplits, "c51_launch_head_forward: more fc1 K-splits than the head kernel sums");
    const int nc = c51_cols(L);
    auto kern = L.quantile ? (nc <= 64 ? c51_head_forward_kernel<2, true> : nc <= 128 ? c51_head_forward_kernel<4, true> : c51_head_forward_kernel<6, true>)
                           : (nc <= 64 ? c51_head_forward_kernel<2, false> : nc <= 128 ? c51_head_forward_kernel<4, false> : c51_head_forward_kernel<6, false>);
    kern<<<(B + kFwdSamples - 1) / kFwdSamples, kFwdThreads, fwd_smem(L.hidden, nc, L.atoms), st>>>(part, splits, split_stride, h1_in, params, L,
                                                                                                    B, h1_out, probs, logp, q);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

int c51_launch_loss(const NetLayout &L, int B, int variant, int loss_sum, int global_batch, double gamma, const float *ps, const float *logps,
                    const float *pn, const float *q_next, const float *q_next_online, const uint8_t *actions, const float *rewards,
                    const uint8_t *terminals, const float *isw, const double *ret, const double *disc, float *dl, float *terms, float *abs_err,
                    float *q_target, cudaStream_t st) {
    const LossArgs a{variant, loss_sum, global_batch, gamma, ps, logps, pn, q_next, q_next_online, actions, rewards, terminals, isw, ret, disc,
                     dl, terms, abs_err, q_target};
    c51_loss_kernel<<<(B + 3) / 4, 128, 0, st>>>(a, L, B);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

int c51_launch_head_backward(const NetLayout &L, int B, const float *h1, const float *dl, const float *params, const float *terms, float *grads,
                             float *loss_out, float *dh1_f32, float *hp, float *hb, void *dh1_16, int f16, float gscale, const AdamPow &ap,
                             cudaStream_t st) {
    const int rows = grads != nullptr ? B : kC51Rows, G = (B + rows - 1) / rows;
    const BwdArgs a{h1, dl, params, terms, B, rows, grads, loss_out, dh1_f32, hp, hb, (unsigned short *)dh1_16, f16, gscale, ap};
    c51_head_backward_kernel<<<dim3(L.hidden / 32 + 1, G), 256, bwd_smem(c51_cols(L)), st>>>(a, L);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

// test hook (include/flappy_b200.h): m_out[B][N] = the fp32 projection of p_next[B][N] under the 1-step (ret == NULL) or n-step target
extern "C" int fb_debug_c51_project(fb_qnet *n, const float *p_next_dev, const float *rewards_dev, const uint8_t *terminals_dev, const double *ret_dev,
                                    const double *disc_dev, double gamma, int batch, float *m_out_dev, void *stream) {
    FB_REQUIRE(n && n->L.atoms > 0, "fb_debug_c51_project: needs a C51 net (fb_qnet_create_c51)");
    FB_REQUIRE(p_next_dev && m_out_dev && batch > 0, "fb_debug_c51_project: bad argument");
    FB_REQUIRE((ret_dev != nullptr) == (disc_dev != nullptr), "fb_debug_c51_project: ret and disc go together");
    FB_REQUIRE(ret_dev != nullptr || (rewards_dev && terminals_dev), "fb_debug_c51_project: rewards and terminals required without ret / disc");
    c51_project_kernel<<<(batch + 3) / 4, 128, 0, (cudaStream_t)stream>>>(p_next_dev, rewards_dev, terminals_dev, ret_dev, disc_dev, gamma,
                                                                              batch, n->L, m_out_dev);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}
