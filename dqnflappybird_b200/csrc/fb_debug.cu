// Host-side test hooks: run the SAME physics / table / exact-pixel code the kernels run
// (fb_env_logic.cuh is __host__ __device__) on the CPU, so the CPU-only test-suite can check
// the derived tables and the step logic against the oracle without a GPU.  Not used by the
// product path.
#include <stddef.h>
#include <string.h>

#include "fb_env_logic.cuh"

extern "C" int fb_debug_host_step(int32_t *state16, int action, const uint8_t *gaps, int gaps_len, uint64_t seed,
                                  uint64_t env_id, float *reward, uint8_t *terminal, int32_t *score) {
    const ExactTables *ex = fb_host_exact_tables();
    if (!ex) { fb_set_error("fb_debug_host_step: load the assets first"); return FB_ERR_ASSETS; }
    FB_REQUIRE(state16 && reward && terminal && score, "fb_debug_host_step: NULL argument");
    if (action != 0 && action != 1) { fb_set_error("Multiple input actions!"); return FB_ERR_ACTION; }
    EnvState s;
    memset(&s, 0, sizeof(s));
    if (!ints_to_state(state16, s)) { fb_set_error("fb_debug_host_step: state outside the reachable range"); return FB_ERR_STATE; }
    GapSource g{gaps, gaps_len, seed, env_id};
    env_step(s, action, g, ex, *reward, *terminal, *score);
    state_to_ints(s, state16);
    return FB_OK;
}

extern "C" int fb_debug_host_reset(int32_t *state16, const uint8_t *gaps, int gaps_len, uint64_t seed, uint64_t env_id) {
    FB_REQUIRE(state16 != nullptr, "fb_debug_host_reset: NULL argument");
    EnvState s;
    memset(&s, 0, sizeof(s));
    GapSource g{gaps, gaps_len, seed, env_id};
    env_reset(s, g);
    state_to_ints(s, state16);
    return FB_OK;
}

// mode 0: table path (obs_row_mask + per-pixel fix of the bird window when flagged), as render_env does;
// mode 1: every pixel by exact arithmetic, base strip included, as env_obs_exact_kernel does.
extern "C" int fb_debug_host_obs(const int32_t *state16, int mode, uint8_t *out) {
    const ObsTables *T = fb_host_obs_tables();
    const ExactTables *ex = fb_host_exact_tables();
    if (!T || !ex) { fb_set_error("fb_debug_host_obs: load the assets first"); return FB_ERR_ASSETS; }
    EnvState s;
    memset(&s, 0, sizeof(s));
    if (!ints_to_state(state16, s)) { fb_set_error("fb_debug_host_obs: state outside the reachable range"); return FB_ERR_STATE; }
    DrawList d = make_draw_list(s);
    if (mode == 1) {
        for (int i = 0; i < kObs; i++)
            for (int j = 0; j < kObs; j++) out[i * kObs + j] = exact_obs_bit(ex, d, s.basex, true, i, j) ? 255 : 0;
        return FB_OK;
    }
    const int j0 = T->birdJ0[d.y];
    for (int i = 0; i < kObs; i++) {
        unsigned long long m = obs_row_mask(*T, d, i);
        int r = i - 16;
        if ((d.np_mixed & 16) && r >= 0 && r < kBirdRows) {
            unsigned byte = 0;
            for (int b = 0; b < 8; b++)
                if (j0 + b < kBaseJ && exact_obs_bit(ex, d, 0, false, i, j0 + b)) byte |= 1u << b;
            m = obs_row_fix(m, byte, j0);
        }
        for (int j = 0; j < kObs; j++) out[i * kObs + j] = (j >= 64 || ((m >> j) & 1)) ? 255 : 0;
    }
    return FB_OK;
}

extern "C" int fb_debug_host_mixed(const int32_t *state16) {
    EnvState s;
    memset(&s, 0, sizeof(s));
    if (!ints_to_state(state16, s)) return -1;
    return (make_draw_list(s).np_mixed & 16) ? 1 : 0;
}

// layout of the C ABI's structs as this library was compiled: sizeof, then the byte offset of every field in declaration order
// -- the CPU test-suite checks the ctypes mirrors (dqnflappybird_b200/_lib.py StepSampling, QnetStepArgs) against it
#define FB_OFF(S, f) (int32_t) offsetof(S, f)
extern "C" int fb_debug_struct_layout(int which, int32_t *out, int capacity) {
    typedef fb_step_sampling S;
    typedef fb_qnet_step_args A;
    const int32_t sampling[] = {(int32_t)sizeof(S), FB_OFF(S, replay), FB_OFF(S, ring_dev), FB_OFF(S, act_dev), FB_OFF(S, rew_dev),
                                FB_OFF(S, term_dev), FB_OFF(S, t), FB_OFF(S, batch), FB_OFF(S, setsize), FB_OFF(S, seed),
                                FB_OFF(S, idx_out_dev), FB_OFF(S, frames_out_dev), FB_OFF(S, act_out_dev), FB_OFF(S, rew_out_dev),
                                FB_OFF(S, term_out_dev), FB_OFF(S, env_out_dev), FB_OFF(S, k_out_dev), FB_OFF(S, prioritized),
                                FB_OFF(S, per_mode), FB_OFF(S, beta), FB_OFF(S, tree_idx_out_dev), FB_OFF(S, is_weights_out_dev),
                                FB_OFF(S, prio_out_dev), FB_OFF(S, is_weights_f32_out_dev), FB_OFF(S, n_step), FB_OFF(S, ret_out_dev),
                                FB_OFF(S, disc_out_dev)};
    const int32_t step[] = {(int32_t)sizeof(A), FB_OFF(A, variant), FB_OFF(A, loss_sum), FB_OFF(A, batch), FB_OFF(A, global_batch),
                            FB_OFF(A, gamma), FB_OFF(A, params_dev), FB_OFF(A, target_params_dev), FB_OFF(A, sampling),
                            FB_OFF(A, frames_dev), FB_OFF(A, sample_stride), FB_OFF(A, chan_off_s), FB_OFF(A, chan_off_next),
                            FB_OFF(A, actions_dev), FB_OFF(A, rewards_dev), FB_OFF(A, terminals_dev), FB_OFF(A, is_weights_dev),
                            FB_OFF(A, grads_dev), FB_OFF(A, loss_out_dev), FB_OFF(A, abs_err_out_dev), FB_OFF(A, q_target_out_dev),
                            FB_OFF(A, m_dev), FB_OFF(A, v_dev), FB_OFF(A, lr), FB_OFF(A, beta1), FB_OFF(A, beta2), FB_OFF(A, eps),
                            FB_OFF(A, grad_scale), FB_OFF(A, beta1_power), FB_OFF(A, beta2_power)};
    FB_REQUIRE(which == 0 || which == 1, "fb_debug_struct_layout: which must be 0 (fb_step_sampling) or 1 (fb_qnet_step_args)");
    const int32_t *v = which == 0 ? sampling : step;
    const int n = which == 0 ? (int)(sizeof(sampling) / sizeof(sampling[0])) : (int)(sizeof(step) / sizeof(step[0]));
    FB_REQUIRE(out != nullptr && capacity >= n, "fb_debug_struct_layout: buffer too small");
    for (int i = 0; i < n; i++) out[i] = v[i];
    return n;
}
#undef FB_OFF
extern "C" int fb_debug_step_sampling_layout(int32_t *out, int capacity) { return fb_debug_struct_layout(0, out, capacity); }

// ---- write-pattern probe (tools/write_bw_probe.py): how fast can the device absorb the env kernel's output pattern? ---------
// n_chunks chunks of 6,400 bytes, chunk k at dst + k * stride_bytes.  mode 0: one warp per chunk, 16-byte streaming stores
// straight from registers; mode 1: one warp per chunk through a shared-memory staging frame and cp.async.bulk (the step
// kernel's path).  No computation: whatever this reaches is the ceiling of a frame-writing kernel for that layout.
__global__ void __launch_bounds__(256) write_probe_kernel(uint8_t *dst, int n_chunks, long long stride_bytes, int mode) {
    extern __shared__ __align__(128) uint8_t stage_all[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *stage = stage_all + warp * 6400;
    const long long W = (long long)gridDim.x * 8, w = (long long)blockIdx.x * 8 + warp;
    const int lo = (int)((long long)n_chunks * w / W), hi = (int)((long long)n_chunks * (w + 1) / W);
    if (mode == 1) {
        for (int i = lane; i < 400; i += 32) reinterpret_cast<uint4 *>(stage)[i] = make_uint4(i, lane, 0xFFFFFFFFu, 0);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
    }
    for (int k = lo; k < hi; k++) {
        uint8_t *out = dst + (long long)k * stride_bytes;
        if (mode == 0) {
            const uint4 v = make_uint4(k, lane, 0xFFFFFFFFu, 0);
#pragma unroll
            for (int it = 0; it < 13; it++) { int c = lane + 32 * it; if (c < 400) __stcs(reinterpret_cast<uint4 *>(out) + c, v); }
        } else if (lane == 0) {
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 6400;" ::"l"(reinterpret_cast<uint64_t>(out)),
                         "r"((uint32_t)__cvta_generic_to_shared(stage)) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (mode == 1 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

extern "C" int fb_debug_write_probe(uint8_t *dst_dev, int n_chunks, long long stride_bytes, int mode, int ctas, void *stream) {
    FB_REQUIRE(dst_dev && n_chunks > 0 && stride_bytes >= 6400 && (mode == 0 || mode == 1) && ctas > 0, "fb_debug_write_probe: bad argument");
    FB_CUDA_OK(cudaFuncSetAttribute(write_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * 6400));
    write_probe_kernel<<<ctas, 256, 8 * 6400, (cudaStream_t)stream>>>(dst_dev, n_chunks, stride_bytes, mode);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}
