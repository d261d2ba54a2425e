// Tensor-core path of the DQN-family Q-network (sm_100a): every convolution / fully connected layer, forward,
// data gradient and weight gradient, is ONE warp-specialised kernel shape -- TMA (cp.async.bulk.tensor) feeds
// 128B-swizzled shared-memory stages, one elected thread issues tcgen05.mma (bf16 x bf16 -> fp32 in TMEM), four
// epilogue warps read the accumulator back with tcgen05.ld and fuse bias / ReLU / masks / layout remaps.
//
// Reference graph: BrainDQN.py:119-163; backward = tf.gradients of it (BrainDQN.py:163).
//
// What makes the convolutions plain TMA GEMMs ("implicit GEMM by row offset"): activations live in HBM as bf16
// matrices [position][channel] whose positions are the cells of a zero-padded grid linearised with a FIXED width,
// so that the input row of filter tap (dh,dw) for output position p is simply p + dh*width + dw:
//   conv1 8x8 s4 pad 2  = 2x2 s1 conv over the space-to-depth tensor X2 [B*441][64]  (21x21 blocks of 4x4x4)
//   conv2 4x4 s2 pad 1  = 2x2 s1 conv over the pooled space-to-depth tensor P2 [B*49][128] (7-wide grid of 2x2x32)
//   conv3 3x3 s1 pad 1  = 3x3 s1 conv over A2 [B*49][64] (7-wide grid, the pad ring is the invalid rows, offset -8)
// Each K-block of 64 channels of one tap is one TMA box at a shifted row coordinate; rows outside the tensor are
// zero-filled by TMA.  Invalid grid positions are computed and discarded (conv1 10 %, conv2/3 2x; those layers
// are < 30 % of the FLOPs).  Data gradients are the same kernel over the gradient tensors with re-packed weights;
// weight gradients contract over positions with both operands MN-major (the same row-major tensors, transposed
// by the descriptor, not in memory) and a deterministic split-K.
//
// Numerics: operands bf16 (inputs {0,255} are exact), accumulation fp32, activations stored bf16 between layers,
// head / TD loss / Adam in fp32 (shared with fb_qnet.cu).  Tolerances vs the float64 oracle: tests/test_qnet_tc_gpu.py.
#include <cudaTypedefs.h>

#include <string.h>

#include <map>
#include <new>
#include <vector>

#include "fb_qnet.cuh"
#include "fb_pack.cuh"
#include "fb_tc.cuh"
#include "fb_tc_conv.cuh"


namespace {

constexpr int kStages = 4;
constexpr int kMaxKb = 32;
constexpr int kG1 = 21, kP1 = 441;        // conv1 block grid
constexpr int kG2 = 7, kP2 = 49;          // 7-wide grid shared by conv2 / conv3 tensors
constexpr int kThreads = 192;             // warp 0 TMA, warp 1 MMA + TMEM owner, warps 2..5 epilogue

// ------------------------------------------------------------------------------------------------ the GEMM
struct GemmParams {
    // MODE 0 (K-major A and B):  D[m][n] = sum_kb sum_k A[m + a_rowoff[kb]][a_col[kb] + k] * Bt[n][64 kb + k];
    // CTA z takes K-blocks [z kper, min(nkb, (z+1) kper))
    int nkb, kper;
    int a_rowoff[kMaxKb];
    int a_col[kMaxKb];
    // MODE 1 (MN-major A and B): D[128 mt + 64 i + j][n] = sum_p A[p + a2_rowoff[mt][i]][a2_col[mt][i] + j] * B[p][n]
    int p_total, klen;
    int a2_rowoff[16][2];
    int a2_col[16][2];
    // shared-memory descriptor strides (bytes); runtime so that the self-test can probe encodings
    uint32_t lbo_a, sbo_a, kstep_a, lbo_b, sbo_b, kstep_b;
    int f16;                    // operand format (tc::pack2): 0 bf16, 1 fp16
};

template <int BN, int MODE, class EP>
__global__ void __launch_bounds__(kThreads) tc_gemm_kernel(const __grid_constant__ CUtensorMap mapA,
                                                           const __grid_constant__ CUtensorMap mapB, const GemmParams g, const EP ep) {
    constexpr uint32_t A_BYTES = 128 * 64 * 2, B_BYTES = BN * 64 * 2, STAGE = A_BYTES + B_BYTES;
    // MODE 0: A and B K-major.  MODE 1: A and B MN-major (contraction over rows).  MODE 2: A K-major, B MN-major
    // (B = a row-major [K][N] matrix used as stored: fc1 forward reads W_fc1 [1600][H] without a transposed copy).
    constexpr uint32_t B_LAYOUT = (MODE == 1 && BN == 32) ? tc::kSwizzle64 : tc::kSwizzle128;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[kStages], bar_empty[kStages], bar_accum;
    __shared__ uint32_t tmem_slot;
    const uint32_t smem = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mt = blockIdx.x, n0 = blockIdx.y * BN;

    int nkb, p_begin = 0, kb0 = 0;
    if (MODE != 1) { kb0 = blockIdx.z * g.kper; nkb = min(g.kper, g.nkb - kb0); }
    else {
        p_begin = blockIdx.z * g.klen;
        int len = min(g.klen, g.p_total - p_begin);
        nkb = (len + 63) >> 6;
    }

    if (threadIdx.x == 0) {
        tc::tma_prefetch_desc(&mapA);
        tc::tma_prefetch_desc(&mapB);
        for (int s = 0; s < kStages; s++) { tc::mbar_init(tc::smem_u32(&bar_full[s]), 1); tc::mbar_init(tc::smem_u32(&bar_empty[s]), 1); }
        tc::mbar_init(tc::smem_u32(&bar_accum), 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tc::smem_u32(&tmem_slot), BN);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_slot;
    tc::pdl_wait();
    tc::pdl_launch();

    if (warp == 0) {
        const bool leader = tc::elect_one();
        for (int kb = 0; kb < nkb; kb++) {
            const int s = kb % kStages;
            const uint32_t ph = (kb / kStages) & 1;
            tc::mbar_wait(tc::smem_u32(&bar_empty[s]), ph ^ 1u);
            if (leader) {
                const uint32_t full = tc::smem_u32(&bar_full[s]);
                const uint32_t sa = smem + s * STAGE, sb = sa + A_BYTES;
                tc::mbar_expect_tx(full, STAGE);
                if (MODE == 0) {
                    tc::tma_load_2d(sa, &mapA, g.a_col[kb0 + kb], mt * 128 + g.a_rowoff[kb0 + kb], full);
                    tc::tma_load_2d(sb, &mapB, (kb0 + kb) * 64, n0, full);
                } else if (MODE == 2) {
                    tc::tma_load_2d(sa, &mapA, g.a_col[kb0 + kb], mt * 128 + g.a_rowoff[kb0 + kb], full);
                    tc::tma_load_2d(sb, &mapB, n0, (kb0 + kb) * 64, full);
                    if (BN == 128) tc::tma_load_2d(sb + 8192, &mapB, n0 + 64, (kb0 + kb) * 64, full);
                } else {
                    const int p = p_begin + kb * 64;
                    tc::tma_load_2d(sa, &mapA, g.a2_col[mt][0], p + g.a2_rowoff[mt][0], full);
                    tc::tma_load_2d(sa + 8192, &mapA, g.a2_col[mt][1], p + g.a2_rowoff[mt][1], full);
                    tc::tma_load_2d(sb, &mapB, n0, p, full);
                    if (BN == 128) tc::tma_load_2d(sb + 8192, &mapB, n0 + 64, p, full);
                }
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        {
            const bool leader = tc::elect_one();
            const uint32_t idesc = tc::instr_desc_16(128, BN, MODE == 1, MODE != 0, g.f16);
            const uint32_t ahi = tc::smem_desc_hi(g.sbo_a, tc::kSwizzle128), bhi = tc::smem_desc_hi(g.sbo_b, B_LAYOUT);
            const uint32_t a_lo0 = tc::smem_desc_lo(smem, g.lbo_a), b_lo0 = tc::smem_desc_lo(smem + A_BYTES, g.lbo_b);
            const uint32_t ka = g.kstep_a >> 4, kbs = g.kstep_b >> 4;
            for (int kb = 0; kb < nkb; kb++) {
                const int s = kb % kStages;
                const uint32_t ph = (kb / kStages) & 1;
                tc::mbar_wait(tc::smem_u32(&bar_full[s]), ph);
                tc::tc_fence_after();
                const uint32_t soff = s * (STAGE >> 4);
                if (leader) {
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        tc::umma_bf16_lohi(tmem, a_lo0 + soff + k * ka, ahi, b_lo0 + soff + k * kbs, bhi, idesc, (kb | k) != 0);
                    tc::umma_commit(tc::smem_u32(&bar_empty[s]));     // frees the stage once these MMAs have read it
                }
                __syncwarp();
            }
            if (leader) tc::umma_commit(tc::smem_u32(&bar_accum));
            __syncwarp();
        }
    } else {
        const int q = warp & 3;                                    // TMEM lane quadrant this warp may read
        tc::mbar_wait(tc::smem_u32(&bar_accum), 0);
        tc::tc_fence_after();
        const int row = mt * 128 + q * 32 + lane;
        if constexpr (EP::kRowMajorF32) {
            // fp32 rows out as whole 128-byte lines: the warp transposes 32 columns of its 32 rows through shared memory (the
            // operand stages are free by now), eight lanes store one row's 128 bytes -- see tc_wgrad_kernel
            float4 *stage = reinterpret_cast<float4 *>(smem_raw + (smem - tc::smem_u32(smem_raw))) + q * 256;
            float *outp = ep.out + (size_t)blockIdx.z * ep.split_stride;
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 32) {
                float v[32];
                if (nkb > 0) tc::tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
                else {
#pragma unroll
                    for (int i = 0; i < 32; i++) v[i] = 0.f;
                }
#pragma unroll
                for (int j = 0; j < 8; j++)
                    stage[lane * 8 + (j ^ (lane & 7))] = make_float4(v[4 * j] * ep.scale, v[4 * j + 1] * ep.scale, v[4 * j + 2] * ep.scale, v[4 * j + 3] * ep.scale);
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int r = (lane >> 3) + 4 * j, c4 = lane & 7, orow = mt * 128 + q * 32 + r;
                    const float4 x = stage[r * 8 + (c4 ^ (r & 7))];
                    if (orow < ep.rows) *reinterpret_cast<float4 *>(outp + (size_t)orow * ep.ld + n0 + c0 + 4 * c4) = x;
                }
                __syncwarp();
            }
        } else {
#pragma unroll 1
            for (int c0 = 0; c0 < BN; c0 += 16) {
                float v[16];
                if (nkb > 0) tc::tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
                else {
#pragma unroll
                    for (int i = 0; i < 16; i++) v[i] = 0.f;
                }
                ep(row, n0 + c0, v, (int)blockIdx.z, nullptr);
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem, BN);
}

template <int BN>
constexpr size_t gemm_smem_bytes() { return exclusive_smem((size_t)kStages * (128 * 64 * 2 + BN * 64 * 2) + 1024); }

template <int BN, int MODE, class EP>
static cudaError_t launch_tc_gemm(const CUtensorMap &ma, const CUtensorMap &mb, const GemmParams &g, dim3 grid, EP ep, cudaStream_t st) {
    static bool configured = false;
    auto kern = tc_gemm_kernel<BN, MODE, EP>;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gemm_smem_bytes<BN>());
        if (e != cudaSuccess) return e;
        configured = true;
    }
    return tc::launch_pdl(kern, grid, dim3(kThreads), gemm_smem_bytes<BN>(), st, ma, mb, g, ep);
}

// ------------------------------------------------------------------------------------------------ epilogues
__device__ __forceinline__ void store_bf16x16(bf16 *dst, const float (&v)[16], int f16) {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; i++) w[i] = tc::pack2(v[2 * i], v[2 * i + 1], f16);
    tc::st_global_256(dst, make_uint4(w[0], w[1], w[2], w[3]), make_uint4(w[4], w[5], w[6], w[7]));      // every caller's dst is 32-byte aligned
}
__device__ __forceinline__ void load_bf16x16(const bf16 *src, float (&v)[16], int f16) {
    uint4 a, b;
    tc::ld_global_nc_256(src, a, b);                 // (activations of an earlier kernel: read-only here; 32-byte aligned at every caller)
    uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; i++) {
        float2 f = tc::unpack2(w[i], f16);
        v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
}

// An epilogue sees 16 consecutive fp32 columns of one output row; `bs` is the layer bias staged in shared memory by the
// kernel when the functor asks for it (bias != nullptr) -- a global load per column per tile was what bounded the tiles.
// sixteen bias values of the staged layer bias, loaded unconditionally and vectorised BEFORE any per-row predicate: with
// the shared-memory loads inside `ok ? ... : 0` the compiler emits one divergent block per pair of columns
__device__ __forceinline__ void load_bias16(const float *bs, int col, float (&b)[16]) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float4 t4 = reinterpret_cast<const float4 *>(bs + col)[k];
        b[4 * k] = t4.x; b[4 * k + 1] = t4.y; b[4 * k + 2] = t4.z; b[4 * k + 3] = t4.w;
    }
}
struct EpiGrid7 {               // conv2: rows on the 7-grid -> A2 [B*49][64], zeros at invalid positions
    bf16 *out; const float *bias; int rows, f16;
    __device__ void operator()(int row, int col, float (&v)[16], int, const float *bs) const {
        float b[16];
        load_bias16(bs, col, b);
        if (row >= rows) return;
        int p = row % kP2;
        const float keep = ((p / kG2) < 5 && (p % kG2) < 5) ? 1.f : 0.f;
#pragma unroll
        for (int i = 0; i < 16; i++) v[i] = fmaxf(v[i] + b[i], 0.f) * keep;
        store_bf16x16(out + (size_t)row * 64 + col, v, f16);
    }
};
struct EpiConv3 {               // rows on the 7-grid -> dense A3 [B][25][64] (TF flatten order h,w,c)
    bf16 *a3; const float *bias; int rows, f16;
    __device__ void operator()(int row, int col, float (&v)[16], int, const float *bs) const {
        float bi[16];
        load_bias16(bs, col, bi);
        if (row >= rows) return;
        int b = row / kP2, p = row - b * kP2, oh = p / kG2, ow = p - oh * kG2;
        if (oh >= 5 || ow >= 5) return;
#pragma unroll
        for (int i = 0; i < 16; i++) v[i] = fmaxf(v[i] + bi[i], 0.f);
        store_bf16x16(a3 + ((size_t)b * 25 + oh * 5 + ow) * 64 + col, v, f16);
    }
};
struct EpiFc1Dgrad {            // dA3 [B][1600] masked by relu(a3) -> dZ3 on the 7-grid [B*49][64]
    bf16 *dz3; const bf16 *a3; int B, f16;
    static constexpr const float *bias = nullptr;
    static constexpr bool kRowMajorF32 = false;
    __device__ void operator()(int row, int col, float (&v)[16], int, const float *) const {
        if (row >= B) return;
        float a[16];
        load_bf16x16(a3 + (size_t)row * kFlat + col, a, f16);
#pragma unroll
        for (int i = 0; i < 16; i++) v[i] = a[i] > 0.f ? v[i] : 0.f;
        int pix = col >> 6, oh = pix / 5, ow = pix - oh * 5;
        store_bf16x16(dz3 + ((size_t)row * kP2 + oh * kG2 + ow) * 64 + (col & 63), v, f16);
    }
};
struct EpiConv3Dgrad {          // dA2 on the 7-grid masked by relu(a2) -> dZ2 [B*49][64], zeros at invalid positions
    bf16 *dz2; const bf16 *a2; int rows, f16;
    static constexpr const float *bias = nullptr;
    __device__ void operator()(int row, int col, float (&v)[16], int, const float *) const {
        if (row >= rows) return;
        int p = row % kP2;
        bool ok = (p / kG2) < 5 && (p % kG2) < 5;
        float a[16];
        load_bf16x16(a2 + (size_t)row * 64 + col, a, f16);
#pragma unroll
        for (int i = 0; i < 16; i++) v[i] = (ok && a[i] > 0.f) ? v[i] : 0.f;
        store_bf16x16(dz2 + (size_t)row * 64 + col, v, f16);
    }
};
struct EpiStoreBf16 {           // conv2 dgrad: dP2 [B*49][128]
    bf16 *out; int rows, ld, f16;
    static constexpr const float *bias = nullptr;
    __device__ void operator()(int row, int col, float (&v)[16], int, const float *) const {
        if (row >= rows) return;
        store_bf16x16(out + (size_t)row * ld + col, v, f16);
    }
};
struct EpiStoreF32 {            // weight-gradient partials [split][rows][ld] and the self-test
    float *out; int rows, ld; size_t split_stride;
    float scale = 1.f;          // a power of two: un-scales gradients that were scaled for the fp16 operand format
    static constexpr const float *bias = nullptr;
    static constexpr bool kRowMajorF32 = true;     // tc_gemm_kernel / tc_wgrad_kernel store it as whole lines (warp transpose)
    __device__ void operator()(int row, int col, float (&v)[16], int split, const float *) const {
        if (row >= rows) return;
        float4 *d = reinterpret_cast<float4 *>(out + (size_t)split * split_stride + (size_t)row * ld + col);
#pragma unroll
        for (int i = 0; i < 4; i++) d[i] = make_float4(v[4 * i] * scale, v[4 * i + 1] * scale, v[4 * i + 2] * scale, v[4 * i + 3] * scale);
    }
};

// ------------------------------------------------------------------------------------------------ glue kernels
// u8 frames (FrameView) -> X2 [B*441][64]: block (bh,bw) of the input padded by 2, channel j = r*16 + s*4 + c
__global__ void pack_x2_kernel(FrameView fv, int B, bf16 *x2, int f16) {
    tc::pdl_wait();
    tc::pdl_launch();
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)B * kP1 * 8) return;
    int t8 = (int)(t & 7);
    size_t blk = t >> 3;
    int b = (int)(blk / kP1), pb = (int)(blk - (size_t)b * kP1), bh = pb / kG1, bw = pb - bh * kG1;
    int r = t8 >> 1, sp = t8 & 1;
    int ih = 4 * bh - 2 + r, iw = 4 * bw - 2 + 2 * sp;
    float px[2][4];
    bool in = (unsigned)ih < 80u && (unsigned)iw < 80u;
#pragma unroll
    for (int c = 0; c < 4; c++) {
        unsigned short two = 0;
        if (in) two = __ldg(reinterpret_cast<const unsigned short *>(fv.chan(b, c) + ih * 80 + iw));
        px[0][c] = (float)(two & 255);
        px[1][c] = (float)(two >> 8);
    }
    uint32_t w[4];
#pragma unroll
    for (int s = 0; s < 2; s++)
#pragma unroll
        for (int h = 0; h < 2; h++) w[s * 2 + h] = tc::pack2(px[s][2 * h], px[s][2 * h + 1], f16);
    *reinterpret_cast<uint4 *>(x2 + blk * 64 + r * 16 + sp * 8) = make_uint4(w[0], w[1], w[2], w[3]);
}

// eight channels of one pooling window: g = gradient of the pooled value, z[k] = the window's four activations (k = row-major
// position); the gradient goes to the FIRST maximum (TF MaxPoolGrad) if it is positive (ReluGrad); bf16 out, 16 bytes a position
__device__ __forceinline__ void unpool_pack8(const float (&g)[8], const float (&z)[4][8], uint4 (&out)[4], int f16) {
    float o[4][8];
#pragma unroll
    for (int i = 0; i < 8; i++) {
        float m = fmaxf(fmaxf(z[0][i], z[1][i]), fmaxf(z[2][i], z[3][i]));
        bool done = false;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            bool hit = !done && z[k][i] == m;
            o[k][i] = (hit && z[k][i] > 0.f) ? g[i] : 0.f;
            done |= hit;
        }
    }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; i++) w[i] = tc::pack2(o[k][2 * i], o[k][2 * i + 1], f16);
        out[k] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}
__device__ __forceinline__ void unpool_route8(const float (&g)[8], const float (&z)[4][8], bf16 *dst, const size_t (&off)[4], int f16) {
    uint4 out[4];
    unpool_pack8(g, z, out, f16);
#pragma unroll
    for (int k = 0; k < 4; k++) *reinterpret_cast<uint4 *>(dst + off[k]) = out[k];
}

// dZ1 = unpool(dP2) * relu'(z1): the gradient goes to the first maximum of each window (TF MaxPoolGrad)
__global__ void unpool_relu_kernel_tc(const bf16 *z1, const bf16 *dp2, int B, bf16 *dz1, int f16) {
    tc::pdl_wait();
    tc::pdl_launch();
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)B * 100 * 4) return;
    int cg = (int)(t & 3);
    size_t pp = t >> 2;
    int b = (int)(pp / 100), q = (int)(pp - (size_t)b * 100), ph = q / 10, pw = q - ph * 10;
    int bh = (ph + 1) >> 1, r = (ph + 1) & 1, bw = (pw + 1) >> 1, s = (pw + 1) & 1;
    float g[8], z[4][8];
    {
        uint4 raw = __ldg(reinterpret_cast<const uint4 *>(dp2 + ((size_t)b * kP2 + bh * kG2 + bw) * 128 + r * 64 + s * 32 + cg * 8));
        const uint32_t *h = reinterpret_cast<const uint32_t *>(&raw);
#pragma unroll
        for (int i = 0; i < 4; i++) { float2 f = tc::unpack2(h[i], f16); g[2 * i] = f.x; g[2 * i + 1] = f.y; }
    }
    size_t base = ((size_t)b * kP1 + (2 * ph) * kG1 + 2 * pw) * kC1 + cg * 8;
    const size_t off[4] = {0, (size_t)kC1, (size_t)kG1 * kC1, (size_t)kG1 * kC1 + kC1};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        uint4 raw = __ldg(reinterpret_cast<const uint4 *>(z1 + base + off[k]));
        const uint32_t *h = reinterpret_cast<const uint32_t *>(&raw);
#pragma unroll
        for (int i = 0; i < 4; i++) { float2 f = tc::unpack2(h[i], f16); z[k][2 * i] = f.x; z[k][2 * i + 1] = f.y; }
    }
    unpool_route8(g, z, dz1 + base, off, f16);
}

// This kernel WRITES the operand copies that its stream successor (a conv kernel) fetches by TMA in its prologue, i.e.
// BEFORE that kernel's griddepcontrol.wait: it must not release its dependents early.  No launch_dependents here -- the
// implicit trigger at grid completion applies, so the successor starts only when every packed weight is in memory
// (tests/test_qnet_tc_gpu.py::test_pack_then_forward_never_reads_stale_operands).
__global__ void pack_weights_kernel(const float *params, QnetLayout L, PackedWeights pw, int fwd_only) {
    tc::pdl_wait();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L.bf1; i += gridDim.x * blockDim.x) scatter_packed(i, params[i], L, pw, fwd_only);
}

// tf.train.AdamOptimizer step (TF 1.12 ApplyAdam, adam_math in fb_qnet.cuh) that also refreshes the bf16 operand
// copies of the parameters it has just written, so the next training step starts without a pack kernel
__device__ __forceinline__ void adam_one(int i, float g, float *__restrict__ p, float *__restrict__ m, float *__restrict__ v, float alpha,
                                         float beta1, float beta2, float eps, float grad_scale, const QnetLayout &L, const PackedWeights &pw) {
    float mi = m[i], vi = v[i];
    float pi = adam_math(g, p[i], mi, vi, alpha, beta1, beta2, eps, grad_scale);
    m[i] = mi; v[i] = vi;
    p[i] = pi;
    scatter_packed(i, pi, L, pw, 0);
}
__global__ void adam_pack_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m, float *__restrict__ v, int n,
                                 float alpha, float beta1, float beta2, float eps, float grad_scale, QnetLayout L, PackedWeights pw) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    adam_one(i, g[i], p, m, v, alpha, beta1, beta2, eps, grad_scale, L, pw);
}

// column sums of bf16 matrices [rows][N] in row chunks -> part[chunk][N] (bias gradients; summed in order by
// finalize_grads_kernel).  One launch covers all jobs; 16-byte loads, a warp reads whole rows.
struct ColsumJob { const bf16 *x; float *part; int rows, N, chunk_rows, first_block; };
struct ColsumJobs { ColsumJob j[3]; int njobs, f16; };
__global__ void __launch_bounds__(256) colsum_kernel(ColsumJobs jobs) {
    tc::pdl_wait();
    tc::pdl_launch();
    __shared__ float red[8][64 + 1];
    int ji = 0;
#pragma unroll
    for (int k = 1; k < 3; k++) if (k < jobs.njobs && (int)blockIdx.x >= jobs.j[k].first_block) ji = k;
    const ColsumJob jb = jobs.j[ji];
    const int chunk = blockIdx.x - jb.first_block;
    const int r0 = chunk * jb.chunk_rows, r1 = min(jb.rows, r0 + jb.chunk_rows);
    const int vec = jb.N >> 3;                       // 16-byte vectors per row: 4 (N = 32) or 8 (N = 64)
    const int rows_per_pass = 256 / vec;
    const int v = threadIdx.x % vec, rl = threadIdx.x / vec;
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = 0.f;
    for (int r = r0 + rl; r < r1; r += 8 * rows_per_pass) {        // eight rows in flight per thread, added in row order as before
        uint4 raw[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int rr = r + u * rows_per_pass;
            raw[u] = rr < r1 ? __ldg(reinterpret_cast<const uint4 *>(jb.x + (size_t)rr * jb.N) + v) : make_uint4(0u, 0u, 0u, 0u);
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            if (r + u * rows_per_pass >= r1) break;
            const uint32_t *h = reinterpret_cast<const uint32_t *>(&raw[u]);
#pragma unroll
            for (int i = 0; i < 4; i++) { float2 f = tc::unpack2(h[i], jobs.f16); acc[2 * i] += f.x; acc[2 * i + 1] += f.y; }
        }
    }
    // lanes with equal (lane % vec) hold the same columns: butterfly over the other lane bits, then across warps
#pragma unroll
    for (int i = 0; i < 8; i++)
        for (int o = 16; o >= vec; o >>= 1) acc[i] += __shfl_xor_sync(~0u, acc[i], o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane < vec)
#pragma unroll
        for (int i = 0; i < 8; i++) red[warp][lane * 8 + i] = acc[i];
    __syncthreads();
    if ((int)threadIdx.x < jb.N) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; w++) t += red[w][threadIdx.x];
        jb.part[(size_t)chunk * jb.N + threadIdx.x] = t;
    }
}

// Head backward in one pass over h1 (BrainDQN.py:151-154 / dueling BrainDuelingDQN_CC.py:68-77): gradients of the head
// weights, dh1 = dQ W^T masked by relu (bf16, the operand of the fc1 gradient GEMMs) and the fc1 bias gradient
// sum_b dh1.  Block = 32 hidden units x 8 row lanes; block gridDim.x-1 does the head bias.
constexpr int kHeadRows = 256;                      // rows of the minibatch per head-backward CTA row group
constexpr int kMaxHeadCtas = 160;                   // fused head kernel: at most one CTA (four samples at a time) per SM
// Fused Adam: AdamPow (fb_qnet.cuh) -- one thread of this kernel, early on the step's critical path, forms this step's alpha.
// operand format of the gradient tensors and the power of two they are scaled by (1 for bf16; fp16's exponent range is narrow:
// dh1 and everything downstream of it carry the factor, the weight / bias gradients are un-scaled where they are finalised)
struct GradFmt { int f16; float scale; };
__global__ void __launch_bounds__(256) head_backward_tc_kernel(const float *__restrict__ h1, const float *__restrict__ dq,
                                                               const float *__restrict__ params, QnetLayout L, int B,
                                                               float *__restrict__ hp /* [G][H][4] */, float *__restrict__ hb /* [G][4] */,
                                                               const float *__restrict__ loss_terms, bf16 *__restrict__ dh1, const AdamPow ap,
                                                               const GradFmt gf) {
    tc::pdl_wait();
    tc::pdl_launch();
    if (ap.on && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
        const float b1p = ap.pow[0], b2p = ap.pow[1];
        *ap.alpha = ap.lr * sqrtf(1.f - b2p) / (1.f - b1p);
        ap.pow[0] = b1p * ap.beta1; ap.pow[1] = b2p * ap.beta2;
    }
    __shared__ float red[8][32][4];
    const int H = L.hidden, grp = blockIdx.y, b0 = grp * kHeadRows, b1 = min(B, b0 + kHeadRows);
    if ((int)blockIdx.x == H / 32) {                 // head bias partials: sum_b dq over this row group
        float s0 = 0.f, s1 = 0.f, sl = 0.f;
        for (int b = b0 + threadIdx.x; b < b1; b += 256) { s0 += dq[b * 2]; s1 += dq[b * 2 + 1]; sl += loss_terms[b]; }
#pragma unroll
        for (int o = 16; o; o >>= 1) { s0 += __shfl_xor_sync(~0u, s0, o); s1 += __shfl_xor_sync(~0u, s1, o); sl += __shfl_xor_sync(~0u, sl, o); }
        if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0][0] = s0; red[threadIdx.x >> 5][0][1] = s1; red[threadIdx.x >> 5][0][2] = sl; }
        __syncthreads();
        if (threadIdx.x == 0) {
            float t0 = 0.f, t1 = 0.f, tl = 0.f;
            for (int w = 0; w < 8; w++) { t0 += red[w][0][0]; t1 += red[w][0][1]; tl += red[w][0][2]; }
            hb[grp * 4] = t0; hb[grp * 4 + 1] = t1; hb[grp * 4 + 2] = tl;
        }
        return;
    }
    const int jl = threadIdx.x & 31, rl = threadIdx.x >> 5, j = blockIdx.x * 32 + jl;
    float w0, w1, wv = 0.f;
    if (!L.dueling) { w0 = params[L.wf2 + j * 2]; w1 = params[L.wf2 + j * 2 + 1]; }
    else { w0 = params[L.wa + j * 2]; w1 = params[L.wa + j * 2 + 1]; wv = params[L.wv + j]; }
    float g0 = 0.f, g1 = 0.f, gv = 0.f, gb = 0.f;
#pragma unroll 8
    for (int b = b0 + rl; b < b1; b += 8) {
        float x = h1[(size_t)b * H + j];
        float d0 = dq[b * 2], d1 = dq[b * 2 + 1], g;
        if (!L.dueling) { g0 = fmaf(x, d0, g0); g1 = fmaf(x, d1, g1); g = d0 * w0 + d1 * w1; }
        else {
            float m = (d0 + d1) * 0.5f;
            g0 = fmaf(x, d0 - m, g0); g1 = fmaf(x, d1 - m, g1); gv = fmaf(x, d0 + d1, gv);
            g = (d0 - m) * w0 + (d1 - m) * w1 + (d0 + d1) * wv;
        }
        g = x > 0.f ? g * gf.scale : 0.f;
        const unsigned short gr = tc::pack1(g, gf.f16);
        reinterpret_cast<unsigned short *>(dh1)[(size_t)b * H + j] = gr;
        gb += tc::round1(g, gf.f16);                 // the bias gradient sums what the weight-gradient GEMM sees (scaled)
    }
    red[rl][jl][0] = g0; red[rl][jl][1] = g1; red[rl][jl][2] = gv; red[rl][jl][3] = gb;
    __syncthreads();
    if (rl == 0) {
        float t0 = 0.f, t1 = 0.f, tv = 0.f, tb = 0.f;
#pragma unroll
        for (int w = 0; w < 8; w++) { t0 += red[w][jl][0]; t1 += red[w][jl][1]; tv += red[w][jl][2]; tb += red[w][jl][3]; }
        *reinterpret_cast<float4 *>(hp + ((size_t)grp * H + j) * 4) = make_float4(t0, t1, tv, tb);
    }
}

// fc1 split-K finish fused with the Q head (BrainDQN.py:146-154; dueling BrainDuelingDQN_CC.py:68-77): one CTA per
// sample sums the K-split partials in order, adds the bias, applies ReLU, keeps h1 (fp32) for backward and reduces
// the two (three) head dot products.
// The TD target / loss of sample b needs only Q(s)[b] and Q(s')[b] (td_loss_kernel in fb_qnet.cu): when `td.on` the CTA that has
// just produced Q(s)[b] also writes dLoss/dQ[b], |error|, y and the sample's loss term (summed later in a fixed order).
struct TdFuse {
    int on, variant, loss_sum, global_batch, isw_mean;
    double gamma;
    const float *q_next, *q_next_online, *rewards, *isw;
    const uint8_t *actions, *terminals;
    float *dq, *abs_err, *q_target, *loss_terms;
    const double *ret, *disc;         // n-step return / discount per sample, or nullptr: the 1-step target (td_target, fb_qnet.cuh)
};
__global__ void __launch_bounds__(128) fc1_head_kernel(const float *__restrict__ part, int splits, size_t split_stride,
                                                      const float *__restrict__ params, QnetLayout L, int B, float *__restrict__ h1,
                                                      float *__restrict__ q, const TdFuse td) {
    tc::pdl_wait();
    tc::pdl_launch();
    __shared__ float red[4][3];
    const int b = blockIdx.x, H = L.hidden;
    float s0 = 0.f, s1 = 0.f, sv = 0.f;
    for (int j = threadIdx.x; j < H; j += 128) {
        float x = params[L.bf1 + j];
#pragma unroll 5
        for (int z = 0; z < splits; z++) x += part[(size_t)z * split_stride + (size_t)b * H + j];
        x = fmaxf(x, 0.f);
        if (h1 != nullptr) h1[(size_t)b * H + j] = x;          // kept for the head backward; acting / target forwards pass nullptr
        if (!L.dueling) { s0 = fmaf(x, params[L.wf2 + j * 2], s0); s1 = fmaf(x, params[L.wf2 + j * 2 + 1], s1); }
        else { s0 = fmaf(x, params[L.wa + j * 2], s0); s1 = fmaf(x, params[L.wa + j * 2 + 1], s1); sv = fmaf(x, params[L.wv + j], sv); }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) { s0 += __shfl_xor_sync(~0u, s0, o); s1 += __shfl_xor_sync(~0u, s1, o); sv += __shfl_xor_sync(~0u, sv, o); }
    if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = s0; red[threadIdx.x >> 5][1] = s1; red[threadIdx.x >> 5][2] = sv; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float t0 = 0.f, t1 = 0.f, tv = 0.f;
        for (int w = 0; w < 4; w++) { t0 += red[w][0]; t1 += red[w][1]; tv += red[w][2]; }
        if (!L.dueling) { q[b * 2] = t0 + params[L.bf2]; q[b * 2 + 1] = t1 + params[L.bf2 + 1]; }
        else {
            float a0 = t0 + params[L.ba], a1 = t1 + params[L.ba + 1], v = tv + params[L.bv];
            float mean = (a0 + a1) * 0.5f;
            q[b * 2] = v + (a0 - mean); q[b * 2 + 1] = v + (a1 - mean);
        }
        if (td.on) {                                  // exactly td_loss_kernel's arithmetic for this sample
            float x;
            if (td.variant == 2) { int am = td.q_next_online[b * 2 + 1] > td.q_next_online[b * 2] ? 1 : 0; x = td.q_next[b * 2 + am]; }
            else x = fmaxf(td.q_next[b * 2], td.q_next[b * 2 + 1]);
            const float y = td_target(x, td.rewards[b], td.terminals[b], td.ret, td.disc, b, td.gamma);
            const int a = td.actions[b] ? 1 : 0;
            const float err = y - q[b * 2 + a];
            float w = td.isw ? td.isw[b] : 1.f;
            if (td.isw && td.isw_mean) { w = 0.f; for (int k = 0; k < B; k++) w += td.isw[k]; w /= (float)B; }    // [B,1] x [B] broadcast (see TdFuse)
            const float scale = td.loss_sum ? 1.f : 1.f / (float)td.global_batch;
            td.dq[b * 2 + a] = -2.f * w * err * scale; td.dq[b * 2 + (1 - a)] = 0.f;
            td.loss_terms[b] = w * err * err * scale;
            if (td.abs_err) td.abs_err[b] = fabsf(err);
            if (td.q_target) td.q_target[b] = y;
        }
    }
}

// The plain head (acting, Q(s')) in the same warp-per-sample form: fc1 split-K finish + bias + ReLU + the head dot products,
// reductions by shuffles.  Measured at minibatch 256: 5 us against 10 us for the CTA-per-sample fc1_head_kernel.
template <int JPL>
__global__ void __launch_bounds__(128) fc1_head_warp_kernel(const float *__restrict__ part, int splits, size_t split_stride,
                                                           const float *__restrict__ params, QnetLayout L, int B, float *__restrict__ h1,
                                                           float *__restrict__ q) {
    tc::pdl_wait();
    tc::pdl_launch();
    constexpr int H = 32 * JPL;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float w0[JPL], w1[JPL], wv[JPL], bias[JPL];
#pragma unroll
    for (int u = 0; u < JPL; u++) {
        const int j = lane + 32 * u;
        bias[u] = params[L.bf1 + j];
        if (!L.dueling) { w0[u] = params[L.wf2 + j * 2]; w1[u] = params[L.wf2 + j * 2 + 1]; wv[u] = 0.f; }
        else { w0[u] = params[L.wa + j * 2]; w1[u] = params[L.wa + j * 2 + 1]; wv[u] = params[L.wv + j]; }
    }
    const float b_q0 = L.dueling ? params[L.ba] : params[L.bf2], b_q1 = L.dueling ? params[L.ba + 1] : params[L.bf2 + 1];
    const float b_v = L.dueling ? params[L.bv] : 0.f;
    const int nwarps = gridDim.x * 4;
    for (int b = blockIdx.x * 4 + warp; b < B; b += nwarps) {
        float x[JPL];
        float s0 = 0.f, s1 = 0.f, sv = 0.f;
#pragma unroll
        for (int u = 0; u < JPL; u++) x[u] = bias[u];
        for (int z = 0; z < splits; z++) {
            const float *pz = part + (size_t)z * split_stride + (size_t)b * H + lane;
#pragma unroll
            for (int u = 0; u < JPL; u++) x[u] += pz[32 * u];
        }
#pragma unroll
        for (int u = 0; u < JPL; u++) {
            x[u] = fmaxf(x[u], 0.f);
            if (h1 != nullptr) h1[(size_t)b * H + lane + 32 * u] = x[u];
            s0 = fmaf(x[u], w0[u], s0); s1 = fmaf(x[u], w1[u], s1); sv = fmaf(x[u], wv[u], sv);
        }
#pragma unroll
        for (int off = 16; off; off >>= 1) { s0 += __shfl_xor_sync(~0u, s0, off); s1 += __shfl_xor_sync(~0u, s1, off); sv += __shfl_xor_sync(~0u, sv, off); }
        if (lane == 0) {
            if (!L.dueling) { q[b * 2] = s0 + b_q0; q[b * 2 + 1] = s1 + b_q1; }
            else { const float a0 = s0 + b_q0, a1 = s1 + b_q1, v = sv + b_v, mean = (a0 + a1) * 0.5f; q[b * 2] = v + (a0 - mean); q[b * 2 + 1] = v + (a1 - mean); }
        }
    }
}

// The training step's head in ONE kernel (hidden = 32 JPL): fc1 split-K finish + bias + ReLU, the Q head, the TD target /
// loss / dLoss/dQ, and the head's backward pass -- dh1 = dQ W^T masked by relu (bf16, the operand of the fc1 gradient GEMMs),
// the head weight gradients and the fc1 bias gradient -- for which h1 never leaves the registers.  One WARP per sample
// (lane = hidden units lane + 32 u): the sample's reductions are shuffles, no block barrier sits between Q(s) and its
// gradient; the per-CTA partial sums [G][H][4], [G][4] are what finalize_grads_kernel adds in a fixed order.  Also carries the
// fused-Adam alpha (AdamPow, as head_backward_tc_kernel did).  Replaces fc1_head_kernel + head_backward_tc_kernel on the
// step's critical path.
struct HeadBwd { bf16 *dh1; float *hp /* [G][H][4] */, *hb /* [G][4]: sum dq0, sum dq1, loss */; GradFmt gf; };
template <int JPL>
__global__ void __launch_bounds__(128) fc1_head_train_kernel(const float *__restrict__ part, int splits, size_t split_stride,
                                                            const float *__restrict__ params, QnetLayout L, int B, float *__restrict__ q,
                                                            const TdFuse td, const HeadBwd o, const AdamPow ap) {
    tc::pdl_wait();
    tc::pdl_launch();
    constexpr int H = 32 * JPL;
    __shared__ float4 red[4][H];
    __shared__ float red_b[4][4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (ap.on && blockIdx.x == 0 && threadIdx.x == 0) {
        const float b1p = ap.pow[0], b2p = ap.pow[1];
        *ap.alpha = ap.lr * sqrtf(1.f - b2p) / (1.f - b1p);
        ap.pow[0] = b1p * ap.beta1; ap.pow[1] = b2p * ap.beta2;
    }
    float w0[JPL], w1[JPL], wv[JPL], bias[JPL], g0[JPL], g1[JPL], gv[JPL], gb[JPL];
#pragma unroll
    for (int u = 0; u < JPL; u++) {
        const int j = lane + 32 * u;
        bias[u] = params[L.bf1 + j];
        if (!L.dueling) { w0[u] = params[L.wf2 + j * 2]; w1[u] = params[L.wf2 + j * 2 + 1]; wv[u] = 0.f; }
        else { w0[u] = params[L.wa + j * 2]; w1[u] = params[L.wa + j * 2 + 1]; wv[u] = params[L.wv + j]; }
        g0[u] = g1[u] = gv[u] = gb[u] = 0.f;
    }
    float wmean = 1.f;
    if (td.isw && td.isw_mean) {                     // ISWeights [B,1] * square(...) [B] broadcasts to [B,B] in the reference
        float s = 0.f;                               // (BrainPrioritizedReplyDQN.py:243-251): every sample is weighted by mean(w)
        for (int b = lane; b < B; b += 32) s += td.isw[b];
#pragma unroll
        for (int off = 16; off; off >>= 1) s += __shfl_xor_sync(~0u, s, off);
        wmean = s / (float)B;
    }
    const float b_q0 = L.dueling ? params[L.ba] : params[L.bf2], b_q1 = L.dueling ? params[L.ba + 1] : params[L.bf2 + 1];
    const float b_v = L.dueling ? params[L.bv] : 0.f;
    float sd0 = 0.f, sd1 = 0.f, sloss = 0.f;
    const int nwarps = gridDim.x * 4;
    for (int b = blockIdx.x * 4 + warp; b < B; b += nwarps) {
        float x[JPL];
        float s0 = 0.f, s1 = 0.f, sv = 0.f;
#pragma unroll
        for (int u = 0; u < JPL; u++) x[u] = bias[u];
        for (int z = 0; z < splits; z++) {
            const float *pz = part + (size_t)z * split_stride + (size_t)b * H + lane;
#pragma unroll
            for (int u = 0; u < JPL; u++) x[u] += pz[32 * u];
        }
#pragma unroll
        for (int u = 0; u < JPL; u++) {
            x[u] = fmaxf(x[u], 0.f);
            s0 = fmaf(x[u], w0[u], s0); s1 = fmaf(x[u], w1[u], s1); sv = fmaf(x[u], wv[u], sv);
        }
#pragma unroll
        for (int off = 16; off; off >>= 1) { s0 += __shfl_xor_sync(~0u, s0, off); s1 += __shfl_xor_sync(~0u, s1, off); sv += __shfl_xor_sync(~0u, sv, off); }
        float q0, q1;
        if (!L.dueling) { q0 = s0 + b_q0; q1 = s1 + b_q1; }
        else { const float a0 = s0 + b_q0, a1 = s1 + b_q1, v = sv + b_v, mean = (a0 + a1) * 0.5f; q0 = v + (a0 - mean); q1 = v + (a1 - mean); }
        // td_loss_kernel's arithmetic (fb_qnet.cu), the same in every lane
        float xn;
        if (td.variant == 2) { const int am = td.q_next_online[b * 2 + 1] > td.q_next_online[b * 2] ? 1 : 0; xn = td.q_next[b * 2 + am]; }
        else xn = fmaxf(td.q_next[b * 2], td.q_next[b * 2 + 1]);
        const float y = td_target(xn, td.rewards[b], td.terminals[b], td.ret, td.disc, b, td.gamma);
        const int a = td.actions[b] ? 1 : 0;
        const float err = y - (a ? q1 : q0);
        const float w = td.isw ? (td.isw_mean ? wmean : td.isw[b]) : 1.f;
        const float scale = td.loss_sum ? 1.f : 1.f / (float)td.global_batch;
        const float g = -2.f * w * err * scale;
        const float d0 = a ? 0.f : g, d1 = a ? g : 0.f;
        sd0 += d0; sd1 += d1; sloss += w * err * err * scale;
        if (lane == 0) {
            q[b * 2] = q0; q[b * 2 + 1] = q1;
            td.dq[b * 2] = d0; td.dq[b * 2 + 1] = d1;
            td.loss_terms[b] = w * err * err * scale;
            if (td.abs_err) td.abs_err[b] = fabsf(err);
            if (td.q_target) td.q_target[b] = y;
        }
        // head backward for this sample (head_backward_tc_kernel's arithmetic)
        const float m = (d0 + d1) * 0.5f;
#pragma unroll
        for (int u = 0; u < JPL; u++) {
            float gh;
            if (!L.dueling) { g0[u] = fmaf(x[u], d0, g0[u]); g1[u] = fmaf(x[u], d1, g1[u]); gh = d0 * w0[u] + d1 * w1[u]; }
            else {
                g0[u] = fmaf(x[u], d0 - m, g0[u]); g1[u] = fmaf(x[u], d1 - m, g1[u]); gv[u] = fmaf(x[u], d0 + d1, gv[u]);
                gh = (d0 - m) * w0[u] + (d1 - m) * w1[u] + (d0 + d1) * wv[u];
            }
            gh = x[u] > 0.f ? gh * o.gf.scale : 0.f;
            reinterpret_cast<unsigned short *>(o.dh1)[(size_t)b * H + lane + 32 * u] = tc::pack1(gh, o.gf.f16);
            gb[u] += tc::round1(gh, o.gf.f16);        // the bias gradient sums what the weight-gradient GEMM sees (scaled)
        }
    }
#pragma unroll
    for (int u = 0; u < JPL; u++) red[warp][lane + 32 * u] = make_float4(g0[u], g1[u], gv[u], gb[u]);
    if (lane == 0) { red_b[warp][0] = sd0; red_b[warp][1] = sd1; red_b[warp][2] = sloss; }
    __syncthreads();
    for (int j = threadIdx.x; j < H; j += 128) {
        float4 t = red[0][j];
#pragma unroll
        for (int k = 1; k < 4; k++) { const float4 v = red[k][j]; t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w; }
        *reinterpret_cast<float4 *>(o.hp + ((size_t)blockIdx.x * H + j) * 4) = t;
    }
    if (threadIdx.x < 3) o.hb[blockIdx.x * 4 + threadIdx.x] = red_b[0][threadIdx.x] + red_b[1][threadIdx.x] + red_b[2][threadIdx.x] + red_b[3][threadIdx.x];
}

// split-K partials, bias partials and head partials -> the flat gradient vector in TF variable order (HWIO).  One CTA
// sums 32 consecutive gradient elements: lane = element (coalesced across the partial buffers), the kFinWarps warps take every
// kFinWarps-th term, and the sub-sums are added in a fixed order (deterministic for a given batch size).  Two warps of 32
// loads in flight each: the whole grid (2,486 CTAs at hidden 512) is resident at once, so the kernel costs one CTA's chain of
// round trips (partials -> Adam state -> stores), not two waves of it -- it is the last stage of every update.
constexpr int kFinWarps = 2, kFinInflight = 40;      // 74 conv1 splits at minibatch 256: one batch of loads per warp
struct FinalizeArgs {
    const float *part1, *part2, *part3;             // [splits][rows][N]
    int s1, s2, s3;                                  // number of splits (fc1's weight gradient is written in place)
    const float *bp1, *bp2, *bp3;                   // bias partials [chunks][N]
    int c1, c2, c3;
    const float *hp, *hb;                           // head partials [G][H][4], [G][4] (dq sums, loss)
    int G;
    float *loss_out;
    float inv_scale;                                // un-scales what came through the (scaled) gradient tensors
};
// With `ad.on` the same launch also applies Adam (fb_qnet_step): the CTA that has just summed 32 gradient elements
// updates those parameters (W_fc1, whose gradient the fc1 GEMM wrote in place, is updated earlier by adam_wf1_kernel).
// alpha was left in device memory by the head kernel, so the whole update replays as one CUDA graph.
// These kernels WRITE the bf16 operand copies: no early launch_dependents (see pack_weights_kernel).
struct AdamDev { int on; float *p, *m, *v; float beta1, beta2, eps, grad_scale; const float *alpha; };
// Adam on W_fc1: its gradient exists early in the backward pass, so these 819,200 of the 898,722 parameters are updated beside
// the convolution gradients instead of after them (the caller orders it after the fc1 data-gradient GEMM, the last reader of
// the bf16 copy it rewrites).
__global__ void __launch_bounds__(256) adam_wf1_kernel(QnetLayout L, const float *__restrict__ grads, const AdamDev ad, const PackedWeights pw) {
    const float alpha = *ad.alpha;
    const int n4 = (L.bf1 - L.wf1) >> 2;            // hidden % 128 == 0: a multiple of four, 16-byte aligned (L.wf1 = 77,984)
    for (int i4 = blockIdx.x * blockDim.x + threadIdx.x; i4 < n4; i4 += gridDim.x * blockDim.x) {
        const int i = L.wf1 + 4 * i4;
        const float4 g = *reinterpret_cast<const float4 *>(grads + i);
        float4 p = *reinterpret_cast<float4 *>(ad.p + i), m = *reinterpret_cast<float4 *>(ad.m + i), v = *reinterpret_cast<float4 *>(ad.v + i);
        const float gg[4] = {g.x, g.y, g.z, g.w};
        float pp[4] = {p.x, p.y, p.z, p.w}, mm[4] = {m.x, m.y, m.z, m.w}, vv[4] = {v.x, v.y, v.z, v.w};
        uint32_t pk[2];
#pragma unroll
        for (int k = 0; k < 4; k++) pp[k] = adam_math(gg[k], pp[k], mm[k], vv[k], alpha, ad.beta1, ad.beta2, ad.eps, ad.grad_scale);
        *reinterpret_cast<float4 *>(ad.p + i) = make_float4(pp[0], pp[1], pp[2], pp[3]);
        *reinterpret_cast<float4 *>(ad.m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
        *reinterpret_cast<float4 *>(ad.v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
#pragma unroll
        for (int k = 0; k < 2; k++) pk[k] = tc::pack2(pp[2 * k], pp[2 * k + 1], pw.f16);
        *reinterpret_cast<uint2 *>(pw.wf1n + 4 * i4) = make_uint2(pk[0], pk[1]);
    }
}
// kC51: the head region reads c51_head_backward_kernel's partials (fb_c51.cu); a separate instantiation, so that the expected-value
// head's code is exactly what it was
template <bool kC51>
__global__ void __launch_bounds__(32 * kFinWarps) finalize_grads_kernel(const FinalizeArgs a, QnetLayout L, float *__restrict__ grads, const AdamDev ad,
                                                                       const PackedWeights pw, const NetLayout Lc /* kC51: the head */) {
    __shared__ float red[kFinWarps][32];
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5, H = L.hidden;
    const int k = blockIdx.x * 32 + lane;            // compact index: [0, wf1) then [bf1, total)
    const int n_compact = L.wf1 + (L.total - L.bf1);
    const int i = k < L.wf1 ? k : k - L.wf1 + L.bf1;
    // the Adam state of these parameters was last written by the PREVIOUS step's launch of this kernel: fetched while this
    // step's weight gradients still run (one round trip off the update's tail)
    float p0 = 0.f, m0 = 0.f, v0 = 0.f;
    if (ad.on && g == 0 && k < n_compact) { p0 = ad.p[i]; m0 = ad.m[i]; v0 = ad.v[i]; }
    tc::pdl_wait();
    if (!ad.on) tc::pdl_launch();
    const float alpha = ad.on ? *ad.alpha : 0.f;
    float s = 0.f;
    // terms z = g, g + kFinWarps, ... of one element, added in that order; kFinInflight loads are issued before the first add
    // (the sums over 49 .. 147 split-K partials were a chain of dependent L2 round trips)
    auto strided_sum = [&](int count, auto &&term) {
        for (int z = g; z < count; z += kFinWarps * kFinInflight) {
            float v[kFinInflight];
#pragma unroll
            for (int u = 0; u < kFinInflight; u++) v[u] = z + kFinWarps * u < count ? term(z + kFinWarps * u) : 0.f;
#pragma unroll
            for (int u = 0; u < kFinInflight; u++) if (z + kFinWarps * u < count) s += v[u];
        }
    };
    if (k < n_compact) {
        if (i < L.b1) {                     // W1 [kh][kw][c][n]
            int e = i - L.w1, n = e & 31, c = (e >> 5) & 3, kw = (e >> 7) & 7, kh = e >> 10;
            int row = ((kh >> 2) * 2 + (kw >> 2)) * 64 + (kh & 3) * 16 + (kw & 3) * 4 + c;
            strided_sum(a.s1, [&](int z) { return a.part1[((size_t)z * 256 + row) * 32 + n]; });
        } else if (i < L.w2) {
            int n = i - L.b1;
            strided_sum(a.c1, [&](int z) { return a.bp1[z * 32 + n]; });
        } else if (i < L.b2) {              // W2 [kh][kw][c][n]
            int e = i - L.w2, n = e & 63, c = (e >> 6) & 31, kw = (e >> 11) & 3, kh = e >> 13;
            int row = ((kh >> 1) * 2 + (kw >> 1)) * 128 + (kh & 1) * 64 + (kw & 1) * 32 + c;
            strided_sum(a.s2, [&](int z) { return a.part2[((size_t)z * 512 + row) * 64 + n]; });
        } else if (i < L.w3) {
            int n = i - L.b2;
            strided_sum(a.c2, [&](int z) { return a.bp2[z * 64 + n]; });
        } else if (i < L.b3) {              // W3 [k][n], k natural
            int e = i - L.w3;
            strided_sum(a.s3, [&](int z) { return a.part3[(size_t)z * 640 * 64 + e]; });
        } else if (i < L.wf1) {
            int n = i - L.b3;
            strided_sum(a.c3, [&](int z) { return a.bp3[z * 64 + n]; });
        } else if (i < L.bf1 + H) {         // fc1 bias
            int j = i - L.bf1;
            if constexpr (kC51) strided_sum(a.G, [&](int z) { return a.hp[z * c51_partial_stride(Lc) + (size_t)(H + 1) * c51_cols(Lc) + j]; });
            else strided_sum(a.G, [&](int z) { return a.hp[((size_t)z * H + j) * 4 + 3]; });
        } else if constexpr (kC51) {        // C51 head: partials [G][c51_partial_stride]
            int j, c;
            c51_column(Lc, i, &j, &c);
            strided_sum(a.G, [&](int z) { return a.hp[z * c51_partial_stride(Lc) + (size_t)j * c51_cols(Lc) + c]; });
        } else if (!L.dueling) {
            if (i < L.bf2) { int e = i - L.wf2; strided_sum(a.G, [&](int z) { return a.hp[((size_t)z * H + (e >> 1)) * 4 + (e & 1)]; }); }
            else { int e = i - L.bf2; strided_sum(a.G, [&](int z) { return a.hb[z * 4 + e]; }); }
        } else {
            if (i < L.bv) { int j = i - L.wv; strided_sum(a.G, [&](int z) { return a.hp[((size_t)z * H + j) * 4 + 2]; }); }
            else if (i < L.wa) { strided_sum(a.G, [&](int z) { return a.hb[z * 4] + a.hb[z * 4 + 1]; }); }
            else if (i < L.ba) { int e = i - L.wa; strided_sum(a.G, [&](int z) { return a.hp[((size_t)z * H + (e >> 1)) * 4 + (e & 1)]; }); }
            else { int e = i - L.ba; strided_sum(a.G, [&](int z) { return (e == 0 ? 0.5f : -0.5f) * (a.hb[z * 4] - a.hb[z * 4 + 1]); }); }
        }
    }
    red[g][lane] = s;
    __syncthreads();
    if (g == 0 && k < n_compact) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kFinWarps; w++) t += red[w][lane];
        if (i < L.bf1 + H) t *= a.inv_scale;         // conv / fc1 weights and biases: sums of scaled gradient tensors (the head's are not)
        grads[i] = t;
        if (ad.on) {
            const float pi = adam_math(t, p0, m0, v0, alpha, ad.beta1, ad.beta2, ad.eps, ad.grad_scale);
            ad.m[i] = m0; ad.v[i] = v0; ad.p[i] = pi;
            scatter_packed(i, pi, L, pw, 0);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && a.loss_out) {       // the loss: row-group sums in order
        float t = 0.f;
        for (int z = 0; z < a.G; z++) t += a.hb[z * 4 + 2];
        *a.loss_out = t;
    }
}

// ------------------------------------------------------------------------------------------------ fused conv backward
// conv3 data gradient -> ReLU mask -> conv2 data gradient -> un-pool + ReLU mask in ONE kernel: three dependent stages of the
// step's critical path (three launches, two HBM/L2 round trips of dZ2 / dP2) become one.  A tile is TWO SAMPLES of the
// 7-wide grid (98 rows of an M = 128 accumulator), so that everything a tile needs from its neighbours is rows that are zero
// by construction (the pad ring of the grid): dZ2 of the tile never leaves the SM between the two GEMMs -- the epilogue of the
// first writes it (bf16, masked) where TMA's 128-byte swizzle would have put it, fence.proxy.async, and the second GEMM reads
// it through shifted descriptors like any slab.  dZ2 also goes to HBM once (the conv2 weight gradient and the conv2 bias
// gradient contract over it); dP2 exists only in TMEM / registers.  Arithmetic and roundings are those of the three separate
// kernels (bit-identical results: tests/test_qnet_tc_gpu.py::test_fused_backward_is_bit_identical).
struct Bwd23Params {
    int n_tiles, B;
    const bf16 *a2;             // [B*49][64]   conv2 activations: ReLU mask of dZ2
    bf16 *dz2;                  // [B*49][64]   out
    const bf16 *z1;             // [B*441][32]  conv1 activations: pooling argmax + ReLU mask
    bf16 *dz1;                  // [B*441][32]  out (invalid grid positions stay zero)
    int f16;
};
constexpr int kBwdRows = 2 * kP2;           // 98 rows of the 7-grid per tile

template <int S>
__global__ void __launch_bounds__(kConvThreads, 1) tc_bwd23_kernel(const __grid_constant__ CUtensorMap mapDz3, const __grid_constant__ CUtensorMap mapW3d,
                                                                    const __grid_constant__ CUtensorMap mapW2d, const Bwd23Params g) {
    constexpr uint32_t W3_BYTES = 9 * 64 * 128, W2_BYTES = 4 * 128 * 128, SLAB1 = 144 * 128, SLAB2 = 136 * 128;
    static_assert(SLAB1 % 1024 == 0 && SLAB2 % 1024 == 0, "swizzle atoms are 1024-byte aligned");   // slab 2: taps reach 8 rows back, 128 + 8 rows
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[S], bar_empty[S], bar_b, bar_acc1_full, bar_acc1_empty, bar_acc2_full, bar_acc2_empty, bar_slab2;
    __shared__ uint32_t tmem_slot;
    uint8_t *smem_gen = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t smem_w3 = tc::smem_u32(smem_gen), smem_w2 = smem_w3 + W3_BYTES, smem_s1 = smem_w2 + W2_BYTES, smem_s2 = smem_s1 + S * SLAB1;
    uint8_t *slab2_gen = smem_gen + W3_BYTES + W2_BYTES + S * SLAB1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        tc::tma_prefetch_desc(&mapDz3); tc::tma_prefetch_desc(&mapW3d); tc::tma_prefetch_desc(&mapW2d);
        for (int s = 0; s < S; s++) { tc::mbar_init(tc::smem_u32(&bar_full[s]), 1); tc::mbar_init(tc::smem_u32(&bar_empty[s]), 1); }
        tc::mbar_init(tc::smem_u32(&bar_b), 1);
        tc::mbar_init(tc::smem_u32(&bar_acc1_full), 1); tc::mbar_init(tc::smem_u32(&bar_acc1_empty), 4);
        tc::mbar_init(tc::smem_u32(&bar_acc2_full), 1); tc::mbar_init(tc::smem_u32(&bar_acc2_empty), 4);
        tc::mbar_init(tc::smem_u32(&bar_slab2), 4);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tc::smem_u32(&tmem_slot), 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_slot, acc1 = tmem, acc2 = tmem + 64;
    if (threadIdx.x == 0) {                          // the weights do not depend on the previous kernel: fetch them first
        tc::mbar_expect_tx(tc::smem_u32(&bar_b), W3_BYTES + W2_BYTES);
        for (int kb = 0; kb < 9; kb++) tc::tma_load_2d(smem_w3 + kb * (64 * 128), &mapW3d, kb * 64, 0, tc::smem_u32(&bar_b));
        for (int kb = 0; kb < 4; kb++) tc::tma_load_2d(smem_w2 + kb * (128 * 128), &mapW2d, kb * 64, 0, tc::smem_u32(&bar_b));
    }
    tc::pdl_wait();
    tc::pdl_launch();

    if (warp == 0) {
        const bool leader = tc::elect_one();
        int i = 0;
        for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, i++) {
            const int s = i % S;
            tc::mbar_wait(tc::smem_u32(&bar_empty[s]), ((i / S) & 1) ^ 1u);
            if (leader) {
                const uint32_t full = tc::smem_u32(&bar_full[s]);
                tc::mbar_expect_tx(full, SLAB1);
                tc::tma_load_2d(smem_s1 + s * SLAB1, &mapDz3, 0, tile * kBwdRows - 8, full);    // rows before / after the tensor: zeros
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        const bool leader = tc::elect_one();
        const uint32_t idesc1 = tc::instr_desc_16(128, 64, 0, 0, g.f16), idesc2 = tc::instr_desc_16(128, 128, 0, 0, g.f16);
        constexpr uint32_t dhi = tc::smem_desc_hi(1024, tc::kSwizzle128);
        const uint32_t w3_lo = tc::smem_desc_lo(smem_w3, 16), w2_lo = tc::smem_desc_lo(smem_w2, 16);
        const uint32_t s1_lo = tc::smem_desc_lo(smem_s1, 16), s2_lo = tc::smem_desc_lo(smem_s2, 16);
        tc::mbar_wait(tc::smem_u32(&bar_b), 0);
        int i = 0;
        for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, i++) {
            const int s = i % S;
            // ---- GEMM 1: dA2[p][c] = sum_{kh,kw,o} dZ3[p + (1-kh) 7 + (1-kw)][o] W3[kh][kw][c][o]   (slab row 0 = position -8)
            tc::mbar_wait(tc::smem_u32(&bar_acc1_empty), (i & 1) ^ 1u);
            tc::mbar_wait(tc::smem_u32(&bar_full[s]), (i / S) & 1);
            tc::tc_fence_after();
            if (leader) {
#pragma unroll
                for (int kb = 0; kb < 9; kb++) {
                    const uint32_t tap = (uint32_t)(((1 - kb / 3) * kG2 + (1 - kb % 3) + 8) * 128) >> 4;
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        tc::umma_bf16_lohi(acc1, s1_lo + s * (SLAB1 >> 4) + tap + 2 * k, dhi, w3_lo + ((kb * 64 * 128 + k * 32) >> 4), dhi, idesc1, (kb | k) != 0);
                }
                tc::umma_commit(tc::smem_u32(&bar_empty[s]));
                tc::umma_commit(tc::smem_u32(&bar_acc1_full));
            }
            __syncwarp();
            // ---- GEMM 2: dP2[p][(r,s,c)] = sum_{dh,dw,o} dZ2[p - 7 dh - dw][o] W2d[(r,s,c)][(dh,dw),o]   (slab-2 row 8 = the tile's row 0)
            tc::mbar_wait(tc::smem_u32(&bar_slab2), i & 1);
            tc::mbar_wait(tc::smem_u32(&bar_acc2_empty), (i & 1) ^ 1u);
            tc::tc_fence_after();
            if (leader) {
#pragma unroll
                for (int kb = 0; kb < 4; kb++) {
                    const uint32_t tap = (uint32_t)((8 - (kb >> 1) * kG2 - (kb & 1)) * 128) >> 4;
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        tc::umma_bf16_lohi(acc2, s2_lo + tap + 2 * k, dhi, w2_lo + ((kb * 128 * 128 + k * 32) >> 4), dhi, idesc2, (kb | k) != 0);
                }
                tc::umma_commit(tc::smem_u32(&bar_acc2_full));
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3, r = q * 32 + lane;            // accumulator row = row r of the tile (TMEM lanes of warp % 4)
        // zero rows of the second slab that no tile ever writes: the 8 rows before the tile (the previous sample's pad ring)
        if (r < 8) {
#pragma unroll
            for (int c = 0; c < 8; c++) *reinterpret_cast<uint4 *>(slab2_gen + r * 128 + c * 16) = make_uint4(0, 0, 0, 0);
        }
        int i = 0;
        for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, i++) {
            const long long grow = (long long)tile * kBwdRows + r;               // row of the [B*49] grid tensors
            const bool in_tile = r < kBwdRows && grow < (long long)g.B * kP2;
            const int p = r % kP2, bh = p / kG2, bw = p - bh * kG2;
            const int b = (int)(tile * 2 + (r >= kP2 ? 1 : 0));
            // ---- epilogue 1: dZ2 = dA2 * relu'(a2), zeros at invalid positions -> HBM and the second slab
            const bool ok = in_tile && bh < 5 && bw < 5;
            uint4 araw[8];                                   // the ReLU mask does not depend on the accumulator: fetched while the MMAs run
            if (ok) {
                const uint4 *am = reinterpret_cast<const uint4 *>(g.a2 + grow * 64);
#pragma unroll
                for (int c = 0; c < 8; c += 2) tc::ld_global_nc_256(am + c, araw[c], araw[c + 1]);
            }
            tc::mbar_wait(tc::smem_u32(&bar_acc1_full), i & 1);
            tc::tc_fence_after();
            float v[64];
            tc::tmem_ld32(acc1 + ((uint32_t)(q * 32) << 16), *reinterpret_cast<float(*)[32]>(&v[0]));
            tc::tmem_ld32(acc1 + ((uint32_t)(q * 32) << 16) + 32, *reinterpret_cast<float(*)[32]>(&v[32]));
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bar_acc1_empty));
            uint4 outw[8];
#pragma unroll
            for (int c = 0; c < 8; c++) outw[c] = make_uint4(0, 0, 0, 0);
            if (ok) {
#pragma unroll
                for (int c = 0; c < 8; c++) {
                    const uint32_t *h = reinterpret_cast<const uint32_t *>(&araw[c]);
                    uint32_t w[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const float2 a = tc::unpack2(h[k], g.f16);
                        w[k] = tc::pack2(a.x > 0.f ? v[c * 8 + 2 * k] : 0.f, a.y > 0.f ? v[c * 8 + 2 * k + 1] : 0.f, g.f16);
                    }
                    outw[c] = make_uint4(w[0], w[1], w[2], w[3]);
                }
            }
            if (in_tile) {
                uint4 *d = reinterpret_cast<uint4 *>(g.dz2 + grow * 64);
#pragma unroll
                for (int c = 0; c < 8; c += 2) tc::st_global_256(d + c, outw[c], outw[c + 1]);
            }
            {   // slab-2 row r + 8, 16-byte chunk c at ((c ^ (row & 7)) << 4): the layout a TMA SWIZZLE_128B load would have produced
                const int R = r + 8;
                uint8_t *rowp = slab2_gen + R * 128;
#pragma unroll
                for (int c = 0; c < 8; c++) *reinterpret_cast<uint4 *>(rowp + ((c ^ (R & 7)) << 4)) = outw[c];
            }
            tc::fence_proxy_async();                      // generic-proxy writes -> visible to the tensor core's async proxy
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bar_slab2));
            // ---- epilogue 2: dZ1 = unpool(dP2) * relu'(z1); row (b, bh, bw) holds the 2x2 block of pooled positions (2bh-1+rr, 2bw-1+ss)
            // the window activations of all four channel groups of one pooled position: 16 independent 16-byte loads in flight (they
            // were four dependent rounds of four -- 16 L2 round trips per thread and tile); the first position's before the wait
            const size_t off[4] = {0, (size_t)kC1, (size_t)kG1 * kC1, (size_t)kG1 * kC1 + kC1};
            uint4 zr[4][4];
            bool valid = false;
            size_t base = 0;
            auto issue = [&](int rs) {
                const int ph = 2 * bh - 1 + (rs >> 1), pw = 2 * bw - 1 + (rs & 1);
                valid = in_tile && (unsigned)ph < 10u && (unsigned)pw < 10u;
                base = valid ? ((size_t)b * kP1 + (2 * ph) * kG1 + 2 * pw) * kC1 : 0;
                if (valid) {
#pragma unroll
                    for (int cp = 0; cp < 2; cp++)
#pragma unroll
                        for (int k = 0; k < 4; k++) tc::ld_global_nc_256(g.z1 + base + off[k] + cp * 16, zr[2 * cp][k], zr[2 * cp + 1][k]);
                }
            };
            issue(0);
            tc::mbar_wait(tc::smem_u32(&bar_acc2_full), i & 1);
            tc::tc_fence_after();
#pragma unroll 1
            for (int rs = 0; rs < 4; rs++) {
                if (rs > 0) issue(rs);
                float gq[32];
                tc::tmem_ld32(acc2 + ((uint32_t)(q * 32) << 16) + (uint32_t)(rs * 32), gq);
                if (rs == 3) {                             // accumulator drained: hand it back before the stores
                    tc::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bar_acc2_empty));
                }
                if (valid) {
#pragma unroll
                    for (int cp = 0; cp < 2; cp++) {                      // two channel groups = 32 bytes of a position: one store
                        uint4 outp[2][4];
#pragma unroll
                        for (int hh = 0; hh < 2; hh++) {
                            const int cg = 2 * cp + hh;
                            float gg[8], z[4][8];
#pragma unroll
                            for (int k = 0; k < 8; k++) gg[k] = tc::round1(gq[cg * 8 + k], g.f16);      // dP2 was a 16-bit tensor
#pragma unroll
                            for (int k = 0; k < 4; k++) {
                                const uint32_t *h = reinterpret_cast<const uint32_t *>(&zr[cg][k]);
#pragma unroll
                                for (int e = 0; e < 4; e++) { const float2 f = tc::unpack2(h[e], g.f16); z[k][2 * e] = f.x; z[k][2 * e + 1] = f.y; }
                            }
                            unpool_pack8(gg, z, outp[hh], g.f16);
                        }
#pragma unroll
                        for (int k = 0; k < 4; k++) tc::st_global_256(g.dz1 + base + off[k] + cp * 16, outp[0][k], outp[1][k]);
                    }
                }
                __syncwarp();
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem, 256);
}

template <int S>
static cudaError_t launch_tc_bwd23(const CUtensorMap &mdz3, const CUtensorMap &mw3d, const CUtensorMap &mw2d, const Bwd23Params &g, int max_ctas,
                                   cudaStream_t st) {
    static bool configured = false;
    auto kern = tc_bwd23_kernel<S>;
    constexpr size_t smem = 9 * 64 * 128 + 4 * 128 * 128 + (size_t)S * 144 * 128 + 136 * 128 + 1024;
    static_assert(smem <= 227 * 1024 && smem > kExclusiveSmem, "shared memory budget");
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    const int grid = g.n_tiles < max_ctas ? g.n_tiles : max_ctas;
    return tc::launch_pdl(kern, dim3(grid), dim3(kConvThreads), smem, st, mdz3, mw3d, mw2d, g);
}

// ------------------------------------------------------------------------------------------------ fused conv2 + conv3 forward
// conv 4x4 s2 + bias + ReLU -> conv 3x3 s1 + bias + ReLU in ONE kernel, the forward twin of tc_bwd23_kernel: a tile is two
// samples of the 7-wide grid; the conv2 activations A2 are handed to the second GEMM through a hand-swizzled shared-memory slab
// (and go to HBM only when a backward pass needs them); A3 leaves in TF flatten order.  One stage less on every forward's
// critical path; arithmetic and roundings are those of the two separate kernels (bit-identical).
struct Fwd23Params {
    int n_tiles, B;
    const float *bias2, *bias3;
    bf16 *a2;                   // [B*49][64] or nullptr (acting / target forward: not needed)
    bf16 *a3;                   // [B][25][64]
    int f16;
};

template <int S>
__global__ void __launch_bounds__(kConvThreads, 1) tc_fwd23_kernel(const __grid_constant__ CUtensorMap mapP2, const __grid_constant__ CUtensorMap mapW2,
                                                                    const __grid_constant__ CUtensorMap mapW3, const Fwd23Params g) {
    // slab 2 (conv3's input): 8 zero rows + the tile's 98 rows + ...; the 3x3 taps reach 16 rows past an accumulator row, so the
    // 128-row MMA reads 144 rows (rows 136..143 feed discarded accumulator rows only)
    constexpr uint32_t W2_BYTES = 8 * 64 * 128, W3_BYTES = 9 * 64 * 128, HALF1 = 136 * 128, SLAB1 = 2 * HALF1, SLAB2 = 144 * 128;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full[S], bar_empty[S], bar_b, bar_acc1_full, bar_acc1_empty, bar_acc2_full, bar_acc2_empty, bar_slab2;
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(16) float bias_s[128];
    uint8_t *smem_gen = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t smem_w2 = tc::smem_u32(smem_gen), smem_w3 = smem_w2 + W2_BYTES, smem_s1 = smem_w3 + W3_BYTES, smem_s2 = smem_s1 + S * SLAB1;
    uint8_t *slab2_gen = smem_gen + W2_BYTES + W3_BYTES + S * SLAB1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    static_assert(SLAB2 % 1024 == 0 && SLAB1 % 1024 == 0, "swizzle atoms are 1024-byte aligned");

    if (threadIdx.x == 0) {
        tc::tma_prefetch_desc(&mapP2); tc::tma_prefetch_desc(&mapW2); tc::tma_prefetch_desc(&mapW3);
        for (int s = 0; s < S; s++) { tc::mbar_init(tc::smem_u32(&bar_full[s]), 1); tc::mbar_init(tc::smem_u32(&bar_empty[s]), 1); }
        tc::mbar_init(tc::smem_u32(&bar_b), 1);
        tc::mbar_init(tc::smem_u32(&bar_acc1_full), 1); tc::mbar_init(tc::smem_u32(&bar_acc1_empty), 4);
        tc::mbar_init(tc::smem_u32(&bar_acc2_full), 1); tc::mbar_init(tc::smem_u32(&bar_acc2_empty), 4);
        tc::mbar_init(tc::smem_u32(&bar_slab2), 4);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tc::smem_u32(&tmem_slot), 128);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_slot, acc1 = tmem, acc2 = tmem + 64;
    if (threadIdx.x == 0) {
        tc::mbar_expect_tx(tc::smem_u32(&bar_b), W2_BYTES + W3_BYTES);
        for (int kb = 0; kb < 8; kb++) tc::tma_load_2d(smem_w2 + kb * (64 * 128), &mapW2, kb * 64, 0, tc::smem_u32(&bar_b));
        for (int kb = 0; kb < 9; kb++) tc::tma_load_2d(smem_w3 + kb * (64 * 128), &mapW3, kb * 64, 0, tc::smem_u32(&bar_b));
    }
    if (threadIdx.x >= 64) bias_s[threadIdx.x - 64] = threadIdx.x < 128 ? g.bias2[threadIdx.x - 64] : g.bias3[threadIdx.x - 128];
    tc::pdl_wait();
    tc::pdl_launch();
    __syncthreads();

    if (warp == 0) {
        const bool leader = tc::elect_one();
        int i = 0;
        for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, i++) {
            const int s = i % S;
            tc::mbar_wait(tc::smem_u32(&bar_empty[s]), ((i / S) & 1) ^ 1u);
            if (leader) {
                const uint32_t full = tc::smem_u32(&bar_full[s]);
                tc::mbar_expect_tx(full, SLAB1);
                tc::tma_load_2d(smem_s1 + s * SLAB1, &mapP2, 0, tile * kBwdRows, full);
                tc::tma_load_2d(smem_s1 + s * SLAB1 + HALF1, &mapP2, 64, tile * kBwdRows, full);
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        const bool leader = tc::elect_one();
        const uint32_t idesc = tc::instr_desc_16(128, 64, 0, 0, g.f16);
        constexpr uint32_t dhi = tc::smem_desc_hi(1024, tc::kSwizzle128);
        const uint32_t w2_lo = tc::smem_desc_lo(smem_w2, 16), w3_lo = tc::smem_desc_lo(smem_w3, 16);
        const uint32_t s1_lo = tc::smem_desc_lo(smem_s1, 16), s2_lo = tc::smem_desc_lo(smem_s2, 16);
        tc::mbar_wait(tc::smem_u32(&bar_b), 0);
        int i = 0;
        for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, i++) {
            const int s = i % S;
            // ---- GEMM 1 (conv2): K-block kb = (tap, column half): rows p + (tap >> 1) 7 + (tap & 1), channels 64 half ..
            tc::mbar_wait(tc::smem_u32(&bar_acc1_empty), (i & 1) ^ 1u);
            tc::mbar_wait(tc::smem_u32(&bar_full[s]), (i / S) & 1);
            tc::tc_fence_after();
            if (leader) {
#pragma unroll
                for (int kb = 0; kb < 8; kb++) {
                    const int tp = kb >> 1;
                    const uint32_t a_rel = (uint32_t)((kb & 1) * (int)HALF1 + ((tp >> 1) * kG2 + (tp & 1)) * 128) >> 4;
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        tc::umma_bf16_lohi(acc1, s1_lo + s * (SLAB1 >> 4) + a_rel + 2 * k, dhi, w2_lo + ((kb * 64 * 128 + k * 32) >> 4), dhi, idesc, (kb | k) != 0);
                }
                tc::umma_commit(tc::smem_u32(&bar_empty[s]));
                tc::umma_commit(tc::smem_u32(&bar_acc1_full));
            }
            __syncwarp();
            // ---- GEMM 2 (conv3): tap (kh,kw) reads slab-2 rows p + 8 + (kh-1) 7 + (kw-1) = p + kh 7 + kw
            tc::mbar_wait(tc::smem_u32(&bar_slab2), i & 1);
            tc::mbar_wait(tc::smem_u32(&bar_acc2_empty), (i & 1) ^ 1u);
            tc::tc_fence_after();
            if (leader) {
#pragma unroll
                for (int kb = 0; kb < 9; kb++) {
                    const uint32_t tap = (uint32_t)(((kb / 3) * kG2 + (kb % 3)) * 128) >> 4;
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        tc::umma_bf16_lohi(acc2, s2_lo + tap + 2 * k, dhi, w3_lo + ((kb * 64 * 128 + k * 32) >> 4), dhi, idesc, (kb | k) != 0);
                }
                tc::umma_commit(tc::smem_u32(&bar_acc2_full));
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3, r = q * 32 + lane;
        if (r < 8) {
#pragma unroll
            for (int c = 0; c < 8; c++) *reinterpret_cast<uint4 *>(slab2_gen + r * 128 + c * 16) = make_uint4(0, 0, 0, 0);
        }
        int i = 0;
        for (int tile = blockIdx.x; tile < g.n_tiles; tile += gridDim.x, i++) {
            const long long grow = (long long)tile * kBwdRows + r;
            const bool in_tile = r < kBwdRows && grow < (long long)g.B * kP2;
            const int p = r % kP2, oh = p / kG2, ow = p - oh * kG2;
            const int b = (int)(tile * 2 + (r >= kP2 ? 1 : 0));
            const bool ok = in_tile && oh < 5 && ow < 5;
            // ---- epilogue 1: A2 = relu(conv2 + b2), zeros at invalid positions
            tc::mbar_wait(tc::smem_u32(&bar_acc1_full), i & 1);
            tc::tc_fence_after();
            float v[64];
            tc::tmem_ld32(acc1 + ((uint32_t)(q * 32) << 16), *reinterpret_cast<float(*)[32]>(&v[0]));
            tc::tmem_ld32(acc1 + ((uint32_t)(q * 32) << 16) + 32, *reinterpret_cast<float(*)[32]>(&v[32]));
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bar_acc1_empty));
            const float keep = ok ? 1.f : 0.f;
            uint4 outw[8];
#pragma unroll
            for (int c = 0; c < 8; c++) {
                const float4 b0 = reinterpret_cast<const float4 *>(bias_s)[2 * c], b1 = reinterpret_cast<const float4 *>(bias_s)[2 * c + 1];
                const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                uint32_t w[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    w[k] = tc::pack2(fmaxf(v[c * 8 + 2 * k] + bb[2 * k], 0.f) * keep, fmaxf(v[c * 8 + 2 * k + 1] + bb[2 * k + 1], 0.f) * keep, g.f16);
                }
                outw[c] = make_uint4(w[0], w[1], w[2], w[3]);
            }
            if (in_tile && g.a2 != nullptr) {
                uint4 *d = reinterpret_cast<uint4 *>(g.a2 + grow * 64);
#pragma unroll
                for (int c = 0; c < 8; c += 2) tc::st_global_256(d + c, outw[c], outw[c + 1]);
            }
            {
                const int R = r + 8;
                uint8_t *rowp = slab2_gen + R * 128;
#pragma unroll
                for (int c = 0; c < 8; c++) *reinterpret_cast<uint4 *>(rowp + ((c ^ (R & 7)) << 4)) = outw[c];
            }
            tc::fence_proxy_async();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bar_slab2));
            // ---- epilogue 2: A3 = relu(conv3 + b3), dense [B][25][64]
            tc::mbar_wait(tc::smem_u32(&bar_acc2_full), i & 1);
            tc::tc_fence_after();
            tc::tmem_ld32(acc2 + ((uint32_t)(q * 32) << 16), *reinterpret_cast<float(*)[32]>(&v[0]));
            tc::tmem_ld32(acc2 + ((uint32_t)(q * 32) << 16) + 32, *reinterpret_cast<float(*)[32]>(&v[32]));
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(tc::smem_u32(&bar_acc2_empty));
            float b3[64];
#pragma unroll
            for (int c = 0; c < 16; c++) {
                const float4 t4 = reinterpret_cast<const float4 *>(bias_s + 64)[c];
                b3[4 * c] = t4.x; b3[4 * c + 1] = t4.y; b3[4 * c + 2] = t4.z; b3[4 * c + 3] = t4.w;
            }
            if (ok) {
                uint4 *d = reinterpret_cast<uint4 *>(g.a3 + ((size_t)b * 25 + oh * 5 + ow) * 64);
#pragma unroll
                for (int c = 0; c < 8; c += 2) {
                    uint32_t w[8];
#pragma unroll
                    for (int k = 0; k < 8; k++) {
                        w[k] = tc::pack2(fmaxf(v[c * 8 + 2 * k] + b3[c * 8 + 2 * k], 0.f), fmaxf(v[c * 8 + 2 * k + 1] + b3[c * 8 + 2 * k + 1], 0.f), g.f16);
                    }
                    tc::st_global_256(d + c, make_uint4(w[0], w[1], w[2], w[3]), make_uint4(w[4], w[5], w[6], w[7]));
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) tc::tmem_dealloc(tmem, 128);
}

template <int S>
static cudaError_t launch_tc_fwd23(const CUtensorMap &mp2, const CUtensorMap &mw2, const CUtensorMap &mw3, const Fwd23Params &g, int max_ctas,
                                   cudaStream_t st) {
    static bool configured = false;
    auto kern = tc_fwd23_kernel<S>;
    constexpr size_t smem = 8 * 64 * 128 + 9 * 64 * 128 + (size_t)S * 2 * 136 * 128 + 144 * 128 + 1024;
    static_assert(smem <= 227 * 1024 && smem > kExclusiveSmem, "shared memory budget");
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    const int grid = g.n_tiles < max_ctas ? g.n_tiles : max_ctas;
    return tc::launch_pdl(kern, dim3(grid), dim3(kConvThreads), smem, st, mp2, mw2, mw3, g);
}

// ------------------------------------------------------------------------------------------------ TMA maps
PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;

int ensure_encode() {
    if (g_encode) return FB_OK;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    FB_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    FB_REQUIRE(fn != nullptr && qres == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled is not available from this driver");
    g_encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
    return FB_OK;
}

// bf16 matrix [rows][cols] row-major, box [box_rows][box_cols]; swizzle 128B (64B when the box is 32 columns wide)
int make_map(CUtensorMap *m, const bf16 *base, long long rows, long long cols, int box_cols, int box_rows) {
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUtensorMapSwizzle sw = box_cols * 2 == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    FB_REQUIRE(box_cols * 2 == 128 || box_cols * 2 == 64, "make_map: box must be 64 or 32 bf16 wide");
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16 *>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { fb_set_error("cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"); return FB_ERR_CUDA; }
    return FB_OK;
}

void set_kmajor(GemmParams &g) { g.kper = kMaxKb; g.lbo_a = 16; g.sbo_a = 1024; g.kstep_a = 32; g.lbo_b = 16; g.sbo_b = 1024; g.kstep_b = 32; }
void set_mnmajor(GemmParams &g, int bn) {
    g.lbo_a = 8192; g.sbo_a = 1024; g.kstep_a = 2048;
    if (bn == 32) { g.lbo_b = 4096; g.sbo_b = 512; g.kstep_b = 1024; }
    else { g.lbo_b = 8192; g.sbo_b = 1024; g.kstep_b = 2048; }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ state
struct TcWeightMaps { CUtensorMap w1p, w2p, w3p, wf1n, w3d, w2d; };
struct FwdWs {                  // forward tensors of one network evaluation (bf16 unless noted), sized for max_batch
    bf16 *x2, *z1, *p2, *a2, *a3;
    float *parth, *h1;          // fc1 K-split partials, h1 (fp32, kept for the head backward)
};
struct TcPlan {                 // everything that depends on the batch size
    int B;
    CUtensorMap x2_s[2], p2_s[2], a2_s[2], a3_k[2];                  // forward operands of workspace 0 / 1
    CUtensorMap dh1_k, dz3_s, dz2_s;                                 // data-gradient operands
    CUtensorMap x2_w, p2_w, a2_w, a3_m;                              // weight-gradient A operands (workspace 0)
    CUtensorMap dz1_b, dz2_b, dz3_b, dh1_b;                          // weight-gradient B operands, 64 rows
    GemmParams fc1, fc1_d, fc1_w;
    ConvParams conv2, conv3, conv3_d, conv2_d;
    WgradParams conv1_w, conv2_w, conv3_w;
    int s1, s2, s3, sf;                                              // split-K counts (conv weight gradients, fc1 forward)
};
struct GraphKey {               // a captured training step is replayed only for byte-identical arguments
    QnetStep a;
    int pack_online, pack_target;
};
struct GraphEntry {
    GraphKey key; int seen; cudaGraphExec_t exec;
    cudaGraph_t graph;                      // kept only while its node handles are needed (the sampling head is patched every step)
    cudaGraphNode_t n_sampler, n_gather;
};
static void destroy_entry(GraphEntry &g) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    if (g.graph) cudaGraphDestroy(g.graph);
    g.exec = nullptr; g.graph = nullptr;
}
// TcState::ev: a training step takes the running slots [0, kEvGather) in order, one per cross-stream edge; the named slots
// after them have fixed uses (the replay gather and the early X2 conversion of a step, the two streams of chunked acting)
constexpr int kEvGather = 12, kEvX2 = 13, kEvChunkIn = 14, kEvChunkOut = 15, kEvSlots = 16;
struct TcState {
    FwdWs ws[2];                // 0: the online net on s (kept for backward); 1: the other forwards, concurrently
    bf16 *dh1, *dz3, *dz2, *dp2, *dz1;
    float *part1, *part2, *part3;
    size_t cap1, cap2, cap3;
    float *bp1, *bp2, *bp3;
    float *hp, *hb;             // head-backward partials per row group
    float *loss_terms;          // per-sample loss terms
    float *adam_pow;            // device: beta1^t, beta2^t of the fused Adam (fb_qnet_step), then this step's alpha
    float pow_host[2];          // what adam_pow will hold once everything enqueued so far has run
    float *pow_pinned;          // 16 x 2 staging slots for re-seeding adam_pow
    int pow_slot;
    PackedWeights pw[2];
    TcWeightMaps wm[2];
    std::map<int, TcPlan> plans;
    int n_sms;
    cudaStream_t aux;           // second stream: target forward / weight gradients run beside the critical path
    cudaStream_t aux2;          // third stream: bias column sums and the early Adam on W_fc1
    cudaStream_t aux4;          // fifth stream: Memory.batch_update (prioritized replay) beside the whole backward pass
    cudaStream_t aux3;          // fourth stream (several GPUs): W_fc1's bucket of the gradient exchange, joined only at the step's end
    cudaStream_t cap;           // capture origin (the caller's stream may be the legacy default stream, which cannot capture)
    cudaEvent_t ev[kEvSlots];
    std::vector<GraphEntry> graphs;
    int use_graph;
    int f16;                    // operand format of every 16-bit tensor of this net: 0 bf16, 1 fp16 (FB_PRECISION_FP16)
    int separate_kernels;       // test hook (fb_debug_tc_separate_kernels): no fused conv2+conv3 forward / conv3-conv2 backward at any batch
    FrameView probe_view;       // frames of this net's last forward (fb_debug_tc_kernel's conv1 probes re-read them)
};

namespace {

constexpr int kChunk1 = 1024, kChunk23 = 256;
constexpr int kFc1Splits = 5;                    // fc1 forward: 25 K-blocks in 5 K-splits of 5
// The fused conv2+conv3 forward / conv3+conv2+un-pool backward kernels (two samples = 98 of 128 accumulator rows per tile, the
// layers of a tile chained inside one CTA) cut launches at minibatch sizes; measured at 4,096 samples they LOSE to the separate,
// fully pipelined kernels (bwd 172 us against 125 us; whole update 721 against 607 us): above this batch the separate kernels run.
constexpr int kFuseMaxBatch = 512;
// the fused head kernel (fc1_head_train_kernel<16>) serves the reference's hidden width; other widths keep the two-kernel form
bool fused_head_ok(const NetLayout &L) { return L.hidden == 512 && L.atoms == 0; }
int head_ctas(const TcState *t, int B) { const int c = (B + 3) / 4, m = t->n_sms < kMaxHeadCtas ? t->n_sms : kMaxHeadCtas; return c < m ? c : m; }

// slab geometry (rows of 128 bytes): tile or K-block rows + the largest tap offset, rounded up to 8
constexpr int kSlab1 = 152, kSlab2 = 136, kSlab3 = 144;          // forward / data gradient, 128-position tiles
constexpr int kSlabW1 = 88, kSlabW2 = 72, kSlabW3 = 88;          // weight gradient, 64-position K-blocks

int plan_splits(long long P, int target, int *klen_out) {
    if (target < 1) target = 1;
    long long klen = (P + target - 1) / target;
    klen = (klen + 63) / 64 * 64;
    if (klen < 64) klen = 64;
    *klen_out = (int)klen;
    return (int)((P + klen - 1) / klen);
}

int make_plan(fb_qnet *n, int B, TcPlan **out) {
    TcState *t = n->tc;
    auto it = t->plans.find(B);
    if (it != t->plans.end()) { *out = &it->second; return FB_OK; }
    if (t->plans.size() > 16) {                  // plans are referenced by captured graphs: drop both together
        for (auto &g : t->graphs) destroy_entry(g);
        t->graphs.clear();
        t->plans.clear();
    }
    TcPlan p{};
    p.B = B;
    const int H = n->L.hidden;
    const long long P1 = (long long)B * kP1, P2 = (long long)B * kP2;
    int rc;
#define MAP(dst, base, rows, cols, bc, br) if ((rc = make_map(&p.dst, base, rows, cols, bc, br))) return rc
    for (int w = 0; w < 2; w++) {
        MAP(x2_s[w], t->ws[w].x2, P1, 64, 64, kSlab1); MAP(p2_s[w], t->ws[w].p2, P2, 128, 64, kSlab2);
        MAP(a2_s[w], t->ws[w].a2, P2, 64, 64, kSlab3); MAP(a3_k[w], t->ws[w].a3, B, kFlat, 64, 128);
    }
    MAP(dh1_k, t->dh1, B, H, 64, 128); MAP(dz3_s, t->dz3, P2, 64, 64, kSlab3); MAP(dz2_s, t->dz2, P2, 64, 64, kSlab2);
    MAP(x2_w, t->ws[0].x2, P1, 64, 64, kSlabW1); MAP(p2_w, t->ws[0].p2, P2, 128, 64, kSlabW2); MAP(a2_w, t->ws[0].a2, P2, 64, 64, kSlabW3);
    MAP(a3_m, t->ws[0].a3, B, kFlat, 64, 64);
    MAP(dz1_b, t->dz1, P1, 32, 32, 64); MAP(dz2_b, t->dz2, P2, 64, 64, 64); MAP(dz3_b, t->dz3, P2, 64, 64, 64); MAP(dh1_b, t->dh1, B, H, 64, 64);
#undef MAP
    // ---- forward: tap (dh,dw) of K-block kb = row offset inside the slab
    p.conv2.n_tiles = (int)((P2 + 127) / 128); p.conv2.slab_row0 = 0;
    for (int k = 0; k < 8; k++) { int tp = k >> 1; p.conv2.kb_rowoff[k] = (tp >> 1) * kG2 + (tp & 1); p.conv2.kb_half[k] = k & 1; }
    p.conv3.n_tiles = p.conv2.n_tiles; p.conv3.slab_row0 = -8;                  // pad ring = the row before / after: offset -8
    for (int k = 0; k < 9; k++) { p.conv3.kb_rowoff[k] = (k / 3) * kG2 + (k % 3); p.conv3.kb_half[k] = 0; }
    set_kmajor(p.fc1); p.fc1.lbo_b = 8192; p.fc1.sbo_b = 1024; p.fc1.kstep_b = 2048;     // B = W_fc1 as stored (MN-major)
    // K-splits of fc1 forward: 5 of 5 K-blocks fill the GPU at minibatch sizes (2 row tiles x 4 column tiles); from 8 row tiles
    // up fewer, longer splits do (2 at 2,048 samples: 128 CTAs of 13 K-blocks, 2/5 of the partial-sum traffic)
    {
        const int mt = (B + 127) / 128, ct = H / 128;
        int sf = kFc1Splits;
        while (sf > 1 && mt * ct * (sf - 1) >= 128) sf--;
        p.sf = sf; p.fc1.nkb = 25; p.fc1.kper = (25 + sf - 1) / sf;
    }
    for (int k = 0; k < 25; k++) { p.fc1.a_rowoff[k] = 0; p.fc1.a_col[k] = k * 64; }
    // ---- data gradients
    set_kmajor(p.fc1_d); p.fc1_d.nkb = H / 64;
    FB_REQUIRE(H / 64 <= kMaxKb, "tensor-core path: hidden must be <= 2048");
    for (int k = 0; k < H / 64; k++) { p.fc1_d.a_rowoff[k] = 0; p.fc1_d.a_col[k] = k * 64; }
    p.conv3_d.n_tiles = p.conv2.n_tiles; p.conv3_d.slab_row0 = -8;              // dz3 row p + (1-kh)*7 + (1-kw)
    for (int k = 0; k < 9; k++) { p.conv3_d.kb_rowoff[k] = (1 - k / 3) * kG2 + (1 - k % 3) + 8; p.conv3_d.kb_half[k] = 0; }
    p.conv2_d.n_tiles = p.conv2.n_tiles; p.conv2_d.slab_row0 = -8;              // dz2 row p - dh*7 - dw
    for (int k = 0; k < 4; k++) { p.conv2_d.kb_rowoff[k] = 8 - (k >> 1) * kG2 - (k & 1); p.conv2_d.kb_half[k] = 0; }
    // ---- weight gradients (contract over positions; accumulator = two taps, or the two column halves of P2)
    p.conv1_w.p_total = (int)P1; p.conv1_w.slab_row0 = 0;
    // split-K: about 24 (conv1) / 4 (conv2, conv3) K-blocks of 64 positions per CTA, one wave of CTAs at most
    auto splits_for = [](long long P, int kb_per_cta) { long long s = (P / 64 + kb_per_cta - 1) / kb_per_cta; return (int)(s < 1 ? 1 : s > 148 ? 148 : s); };
    // conv1: <= 24 K-blocks per CTA once that still gives 64 CTAs (74 at minibatch 256: it runs beside the conv2 / conv3 weight
    // gradients, 49 CTAs each, and every one of these CTAs owns an SM -- 147 + 49 + 49 queued for 148), else <= 8 per CTA
    { int s24 = splits_for(P1, 24), s8 = splits_for(P1, 8);
      p.s1 = plan_splits(P1, s24 >= 64 ? s24 : (s8 < 64 ? s8 : 64), &p.conv1_w.klen); }
    p.conv1_w.acc_rowoff[0] = 0; p.conv1_w.acc_lbo[0] = 128; p.conv1_w.acc_rowoff[1] = kG1; p.conv1_w.acc_lbo[1] = 128;
    p.conv2_w.p_total = (int)P2; p.conv2_w.slab_row0 = 0;
    p.s2 = plan_splits(P2, splits_for(P2, 4), &p.conv2_w.klen);
    for (int a = 0; a < 4; a++) { p.conv2_w.acc_rowoff[a] = (a >> 1) * kG2 + (a & 1); p.conv2_w.acc_lbo[a] = 0; }
    p.conv3_w.p_total = (int)P2; p.conv3_w.slab_row0 = -8;
    p.s3 = plan_splits(P2, splits_for(P2, 4), &p.conv3_w.klen);
    {   // taps 0..8 at rows {0,1,2,7,8,9,14,15,16}; pairs (0,1) (2,3) (4,5) (6,7) (8,-): second atom LBO bytes further
        const int off[5] = {0, 2, 8, 14, 16};
        const uint32_t lbo[5] = {128, 5 * 128, 128, 128, 128};
        for (int a = 0; a < 5; a++) { p.conv3_w.acc_rowoff[a] = off[a]; p.conv3_w.acc_lbo[a] = lbo[a]; }
    }
    set_mnmajor(p.fc1_w, 128); p.fc1_w.p_total = B; p.fc1_w.klen = (B + 63) / 64 * 64;
    for (int mt = 0; mt < 13; mt++) for (int i = 0; i < 2; i++) { p.fc1_w.a2_rowoff[mt][i] = 0; p.fc1_w.a2_col[mt][i] = mt * 128 + i * 64; }
    FB_REQUIRE((size_t)p.s1 <= t->cap1 && (size_t)p.s2 <= t->cap2 && (size_t)p.s3 <= t->cap3, "tensor-core path: split-K workspace too small");
    p.conv2.f16 = p.conv3.f16 = p.conv3_d.f16 = p.conv2_d.f16 = t->f16;
    p.conv1_w.f16 = p.conv2_w.f16 = p.conv3_w.f16 = t->f16;
    p.fc1.f16 = p.fc1_d.f16 = p.fc1_w.f16 = t->f16;
    auto res = t->plans.emplace(B, p);
    *out = &res.first->second;
    return FB_OK;
}

}  // namespace

int tc_state_create(fb_qnet *n) {
    if (n->tc) return FB_OK;
    FB_REQUIRE(n->L.hidden % 128 == 0 && n->L.hidden <= 2048, "tensor-core path needs hidden % 128 == 0 and hidden <= 2048");
    int rc = ensure_encode();
    if (rc) return rc;
    TcState *t = new (std::nothrow) TcState();
    FB_REQUIRE(t != nullptr, "tc_state_create: out of host memory");
    const size_t B = (size_t)n->max_batch, H = (size_t)n->L.hidden;
    auto alloc_bf = [](bf16 **p, size_t elems) {
        cudaError_t e = cudaMalloc(p, elems * sizeof(bf16));
        if (e == cudaSuccess) e = cudaMemset(*p, 0, elems * sizeof(bf16));
        return e;
    };
    auto alloc_f = [](float **p, size_t elems) {
        cudaError_t e = cudaMalloc(p, elems * sizeof(float));
        if (e == cudaSuccess) e = cudaMemset(*p, 0, elems * sizeof(float));
        return e;
    };
    for (int w = 0; w < 2; w++) {
        FwdWs &f = t->ws[w];
        FB_CUDA_OK(alloc_bf(&f.x2, B * kP1 * 64)); FB_CUDA_OK(alloc_bf(&f.z1, B * kP1 * 32)); FB_CUDA_OK(alloc_bf(&f.p2, B * kP2 * 128));
        FB_CUDA_OK(alloc_bf(&f.a2, B * kP2 * 64)); FB_CUDA_OK(alloc_bf(&f.a3, B * kFlat));
        FB_CUDA_OK(alloc_f(&f.parth, (size_t)kFc1Splits * B * H)); FB_CUDA_OK(alloc_f(&f.h1, B * H));
    }
    FB_CUDA_OK(alloc_bf(&t->dh1, B * H));
    FB_CUDA_OK(alloc_bf(&t->dz3, B * kP2 * 64)); FB_CUDA_OK(alloc_bf(&t->dz2, B * kP2 * 64)); FB_CUDA_OK(alloc_bf(&t->dp2, B * kP2 * 128));
    FB_CUDA_OK(alloc_bf(&t->dz1, B * kP1 * 32));
    t->cap1 = 150; t->cap2 = 150; t->cap3 = 150;              // plan_splits never exceeds its target
    FB_CUDA_OK(alloc_f(&t->part1, t->cap1 * 256 * 32)); FB_CUDA_OK(alloc_f(&t->part2, t->cap2 * 512 * 64));
    FB_CUDA_OK(alloc_f(&t->part3, t->cap3 * 640 * 64));
    FB_CUDA_OK(alloc_f(&t->bp1, ((B * kP1 + kChunk1 - 1) / kChunk1) * 32)); FB_CUDA_OK(alloc_f(&t->bp2, ((B * kP2 + kChunk23 - 1) / kChunk23) * 64));
    FB_CUDA_OK(alloc_f(&t->bp3, ((B * kP2 + kChunk23 - 1) / kChunk23) * 64));
    {   // head partials: one per row group (head_backward_tc_kernel) or per CTA of the fused head kernel (at most kMaxHeadCtas)
        const size_t G = (B + kHeadRows - 1) / kHeadRows > (size_t)kMaxHeadCtas ? (B + kHeadRows - 1) / kHeadRows : (size_t)kMaxHeadCtas;
        FB_CUDA_OK(alloc_f(&t->hp, G * H * 4)); FB_CUDA_OK(alloc_f(&t->hb, G * 4 + 4));
    }
    FB_CUDA_OK(alloc_f(&t->loss_terms, B));
    FB_CUDA_OK(alloc_f(&t->adam_pow, 4));
    FB_CUDA_OK(cudaMallocHost(&t->pow_pinned, 32 * sizeof(float)));
    t->pow_host[0] = t->pow_host[1] = -1.f; t->pow_slot = 0;
    for (int s = 0; s < 2; s++) {
        PackedWeights &w = t->pw[s];
        FB_CUDA_OK(alloc_bf(&w.w1p, kC1 * kK1)); FB_CUDA_OK(alloc_bf(&w.w2p, kC2 * kK2)); FB_CUDA_OK(alloc_bf(&w.w3p, kC3 * kK3));
        FB_CUDA_OK(alloc_bf(&w.wf1n, kFlat * H)); FB_CUDA_OK(alloc_bf(&w.w3d, kC3 * kK3));
        FB_CUDA_OK(alloc_bf(&w.w2d, 128 * 256));
        TcWeightMaps &m = t->wm[s];
        if ((rc = make_map(&m.w1p, w.w1p, kC1, kK1, 64, 32))) return rc;
        if ((rc = make_map(&m.w2p, w.w2p, kC2, kK2, 64, 64))) return rc;
        if ((rc = make_map(&m.w3p, w.w3p, kC3, kK3, 64, 64))) return rc;
        if ((rc = make_map(&m.wf1n, w.wf1n, kFlat, (long long)H, 64, 64))) return rc;
        if ((rc = make_map(&m.w3d, w.w3d, kC3, kK3, 64, 64))) return rc;
        if ((rc = make_map(&m.w2d, w.w2d, 128, 256, 64, 128))) return rc;
    }
    int dev = 0;
    FB_CUDA_OK(cudaGetDevice(&dev));
    FB_CUDA_OK(cudaDeviceGetAttribute(&t->n_sms, cudaDevAttrMultiProcessorCount, dev));
    {   // the side streams run at the LOWEST priority, the capture origin at the highest: when a critical-path kernel and a side
        // kernel are ready together the block scheduler places the critical one first (measured: the Q(s') conv1, 576 threads
        // and the whole register file per SM, held up the 256-thread X2 conversion of the Q(s) path by 7.6 us)
        int lo = 0, hi = 0;
        FB_CUDA_OK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        FB_CUDA_OK(cudaStreamCreateWithPriority(&t->aux, cudaStreamNonBlocking, lo));
        FB_CUDA_OK(cudaStreamCreateWithPriority(&t->aux2, cudaStreamNonBlocking, hi));     // short kernels finalize waits for
        FB_CUDA_OK(cudaStreamCreateWithPriority(&t->aux3, cudaStreamNonBlocking, hi));
        FB_CUDA_OK(cudaStreamCreateWithPriority(&t->aux4, cudaStreamNonBlocking, lo));
        FB_CUDA_OK(cudaStreamCreateWithPriority(&t->cap, cudaStreamNonBlocking, hi));
    }
    for (auto &e : t->ev) FB_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    t->use_graph = 1;
    n->tc = t;
    return FB_OK;
}

void tc_state_destroy(fb_qnet *n) {
    TcState *t = n->tc;
    if (!t) return;
    for (auto &g : t->graphs) destroy_entry(g);
    for (int w = 0; w < 2; w++) {
        FwdWs &f = t->ws[w];
        void *fs[] = {f.x2, f.z1, f.p2, f.a2, f.a3, f.parth, f.h1};
        for (void *p : fs) cudaFree(p);
    }
    void *ps[] = {t->dh1, t->dz3, t->dz2, t->dp2, t->dz1, t->part1, t->part2, t->part3, t->bp1, t->bp2, t->bp3, t->hp, t->hb, t->loss_terms,
                  t->adam_pow};
    for (void *p : ps) cudaFree(p);
    if (t->pow_pinned) cudaFreeHost(t->pow_pinned);
    for (int s = 0; s < 2; s++) {
        PackedWeights &w = t->pw[s];
        void *ws[] = {w.w1p, w.w2p, w.w3p, w.wf1n, w.w3d, w.w2d};
        for (void *p : ws) cudaFree(p);
    }
    for (auto &e : t->ev) if (e) cudaEventDestroy(e);
    if (t->aux) cudaStreamDestroy(t->aux);
    if (t->aux2) cudaStreamDestroy(t->aux2);
    if (t->aux3) cudaStreamDestroy(t->aux3);
    if (t->aux4) cudaStreamDestroy(t->aux4);
    if (t->cap) cudaStreamDestroy(t->cap);
    delete t;
    n->tc = nullptr;
}

int tc_pack_weights(fb_qnet *n, const float *params_dev, int slot, cudaStream_t st) {
    FB_REQUIRE(n->tc != nullptr && (slot == 0 || slot == 1), "tc_pack_weights: bad argument");
    FB_CUDA_OK(tc::launch_pdl(pack_weights_kernel, dim3(592), dim3(256), 0, st, params_dev, n->L, n->tc->pw[slot], slot == 1 ? 1 : 0));
    return FB_OK;
}

extern "C" int fb_debug_poison_packed(fb_qnet *n, int slot, void *stream) {
    FB_REQUIRE(n != nullptr && n->tc != nullptr && (slot == 0 || slot == 1), "fb_debug_poison_packed: needs the tensor-core path and slot 0 / 1");
    const PackedWeights &w = n->tc->pw[slot];
    cudaStream_t st = (cudaStream_t)stream;
    const size_t H = (size_t)n->L.hidden;
    FB_CUDA_OK(cudaMemsetAsync(w.w1p, 0xFF, sizeof(bf16) * kC1 * kK1, st)); FB_CUDA_OK(cudaMemsetAsync(w.w2p, 0xFF, sizeof(bf16) * kC2 * kK2, st));
    FB_CUDA_OK(cudaMemsetAsync(w.w3p, 0xFF, sizeof(bf16) * kC3 * kK3, st)); FB_CUDA_OK(cudaMemsetAsync(w.wf1n, 0xFF, sizeof(bf16) * kFlat * H, st));
    FB_CUDA_OK(cudaMemsetAsync(w.w3d, 0xFF, sizeof(bf16) * kC3 * kK3, st)); FB_CUDA_OK(cudaMemsetAsync(w.w2d, 0xFF, sizeof(bf16) * 128 * 256, st));
    return FB_OK;
}

bool tc_online_operands(fb_qnet *n, PackedWeights *out) {
    if (!n || !tc_precision(n->precision) || !n->tc) return false;
    *out = n->tc->pw[0];
    return true;
}

int tc_adam(fb_qnet *n, float *params_dev, const float *grads_dev, float *m_dev, float *v_dev, float alpha, float beta1, float beta2,
            float eps, float grad_scale, cudaStream_t st) {
    FB_REQUIRE(n->tc != nullptr, "tc_adam: no tensor-core state");
    const int cnt = n->L.total;
    adam_pack_kernel<<<(cnt + 255) / 256, 256, 0, st>>>(params_dev, grads_dev, m_dev, v_dev, cnt, alpha, beta1, beta2, eps, grad_scale, n->L,
                                                        n->tc->pw[0]);
    FB_CUDA_OK(cudaGetLastError());
    if (n->packed_src[1] == params_dev) n->packed_src[1] = nullptr;
    n->packed_src[0] = params_dev;          // slot 0 now mirrors the updated vector
    return FB_OK;
}

// which bf16 operand copy serves params_dev (want_slot < 0: whichever already holds it, else slot 0), refreshed if stale
int tc_slot_for(fb_qnet *n, const float *params_dev, int want_slot, cudaStream_t st, int *slot_out) {
    int slot = want_slot;
    if (slot < 0) slot = (n->packed_src[1] == params_dev && n->packed_src[0] != params_dev) ? 1 : 0;
    if (n->packed_src[slot] != params_dev) {
        int rc = tc_pack_weights(n, params_dev, slot, st);
        if (rc) return rc;
        n->packed_src[slot] = params_dev;
    }
    *slot_out = slot;
    return FB_OK;
}

// The training forward on s (train_step_launch): its activations feed the backward pass (Z1, A2, h1 and, for the conv1 weight
// gradient, X2 are kept), and its head kernel also forms the TD target / loss -- after waiting for `join`, the end of the Q(s')
// forward on the other stream.  nullptr: a forward with no backward pass (acting, Q(s')).
struct TrainFwd {
    TdFuse td;
    cudaEvent_t join;
    AdamPow ap;
    float gscale;               // power of two carried by the gradient tensors (GradFmt)
    bool x2_early;              // conv1 from the u8 frames, X2 packed early by the caller; else X2 is packed here and feeds conv1
};
// probs: a C51 net's p [B][2][N] (may be nullptr; the training forward keeps p and log p of s in the net's own buffers)
static int run_forward(fb_qnet *n, int slot, int w, const float *params_dev, FrameView fv, int B, float *q_out, const TrainFwd *tr,
                       cudaStream_t st, float *probs = nullptr) {
    TcState *t = n->tc;
    FB_REQUIRE(t != nullptr && B > 0 && B <= n->max_batch && (w == 0 || w == 1), "tc_forward: bad argument");
    TcPlan *p;
    int rc = make_plan(n, B, &p);
    if (rc) return rc;
    const NetLayout &L = n->L;
    const TcWeightMaps &wm = t->wm[slot];
    const FwdWs &f = t->ws[w];
    const int P1 = B * kP1, P2 = B * kP2;
    const bool keep = tr != nullptr;
    t->probe_view = fv;
    // conv1 with the 2x2 max-pool in its epilogue (Z1 is written only when a backward pass needs it; no pooling pass), its slab
    // built in the kernel straight from the u8 frames -- except in a training forward without x2_early: there X2 is materialised
    // once (the conv1 weight gradient contracts over it by TMA) and feeds the slab
    const Conv1FusedParams c1{fv, B, params_dev + L.b1, keep ? f.z1 : nullptr, f.p2, t->f16};
    if (keep && !tr->x2_early) {
        FB_CUDA_OK(tc::launch_pdl(pack_x2_kernel, dim3((unsigned)(((size_t)P1 * 8 + 255) / 256)), dim3(256), 0, st, fv, B, f.x2, t->f16));
        FB_CUDA_OK((launch_tc_conv1_fused<6, true>(p->x2_s[w], wm.w1p, c1, t->n_sms, st)));
    } else {
        FB_CUDA_OK((launch_tc_conv1_fused<4, false>(p->x2_s[w], wm.w1p, c1, t->n_sms, st)));
    }
    if (B <= kFuseMaxBatch && !t->separate_kernels) {
        FB_CUDA_OK((launch_tc_fwd23<2>(p->p2_s[w], wm.w2p, wm.w3p, Fwd23Params{(B + 1) / 2, B, params_dev + L.b2, params_dev + L.b3, keep ? f.a2 : nullptr, f.a3, t->f16},
                                       t->n_sms, st)));
    } else {
        FB_CUDA_OK((launch_tc_conv<64, kSlab2, 2, 8, 3, 1>(p->p2_s[w], wm.w2p, p->conv2, t->n_sms, EpiGrid7{f.a2, params_dev + L.b2, P2, t->f16}, st)));
        FB_CUDA_OK((launch_tc_conv<64, kSlab3, 1, 9, 4, 1>(p->a2_s[w], wm.w3p, p->conv3, t->n_sms, EpiConv3{f.a3, params_dev + L.b3, P2, t->f16}, st)));
    }
    FB_CUDA_OK((launch_tc_gemm<128, 2>(p->a3_k[w], wm.wf1n, p->fc1, dim3((B + 127) / 128, L.hidden / 128, p->sf),
                                       EpiStoreF32{f.parth, B, L.hidden, (size_t)n->max_batch * L.hidden}, st)));
    if (keep) FB_CUDA_OK(cudaStreamWaitEvent(st, tr->join, 0));
    if (L.atoms) {                             // C51 / QR head (fb_c51.cu); training: h1, p and log p (QR: theta) of s kept, then the loss
        const size_t sstride = (size_t)n->max_batch * L.hidden;
        rc = c51_launch_head_forward(f.parth, p->sf, sstride, nullptr, params_dev, L, B, keep ? f.h1 : nullptr, keep ? n->c51_ps : probs,
                                     keep ? n->c51_logps : nullptr, q_out, st);
        if (rc || !keep) return rc;
        const TdFuse &td = tr->td;
        if (L.quantile)                        // quantile-Huber loss (fb_qr.cu)
            return qr_launch_loss(L, B, td.variant, td.loss_sum, td.global_batch, td.gamma, n->c51_ps, n->c51_pn, td.q_next, td.q_next_online,
                                  td.actions, td.rewards, td.terminals, td.isw, td.ret, td.disc, n->c51_dl, n->c51_terms, td.abs_err, td.q_target, st);
        return c51_launch_loss(L, B, td.variant, td.loss_sum, td.global_batch, td.gamma, n->c51_ps, n->c51_logps, n->c51_pn, td.q_next,
                               td.q_next_online, td.actions, td.rewards, td.terminals, td.isw, td.ret, td.disc, n->c51_dl, n->c51_terms,
                               td.abs_err, td.q_target, st);
    }
    if (keep && fused_head_ok(L))              // training step: head forward + TD loss + head backward in one kernel
        FB_CUDA_OK(tc::launch_pdl(fc1_head_train_kernel<16>, dim3(head_ctas(t, B)), dim3(128), 0, st, f.parth, p->sf,
                                  (size_t)n->max_batch * L.hidden, params_dev, L, B, q_out, tr->td, HeadBwd{t->dh1, t->hp, t->hb, GradFmt{t->f16, tr->gscale}},
                                  tr->ap));
    else if (!keep && fused_head_ok(L)) {
        const int ctas = (B + 3) / 4 < 4 * t->n_sms ? (B + 3) / 4 : 4 * t->n_sms;
        FB_CUDA_OK(tc::launch_pdl(fc1_head_warp_kernel<16>, dim3(ctas), dim3(128), 0, st, f.parth, p->sf, (size_t)n->max_batch * L.hidden,
                                  params_dev, L, B, (float *)nullptr, q_out));
    } else
        FB_CUDA_OK(tc::launch_pdl(fc1_head_kernel, dim3(B), dim3(128), 0, st, f.parth, p->sf, (size_t)n->max_batch * L.hidden, params_dev, L, B,
                                  keep ? f.h1 : nullptr, q_out, keep ? tr->td : TdFuse{}));
    return FB_OK;
}
int tc_forward(fb_qnet *n, int slot, int w, const float *params_dev, FrameView fv, int B, float *q_out, cudaStream_t st, float *probs) {
    return run_forward(n, slot, w, params_dev, fv, B, q_out, nullptr, st, probs);
}

// Acting over more samples than one workspace holds: chunks alternate between the two forward workspaces and the two
// streams, so one chunk's latency chain (seven kernels) overlaps the other's.
int tc_forward_chunks(fb_qnet *n, int slot, const float *params_dev, const uint8_t *frames_dev, long long sample_stride,
                      const int32_t *chan_off, int batch, float *q_out_dev, cudaStream_t st, float *probs_dev) {
    TcState *t = n->tc;
    FB_REQUIRE(t != nullptr, "tc_forward_chunks: no tensor-core state");
    const int nchunks = (batch + n->max_batch - 1) / n->max_batch;
    const bool two = nchunks > 1;
    if (two) { FB_CUDA_OK(cudaEventRecord(t->ev[kEvChunkIn], st)); FB_CUDA_OK(cudaStreamWaitEvent(t->aux, t->ev[kEvChunkIn], 0)); }
    int c = 0;
    for (int b0 = 0; b0 < batch; b0 += n->max_batch, c++) {
        const int B = min(n->max_batch, batch - b0), w = two ? (c & 1) : 0;
        FrameView fv;
        fv.base = frames_dev + (size_t)b0 * sample_stride; fv.sample_stride = sample_stride; fv.tab = nullptr; fv.tab_stride = 0;
        for (int k = 0; k < 4; k++) fv.chan_off[k] = chan_off[k];
        int rc = tc_forward(n, slot, w, params_dev, fv, B, q_out_dev + (size_t)b0 * 2, w ? t->aux : st,
                            probs_dev ? probs_dev + (size_t)b0 * 2 * n->L.atoms : nullptr);
        if (rc) return rc;
    }
    if (two) { FB_CUDA_OK(cudaEventRecord(t->ev[kEvChunkOut], t->aux)); FB_CUDA_OK(cudaStreamWaitEvent(st, t->ev[kEvChunkOut], 0)); }
    return FB_OK;
}

namespace {

// One training step's device work (BrainDQN.py:195-223 and the variants).  Two streams: the critical path
// (online forward on s -> TD loss -> data gradients -> conv1 weight gradient -> finalize) stays on `st`; the Q(s')
// forward(s) and the other weight gradients run beside it on the auxiliary stream.  The same code is what a CUDA
// graph captures.
int train_step_launch(fb_qnet *n, const QnetStep &a, int pack_online, int pack_target, cudaStream_t st) {
    TcState *t = n->tc;
    TcPlan *p;
    int rc = make_plan(n, a.B, &p);
    if (rc) return rc;
    const NetLayout &L = n->L;
    const TcWeightMaps &wm = t->wm[0];
    const FwdWs &f = t->ws[0];
    const int B = a.B, H = L.hidden, P1 = B * kP1, P2 = B * kP2;
    cudaStream_t sx = t->aux;
    int e = 0;                                  // next running event slot
    auto record = [&](cudaStream_t on, cudaEvent_t *ev) -> int {            // the next running slot, recorded on `on`
        FB_REQUIRE(e < kEvGather, "train_step_launch: out of running event slots (the next one is the replay gather's)");
        *ev = t->ev[e++];
        FB_CUDA_OK(cudaEventRecord(*ev, on));
        return FB_OK;
    };
    auto fork = [&](cudaStream_t from, cudaStream_t to, cudaEvent_t *ev_out = nullptr) -> int {   // `to` waits for everything issued on `from`
        cudaEvent_t ev;
        int r = record(from, &ev);
        if (r) return r;
        FB_CUDA_OK(cudaStreamWaitEvent(to, ev, 0));
        if (ev_out) *ev_out = ev;
        return FB_OK;
    };
    // the minibatch itself.  The sampler leaves the ring offsets of the drawn frames behind (a.fs.tab): the convolutions read the
    // frames in place, and the gather into the caller-visible minibatch buffers (frames, actions, rewards, terminals -- the head
    // kernel needs the last three) runs on a side stream beside the forward passes: one dependent stage less (5.5 us)
    const bool sampled = a.pro.replay != nullptr;
    if (sampled) {
        rc = replay_launch_sample(a.pro, true, st); if (rc) return rc;
        FB_CUDA_OK(cudaEventRecord(t->ev[kEvGather], st));
        FB_CUDA_OK(cudaStreamWaitEvent(t->aux4, t->ev[kEvGather], 0));
        rc = replay_launch_gather(a.pro, a.gamma, t->aux4); if (rc) return rc;
        FB_CUDA_OK(cudaEventRecord(t->ev[kEvGather], t->aux4));
    }
    if (pack_online) { rc = tc_pack_weights(n, a.params, 0, st); if (rc) return rc; }
    if ((rc = fork(st, sx))) return rc;
    // ---- aux: Q(s') with the net the variant names (and the online net too for Double)
    if (a.variant != 0 && pack_target) { rc = tc_pack_weights(n, a.target, 1, sx); if (rc) return rc; }
    if (a.variant == 2) { rc = tc_forward(n, 0, 1, a.params, a.fn, B, n->q_next_online, sx); if (rc) return rc; }
    rc = a.variant == 0 ? tc_forward(n, 0, 1, a.params, a.fn, B, n->q_next, sx, n->c51_pn) : tc_forward(n, 1, 1, a.target, a.fn, B, n->q_next, sx, n->c51_pn);
    if (rc) return rc;
    if (sampled) FB_CUDA_OK(cudaStreamWaitEvent(sx, t->ev[kEvGather], 0));     // the event below then also says: minibatch buffers complete
    // ---- main: Q(s) with the online net; its activations stay in workspace 0 for the backward pass
    // the TD target, loss and dLoss/dQ come out of its head kernel, which first waits for Q(s') from the other stream
    cudaEvent_t q_next_done;
    if ((rc = record(sx, &q_next_done))) return rc;
    // Q(s)'s conv1 from the u8 frames too, X2 packed early on the stream of the replay gather -- up to minibatch 512 when the step
    // draws its own minibatch.  Measured: it wins there (100.9 vs 102.9 us per update at 256) and loses above (1,024: 235 vs
    // 213 us; 4,096: 689 vs 635 us -- the u8 path is bound by shared memory, the X2 path by HBM); on a caller-supplied minibatch
    // no gather runs ahead of the X2 conversion to keep its 3,528 CTAs out of the way of the two conv1 launches (105 vs 98 us)
    const bool x2_early = sampled && B <= kFuseMaxBatch;
    if (x2_early) {                            // X2 of s for the conv1 weight gradient: early, on the stream of the replay gather
        FB_CUDA_OK(cudaEventRecord(t->ev[kEvX2], st));         // (st has seen the sampler; nothing else of this step yet)
        FB_CUDA_OK(cudaStreamWaitEvent(t->aux4, t->ev[kEvX2], 0));
        pack_x2_kernel<<<dim3((unsigned)(((size_t)P1 * 8 + 255) / 256)), dim3(256), 0, t->aux4>>>(a.fs, B, f.x2, t->f16);
        FB_CUDA_OK(cudaGetLastError());
        FB_CUDA_OK(cudaEventRecord(t->ev[kEvX2], t->aux4));
    }
    TrainFwd tr{};
    tr.td = TdFuse{1, a.variant, a.loss_sum, a.global_batch, n->per_broadcast, a.gamma, n->q_next, n->q_next_online, a.rewards, a.isw, a.actions,
                   a.terminals, n->dq, a.abs_err, a.q_target, t->loss_terms, a.ret, a.disc};
    tr.join = q_next_done;
    tr.ap = AdamPow{a.ad.on, t->adam_pow, t->adam_pow + 2, a.ad.lr, a.ad.beta1, a.ad.beta2};
    // fp16 operands: gradient tensors carry a power-of-two factor that keeps them in fp16's normal range (dq ~ err / batch for the
    // mean losses); it is removed exactly where weight / bias gradients are finalised.  bf16: 1.
    float gscale = 1.f;
    if (t->f16) { gscale = 8.f; if (!a.loss_sum) { int gb = a.global_batch > 0 ? a.global_batch : B; while (gscale < 8.f * (float)gb) gscale *= 2.f; } }
    tr.gscale = gscale;
    tr.x2_early = x2_early;
    rc = run_forward(n, 0, 0, a.params, a.fs, B, n->q, &tr, st); if (rc) return rc;
    // Memory.batch_update (BrainPrioritizedReplyDQN.py:316) needs only |TD error|, which the head kernel has just written: it runs on
    // a stream of its own beside the whole backward pass (measured: 26 us at the step's tail otherwise) and joins at the end
    const bool per_on_side = sampled && a.pro.prioritized;
    cudaEvent_t head_done = nullptr;
    if (per_on_side && (rc = record(st, &head_done))) return rc;        // launched below, after the fc1 gradient GEMMs
    // ---- backward.  The head's backward pass rode in the forward's last kernel when hidden = 512 (fc1_head_train_kernel);
    // otherwise: fp32 gradients of the head variables and the fc1 bias straight into partials, dh1 as bf16
    const bool fused_head = fused_head_ok(L);
    const int G = L.atoms ? (B + kC51Rows - 1) / kC51Rows : fused_head ? head_ctas(t, B) : (B + kHeadRows - 1) / kHeadRows;
    if (L.atoms) {                              // C51: dh1 and the head's partials per row group (fb_c51.cu)
        rc = c51_launch_head_backward(L, B, f.h1, n->c51_dl, a.params, n->c51_terms, nullptr, nullptr, nullptr, n->c51_hp, n->c51_hb, t->dh1,
                                      t->f16, gscale, tr.ap, st);
        if (rc) return rc;
    } else if (!fused_head)
        FB_CUDA_OK(tc::launch_pdl(head_backward_tc_kernel, dim3(H / 32 + 1, G), dim3(256), 0, st, f.h1, n->dq, a.params, L, B, t->hp, t->hb,
                                  t->loss_terms, t->dh1, tr.ap, GradFmt{t->f16, gscale}));
    cudaStream_t sy = t->aux2;                  // third stream: bias column sums and the early Adam on W_fc1, all off the critical path
    if ((rc = fork(st, sx))) return rc;
    // fc1: dW = a3^T dh1 (aux, written in place), dz3 = (dh1 Wf1^T) * relu'(a3)
    FB_CUDA_OK((launch_tc_gemm<128, 1>(p->a3_m, p->dh1_b, p->fc1_w, dim3(13, H / 128, 1), EpiStoreF32{a.grads + L.wf1, kFlat, H, 0, 1.f / gscale}, sx)));
    cudaEvent_t fc1w_done;
    if ((rc = record(sx, &fc1w_done))) return rc;                      // W_fc1's gradient is final
    FB_CUDA_OK((launch_tc_gemm<64, 0>(p->dh1_k, wm.wf1n, p->fc1_d, dim3((B + 127) / 128, kFlat / 64, 1), EpiFc1Dgrad{t->dz3, f.a3, B, t->f16}, st)));
    cudaEvent_t fc1d_done;
    if ((rc = fork(st, sx, &fc1d_done))) return rc;
    if (per_on_side) {
        // (captured AFTER the two fc1 GEMMs: its one 1,024-thread CTA fits only on the SMs the fused backward kernel leaves free,
        // and a kernel that cannot be placed held back the launches captured behind it -- the fc1 weight gradient started 5 us late)
        FB_CUDA_OK(cudaStreamWaitEvent(t->aux4, head_done, 0));
        rc = replay_launch_per_update(a.pro, a.abs_err, t->aux4); if (rc) return rc;
    }
    FB_CUDA_OK(cudaStreamWaitEvent(sy, fc1d_done, 0));              // sy: after the fc1 data gradient (dz3 complete, wf1n no longer read)
    const int c1 = (P1 + kChunk1 - 1) / kChunk1, c23 = (P2 + kChunk23 - 1) / kChunk23;
    auto colsum_on = [&](const bf16 *x, float *part, int rows, int N, int chunk_rows, int chunks) -> cudaError_t {
        ColsumJobs cj{};
        cj.njobs = 1; cj.f16 = t->f16;
        cj.j[0] = ColsumJob{x, part, rows, N, chunk_rows, 0};
        colsum_kernel<<<chunks, 256, 0, sy>>>(cj);
        return cudaGetLastError();
    };
    FB_CUDA_OK(colsum_on(t->dz3, t->bp3, P2, 64, kChunk23, c23));
    FB_REQUIRE(a.xch == nullptr || !a.ad.on || a.grads == dist_current_grads(a.xch), "training step with an exchange: gradients must go to its current buffer");
    AdamDev ad{a.ad.on && a.xch == nullptr, const_cast<float *>(a.params), a.ad.m, a.ad.v, a.ad.beta1, a.ad.beta2, a.ad.eps, a.ad.grad_scale, t->adam_pow + 2};
    FB_CUDA_OK((launch_tc_wgrad<64, 5, kSlabW3, 1, 6>(p->a2_w, p->dz3_b, p->conv3_w, p->s3, EpiStoreF32{t->part3, 640, 64, (size_t)640 * 64}, sx)));
    if (a.ad.on) {
        // Adam on W_fc1 (91 % of the parameters) on a stream of its own, as soon as its gradient is final (fc1 weight-gradient GEMM,
        // sx) and its bf16 / fp16 copy has been read for the last time (fc1 data-gradient GEMM): beside everything that is left of
        // the step -- nothing downstream reads W_fc1 or its gradient again; it joins at the step's end.  On several GPUs the same
        // slot holds W_fc1's bucket of the gradient exchange (sum over NVLink peer memory + Adam).
        FB_CUDA_OK(cudaStreamWaitEvent(t->aux3, fc1d_done, 0));
        FB_CUDA_OK(cudaStreamWaitEvent(t->aux3, fc1w_done, 0));
        if (a.xch != nullptr) {
            rc = dist_launch_bucket(a.xch, n, 0, const_cast<float *>(a.params), a.ad.m, a.ad.v, t->adam_pow + 2, a.ad.beta1, a.ad.beta2, a.ad.eps,
                                    a.ad.grad_scale, t->aux3);
            if (rc) return rc;
        } else {
            adam_wf1_kernel<<<4 * t->n_sms, 256, 0, t->aux3>>>(L, a.grads, ad, t->pw[0]);
            FB_CUDA_OK(cudaGetLastError());
        }
    }
    if (B <= kFuseMaxBatch && !t->separate_kernels) {
        // conv3 data gradient + ReLU mask + conv2 data gradient + un-pool in one kernel (tc_bwd23_kernel)
        FB_CUDA_OK((launch_tc_bwd23<2>(p->dz3_s, wm.w3d, wm.w2d, Bwd23Params{(B + 1) / 2, B, f.a2, t->dz2, f.z1, t->dz1, t->f16}, t->n_sms, st)));
        cudaEvent_t dgrad_done;
        if ((rc = fork(st, sx, &dgrad_done))) return rc;
        FB_CUDA_OK(cudaStreamWaitEvent(sy, dgrad_done, 0));             // sx, sy: dz2 and dz1 complete
        FB_CUDA_OK(colsum_on(t->dz1, t->bp1, P1, 32, kChunk1, c1));
        FB_CUDA_OK(colsum_on(t->dz2, t->bp2, P2, 64, kChunk23, c23));
        FB_CUDA_OK((launch_tc_wgrad<64, 4, kSlabW2, 2, 4>(p->p2_w, p->dz2_b, p->conv2_w, p->s2, EpiStoreF32{t->part2, 512, 64, (size_t)512 * 64}, sx)));
    } else {
        FB_CUDA_OK((launch_tc_conv<64, kSlab3, 1, 9, 4, 1>(p->dz3_s, wm.w3d, p->conv3_d, t->n_sms, EpiConv3Dgrad{t->dz2, f.a2, P2, t->f16}, st)));
        cudaEvent_t dgrad_done;
        if ((rc = fork(st, sx, &dgrad_done))) return rc;
        FB_CUDA_OK(cudaStreamWaitEvent(sy, dgrad_done, 0));             // sy: after the conv3 data gradient (dz2 complete)
        FB_CUDA_OK(colsum_on(t->dz2, t->bp2, P2, 64, kChunk23, c23));
        FB_CUDA_OK((launch_tc_wgrad<64, 4, kSlabW2, 2, 4>(p->p2_w, p->dz2_b, p->conv2_w, p->s2, EpiStoreF32{t->part2, 512, 64, (size_t)512 * 64}, sx)));
        FB_CUDA_OK((launch_tc_conv<128, kSlab2, 1, 4, 4, 1>(p->dz2_s, wm.w2d, p->conv2_d, t->n_sms, EpiStoreBf16{t->dp2, P2, 128, t->f16}, st)));
        FB_CUDA_OK(tc::launch_pdl(unpool_relu_kernel_tc, dim3((unsigned)(((size_t)B * 400 + 255) / 256)), dim3(256), 0, st, f.z1, t->dp2, B, t->dz1, t->f16));
        if ((rc = fork(st, sy))) return rc;                             // sy: after the un-pool (dz1 complete)
        FB_CUDA_OK(colsum_on(t->dz1, t->bp1, P1, 32, kChunk1, c1));
    }
    // conv1 weight gradient (no input gradient there); the bias gradients = column sums of the dZ tensors ran beside it
    if (x2_early) FB_CUDA_OK(cudaStreamWaitEvent(st, t->ev[kEvX2], 0));
    // launched plainly up to minibatch 512: launched early, its 147 CTAs sat on SMs waiting for the fused data-gradient kernel while
    // the conv3 weight gradient, which was ready, queued behind them (121 -> 114.5 us per update, measured; the fused backward, the
    // other weight gradients and finalize launched plainly measured slower or equal).  Large minibatches fill the GPU by
    // themselves: early launch pays there.
    tc::pdl_next_launch_plain(B <= kFuseMaxBatch);
    FB_CUDA_OK((launch_tc_wgrad<32, 2, kSlabW1, 1, 6>(p->x2_w, p->dz1_b, p->conv1_w, p->s1, EpiStoreF32{t->part1, 256, 32, (size_t)256 * 32}, st)));
    if ((rc = fork(sx, st))) return rc;
    if ((rc = fork(sy, st))) return rc;
    FinalizeArgs fa{t->part1, t->part2, t->part3, p->s1, p->s2, p->s3, t->bp1, t->bp2, t->bp3, c1, c23, c23, L.atoms ? n->c51_hp : t->hp,
                    L.atoms ? n->c51_hb : t->hb, G, a.loss_out, 1.f / gscale};
    const int n_compact = L.wf1 + (L.total - L.bf1);
    const int nb_fin = (n_compact + 31) / 32;
    FB_CUDA_OK(tc::launch_pdl(L.atoms ? finalize_grads_kernel<true> : finalize_grads_kernel<false>, dim3(nb_fin), dim3(32 * kFinWarps), 0, st, fa,
                              L, a.grads, ad, t->pw[0], L));
    if (a.ad.on && a.xch != nullptr) {          // the rest of the vector (79,522 parameters): the only exchange left at the tail
        rc = dist_launch_bucket(a.xch, n, 1, const_cast<float *>(a.params), a.ad.m, a.ad.v, t->adam_pow + 2, a.ad.beta1, a.ad.beta2, a.ad.eps,
                                a.ad.grad_scale, st);
        if (rc) return rc;
    }
    if (a.ad.on && (rc = fork(t->aux3, st))) return rc;          // W_fc1's Adam / exchange bucket joins here, at the very end
    if (per_on_side && (rc = fork(t->aux4, st))) return rc;      // Memory.batch_update (started right after the head) joins here
    return FB_OK;
}

bool same_key(const GraphKey &x, const GraphKey &y) { return memcmp(&x, &y, sizeof(GraphKey)) == 0; }

}  // namespace

int tc_set_format(fb_qnet *n, int f16) {
    TcState *t = n->tc;
    FB_REQUIRE(t != nullptr, "tc_set_format: no tensor-core state");
    f16 = f16 ? 1 : 0;
    if (t->f16 != f16) {                         // plans carry the format, graphs the plans, the operand copies the encoding
        for (auto &g : t->graphs) destroy_entry(g);
        t->graphs.clear();
        t->plans.clear();
        n->packed_src[0] = n->packed_src[1] = nullptr;
    }
    t->f16 = f16; t->pw[0].f16 = f16; t->pw[1].f16 = f16;
    return FB_OK;
}

int tc_drop_graphs(fb_qnet *n) {
    if (n->tc) { for (auto &g : n->tc->graphs) destroy_entry(g); n->tc->graphs.clear(); }
    return FB_OK;
}

// test hook: the separate conv2 / conv3 forward kernels and the separate conv3 data gradient / conv2 data gradient / un-pool
// kernels at every minibatch, where the fused ones would run -- the reference the fused kernels are held to bit for bit
extern "C" int fb_debug_tc_separate_kernels(fb_qnet *n, int on) {
    FB_REQUIRE(n != nullptr && n->tc != nullptr, "fb_debug_tc_separate_kernels: needs a tensor-core precision");
    n->tc->separate_kernels = on ? 1 : 0;
    return tc_drop_graphs(n);
}

extern "C" int fb_qnet_use_graphs(fb_qnet *n, int enable) {
    FB_REQUIRE(n != nullptr, "fb_qnet_use_graphs: NULL argument");
    if (n->tc) n->tc->use_graph = enable ? 1 : 0;
    return tc_drop_graphs(n);
}

// One training step (fb_qnet_step).  With Adam, beta*_power are the caller's (QNetwork keeps them like TF's beta1_power /
// beta2_power variables); the device copy is re-seeded only when it does not already hold them (first step, load_state_dict, a
// separate fb_qnet_adam in between).
int tc_step(fb_qnet *n, const QnetStep &a, float beta1_power, float beta2_power, cudaStream_t st) {
    TcState *t = n->tc;
    if (a.ad.on) {
        if (t->pow_host[0] != beta1_power || t->pow_host[1] != beta2_power) {
            float *slot = t->pow_pinned + 2 * (t->pow_slot++ & 15);
            slot[0] = beta1_power; slot[1] = beta2_power;
            FB_CUDA_OK(cudaMemcpyAsync(t->adam_pow, slot, 2 * sizeof(float), cudaMemcpyHostToDevice, st));
        }
        t->pow_host[0] = t->pow_host[1] = -1.f;  // unknown unless the step below is enqueued in full
    }
    GraphKey key;
    memset(&key, 0, sizeof(key));
    memcpy(&key.a, &a, sizeof(a));               // every argument, padding included (zero: fb_qnet_step zero-fills `a`) ...
    key.a.pro.t = 0; key.a.pro.beta = 0.0;       // ... but the two that are patched into the sampler / gather nodes every step
    key.pack_online = n->packed_src[0] != a.params;
    key.pack_target = a.variant != 0 && n->packed_src[1] != a.target;
    int rc = FB_OK;
    GraphEntry *ge = nullptr;
    if (t->use_graph) {
        for (auto &g : t->graphs) if (same_key(g.key, key)) { ge = &g; break; }
        if (!ge) {
            if (t->graphs.size() >= 8) { for (auto &g : t->graphs) destroy_entry(g); t->graphs.clear(); }
            t->graphs.push_back(GraphEntry{key, 0, nullptr, nullptr, nullptr, nullptr});
            ge = &t->graphs.back();
        }
    }
    if (ge && ge->exec) {
        if (a.pro.replay != nullptr) { rc = replay_patch_nodes(ge->exec, ge->n_sampler, ge->n_gather, a.pro, a.gamma); if (rc) return rc; }
        FB_CUDA_OK(cudaGraphLaunch(ge->exec, st));
    } else if (ge && ge->seen >= 1) {            // second identical call: capture (everything lazy was initialised by the first)
        cudaGraph_t graph = nullptr;
        FB_CUDA_OK(cudaStreamBeginCapture(t->cap, cudaStreamCaptureModeRelaxed));
        rc = train_step_launch(n, a, key.pack_online, key.pack_target, t->cap);
        cudaError_t ce = cudaStreamEndCapture(t->cap, &graph);
        if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
        FB_CUDA_OK(ce);
        cudaError_t ie = cudaGraphInstantiate(&ge->exec, graph, 0);
        if (ie == cudaSuccess && a.pro.replay != nullptr) {       // remember the two replay nodes: their `t` changes every step
            size_t nn = 0;
            cudaGraphGetNodes(graph, nullptr, &nn);
            std::vector<cudaGraphNode_t> nodes(nn);
            if (nn) cudaGraphGetNodes(graph, nodes.data(), &nn);
            for (size_t i = 0; i < nn; i++) {
                cudaGraphNodeType ty;
                if (cudaGraphNodeGetType(nodes[i], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
                cudaKernelNodeParams kp{};
                if (cudaGraphKernelNodeGetParams(nodes[i], &kp) != cudaSuccess) continue;
                if (replay_is_sampler(kp.func)) ge->n_sampler = nodes[i];
                else if (replay_is_gather(kp.func)) ge->n_gather = nodes[i];
            }
            if (!ge->n_sampler || !ge->n_gather) { cudaGraphExecDestroy(ge->exec); ge->exec = nullptr; ie = cudaErrorUnknown; }
        }
        if (ie == cudaSuccess && a.pro.replay != nullptr) ge->graph = graph;      // its node handles stay in use
        else cudaGraphDestroy(graph);
        FB_CUDA_OK(ie);
        FB_CUDA_OK(cudaGraphLaunch(ge->exec, st));
    } else {
        rc = train_step_launch(n, a, key.pack_online, key.pack_target, st);
        if (rc) return rc;
        if (ge) ge->seen++;
    }
    n->packed_src[0] = a.params;            // (with a fused Adam the kernel has re-packed what it updated)
    if (a.variant != 0) n->packed_src[1] = a.target;
    if (a.ad.on && n->packed_src[1] == a.params) n->packed_src[1] = nullptr;
    if (a.ad.on) { t->pow_host[0] = beta1_power * a.ad.beta1; t->pow_host[1] = beta2_power * a.ad.beta2; }
    return FB_OK;
}

// ------------------------------------------------------------------------------------------------ kernel probe
// Re-launches ONE GEMM kernel of the path `reps` times on whatever the workspaces hold (after a forward / training
// step at the same batch), so that bench.py and ncu can time it in isolation.  which: 1 conv2 forward, 2 conv3 forward,
// 3 fc1 forward, 4 conv1 weight gradient, 5 conv3 data gradient, 6 fc1 data gradient; 7..11 the fused conv1 on the frames of
// this net's last forward: from the u8 frames without / with Z1 (7 / 8), from X2 without / with Z1 (9 / 10), from X2 without
// pooling (11).  0 was conv1 as a kernel of its own, which the library no longer has.
extern "C" int fb_debug_tc_kernel(fb_qnet *n, int which, int B, int reps, const float *params_dev, void *stream) {
    FB_REQUIRE(n && n->tc && params_dev && B > 0 && B <= n->max_batch && reps > 0, "fb_debug_tc_kernel: bad argument");
    FB_REQUIRE(which != 0, "fb_debug_tc_kernel: kernel 0, the separate conv1 forward kernel, is retired (7..11 time the fused conv1)");
    FB_REQUIRE(which >= 1 && which <= 11, "fb_debug_tc_kernel: which must be 1..11");
    TcState *t = n->tc;
    TcPlan *p;
    int rc = make_plan(n, B, &p);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const QnetLayout &L = n->L;
    const TcWeightMaps &wm = t->wm[0];
    const FwdWs &f = t->ws[0];
    const int H = L.hidden, P2 = B * kP2;
    for (int r = 0; r < reps; r++) {
        switch (which) {
            case 1: FB_CUDA_OK((launch_tc_conv<64, kSlab2, 2, 8, 3, 1>(p->p2_s[0], wm.w2p, p->conv2, t->n_sms, EpiGrid7{f.a2, params_dev + L.b2, P2, t->f16}, st))); break;
            case 2: FB_CUDA_OK((launch_tc_conv<64, kSlab3, 1, 9, 4, 1>(p->a2_s[0], wm.w3p, p->conv3, t->n_sms, EpiConv3{f.a3, params_dev + L.b3, P2, t->f16}, st))); break;
            case 3: FB_CUDA_OK((launch_tc_gemm<128, 2>(p->a3_k[0], wm.wf1n, p->fc1, dim3((B + 127) / 128, H / 128, p->sf),
                                                       EpiStoreF32{f.parth, B, H, (size_t)n->max_batch * H}, st))); break;
            case 4: FB_CUDA_OK((launch_tc_wgrad<32, 2, kSlabW1, 1, 6>(p->x2_w, p->dz1_b, p->conv1_w, p->s1, EpiStoreF32{t->part1, 256, 32, (size_t)256 * 32}, st))); break;
            case 5: FB_CUDA_OK((launch_tc_conv<64, kSlab3, 1, 9, 4, 1>(p->dz3_s, wm.w3d, p->conv3_d, t->n_sms, EpiConv3Dgrad{t->dz2, f.a2, P2, t->f16}, st))); break;
            case 6: FB_CUDA_OK((launch_tc_gemm<64, 0>(p->dh1_k, wm.wf1n, p->fc1_d, dim3((B + 127) / 128, kFlat / 64, 1), EpiFc1Dgrad{t->dz3, f.a3, B, t->f16}, st))); break;
            case 7: FB_CUDA_OK((launch_tc_conv1_fused<4, false>(p->x2_s[0], wm.w1p, Conv1FusedParams{t->probe_view, B, params_dev + L.b1, nullptr, f.p2, t->f16}, t->n_sms, st))); break;
            case 8: FB_CUDA_OK((launch_tc_conv1_fused<4, false>(p->x2_s[0], wm.w1p, Conv1FusedParams{t->probe_view, B, params_dev + L.b1, f.z1, f.p2, t->f16}, t->n_sms, st))); break;
            case 9: FB_CUDA_OK((launch_tc_conv1_fused<6, true>(p->x2_s[0], wm.w1p, Conv1FusedParams{t->probe_view, B, params_dev + L.b1, nullptr, f.p2, t->f16}, t->n_sms, st))); break;
            case 10: FB_CUDA_OK((launch_tc_conv1_fused<6, true>(p->x2_s[0], wm.w1p, Conv1FusedParams{t->probe_view, B, params_dev + L.b1, f.z1, f.p2, t->f16}, t->n_sms, st))); break;
            case 11: FB_CUDA_OK((launch_tc_conv1_fused<6, true>(p->x2_s[0], wm.w1p, Conv1FusedParams{t->probe_view, B, params_dev + L.b1, nullptr, nullptr, t->f16}, t->n_sms, st))); break;
        }
    }
    return FB_OK;
}

// ------------------------------------------------------------------------------------------------ slab probe
// Experiment behind the "one slab, many taps" plan: A rows [0,256) are loaded ONCE (two 128-row boxes, 128B swizzle)
// and the MMA reads rows [shift, shift+128) by starting its descriptor shift*128 bytes into the slab.  Valid only if
// the hardware applies the swizzle to absolute shared-memory address bits (as TMA does when it writes).
namespace {
__global__ void __launch_bounds__(128) tc_slab_probe_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                                                            int shift, uint32_t base_offset, float *d) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar_full, bar_done;
    __shared__ uint32_t tmem_slot;
    const uint32_t smem = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) { tc::mbar_init(tc::smem_u32(&bar_full), 1); tc::mbar_init(tc::smem_u32(&bar_done), 1); tc::fence_barrier_init(); }
    if (warp == 0) tc::tmem_alloc(tc::smem_u32(&tmem_slot), 64);
    tc::tc_fence_before(); __syncthreads(); tc::tc_fence_after();
    const uint32_t tmem = tmem_slot, sa = smem, sb = smem + 32768;
    if (threadIdx.x == 0) {
        tc::mbar_expect_tx(tc::smem_u32(&bar_full), 32768 + 8192);
        tc::tma_load_2d(sa, &mapA, 0, 0, tc::smem_u32(&bar_full));
        tc::tma_load_2d(sa + 16384, &mapA, 0, 128, tc::smem_u32(&bar_full));
        tc::tma_load_2d(sb, &mapB, 0, 0, tc::smem_u32(&bar_full));
        tc::mbar_wait(tc::smem_u32(&bar_full), 0);
        tc::tc_fence_after();
        constexpr uint32_t idesc = tc::instr_desc_bf16(128, 64, 0, 0);
        for (int k = 0; k < 4; k++) {
            uint64_t ad = tc::smem_desc(sa + shift * 128 + k * 32, 16, 1024, tc::kSwizzle128) | ((uint64_t)(base_offset & 7u) << 49);
            uint64_t bd = tc::smem_desc(sb + k * 32, 16, 1024, tc::kSwizzle128);
            tc::umma_bf16(tmem, ad, bd, idesc, k != 0);
        }
        tc::umma_commit(tc::smem_u32(&bar_done));
    }
    tc::mbar_wait(tc::smem_u32(&bar_done), 0);
    tc::tc_fence_after();
    for (int c0 = 0; c0 < 64; c0 += 16) {
        float v[16];
        tc::tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
        for (int i = 0; i < 16; i++) d[(warp * 32 + lane) * 64 + c0 + i] = v[i];
    }
    tc::tc_fence_before(); __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem, 64);
}
}  // namespace

// D[128][64] = A[shift .. shift+128)[64] * Bt[64][64]^T with A [256][64] resident as one slab (see above)
extern "C" int fb_debug_tc_slab(int shift, int base_offset, const void *a_dev, const void *b_dev, float *d_dev, void *stream) {
    FB_REQUIRE(a_dev && b_dev && d_dev && shift >= 0 && shift <= 128, "fb_debug_tc_slab: bad argument");
    int rc = ensure_encode();
    if (rc) return rc;
    CUtensorMap ma, mb;
    if ((rc = make_map(&ma, (const bf16 *)a_dev, 256, 64, 64, 128))) return rc;
    if ((rc = make_map(&mb, (const bf16 *)b_dev, 64, 64, 64, 64))) return rc;
    FB_CUDA_OK(cudaFuncSetAttribute(tc_slab_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768 + 8192 + 1024));
    tc_slab_probe_kernel<<<1, 128, 32768 + 8192 + 1024, (cudaStream_t)stream>>>(ma, mb, shift, (uint32_t)base_offset, d_dev);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

// ------------------------------------------------------------------------------------------------ MMA rate probe
// cycles per tcgen05.mma (M = 128, K = 16, bf16) as a function of N, operand major-ness and the number of independent
// accumulators, on whatever bytes shared memory holds: `iters` back-to-back MMAs by one thread, one commit, clock64.
namespace {
__global__ void __launch_bounds__(128) tc_mma_rate_kernel(int n, int mn_major, int naccs, int iters, int same_operands, long long *cycles) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const uint32_t smem = (tc::smem_u32(smem_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < 48 * 1024 / 4; i += 128) reinterpret_cast<uint32_t *>(smem_raw)[i] = 0x3c003c00u;   // finite bf16s
    if (threadIdx.x == 0) { tc::mbar_init(tc::smem_u32(&bar), 1); tc::fence_barrier_init(); }
    if (warp == 0) tc::tmem_alloc(tc::smem_u32(&tmem_slot), 512);
    tc::fence_proxy_async();
    tc::tc_fence_before(); __syncthreads(); tc::tc_fence_after();
    const uint32_t tmem = tmem_slot;
    if (warp == 1) {                                  // whole warp converged; one elected lane issues (CUTLASS style)
        const uint32_t idesc = tc::instr_desc_bf16(128, n, mn_major, mn_major);
        const uint32_t hi = tc::smem_desc_hi(1024, tc::kSwizzle128);
        const uint32_t a0 = tc::smem_desc_lo(smem, mn_major ? 8192 : 16), b0 = tc::smem_desc_lo(smem + 16384, mn_major ? 8192 : 16);
        const uint32_t step = same_operands ? 0 : (mn_major ? 128 : 2);      // K advance of one MMA, 16-byte units
        const uint32_t d1 = naccs > 1 ? (uint32_t)n : 0, d2 = naccs > 2 ? 2u * n : 0, d3 = naccs > 3 ? 3u * n : d1;
        uint32_t elected;
        asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}" : "=r"(elected));
        long long t0 = clock64();
        for (int i = 0; i < iters; i += 8) {
            if (elected) {
                tc::umma_bf16_lohi(tmem, a0, hi, b0, hi, idesc, 1);
                tc::umma_bf16_lohi(tmem + d1, a0 + step, hi, b0 + step, hi, idesc, 1);
                tc::umma_bf16_lohi(tmem + d2, a0 + 2 * step, hi, b0 + 2 * step, hi, idesc, 1);
                tc::umma_bf16_lohi(tmem + d3, a0 + 3 * step, hi, b0 + 3 * step, hi, idesc, 1);
                tc::umma_bf16_lohi(tmem, a0, hi, b0, hi, idesc, 1);
                tc::umma_bf16_lohi(tmem + d1, a0 + step, hi, b0 + step, hi, idesc, 1);
                tc::umma_bf16_lohi(tmem + d2, a0 + 2 * step, hi, b0 + 2 * step, hi, idesc, 1);
                tc::umma_bf16_lohi(tmem + d3, a0 + 3 * step, hi, b0 + 3 * step, hi, idesc, 1);
            }
            __syncwarp();
        }
        long long t_issue = clock64();
        if (elected) tc::umma_commit(tc::smem_u32(&bar));
        __syncwarp();
        tc::mbar_wait(tc::smem_u32(&bar), 0);
        long long t1 = clock64();
        if (elected) { cycles[0] = t1 - t0; cycles[1] = t_issue - t0; }
    }
    tc::tc_fence_before(); __syncthreads();
    if (warp == 0) tc::tmem_dealloc(tmem, 512);
}
}  // namespace

extern "C" int fb_debug_tc_mma_rate(int n, int mn_major, int naccs, int iters, int same_operands, long long *cycles_dev, void *stream) {
    FB_REQUIRE(cycles_dev && n >= 16 && n <= 256 && n % 16 == 0 && naccs >= 1 && naccs * n <= 512 && iters > 0, "fb_debug_tc_mma_rate: bad argument");
    FB_CUDA_OK(cudaFuncSetAttribute(tc_mma_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    tc_mma_rate_kernel<<<1, 128, 64 * 1024, (cudaStream_t)stream>>>(n, mn_major, naccs, iters, same_operands, cycles_dev);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

// ------------------------------------------------------------------------------------------------ self-test hook
// Raw GEMM on caller matrices through the same kernel, so that the descriptor encodings are pinned on their own:
//   mode 0: D[M][N] = A[M][K] * Bt[N][K]^T          (both K-major)
//   mode 1: D[M][N] = A[K][M]^T * B[K][N]           (both MN-major; contraction over rows)
// bn in {32, 64, 128}; N % bn == 0; strides6 (may be NULL) overrides {lbo_a, sbo_a, kstep_a, lbo_b, sbo_b, kstep_b}.
extern "C" int fb_debug_tc_gemm(int mode, int bn, int M, int N, int K, const void *a_dev, const void *b_dev, float *d_dev,
                                const uint32_t *strides6, void *stream) {
    FB_REQUIRE(a_dev && b_dev && d_dev && (mode == 0 || mode == 1) && (bn == 32 || bn == 64 || bn == 128) && N % bn == 0,
               "fb_debug_tc_gemm: bad argument");
    int rc = ensure_encode();
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    CUtensorMap ma, mb;
    GemmParams g{};
    const bf16 *A = (const bf16 *)a_dev, *Bm = (const bf16 *)b_dev;
    dim3 grid;
    if (mode == 0) {
        FB_REQUIRE(K % 64 == 0 && K / 64 <= kMaxKb, "fb_debug_tc_gemm: K must be a multiple of 64, at most 2048");
        if ((rc = make_map(&ma, A, M, K, 64, 128))) return rc;
        if ((rc = make_map(&mb, Bm, N, K, 64, bn))) return rc;
        set_kmajor(g);
        g.nkb = K / 64;
        for (int k = 0; k < g.nkb; k++) { g.a_rowoff[k] = 0; g.a_col[k] = k * 64; }
        grid = dim3((M + 127) / 128, N / bn, 1);
    } else {
        FB_REQUIRE((M + 127) / 128 <= 16, "fb_debug_tc_gemm: M must be at most 2048 in mode 1");
        if ((rc = make_map(&ma, A, K, M, 64, 64))) return rc;
        if ((rc = make_map(&mb, Bm, K, N, bn == 32 ? 32 : 64, 64))) return rc;
        set_mnmajor(g, bn);
        g.p_total = K; g.klen = (K + 63) / 64 * 64;
        for (int mt = 0; mt < (M + 127) / 128; mt++) for (int i = 0; i < 2; i++) { g.a2_rowoff[mt][i] = 0; g.a2_col[mt][i] = mt * 128 + i * 64; }
        grid = dim3((M + 127) / 128, N / bn, 1);
    }
    if (strides6) { g.lbo_a = strides6[0]; g.sbo_a = strides6[1]; g.kstep_a = strides6[2]; g.lbo_b = strides6[3]; g.sbo_b = strides6[4]; g.kstep_b = strides6[5]; }
    EpiStoreF32 ep{d_dev, M, N, 0};
    cudaError_t e;
    if (mode == 0) e = bn == 32 ? launch_tc_gemm<32, 0>(ma, mb, g, grid, ep, st) : bn == 64 ? launch_tc_gemm<64, 0>(ma, mb, g, grid, ep, st) : launch_tc_gemm<128, 0>(ma, mb, g, grid, ep, st);
    else e = bn == 32 ? launch_tc_gemm<32, 1>(ma, mb, g, grid, ep, st) : bn == 64 ? launch_tc_gemm<64, 1>(ma, mb, g, grid, ep, st) : launch_tc_gemm<128, 1>(ma, mb, g, grid, ep, st);
    FB_CUDA_OK(e);
    return FB_OK;
}
