// Device-resident replay memory.
//
// Replaces
//   BrainDQN.py:69-72,197-201           collections.deque of (s, a, r, s', terminal) + random.sample
//   BrainPrioritizedReplyDQN.py:32-104  SumTree (add / update / get_leaf / get_min_prob / total_p)
//   BrainPrioritizedReplyDQN.py:107-151 Memory (store / sample / batch_update)
//
// Storage.  Frames live once, in the env's own ring u8[N][L][80][80]: frame f_t of env e is slot
// t % L.  Transition k >= 1 of env e is (s_{k-1}, a_k, r_k, s_k, term_k) with s_k = frames
// k-3..k (times < 0 clamp to f_0, the setInitState replication of BrainDQN.py:239), i.e. 5
// consecutive ring slots; a/r/term of step k sit in [L][N] arrays at row k % L and are written there
// directly by the act / step kernels ("append" moves no frame bytes).  With capacity C <= L-4
// transitions per env the live set at time t is k in [max(1, t-C+1), t]; the population index of
// random.sample / the SumTree data index is   j = e * cnt + (k - k_lo)   resp.   e * C + (k-1) % C,
// which for N = 1 is exactly the reference's deque / data_pointer order.
//
// n-step returns (fb_step_sampling.n_step = n >= 1) need nothing stored beyond that: transition k becomes
// (s_{k-1}, a_k, R_k, s_{k+n-1}, disc_k) -- the same lookup, n reward / terminal rows and a later frame window.  It can be drawn
// once its horizon is complete (k + n - 1 <= t), so every index is decoded at t_eff = t - n + 1: the uniform population at t
// is exactly the 1-step population at t_eff, and a prioritized memory stores transition t_eff at time t.  Frames then span
// s_{k-1} .. s_{k+n-1}, hence L >= C + n + 3.  The gather copies F = 4 + min(n, 4) frames per sample (times k-4..k-1, then
// k-4+n .. k-1+n without the overlap) and one thread per sample walks the n rows for R_k and disc_k in float64.
#include <new>

#include "fb_common.cuh"

// ------------------------------------------------------------------------------ uniform sampling
// random.sample(population, k) of CPython (Lib/random.py), driven by the 32-bit word stream
// Philox(seed, purpose 3, stream 0):  _randbelow(n) = getrandbits(n.bit_length()) with rejection,
// getrandbits(b) = word >> (32 - b).
//   n <= setsize : partial shuffle of a pool   (sequential, one thread; only during warm-up sizes)
//   n >  setsize : draw j = _randbelow(n), retry while j was already selected.  Acceptance of a word
//                  is "in range and first occurrence", which does not depend on evaluation order, so a
//                  whole CTA draws candidates in parallel, resolves first occurrences through a shared
//                  hash table (atomicMin on the candidate index) and compacts in candidate order.
constexpr int kSampThreads = 256, kCandPerThread = 4, kCandPerRound = kSampThreads * kCandPerThread;
constexpr int kHashSize = 4096;            // distinct keys ever inserted < max batch 512 + one round (1024)
constexpr uint32_t kEmpty = 0xFFFFFFFFu;

// The stream position is 64 bits: its low word indexes the Philox block / lane as before, its high word goes into the counter
// lanes that carry the env id for the per-env streams (these two streams have none), so the sequence never repeats -- a 32-bit
// position wrapped after 2^32 words, ~8 M updates of minibatch 256.  Below 2^32 words the stream is the one the oracle draws.
__device__ __forceinline__ uint32_t sample_word(uint64_t seed, unsigned long long pos) { return stream_word(seed, 3u, pos >> 32, (uint32_t)pos); }
__device__ __forceinline__ uint32_t per_word(uint64_t seed, unsigned long long pos) { return stream_word(seed, 4u, pos >> 32, (uint32_t)pos); }

// index -> (env, time): a population index of random.sample over the deque (per == 0), or a SumTree data index (per == 1)
__device__ __forceinline__ void decode_transition(int per, long long t, int cap, long long j, int *e, long long *k) {
    const uint32_t ju = (uint32_t)j;                      // indices are int32 (capacity < 2^30): 32-bit divisions
    if (!per) {
        long long k_lo = t - cap + 1; if (k_lo < 1) k_lo = 1;
        const uint32_t cnt = (uint32_t)(t - k_lo + 1);
        *e = (int)(ju / cnt); *k = k_lo + (long long)(ju % cnt);
    } else {
        *e = (int)(ju / (uint32_t)cap);
        const long long p = (long long)(ju % (uint32_t)cap), back = (t - 1 - p) % cap;
        *k = t - back;
    }
}
// Frame f of a sample's minibatch row, as a time offset from its transition k: s = k-4..k-1 (f < 4), s' = the n-step window
// k-4+n .. k-1+n without the frames s already holds (n <= 4: one consecutive run of F = 4 + n frames; n > 4: two runs of four).
// n = 1 is the 1-step row: five consecutive frames k-4..k.
__host__ __device__ __forceinline__ int frames_per_sample(int n) { return 4 + (n < 4 ? n : 4); }
__device__ __forceinline__ int frame_time_offset(int f, int n) { return f < 4 ? f - 4 : f - 4 + n - (n < 4 ? n : 4); }

// Where the F frames of each drawn transition live in the ring (byte offsets), written by the sampler itself: the training
// step's first convolution reads them in place, so the gather that fills the caller-visible minibatch buffers runs beside the
// forward passes instead of ahead of them.  tab == nullptr: not wanted.  t: the time indices are decoded at (t_eff for
// n-step); n: the horizon (1 for the 1-step transitions).
struct FrameTabArgs { long long *tab; long long t; int cap, L, per, n; };
__device__ __forceinline__ void write_frame_tab(const FrameTabArgs &ft, int b, long long j) {
    int e; long long k;
    decode_transition(ft.per, ft.t, ft.cap, j, &e, &k);
    const int F = frames_per_sample(ft.n);
    long long *row = ft.tab + (size_t)b * F;
    if (k >= 4) {
        int slot = (int)((k - 4) % ft.L);                 // one 64-bit remainder, then the ring is walked
#pragma unroll
        for (int f = 0; f < 8; f++) {
            if (f >= F) break;
            if (f == 4 && ft.n > 4) slot = (int)((k - 4 + ft.n) % ft.L);   // the second run of four (n > 4)
            row[f] = ((long long)e * ft.L + slot) * 6400;
            if (++slot == ft.L) slot = 0;
        }
    } else {
#pragma unroll
        for (int f = 0; f < 8; f++) {
            if (f >= F) break;
            long long tf = k + frame_time_offset(f, ft.n); if (tf < 0) tf = 0;     // setInitState replication of frame 0
            row[f] = ((long long)e * ft.L + tf % ft.L) * 6400;
        }
    }
}

__global__ void __launch_bounds__(kSampThreads) sample_uniform_kernel(uint32_t n, int batch, uint32_t setsize, uint64_t seed,
                                                                      unsigned long long *word_pos, int32_t *out, FrameTabArgs ft) {
    __shared__ uint32_t hbuf[2 * kHashSize];
    uint32_t *hkey = hbuf, *hidx = hbuf + kHashSize;
    __shared__ uint32_t warp_tot[kSampThreads / 32];
    __shared__ uint32_t s_taken, s_consumed;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned long long pos0 = *word_pos;
    if (n <= setsize) {                    // pool branch (Lib/random.py: "An n-length list is smaller than a k-length set")
        uint32_t *pool = hbuf;             // n <= setsize <= 2 * kHashSize
        for (uint32_t i = tid; i < n; i += kSampThreads) pool[i] = i;
        __syncthreads();
        if (tid == 0) {
            unsigned long long pos = pos0;
            for (int i = 0; i < batch; i++) {
                uint32_t m = n - (uint32_t)i, bits = 32 - __clz(m), j;
                do { j = sample_word(seed, pos++) >> (32 - bits); } while (j >= m);
                out[i] = (int32_t)pool[j];
                pool[j] = pool[m - 1];
            }
            *word_pos = pos;
        }
        __syncthreads();
        if (ft.tab) for (int b = tid; b < batch; b += kSampThreads) write_frame_tab(ft, b, out[b]);
        return;
    }
    const uint32_t bits = 32 - __clz(n);
    for (int i = tid; i < kHashSize; i += kSampThreads) { hkey[i] = kEmpty; hidx[i] = kEmpty; }
    if (tid == 0) { s_taken = 0; s_consumed = 0; }
    __syncthreads();
    for (uint32_t round = 0;; round++) {
        const uint32_t base = round * kCandPerRound + tid * kCandPerThread;     // candidate index = word offset from pos0
        uint32_t r[kCandPerThread], slot[kCandPerThread];
#pragma unroll
        for (int c = 0; c < kCandPerThread; c++) {
            r[c] = sample_word(seed, pos0 + base + c) >> (32 - bits);
            slot[c] = kEmpty;
            if (r[c] < n) {
                uint32_t h = (r[c] * 2654435761u) >> 20;                          // 12 bits
                for (;;) {
                    uint32_t prev = atomicCAS(&hkey[h], kEmpty, r[c]);
                    if (prev == kEmpty || prev == r[c]) { atomicMin(&hidx[h], base + c); slot[c] = h; break; }
                    h = (h + 1) & (kHashSize - 1);
                }
            }
        }
        __syncthreads();
        uint32_t acc[kCandPerThread], cnt = 0;
#pragma unroll
        for (int c = 0; c < kCandPerThread; c++) { acc[c] = slot[c] != kEmpty && hidx[slot[c]] == base + c; cnt += acc[c]; }
        uint32_t incl = cnt;                                                     // block-wide exclusive scan of cnt
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(~0u, incl, o); if (lane >= o) incl += v; }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        uint32_t before = s_taken;
        for (int w = 0; w < warp; w++) before += warp_tot[w];
        uint32_t rank = before + incl - cnt;
#pragma unroll
        for (int c = 0; c < kCandPerThread; c++)
            if (acc[c]) {
                if (rank < (uint32_t)batch) out[rank] = (int32_t)r[c];
                if (rank == (uint32_t)batch - 1) s_consumed = base + c + 1;
                rank++;
            }
        __syncthreads();
        if (tid == 0) { uint32_t tot = 0; for (int w = 0; w < kSampThreads / 32; w++) tot += warp_tot[w]; s_taken += tot; }
        __syncthreads();
        if (s_taken >= (uint32_t)batch) break;
    }
    if (tid == 0) *word_pos = pos0 + s_consumed;
    if (ft.tab) for (int b = tid; b < batch; b += kSampThreads) write_frame_tab(ft, b, out[b]);      // out[] is complete: last barrier above
}

// ------------------------------------------------------------------------------ gather
struct GatherArgs {
    const uint8_t *ring; int N, L;
    const uint8_t *act; const float *rew; const uint8_t *term;       // [L][N]
    long long t;                 // time the indices are decoded at: the newest stored transition (t_eff = t - n + 1 for n-step)
    int cap;                     // C, transitions kept per env
    int per;                     // 0: idx is a population index of random.sample; 1: a SumTree data index
    const int32_t *idx; int batch;
    uint8_t *frames;             // [batch][F][80][80], F = frames_per_sample(n)
    uint8_t *a_out; float *r_out; uint8_t *t_out;
    int32_t *env_out, *k_out;    // optional
    int n;                       // horizon: 1 (1-step), or the n-step n, for which ret_out / disc_out are written
    double gamma;
    double *ret_out, *disc_out;  // f64[batch] or nullptr (1-step)
};

// one CTA per (sample, frame): 6,400 bytes, every thread's loads issued together (the ring is HBM-cold)
__global__ void __launch_bounds__(128) gather_kernel(GatherArgs g) {
    const int b = blockIdx.x, f = blockIdx.y, F = gridDim.y;
    if (b >= g.batch) return;
    long long k; int e;
    decode_transition(g.per, g.t, g.cap, g.idx[b], &e, &k);
    long long tf = k + frame_time_offset(f, g.n); if (tf < 0) tf = 0;   // setInitState replication of frame 0
    const uint4 *src = reinterpret_cast<const uint4 *>(g.ring) + ((size_t)e * g.L + (size_t)(tf % g.L)) * 400;
    uint4 *dst = reinterpret_cast<uint4 *>(g.frames) + (size_t)b * F * 400 + f * 400;
    uint4 v[4];
#pragma unroll
    for (int q = 0; q < 4; q++) { int i = threadIdx.x + q * 128; v[q] = i < 400 ? __ldg(src + i) : make_uint4(0u, 0u, 0u, 0u); }
#pragma unroll
    for (int q = 0; q < 4; q++) { int i = threadIdx.x + q * 128; if (i < 400) dst[i] = v[q]; }
    if (f == 0 && threadIdx.x == 0) {
        size_t m = (size_t)(k % g.L) * g.N + e;
        g.a_out[b] = g.act[m]; g.r_out[b] = g.rew[m]; g.t_out[b] = g.term[m];
        if (g.env_out) g.env_out[b] = e;
        if (g.k_out) g.k_out[b] = (int32_t)k;
        if (g.ret_out) {
            // R = sum_{i<m} gamma^i r_{k+i}, accumulated forward in float64 (no fused multiply-add: the oracle's roundings),
            // cut after the first terminal; disc = 0 after a terminal, else the running product gamma^n
            double R = 0.0, gm = 1.0;
            bool hit = false;
            int row = (int)(k % g.L);
            for (int i = 0; i < g.n && !hit; i++) {
                const size_t mi = (size_t)row * g.N + e;
                const float rf = g.rew[mi];
                R = __dadd_rn(R, __dmul_rn(gm, rf == 0.1f ? 0.1 : (double)rf));      // the env returns the Python float 0.1
                gm = __dmul_rn(gm, g.gamma);
                hit = g.term[mi] != 0;
                if (++row == g.L) row = 0;
            }
            g.ret_out[b] = R;
            g.disc_out[b] = hit ? 0.0 : gm;
        }
    }
}

// ------------------------------------------------------------------------------ SumTree
// tree: f64[2*cap-1], node 0 the root, leaves [cap-1, 2cap-2] (BrainPrioritizedReplyDQN.py:39-47).
// Beside it live two more trees of the same shape, maintained by the same kernels along the same leaf-to-root paths:
//   mn[node] = smallest POSITIVE leaf below it (+inf if none)   -> Memory.sample's get_min_prob (:70-71), an O(capacity) min()
//   mx[node] = largest leaf below it                             -> Memory.store's np.max over all leaves (:122)
// so both are read from the root in O(1); round 1 re-scanned every leaf before every sample / store (7.9 MB per update at
// 983,040 leaves against ~70 KB algorithmic).  min / max are exact, so their order of evaluation is free.
__device__ __forceinline__ int node_depth(int idx) { return 31 - __clz(idx + 1); }
__device__ __forceinline__ int ancestor_at(int idx, int depth_idx, int d) { return ((idx + 1) >> (depth_idx - d)) - 1; }
__device__ __forceinline__ double pos_or_inf(double p) { return p > 0.0 ? p : __longlong_as_double(0x7FF0000000000000ll); }

struct Node3 { double s, mn, mx; };
__device__ __forceinline__ void set_leaf(double *tree, double *mn, double *mx, int leaf, double p) { tree[leaf] = p; mn[leaf] = pos_or_inf(p); mx[leaf] = p; }
__device__ __forceinline__ void pull_node(double *tree, double *mn, double *mx, int node) {       // parent = f(children), exact
    const int l = 2 * node + 1;
    tree[node] = tree[l] + tree[l + 1];
    mn[node] = fmin(mn[l], mn[l + 1]);
    mx[node] = fmax(mx[l], mx[l + 1]);
}

// One CTA applies `count` leaf updates tree[leaf_i] = p_i and repairs the inner nodes.
//   mode 0 "reference": SumTree.update semantics, item after item: change = p - tree[leaf];
//          every ancestor += change (BrainPrioritizedReplyDQN.py:62-68).  The additions into one node
//          happen in item order (thread d owns depth d and walks the items in order, keeping the
//          running node value in a register), so the float64 rounding history equals the reference's.
//   mode 1 "rebuild": leaves are set, then every touched ancestor is recomputed as left + right,
//          deepest level first.  Deterministic, parallel, no drift; used for N > 1 at scale.
// leaves: tree indices.  prio: f64[count] or nullptr -> Memory.store: the max leaf (root of mx), 1.0 if all zero (:121-125).
// abs_err (f32, optional): Memory.batch_update's transform (:146-149) p = min(|err| + 0.01, 1)^0.6 in float32, computed
// here into prio_scratch instead of by a kernel of its own.
constexpr int kMaxDupScan = 512;
constexpr int kTopDepth = 11, kTopNodes = (1 << kTopDepth) - 1;          // depths 0..10 of the tree: 2,047 nodes
__global__ void __launch_bounds__(1024) tree_update_kernel(double *tree, double *mn, double *mx, int cap, const int32_t *leaves, const double *prio,
                                                           int count, int mode, double *change_scratch, const float *abs_err,
                                                           double *prio_scratch) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    Node3 *s_top = reinterpret_cast<Node3 *>(s_raw);                      // depths 0..10 of the three trees (mode 1)
    const int tid = threadIdx.x;
    const int max_depth = node_depth(2 * cap - 2);
    __shared__ double s_store;
    __shared__ int s_leaf[kMaxDupScan];
    if (tid == 0) { double p = mx[0]; s_store = p == 0.0 ? 1.0 : p; }     // Memory.store :121-125
    if (abs_err != nullptr) {
        for (int i = tid; i < count; i += blockDim.x) prio_scratch[i] = (double)powf(fminf(abs_err[i] + 0.01f, 1.0f), 0.6f);
        prio = prio_scratch;
    }
    __syncthreads();
    if (mode == 0) {
        if (tid == 0)
            for (int i = 0; i < count; i++) {
                int leaf = leaves[i];
                double p = prio ? prio[i] : s_store;
                change_scratch[i] = p - tree[leaf];
                set_leaf(tree, mn, mx, leaf, p);
            }
        __syncthreads();
        if (tid < max_depth) {              // thread d repairs depth d of the SUM tree in the reference's order
            int d = tid, cur = -1; double val = 0.0;
            for (int i = 0; i < count; i++) {
                int leaf = leaves[i], dl = node_depth(leaf);
                if (dl <= d) continue;
                int node = ancestor_at(leaf, dl, d);
                if (node != cur) { if (cur >= 0) tree[cur] = val; cur = node; val = tree[node]; }
                val += change_scratch[i];
            }
            if (cur >= 0) tree[cur] = val;
        }
        __syncthreads();
        for (int d = max_depth - 1; d >= 0; d--) {                         // min / max trees: exact, level by level
            for (int i = tid; i < count; i += blockDim.x) {
                int leaf = leaves[i], dl = node_depth(leaf);
                if (dl > d) { int node = ancestor_at(leaf, dl, d), l = 2 * node + 1; mn[node] = fmin(mn[l], mn[l + 1]); mx[node] = fmax(mx[l], mx[l + 1]); }
            }
            __syncthreads();
        }
        return;
    }
    const bool in_smem = prio != nullptr && count <= kMaxDupScan;     // a minibatch: scan for duplicates from shared memory
    if (in_smem) { for (int i = tid; i < count; i += blockDim.x) s_leaf[i] = leaves[i]; __syncthreads(); }
    for (int i = tid; i < count; i += blockDim.x) {
        if (!prio) { set_leaf(tree, mn, mx, leaves[i], s_store); continue; }      // stores: distinct leaves, one value
        const int mine = leaves[i];
        int later = 0;                                            // duplicates in a minibatch: the last one wins, as in
        if (in_smem) { for (int j = i + 1; j < count; j++) later += (s_leaf[j] == mine); }     // the reference's sequential loop (:150-151)
        else { for (int j = i + 1; j < count; j++) if (leaves[j] == mine) { later = 1; break; } }
        if (later == 0) set_leaf(tree, mn, mx, mine, prio[i]);
    }
    __syncthreads();
    // deep levels in global memory (one dependent L2 round trip per level), then depths <= 10 from a shared-memory copy
    const int top = max_depth - 1 < kTopDepth ? max_depth - 1 : kTopDepth - 1;      // deepest level handled in shared memory
    for (int d = max_depth - 1; d > top; d--) {
        for (int i = tid; i < count; i += blockDim.x) {
            int leaf = leaves[i], dl = node_depth(leaf);
            if (dl > d) pull_node(tree, mn, mx, ancestor_at(leaf, dl, d));
        }
        __syncthreads();
    }
    const int n_top = (2 << top) - 1, n_all = 2 * cap - 1;                         // nodes of depths 0..top
    for (int j = tid; j < n_top && j < n_all; j += blockDim.x) s_top[j] = Node3{tree[j], mn[j], mx[j]};
    __syncthreads();
    for (int d = top; d >= 0; d--) {
        for (int i = tid; i < count; i += blockDim.x) {
            int leaf = leaves[i], dl = node_depth(leaf);
            if (dl > d) {
                int node = ancestor_at(leaf, dl, d), cl = 2 * node + 1;
                const Node3 a = cl < n_top ? s_top[cl] : Node3{tree[cl], mn[cl], mx[cl]};
                const Node3 b = cl + 1 < n_top ? s_top[cl + 1] : Node3{tree[cl + 1], mn[cl + 1], mx[cl + 1]};
                const Node3 v{a.s + b.s, fmin(a.mn, b.mn), fmax(a.mx, b.mx)};
                s_top[node] = v; tree[node] = v.s; mn[node] = v.mn; mx[node] = v.mx;
            }
        }
        __syncthreads();
    }
}

// Memory.store for one transition of EVERY env (mode "rebuild", N >= kStoreMultiMin): N leaves, one per env, at
//   leaf(e) = cap - 1 + e C + off.   Round 1 walked them through ONE CTA, level after level.  Here the tree is cut at depth
// kTopDepth: each of the 2,048 sub-trees below is private to one CTA (CTA b owns sub-trees [b S, (b+1) S)), which finds its envs
// by arithmetic (a sub-tree's leaves are two contiguous index ranges, one per leaf level), sets their leaves and pulls the
// touched ancestors level by level with CTA-local barriers only; the CTA that finishes last repairs depths 10..0 in shared memory.
constexpr int kStoreMultiMin = 2048;
__global__ void __launch_bounds__(256) per_store_multi_kernel(double *tree, double *mn, double *mx, int cap, int N, int C, int off,
                                                              unsigned int *done_counter) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    Node3 *s_top = reinterpret_cast<Node3 *>(s_raw);
    __shared__ double s_store;
    __shared__ int s_last;
    const int tid = threadIdx.x, n_all = 2 * cap - 1, max_depth = node_depth(n_all - 1);
    if (tid == 0) { double p = mx[0]; s_store = p == 0.0 ? 1.0 : p; }     // the max leaf BEFORE this store: read by every CTA before any
    __syncthreads();                                                      // CTA can have changed the root (only the last CTA writes it)
    const double p_store = s_store;
    const int n_sub = 1 << kTopDepth;                                      // sub-trees rooted at depth kTopDepth
    const int j0 = (int)((long long)blockIdx.x * n_sub / gridDim.x), j1 = (int)((long long)(blockIdx.x + 1) * n_sub / gridDim.x);
    // envs whose leaf lies below sub-trees [j0, j1): per leaf level dl the node range [(a0+1) 2^k - 1, (a1+1) 2^k - 1), k = dl - kTopDepth
    int e_lo[2], e_hi[2], dls[2];
    for (int q = 0; q < 2; q++) {
        const int dl = max_depth - 1 + q, k = dl - kTopDepth;
        long long lo = ((long long)(n_sub - 1 + j0 + 1) << k) - 1, hi = ((long long)(n_sub - 1 + j1 + 1) << k) - 1;      // [lo, hi)
        if (lo < cap - 1) lo = cap - 1;
        if (hi > n_all) hi = n_all;
        dls[q] = dl;
        if (hi <= lo) { e_lo[q] = 0; e_hi[q] = 0; continue; }
        // leaf(e) in [lo, hi)  <=>  e C + off in [lo - (cap-1), hi - (cap-1))
        const long long a = lo - (cap - 1) - off, b = hi - (cap - 1) - off;
        long long el = a <= 0 ? 0 : (a + C - 1) / C, eh = b <= 0 ? 0 : (b + C - 1) / C;
        if (eh > N) eh = N;
        if (el > eh) el = eh;
        e_lo[q] = (int)el; e_hi[q] = (int)eh;
    }
    for (int q = 0; q < 2; q++)
        for (int e = e_lo[q] + tid; e < e_hi[q]; e += blockDim.x) set_leaf(tree, mn, mx, cap - 1 + e * C + off, p_store);
    __syncthreads();
    for (int d = max_depth - 1; d >= kTopDepth; d--) {
        for (int q = 0; q < 2; q++) {
            const int dl = dls[q];
            if (dl <= d) continue;
            for (int e = e_lo[q] + tid; e < e_hi[q]; e += blockDim.x) {
                const int leaf = cap - 1 + e * C + off, node = ancestor_at(leaf, dl, d);
                // several envs share an ancestor: the first env below it (in this level's range) pulls it
                if (e > e_lo[q] && ancestor_at(leaf - C, dl, d) == node) continue;
                pull_node(tree, mn, mx, node);
            }
        }
        __syncthreads();
    }
    // ---- the CTA that finishes last repairs depths kTopDepth-1 .. 0
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(done_counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const int base = n_sub - 1;                                            // first node of depth kTopDepth
    for (int d = kTopDepth - 1; d >= 0; d--) {
        const int first = (1 << d) - 1, cnt = 1 << d;
        for (int i = tid; i < cnt; i += blockDim.x) {
            const int node = first + i, cl = 2 * node + 1;
            Node3 a, b;
            if (d == kTopDepth - 1) { a = Node3{__ldcg(tree + cl), __ldcg(mn + cl), __ldcg(mx + cl)}; b = Node3{__ldcg(tree + cl + 1), __ldcg(mn + cl + 1), __ldcg(mx + cl + 1)}; }
            else { a = s_top[cl]; b = s_top[cl + 1]; }
            const Node3 v{a.s + b.s, fmin(a.mn, b.mn), fmax(a.mx, b.mx)};
            s_top[node] = v; tree[node] = v.s; mn[node] = v.mn; mx[node] = v.mx;
        }
        __syncthreads();
    }
    (void)base;
    if (tid == 0) *done_counter = 0u;
}

// Memory.sample (BrainPrioritizedReplyDQN.py:127-144): stratified v_i = uniform(i seg, (i+1) seg) with
// np.random.uniform's 53-bit construction from two stream words (purpose 4), SumTree.get_leaf descent
// (:73-100, "v <= tree[left]" goes left), ISWeights = (p/total / min_prob)^-beta in float64.
// One WARP per sample.  Depths 0..10 come from a shared-memory copy; below that the warp fetches the next FIVE levels under
// its current node at once (62 nodes, two per lane, one L2 round trip) and walks them with shuffles -- the comparisons and
// subtractions are the reference's, in the reference's order, only the loads are batched: 2 round trips instead of 10 at
// 983,040 leaves.  min_prob comes from the root of the min tree.  The CTA that finishes last advances the stream position.
constexpr int kSampleWarps = 8;
__global__ void __launch_bounds__(32 * kSampleWarps) per_sample_kernel(const double *tree, const double *min_p_src, int cap, int batch, double beta,
                                                                       uint64_t seed, unsigned long long *word_pos, unsigned int *done_counter, int32_t *tree_idx,
                                                                       int32_t *data_idx, double *isw, double *prio_out, float *isw_f32, FrameTabArgs ft) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * kSampleWarps + warp;
    const int n_nodes = 2 * cap - 1;
    __shared__ double s_top[kTopNodes];                                      // depths 0..10: one round trip instead of eleven
    __shared__ int s_last;
    const int n_top = n_nodes < kTopNodes ? n_nodes : kTopNodes;
    for (int j = threadIdx.x; j < n_top; j += blockDim.x) s_top[j] = tree[j];
    __syncthreads();
    const double total = s_top[0];
    const unsigned long long pos0 = *word_pos;
    if (i < batch) {
        double seg = total / (double)batch, a = seg * (double)i, b = seg * (double)(i + 1);
        uint32_t w0 = per_word(seed, pos0 + 2 * i) >> 5, w1 = per_word(seed, pos0 + 2 * i + 1) >> 6;
        double u = ((double)w0 * 67108864.0 + (double)w1) / 9007199254740992.0;
        double v = a + (b - a) * u;
        int parent = 0;
        for (;;) {                                                           // SumTree.get_leaf (:73-100) through the cached levels
            int cl = 2 * parent + 1;
            if (cl + 1 >= n_top) break;
            double left = s_top[cl];
            if (v <= left) parent = cl; else { v -= left; parent = cl + 1; }
        }
        while (2 * parent + 1 < n_nodes) {                                   // five levels per round trip
            // heap position t >= 1 inside the sub-tree of `parent` (t = 1): node(t) = ((parent + 1) << floor(log2 t)) - 1 + (t - 2^floor(log2 t))
            double val[2];
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int t = lane + 2 + 32 * h;                             // t = 2..33, 34..65 (t <= 63 used)
                const int lv = 31 - __clz(t);
                const long long node = (((long long)parent + 1) << lv) - 1 + (t - (1 << lv));
                val[h] = (t <= 63 && node < n_nodes) ? tree[node] : 0.0;
            }
            int t = 1;
#pragma unroll
            for (int k = 0; k < 5; k++) {
                const int cl = 2 * parent + 1;
                if (cl >= n_nodes) break;                                    // warp-uniform: reached a leaf
                const int tl = 2 * t;                                        // left child inside the fetched block
                const double lo = __shfl_sync(0xFFFFFFFFu, val[0], (tl - 2) & 31), hi = __shfl_sync(0xFFFFFFFFu, val[1], (tl - 34) & 31);
                const double left = tl <= 33 ? lo : hi;
                if (v <= left) { parent = cl; t = tl; } else { v -= left; parent = cl + 1; t = tl + 1; }
            }
        }
        if (lane == 0) {
            const double p = tree[parent];
            const double min_p = *min_p_src;               // root of this shard's min tree, or the min over all shards (fb_per_set_global_min)
            const double prob = p / total, min_prob = min_p / total;
            tree_idx[i] = parent;
            data_idx[i] = parent - (cap - 1);
            if (ft.tab) write_frame_tab(ft, i, parent - (cap - 1));
            const double w = pow(prob / min_prob, -beta);
            isw[i] = w;
            if (isw_f32) isw_f32[i] = (float)w;             // the ISWeights placeholder is tf.float32 (BrainPrioritizedReplyDQN.py:243)
            if (prio_out) prio_out[i] = p;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(done_counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (s_last && threadIdx.x == 0) { *word_pos = pos0 + 2ull * (unsigned long long)batch; *done_counter = 0u; }     // every CTA has read pos0 by now
}

__global__ void store_leaves_kernel(int N, int C, long long k, int32_t *leaves) {   // leaf of transition k for every env
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    leaves[e] = (N * C - 1) + e * C + (int)((k - 1) % C);
}

__global__ void fill_inf_kernel(double *p, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = __longlong_as_double(0x7FF0000000000000ll);
}
constexpr size_t kTopSmem = sizeof(Node3) * kTopNodes;          // 49,128 bytes: depths 0..10 of the three trees
static int node_depth_host(int idx) { int d = 0; for (unsigned v = (unsigned)idx + 1; v > 1; v >>= 1) d++; return d; }

// ------------------------------------------------------------------------------ C ABI
struct fb_replay {
    int N, L, C, cap;
    double *tree;                    // PER only
    double *mn, *mx;                 // min-positive / max trees of the same shape (see the SumTree section)
    long long *frame_tab;            // [512][F <= 8] ring offsets of the drawn transitions' frames (see FrameTabArgs)
    const double *gmin;              // nullptr, or the caller's device scalar: smallest positive leaf over ALL shards (several GPUs)
    unsigned int *counters;          // [0] per_store_multi_kernel, [1] per_sample_kernel: "last CTA" counters, self-resetting
    int32_t *leaves; double *prio; double *change;   // scratch, max(N, max_batch)
    unsigned long long *word_pos;    // [0] uniform stream, [1] PER stream (64-bit word positions)
    int scratch_n;
};

extern "C" int fb_replay_create(int n_envs, int ring_len, int capacity_per_env, int prioritized, int max_batch, fb_replay **out) {
    FB_REQUIRE(out && n_envs > 0 && ring_len >= 5 && capacity_per_env >= 1 && capacity_per_env <= ring_len - 4 && max_batch > 0 && max_batch <= 512,
               "fb_replay_create: need ring_len >= capacity_per_env + 4 and 0 < max_batch <= 512");
    FB_REQUIRE((long long)n_envs * capacity_per_env < (1ll << 30), "fb_replay_create: capacity too large");
    fb_replay *r = new (std::nothrow) fb_replay();
    FB_REQUIRE(r != nullptr, "fb_replay_create: out of host memory");
    r->N = n_envs; r->L = ring_len; r->C = capacity_per_env; r->cap = n_envs * capacity_per_env; r->tree = nullptr;
    r->scratch_n = n_envs > max_batch ? n_envs : max_batch;
    FB_CUDA_OK(cudaMalloc(&r->word_pos, 2 * sizeof(unsigned long long)));
    FB_CUDA_OK(cudaMemset(r->word_pos, 0, 2 * sizeof(unsigned long long)));
    r->mn = r->mx = nullptr; r->gmin = nullptr;
    FB_CUDA_OK(cudaMalloc(&r->frame_tab, 512 * 8 * sizeof(long long)));
    FB_CUDA_OK(cudaMemset(r->frame_tab, 0, 512 * 8 * sizeof(long long)));
    FB_CUDA_OK(cudaMalloc(&r->counters, 2 * sizeof(unsigned int)));
    FB_CUDA_OK(cudaMemset(r->counters, 0, 2 * sizeof(unsigned int)));
    FB_CUDA_OK(cudaMalloc(&r->leaves, sizeof(int32_t) * r->scratch_n));
    FB_CUDA_OK(cudaMalloc(&r->prio, sizeof(double) * r->scratch_n));
    FB_CUDA_OK(cudaMalloc(&r->change, sizeof(double) * r->scratch_n));
    if (prioritized) {
        const size_t nn = 2 * (size_t)r->cap - 1;
        FB_CUDA_OK(cudaMalloc(&r->tree, sizeof(double) * nn));
        FB_CUDA_OK(cudaMemset(r->tree, 0, sizeof(double) * nn));
        FB_CUDA_OK(cudaMalloc(&r->mn, sizeof(double) * nn));
        FB_CUDA_OK(cudaMalloc(&r->mx, sizeof(double) * nn));
        FB_CUDA_OK(cudaMemset(r->mx, 0, sizeof(double) * nn));
        fill_inf_kernel<<<(unsigned)((nn + 255) / 256), 256>>>(r->mn, nn);
        FB_CUDA_OK(cudaGetLastError());
        FB_CUDA_OK(cudaFuncSetAttribute(tree_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTopSmem));
        FB_CUDA_OK(cudaFuncSetAttribute(per_store_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTopSmem));
        FB_CUDA_OK(cudaDeviceSynchronize());
    }
    *out = r;
    return FB_OK;
}

extern "C" int fb_replay_destroy(fb_replay *r) {
    if (!r) return FB_OK;
    cudaFree(r->frame_tab); cudaFree(r->tree); cudaFree(r->mn); cudaFree(r->mx); cudaFree(r->counters); cudaFree(r->leaves); cudaFree(r->prio); cudaFree(r->change); cudaFree(r->word_pos);
    delete r;
    return FB_OK;
}

extern "C" int fb_replay_sample_uniform(fb_replay *r, long long t, int batch, uint32_t setsize, uint64_t seed,
                                        int32_t *idx_out_dev, void *stream) {
    FB_REQUIRE(r && idx_out_dev && batch > 0 && batch <= 512, "fb_replay_sample_uniform: bad argument");
    long long k_lo = t - r->C + 1; if (k_lo < 1) k_lo = 1;
    long long n = (t - k_lo + 1) * r->N;
    if (t < 1 || n < batch) { fb_set_error("Sample larger than population or is negative"); return FB_ERR_INVALID; }   // random.sample's ValueError
    FB_REQUIRE(setsize <= 2u * kHashSize, "fb_replay_sample_uniform: setsize too large");
    sample_uniform_kernel<<<1, kSampThreads, 0, (cudaStream_t)stream>>>((uint32_t)n, batch, setsize, seed, r->word_pos, idx_out_dev, FrameTabArgs{nullptr, 0, 0, 0, 0, 1});
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

extern "C" int fb_replay_gather(fb_replay *r, const uint8_t *ring_dev, const uint8_t *act_dev, const float *rew_dev,
                                const uint8_t *term_dev, long long t, int prioritized_index, const int32_t *idx_dev, int batch,
                                uint8_t *frames_out_dev, uint8_t *act_out_dev, float *rew_out_dev, uint8_t *term_out_dev,
                                int32_t *env_out_dev, int32_t *k_out_dev, void *stream) {
    FB_REQUIRE(r && ring_dev && act_dev && rew_dev && term_dev && idx_dev && frames_out_dev && act_out_dev && rew_out_dev && term_out_dev && batch > 0,
               "fb_replay_gather: bad argument");
    GatherArgs g{ring_dev, r->N, r->L, act_dev, rew_dev, term_dev, t, r->C, prioritized_index, idx_dev, batch,
                 frames_out_dev, act_out_dev, rew_out_dev, term_out_dev, env_out_dev, k_out_dev, 1, 0.0, nullptr, nullptr};
    gather_kernel<<<dim3(batch, 5), 128, 0, (cudaStream_t)stream>>>(g);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

static void launch_per_sample(fb_replay *r, int batch, double beta, uint64_t seed, int32_t *tree_idx, int32_t *data_idx, double *isw, double *prio,
                              float *isw32, cudaStream_t st, FrameTabArgs ft = FrameTabArgs{nullptr, 0, 0, 0, 0, 1}) {
    per_sample_kernel<<<(batch + kSampleWarps - 1) / kSampleWarps, 32 * kSampleWarps, 0, st>>>(r->tree, r->gmin ? r->gmin : r->mn, r->cap, batch, beta, seed, r->word_pos + 1,
                                                                                               r->counters + 1, tree_idx, data_idx, isw, prio, isw32, ft);
}

// ---- sampling + gather as the head of a captured training step (fb_qnet_step with `sampling`) -------------------------
// n_step == 0: the 1-step transitions; n_step >= 1: everything is decoded at t_eff = t - n + 1 (see the top of this file)
static int horizon(const fb_step_sampling &p) { return p.n_step > 0 ? p.n_step : 1; }
static long long decode_time(const fb_step_sampling &p) { return p.t - horizon(p) + 1; }
int replay_frames_per_sample(const fb_step_sampling &p) { return frames_per_sample(horizon(p)); }
static bool sampling_population(const fb_step_sampling &p, uint32_t *n_out) {
    const long long t = decode_time(p);
    long long k_lo = t - p.replay->C + 1; if (k_lo < 1) k_lo = 1;
    long long n = (t - k_lo + 1) * p.replay->N;
    *n_out = (uint32_t)n;
    return t >= 1 && n >= p.batch;
}
static GatherArgs sampling_gather_args(const fb_step_sampling &p, double gamma) {
    const fb_replay *r = p.replay;
    const bool nstep = p.n_step > 0;
    return GatherArgs{p.ring_dev, r->N, r->L, p.act_dev, p.rew_dev, p.term_dev, decode_time(p), r->C, p.prioritized ? 1 : 0, p.idx_out_dev, p.batch,
                      p.frames_out_dev, p.act_out_dev, p.rew_out_dev, p.term_out_dev, p.env_out_dev, p.k_out_dev,
                      horizon(p), gamma, nstep ? p.ret_out_dev : nullptr, nstep ? p.disc_out_dev : nullptr};
}
static FrameTabArgs sampling_frame_tab(const fb_step_sampling &p, bool want) {
    const fb_replay *r = p.replay;
    return FrameTabArgs{want ? r->frame_tab : nullptr, decode_time(p), r->C, r->L, p.prioritized ? 1 : 0, horizon(p)};
}
// the sampler alone; with_tab: it also leaves the ring offsets of the drawn frames in replay_frame_tab()
int replay_launch_sample(const fb_step_sampling &p, bool with_tab, cudaStream_t st) {
    FB_REQUIRE(p.replay && p.ring_dev && p.act_dev && p.rew_dev && p.term_dev && p.idx_out_dev && p.frames_out_dev && p.act_out_dev &&
               p.rew_out_dev && p.term_out_dev && p.batch > 0 && p.batch <= 512, "step sampling: bad argument");
    fb_replay *r = p.replay;
    if (p.n_step != 0) {
        FB_REQUIRE(p.n_step >= 1 && p.n_step <= 16, "step sampling: n_step must be 0 (1-step) or 1..16");
        FB_REQUIRE(p.ret_out_dev && p.disc_out_dev, "step sampling: n-step returns need ret_out_dev and disc_out_dev");
        FB_REQUIRE(r->L >= r->C + p.n_step + 3, "step sampling: n-step returns need ring_len >= capacity_per_env + n_step + 3");
    }
    if (p.prioritized) {
        FB_REQUIRE(r->tree && p.tree_idx_out_dev && p.is_weights_out_dev && p.is_weights_f32_out_dev && (p.per_mode == 0 || p.per_mode == 1) &&
                   p.batch <= r->scratch_n, "step sampling: prioritized replay arguments");
        launch_per_sample(r, p.batch, p.beta, p.seed, p.tree_idx_out_dev, p.idx_out_dev, p.is_weights_out_dev, p.prio_out_dev, p.is_weights_f32_out_dev, st,
                          sampling_frame_tab(p, with_tab));
    } else {
        FB_REQUIRE(p.setsize <= 2u * kHashSize, "step sampling: setsize too large");
        uint32_t n;
        if (!sampling_population(p, &n)) { fb_set_error("Sample larger than population or is negative"); return FB_ERR_INVALID; }
        sample_uniform_kernel<<<1, kSampThreads, 0, st>>>(n, p.batch, p.setsize, p.seed, r->word_pos, p.idx_out_dev, sampling_frame_tab(p, with_tab));
    }
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}
int replay_launch_gather(const fb_step_sampling &p, double gamma, cudaStream_t st) {
    gather_kernel<<<dim3(p.batch, replay_frames_per_sample(p)), 128, 0, st>>>(sampling_gather_args(p, gamma));
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}
int replay_launch_sample_gather(const fb_step_sampling &p, double gamma, cudaStream_t st) {
    int rc = replay_launch_sample(p, false, st);
    return rc ? rc : replay_launch_gather(p, gamma, st);
}
const long long *replay_frame_tab(const fb_replay *r) { return r->frame_tab; }
int replay_launch_per_update(const fb_step_sampling &p, const float *abs_err_dev, cudaStream_t st) {
    FB_REQUIRE(p.prioritized && abs_err_dev, "step sampling: Memory.batch_update needs the step's |TD errors| (abs_err_out_dev)");
    fb_replay *r = p.replay;
    tree_update_kernel<<<1, 1024, kTopSmem, st>>>(r->tree, r->mn, r->mx, r->cap, p.tree_idx_out_dev, nullptr, p.batch, p.per_mode, r->change, abs_err_dev, r->prio);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}
bool replay_is_sampler(const void *func) { return func == (const void *)sample_uniform_kernel || func == (const void *)per_sample_kernel; }
bool replay_is_gather(const void *func) { return func == (const void *)gather_kernel; }
// (a captured step always has its sampler leave the frame offsets behind: the tensor-core step reads the frames in place)
int replay_patch_nodes(cudaGraphExec_t exec, cudaGraphNode_t sampler, cudaGraphNode_t gather, const fb_step_sampling &p, double gamma) {
    fb_replay *r = p.replay;
    cudaKernelNodeParams kp{};
    int batch = p.batch; uint64_t seed = p.seed; int32_t *idx = p.idx_out_dev;
    FrameTabArgs ft = sampling_frame_tab(p, true);
    if (p.prioritized) {
        const double *tree = r->tree, *mn = r->gmin ? r->gmin : r->mn; int cap = r->cap; double beta = p.beta; unsigned long long *word_pos = r->word_pos + 1;
        unsigned int *done = r->counters + 1;
        int32_t *tree_idx = p.tree_idx_out_dev; double *isw = p.is_weights_out_dev, *prio = p.prio_out_dev; float *isw32 = p.is_weights_f32_out_dev;
        void *sargs[] = {&tree, &mn, &cap, &batch, &beta, &seed, &word_pos, &done, &tree_idx, &idx, &isw, &prio, &isw32, &ft};
        kp.func = (void *)per_sample_kernel; kp.gridDim = dim3((p.batch + kSampleWarps - 1) / kSampleWarps); kp.blockDim = dim3(32 * kSampleWarps); kp.kernelParams = sargs;
        FB_CUDA_OK(cudaGraphExecKernelNodeSetParams(exec, sampler, &kp));
    } else {
        uint32_t n;
        if (!sampling_population(p, &n)) { fb_set_error("Sample larger than population or is negative"); return FB_ERR_INVALID; }
        uint32_t setsize = p.setsize; unsigned long long *word_pos = r->word_pos;
        void *sargs[] = {&n, &batch, &setsize, &seed, &word_pos, &idx, &ft};
        kp.func = (void *)sample_uniform_kernel; kp.gridDim = dim3(1); kp.blockDim = dim3(kSampThreads); kp.kernelParams = sargs;
        FB_CUDA_OK(cudaGraphExecKernelNodeSetParams(exec, sampler, &kp));
    }
    GatherArgs g = sampling_gather_args(p, gamma);            // (t_eff, and with it the n-step window, moves with t)
    void *gargs[] = {&g};
    kp.func = (void *)gather_kernel; kp.gridDim = dim3(p.batch, replay_frames_per_sample(p)); kp.blockDim = dim3(128); kp.kernelParams = gargs;
    FB_CUDA_OK(cudaGraphExecKernelNodeSetParams(exec, gather, &kp));
    return FB_OK;
}


// Memory.store for transition k of every env (env order): priority = max leaf (1.0 if all zero)
extern "C" int fb_per_store(fb_replay *r, long long k, int mode, void *stream) {
    FB_REQUIRE(r && r->tree && k >= 1 && (mode == 0 || mode == 1), "fb_per_store: bad argument (is the replay prioritized?)");
    cudaStream_t st = (cudaStream_t)stream;
    if (mode == 1 && r->N >= kStoreMultiMin && node_depth_host(2 * r->cap - 2) > kTopDepth + 1) {      // one CTA per group of sub-trees
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        per_store_multi_kernel<<<sms, 256, kTopSmem, st>>>(r->tree, r->mn, r->mx, r->cap, r->N, r->C, (int)((k - 1) % r->C), r->counters);
        FB_CUDA_OK(cudaGetLastError());
        return FB_OK;
    }
    store_leaves_kernel<<<(r->N + 255) / 256, 256, 0, st>>>(r->N, r->C, k, r->leaves);
    tree_update_kernel<<<1, 1024, kTopSmem, st>>>(r->tree, r->mn, r->mx, r->cap, r->leaves, nullptr, r->N, mode, r->change, nullptr, nullptr);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

extern "C" int fb_per_sample(fb_replay *r, int batch, double beta, uint64_t seed, int32_t *tree_idx_dev, int32_t *data_idx_dev,
                             double *is_weights_dev, double *prio_out_dev, float *is_weights_f32_dev, void *stream) {
    FB_REQUIRE(r && r->tree && batch > 0 && batch <= 512 && tree_idx_dev && data_idx_dev && is_weights_dev, "fb_per_sample: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    launch_per_sample(r, batch, beta, seed, tree_idx_dev, data_idx_dev, is_weights_dev, prio_out_dev, is_weights_f32_dev, st);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

// Memory.batch_update: either from |TD errors| (abs_err_dev f32, transform on device) or from given priorities
extern "C" int fb_per_update(fb_replay *r, const int32_t *tree_idx_dev, const float *abs_err_dev, const double *prio_dev, int batch,
                             int mode, void *stream) {
    FB_REQUIRE(r && r->tree && tree_idx_dev && (abs_err_dev || prio_dev) && batch > 0 && batch <= r->scratch_n && (mode == 0 || mode == 1),
               "fb_per_update: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    tree_update_kernel<<<1, 1024, kTopSmem, st>>>(r->tree, r->mn, r->mx, r->cap, tree_idx_dev, prio_dev, batch, mode, r->change,
                                                  prio_dev ? nullptr : abs_err_dev, r->prio);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}

extern "C" int fb_per_tree_copy(fb_replay *r, double *out_dev, int n_nodes, void *stream) {
    FB_REQUIRE(r && r->tree && out_dev && n_nodes == 2 * r->cap - 1, "fb_per_tree_copy: bad argument");
    FB_CUDA_OK(cudaMemcpyAsync(out_dev, r->tree, sizeof(double) * (size_t)n_nodes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return FB_OK;
}

// which = 1: the min-positive tree, 2: the max tree (same shape as the SumTree; test hook for their invariants)
extern "C" int fb_per_aux_tree_copy(fb_replay *r, int which, double *out_dev, int n_nodes, void *stream) {
    FB_REQUIRE(r && r->tree && out_dev && n_nodes == 2 * r->cap - 1 && (which == 1 || which == 2), "fb_per_aux_tree_copy: bad argument");
    FB_CUDA_OK(cudaMemcpyAsync(out_dev, which == 1 ? r->mn : r->mx, sizeof(double) * (size_t)n_nodes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return FB_OK;
}

// Several GPUs: Memory.sample's min_prob is a property of the WHOLE memory (BrainPrioritizedReplyDQN.py:131 takes the min over every
// leaf), and ISWeights = (p_i / min_p)^-beta does not depend on total_p, so one scalar makes the shards' weights those of one
// global memory.  fb_per_min_root copies this shard's min (the root of its min tree; +inf if it holds no positive leaf) to a
// caller-owned device scalar; the caller reduces it over the ranks (MIN) and hands the result to fb_per_set_global_min, whose
// pointer every later sample reads instead of the local root (nullptr: back to the local root).
extern "C" int fb_per_min_root(fb_replay *r, double *out_dev, void *stream) {
    FB_REQUIRE(r && r->tree && out_dev, "fb_per_min_root: bad argument");
    FB_CUDA_OK(cudaMemcpyAsync(out_dev, r->mn, sizeof(double), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return FB_OK;
}
extern "C" int fb_per_set_global_min(fb_replay *r, const double *global_min_dev) {
    FB_REQUIRE(r && r->tree, "fb_per_set_global_min: bad argument");
    r->gmin = global_min_dev;
    return FB_OK;
}

extern "C" int fb_replay_rng_pos(fb_replay *r, uint64_t *pos_host2, int set, void *stream) {
    FB_REQUIRE(r && pos_host2, "fb_replay_rng_pos: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    if (set) FB_CUDA_OK(cudaMemcpyAsync(r->word_pos, pos_host2, 2 * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    else FB_CUDA_OK(cudaMemcpyAsync(pos_host2, r->word_pos, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    FB_CUDA_OK(cudaStreamSynchronize(st));
    return FB_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// Logging surface (SURVEY 8f N3; BrainDQN.py:88-93): on a terminal the reference appends curScore to score_every_episode and
// timeStep to time_steps_when_episode_end.  Batched: every env that ended an episode this step appends (time_step, env,
// score) to a device log through one warp-aggregated atomic; the host sorts by (time_step, env) when it flushes, so the
// order is deterministic.  *count_dev keeps counting past the capacity (the host reports the overflow); no host sync.
__global__ void log_episodes_kernel(const uint8_t *__restrict__ terminal, const int32_t *__restrict__ score, int n, int first_env,
                                    int time_step, int32_t *__restrict__ log, int *__restrict__ count, int cap) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const bool hit = e < n && terminal[e] != 0;
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (m == 0) return;
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(count, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (hit) {
        const int at = base + __popc(m & ((1u << lane) - 1u));
        if (at < cap) { log[3 * at] = time_step; log[3 * at + 1] = first_env + e; log[3 * at + 2] = score[e]; }
    }
}

extern "C" int fb_log_episodes(const uint8_t *terminal_dev, const int32_t *score_dev, int n_envs, int first_env_id, int time_step,
                               int32_t *log_dev, int *count_dev, int capacity, void *stream) {
    FB_REQUIRE(terminal_dev && score_dev && log_dev && count_dev && n_envs > 0 && capacity > 0, "fb_log_episodes: bad argument");
    log_episodes_kernel<<<(n_envs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(terminal_dev, score_dev, n_envs, first_env_id, time_step,
                                                                                log_dev, count_dev, capacity);
    FB_CUDA_OK(cudaGetLastError());
    return FB_OK;
}
