// Shared host/device helpers for the dmdqn_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/dmdqn_b200.h"

namespace dmdqn {

void set_error(const char* fmt, ...);

#define DMDQN_CHECK_ARG(cond, ...)                                  \
    do {                                                            \
        if (!(cond)) {                                              \
            ::dmdqn::set_error(__VA_ARGS__);                        \
            return DMDQN_ERR_ARG;                                   \
        }                                                           \
    } while (0)

#define DMDQN_CUDA(expr)                                                              \
    do {                                                                              \
        cudaError_t _e = (expr);                                                      \
        if (_e != cudaSuccess) {                                                      \
            ::dmdqn::set_error("%s failed: %s", #expr, cudaGetErrorString(_e));       \
            return DMDQN_ERR_CUDA;                                                    \
        }                                                                             \
    } while (0)

// Float offsets of W1|b1|W2|b2|W3|b3 inside one parameter block (include/dmdqn_b200.h).  `end` closes the range the
// Adam kernels update: b3 + 4, or with the dueling value head wv[H] | bv | pad[3] after b3, b3 + 8 + H.
struct Layout {
    int64_t w1, b1, w2, b2, w3, b3, stride;
    int64_t end;
};
__host__ __device__ inline Layout make_layout(int dp, int h, bool dueling = false) {
    Layout l;
    l.w1 = 0;
    l.b1 = (int64_t)dp * h;
    l.w2 = l.b1 + h;
    l.b2 = l.w2 + (int64_t)h * h;
    l.w3 = l.b2 + h;
    l.b3 = l.w3 + (int64_t)h * 4;
    l.end = l.b3 + 4 + (dueling ? h + 4 : 0);
    l.stride = (l.end + 31) / 32 * 32;  // blocks start on 128-byte lines
    return l;
}
// Dueling value head: wv[H] right after b3 (16-byte aligned), bv after it.
__host__ __device__ inline int64_t layout_wv(const Layout& l) { return l.b3 + 4; }
__host__ __device__ inline int64_t layout_bv(const Layout& l, int h) { return l.b3 + 4 + h; }

// The dueling fold (include/dmdqn_b200.h): the mean over the first A of four values, summed left to right in fp32 and
// divided by A, and the effective head value (x - mean) + v.  Shared by the fold kernel, act and both head updates.
// (The loops are unrolled with predicated terms so that the four values stay in registers.)
__host__ __device__ __forceinline__ float head_sum(const float (&x)[4], int A) {
    float s = x[0];
#pragma unroll
    for (int b = 1; b < 4; ++b)
        if (b < A) s += x[b];
    return s;
}
// W3e / b3e of one row of four advantage values x and its value weight v (columns >= A are 0)
__host__ __device__ __forceinline__ void head_fold(float (&x)[4], float v, int A) {
    const float m = head_sum(x, A) / (float)A;
#pragma unroll
    for (int a = 0; a < 4; ++a) x[a] = a < A ? (x[a] - m) + v : 0.f;
}
// The projection of the folded head's gradient G onto the advantage row (in place) and the value weight (returned)
__host__ __device__ __forceinline__ float head_project(float (&g)[4], int A) {
    const float s = head_sum(g, A), m = s / (float)A;
#pragma unroll
    for (int a = 0; a < 4; ++a) g[a] = a < A ? g[a] - m : 0.f;
    return s;
}

// Noisy networks (include/dmdqn_b200.h dmdqn_noisy): Philox4x32-10 (Salmon et al. 2011, Random123's constants and round
// order, the same function as curand_Philox4x32_10), usable on the host so that a host build can check it.
__host__ __device__ __forceinline__ uint32_t philox_mulhi(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
__host__ __device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        if (r) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
        const uint32_t hi0 = philox_mulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = philox_mulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    }
    return c;
}

// Offsets (floats) of the eight factor vectors inside one network's noise record for one set (include/dmdqn_b200.h
// dmdqn_noise_record): off[2 * layer + side], layer 0..3 = W1, W2, W3, value head, side 0 = inputs, 1 = outputs; off[8]
// is the end of the last vector, `stride` the record's stride (a network's two sets are adjacent records).
struct NoiseRec {
    int32_t off[9];
    int32_t stride;
};
__host__ __device__ inline NoiseRec make_noise_rec(int dp, int h) {
    const int32_t len[8] = {dp, h, h, h, h, 4, h, 4};
    NoiseRec r;
    r.off[0] = 0;
    for (int v = 0; v < 8; ++v) r.off[v + 1] = r.off[v] + len[v];
    r.stride = (r.off[8] + 31) / 32 * 32;
    return r;
}

// f(z) of one factor entry: z = Box-Muller in float64 on the Philox words (x, y) of counter {i, layer<<2 | side<<1 | set,
// t, "nois"} under the network's key (low word first), rounded to fp32; f(z) = sgn(z) sqrt|z| in fp32.
__device__ __forceinline__ float noise_factor(uint64_t key, uint32_t i, int vec, int set, uint32_t t) {
    const uint4 w = philox4x32_10(make_uint4(i, (uint32_t)((vec >> 1) << 2 | (vec & 1) << 1 | set), t, 0x6e6f6973u),
                                  make_uint2((uint32_t)key, (uint32_t)(key >> 32)));
    const double u1 = ((double)w.x + 0.5) * 0x1p-32, u2 = (double)w.y * 0x1p-32;
    const float z = (float)(sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2));
    return z >= 0.f ? sqrtf(z) : -sqrtf(-z);
}

// The whole record of one network and set into `rec` (shared memory), every thread of the block taking part; entries for
// padding (W1 input rows >= obs_dim, W3 output columns >= A, the value head's outputs >= 1, the tail up to the stride) are 0.
__device__ __forceinline__ void noise_record_build(float* rec, const NoiseRec& R, int obs_dim, int n_actions, uint64_t key,
                                                   uint32_t t, int set) {
    for (int e = threadIdx.x; e < R.stride; e += blockDim.x) {
        int v = 0;
        while (v < 8 && e >= R.off[v + 1]) ++v;
        const int i = e - R.off[v];
        const int valid = v == 0 ? obs_dim : v == 5 ? n_actions : v == 7 ? 1 : R.off[v + 1] - R.off[v];
        rec[e] = v < 8 && i < valid ? noise_factor(key, (uint32_t)i, v, set, t) : 0.f;
    }
}

// The weight noise of the four floats at offset e (a multiple of 4) of a parameter block: f_in[i] * f_out[j] for a weight,
// f_out[j] for a bias, 0 on padding.  rec: the record of the set (include/dmdqn_b200.h: wv is the value head's input side
// and column 0 of its output side, bv with its three pad floats takes the output side's four entries).
__device__ __forceinline__ float4 noise_eps4(const float* rec, const NoiseRec& R, const Layout& L, int H, bool dueling, int64_t e) {
    auto outer = [&](float fi, const float* fo) {
        return make_float4(__fmul_rn(fi, fo[0]), __fmul_rn(fi, fo[1]), __fmul_rn(fi, fo[2]), __fmul_rn(fi, fo[3]));
    };
    auto vec = [](const float* f) { return make_float4(f[0], f[1], f[2], f[3]); };
    if (e < L.b1) return outer(rec[R.off[0] + e / H], rec + R.off[1] + e % H);
    if (e < L.w2) return vec(rec + R.off[1] + (e - L.b1));
    if (e < L.b2) return outer(rec[R.off[2] + (e - L.w2) / H], rec + R.off[3] + (e - L.w2) % H);
    if (e < L.w3) return vec(rec + R.off[3] + (e - L.b2));
    if (e < L.b3) return outer(rec[R.off[4] + (e - L.w3) / 4], rec + R.off[5]);
    if (e < L.b3 + 4) return vec(rec + R.off[5]);
    if (dueling && e < layout_bv(L, H)) {
        const float fo = rec[R.off[7]];
        const float* fi = rec + R.off[6] + (e - layout_wv(L));
        return make_float4(__fmul_rn(fi[0], fo), __fmul_rn(fi[1], fo), __fmul_rn(fi[2], fo), __fmul_rn(fi[3], fo));
    }
    if (dueling && e == layout_bv(L, H)) return vec(rec + R.off[7]);
    return make_float4(0.f, 0.f, 0.f, 0.f);
}

// mu + sigma * eps as the header states it: one rounded product, then one rounded sum
__device__ __forceinline__ float noisy_weight(float mu, float sigma, float eps) { return __fadd_rn(mu, __fmul_rn(sigma, eps)); }

// Tile geometry of the fused MLP kernels for hidden width H (DESIGN.md "K3/K4 tiling").
// A CTA owns BM batch rows and all H output columns; each thread an 8x8 register tile.
template <int H>
struct Tile {
    static constexpr int WN = H / 64;               // warps along the output columns
    static constexpr int WM = (H >= 512) ? 1 : 2;   // warps along the batch rows
    static constexpr int NT = 32 * WN * WM;         // threads per CTA
    static constexpr int BM = 32 * WM;              // batch rows per CTA
    static constexpr int KC = 16;                   // K rows of the streamed operand per stage
    static constexpr int LDH = H + 4;               // smem row stride of activations
    static constexpr int LDW = H + 4;               // smem row stride of a weight chunk
};

inline int row_tiles(int batch, int bm) { return (batch + bm - 1) / bm; }

// Workspace carve-up (device scratch of sample/learn), offsets in bytes, 256-aligned.
struct Workspace {
    size_t rows, r_hat, act_b, done_b, active, y, q_all, q_next, tq_all;
    size_t h1, dh1, dh2;              // [n_nets][B][H] floats each ([H][B] per network on the tcgen05 path)
    size_t tc_error;                  // int: set by a tcgen05 kernel whose mbarrier wait timed out, or by K5 on a peer timeout
    size_t mask2;                     // tcgen05 path: relu'(h2) bits, uint32 [n_nets][B][H/32]
    size_t ga;                        // tcgen05 path: float2 [n_nets][B] {dL/dq of the taken action, action bits}
    size_t w3_copy;                   // tcgen05 path: W3 as K4a saw it, [n_nets][H][4] (K4b rebuilds dh2 while W3 is being updated)
    size_t adam_sc;                   // [n_nets] float4 {alpha_t, eps_eff, sync mode bits, -}: the step's Adam scalars, written
                                      // by the sample kernel for the active networks, read by every Adam kernel (adam_step)
    size_t part_loss;                 // [n_nets][T][8]
    size_t part_b3;                   // [n_nets][T][4]
    size_t part_w3;                   // [n_nets][T][H][4]
    size_t part_b2, part_b1;          // [n_nets][T][H]
    size_t is_w;                      // [n_nets][B] float: importance weights of a prioritized sample (written by the sample
                                      // kernel, read by K4a)
    size_t sync;                      // tcgen05 path, int32: [0] K4b work counter, [1..3] spare, [4 ..] k4a_done[n_nets], then
                                      // k3_done[n_nets][T]; zeroed by the sample kernel (dataflow flags between the learn kernels)
    size_t nrows, disc_b;             // [n_nets][B] int32 bootstrap row (agent*C + slot) and float discount of each row's TD
                                      // target (the drawn row and gamma * (1 - done) for one-step targets; see dmdqn_sample)
    size_t head;                      // dueling: float [2][n_nets][4H + 4], W3e | b3e of the online and the target network
                                      // (the fold kernel's output, read by K3 / K4a); carved last so no other offset moves
    size_t total;
    int tiles;                        // T: row tiles per network of the FFMA kernels (Tile<H>::BM rows); the tcgen05 path's
                                      // 128-row tiles are fewer, so its partials fit the same arrays
};
inline int tile_bm(int h) { return h >= 512 ? 32 : 64; }
inline Workspace make_workspace(const dmdqn_dims& d) {
    Workspace w;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t nb = (size_t)d.n_nets * d.batch;
    w.tiles = row_tiles(d.batch, tile_bm(d.hidden));
    const size_t nt = (size_t)d.n_nets * w.tiles;
    w.rows = take(nb * 4);
    w.r_hat = take(nb * 4);
    w.act_b = take(nb * 4);
    w.done_b = take(nb * 4);
    w.active = take((size_t)d.n_nets * 4);
    w.y = take(nb * 4);
    w.q_all = take(nb * 16);
    w.q_next = take(nb * 16);
    w.tq_all = take(nb * 16);
    w.h1 = take(nb * d.hidden * 4);
    w.tc_error = take(4);
    w.adam_sc = take((size_t)d.n_nets * 16);
    w.mask2 = take(nb * (size_t)(d.hidden / 32) * 4);
    w.ga = take(nb * 8);
    w.w3_copy = take((size_t)d.n_nets * d.hidden * 16);
    w.dh1 = take(nb * d.hidden * 4);
    w.dh2 = take(nb * d.hidden * 4);
    w.part_loss = take(nt * 8 * 4);
    w.part_b3 = take(nt * 4 * 4);
    w.part_w3 = take(nt * d.hidden * 4 * 4);
    w.part_b2 = take(nt * d.hidden * 4);
    w.part_b1 = take(nt * d.hidden * 4);
    w.is_w = take(nb * 4);
    w.sync = take((4 + (size_t)d.n_nets + nt) * 4);
    w.nrows = take(nb * 4);
    w.disc_b = take(nb * 4);
    w.head = take(2 * (size_t)d.n_nets * (4 * (size_t)d.hidden + 4) * 4);
    w.total = off;
    return w;
}

int validate_dims(const dmdqn_dims* d);

constexpr int kAllStages = DMDQN_STAGE_SAMPLE | DMDQN_STAGE_TARGET | DMDQN_STAGE_ONLINE | DMDQN_STAGE_WGRAD;   // dmdqn_learn

// Arguments of every learn kernel of both paths (learn.cu, learn_tc.cu) and of the Adam kernels that finish a
// shared-parameter step; make_learn_args resolves the workspace pointers.  The tcgen05 launcher adds its own part:
// tc_tiles, chain and the k4a_done / k3_done flag pointers.
struct LearnArgs {
    dmdqn_dims d;
    Layout L;
    dmdqn_replay rp;
    dmdqn_nets nets;
    int loss, double_dqn;
    int loss_batch;                   // batch the loss mean runs over (== batch, or the global batch when ranks split it)
    float one_m_b1, one_m_b2, tau;    // Adam constants of the call; the per-step scalars are in adam_sc
    int ws_tiles;                     // Workspace::tiles: row tiles of the FFMA kernels, the per-network stride of k3_done
    int tc_tiles;                     // tcgen05 path: 128-row tiles per network (its K3 / K4a items and part_* slots)
    const int32_t *rows, *nrows, *act_b, *active;     // nrows: bootstrap rows, whose next_obs K3 reads as s'
    const float *r_hat, *disc_b;                       // TD target y = r_hat + disc_b * Q_tgt(s')
    const float4* adam_sc;
    float *y, *q_all, *q_next, *tq_all, *h1, *dh1, *dh2;
    float *part_loss, *part_b3, *part_w3, *part_b2, *part_b1;
    uint32_t* mask2;                  // relu'(h2) bits [n_nets][B][H/32]: the eight words of a batch row are adjacent
    float2* ga;                       // [n_nets][B] {dL/dq of the taken action, action as int bits}: what K4b needs per row
    float* w3_copy;                   // [n_nets][H][4]
    int* error;                       // Workspace::tc_error
    float* metrics;
    float* grads;                     // non-NULL: K4b stores dL/dtheta here instead of applying Adam (shared parameters)
    // Dataflow between the tcgen05 learn kernels of one dmdqn_learn call (`chain`: the sample kernel of the same call has
    // reset the flags): K4a / K4b are programmatic dependent launches whose CTAs start on SMs the previous kernel has left
    // and wait per (network, tile) / per network instead of for the whole previous grid.
    int chain;
    int *sched, *k4a_done, *k3_done;
    // Prioritized replay (per = 1 only in DMDQN_SAMPLE_PRIORITIZED): K4a weights each row by is_w and writes its priority
    int per;
    const float* is_w;                // Workspace::is_w
    double per_alpha, per_eps;  // Workspace::sync: K4b work counter | K4a items finished per network | K3 items finished
                                      // per (network, tile)
    // Where K3 / K4a read the head W3[H][4] | b3[4] of network g: head[0] (online) / head[1] (target) + g * head_stride.
    // Plain: theta / theta_tgt + L.w3 with the parameter stride; dueling: the folded W3e | b3e in Workspace::head.  (The
    // plain tcgen05 K3 / K4a instantiations read the head from the parameter block directly: learn_tc.cu head_w3.)
    const float* head[2];
    int64_t head_stride;
    int dueling;                      // K4b projects the head gradient onto W3 / b3 / wv / bv
};
LearnArgs make_learn_args(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                          char* ws, const Workspace& w, float* metrics, float* grads, int loss_batch);

// Prioritized replay, K4a of both paths: the priority of the transition behind row `row` (agent * C + slot) from its TD
// error, (float)pow(|delta| + eps, alpha) in float64, and the agent's running maximum (positive floats order like their
// int bits, so atomicMax gives the same result in any order).  A non-finite priority is not stored.
__device__ __forceinline__ void per_store_priority(const LearnArgs& A, int row, float delta) {
    const float p = (float)pow(fabs((double)delta) + A.per_eps, A.per_alpha);
    if (!isfinite(p)) return;
    A.rp.priority[row] = p;
    atomicMax(reinterpret_cast<int*>(A.rp.priority_max) + row / A.d.capacity, __float_as_int(p));
}

// Adam scalars of one network's step.  alpha_t, eps_eff and the sync mode are evaluated once per network by the sample
// kernel into adam_sc; every Adam kernel loads them here.
struct AdamStep {
    float alpha, eps, one_m_b1, one_m_b2, tau;
    int sync;                         // 0 none, 1 hard copy, 2 Polyak
};
__device__ __forceinline__ AdamStep adam_step(const LearnArgs& A, int g) {
    const float4 sc = __ldg(A.adam_sc + g);
    return {sc.x, sc.y, A.one_m_b1, A.one_m_b2, A.tau, __float_as_int(sc.z)};
}

// Metrics row of network g (include/dmdqn_b200.h) from its `tiles` loss partials, summed in tile order in float64.
// `ld` reads one partial: the tcgen05 K4b reads through L2 (K4a CTAs of the same chain may have written them while it ran).
// The loop stays rolled: it runs on one thread per network, and unrolled it cost the tcgen05 K4b spill bytes.
template <typename Load>
__device__ __forceinline__ void finish_metrics(const LearnArgs& A, int g, int tiles, Load ld) {
    double ls = 0, qs = 0, qq = 0, hist[4] = {0, 0, 0, 0};
#pragma unroll 1
    for (int r = 0; r < tiles; ++r) {
        const float* pl = A.part_loss + ((size_t)g * tiles + r) * 8;
        ls += ld(pl); qs += ld(pl + 1); qq += ld(pl + 2);
        for (int a = 0; a < 4; ++a) hist[a] += ld(pl + 3 + a);
    }
    const double cnt = (double)A.d.batch * A.d.n_actions, mean = qs / cnt, var = fmax(qq / cnt - mean * mean, 0.0);
    float* m = A.metrics + g * DMDQN_METRICS_STRIDE;
    m[0] = (float)(ls / A.loss_batch);                // batch-mean loss (dqn_agent.py:352)
    m[1] = (float)mean;
    m[2] = (float)sqrt(var);
    for (int a = 0; a < 4; ++a) m[3 + a] = (float)hist[a];
    m[7] = 1.f;
}

// Per-DEVICE launch state.  The dynamic shared-memory opt-in (cudaFuncSetAttribute) and the SM count belong to a
// device, not to the process: a host that drives several GPUs from one process (one AgentGroup per device) must
// opt in on each of them.  `cache` is a zero-initialised static array owned by the call site, indexed by device
// ordinal; the worst a race between two host threads can do is set the same attribute twice.
constexpr int kMaxDevices = 64;
int device_sm_count(int* n_sm);
int opt_in_dynamic_smem(const void* kernel, size_t bytes, size_t (&cache)[kMaxDevices]);

// Launchers implemented in the .cu files.
int launch_featurize(int32_t n, const int32_t* halting, const int32_t* phase, const double* next_switch,
                     const double* phase_dur, double sim_time, const uint8_t* signal_valid,
                     const int32_t* nbr_idx, const int32_t* phase_lut, const double* snapshot,
                     double lw, double gw, double* own_out, float* obs_out, int32_t obs_out_stride,
                     double* reward_out, double* global_out, int64_t* scratch, cudaStream_t s);
int launch_featurize_alt(int32_t n, const int32_t* halting, const int32_t* phase, const double* next_switch,
                         const uint8_t* signal_valid, double sim_time, const int32_t* nbr_idx, const double* prev_own,
                         double* own_out, float* obs_out, int32_t obs_out_stride, double* reward_out, cudaStream_t s);
int launch_act(const dmdqn_dims& d, const dmdqn_nets& nets, const float* obs, int32_t stride,
               const double* eps, const uint32_t* w1, const uint32_t* w2, int32_t* actions, float* q_out, bool dueling,
               cudaStream_t s, const dmdqn_noisy* noisy = nullptr);
int launch_noisy_fold(const dmdqn_dims& d, bool dueling, const dmdqn_nets& nets, const dmdqn_noisy& nz, cudaStream_t s);
int launch_noisy_adam_apply(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const dmdqn_noisy& nz,
                            const float* grads, char* ws, const Workspace& w, cudaStream_t s);
int launch_push(const dmdqn_dims& d, const dmdqn_replay& rp, const float* obs, const int32_t* act,
                const double* rew, const float* next_obs, const uint8_t* done, int32_t in_stride,
                const uint8_t* mask, cudaStream_t s);
int launch_sample(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                  const void* draws, const uint8_t* learn_mask, int advance, char* ws, const Workspace& w,
                  cudaStream_t s);
int launch_gather(const dmdqn_dims& d, const dmdqn_replay& rp, const char* ws, const Workspace& w,
                  float* states, int32_t* actions, float* rewards, float* next_states, float* dones,
                  int32_t* active_out, cudaStream_t s);
int launch_learn(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                 float* metrics, char* ws, const Workspace& w, int stages, float* grads, int loss_batch, cudaStream_t s);
bool tc_supported(const dmdqn_dims& d);
int launch_learn_tc(const LearnArgs& A, int precision, int stages, cudaStream_t s);
int launch_adam_apply(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const float* grads, char* ws,
                      const Workspace& w, cudaStream_t s);
int launch_clip_adam_apply(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const float* grads,
                           double clipnorm, float* norms_out, char* ws, const Workspace& w, cudaStream_t s);
int launch_sync_target(const dmdqn_dims& d, const dmdqn_nets& nets, const uint8_t* mask, double tau, bool dueling,
                       cudaStream_t s);
int launch_fold(const dmdqn_dims& d, const dmdqn_nets& nets, char* ws, const Workspace& w, cudaStream_t s);
int launch_peer_adam(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const dmdqn_peers& peers,
                     const float* my_loss_src, float* loss_out, char* ws, const Workspace& w, cudaStream_t s);

}  // namespace dmdqn
