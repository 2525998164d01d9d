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

// Every parameter block (include/dmdqn_b200.h) is W1|b1|W2|b2|W3|b3, then an optional value stream or cosine embedding.
// The head shape decides the offsets: n atoms per action (1: a scalar head), np the column stride per action (1, or n
// rounded up to a multiple of 4), value: Wv[H][np] | bv[round4(np)] after b3 (dueling and Rainbow), n_cos > 0: Wphi[n_cos][H]
// | bphi[H] after b3 (IQN).  The plain, dueling, C51 / QR-DQN, IQN and Rainbow blocks are (1, 1, -, 0), (1, 1, value, 0),
// (N, Np, -, 0), (1, 1, -, n_cos) and (N, Np, value, 0).
struct HeadShape {
    int n = 1, np = 1;
    bool value = false;
    int n_cos = 0;
};
inline int dist_np(int n_atoms) { return (n_atoms + 3) / 4 * 4; }
inline HeadShape atom_shape(int n_atoms, bool value) { return {n_atoms, dist_np(n_atoms), value, 0}; }
// Float offsets inside one block.  `end` closes the range the Adam kernels update; wv / bv and wphi / bphi equal the end
// of the head (b3 + 4 * np) when the block has no value stream or embedding.
struct Layout {
    int64_t w1, b1, w2, b2, w3, b3, stride;
    int64_t end;
    int64_t wv, bv, wphi, bphi;
};
__host__ __device__ inline Layout make_layout(int dp, int h, HeadShape hs = {}) {
    Layout l;
    l.w1 = 0;
    l.b1 = (int64_t)dp * h;
    l.w2 = l.b1 + h;
    l.b2 = l.w2 + (int64_t)h * h;
    l.w3 = l.b2 + h;
    l.b3 = l.w3 + (int64_t)h * 4 * hs.np;
    l.end = l.b3 + 4 * hs.np;
    l.wv = l.bv = l.wphi = l.bphi = l.end;
    if (hs.value) {
        l.bv = l.wv + (int64_t)h * hs.np;
        l.end = l.bv + (hs.np + 3) / 4 * 4;
    } else if (hs.n_cos) {
        l.bphi = l.wphi + (int64_t)hs.n_cos * h;
        l.end = l.bphi + h;
    }
    l.stride = (l.end + 31) / 32 * 32;  // blocks start on 128-byte lines
    return l;
}

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
// is the end of the last vector, `stride` the record's stride (a network's two sets are adjacent records).  The head's
// output vector has 4 * np entries (column a * np + j), the value head's round4(np) (entry j = atom j).
struct NoiseRec {
    int32_t off[9];
    int32_t stride;
};
__host__ __device__ inline NoiseRec make_noise_rec(int dp, int h, HeadShape hs = {}) {
    const int32_t len[8] = {dp, h, h, h, h, 4 * hs.np, h, (hs.np + 3) / 4 * 4};
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
// padding are 0: W1 input rows >= obs_dim, head output columns a * np + j with a >= A or j >= n_atoms, value head outputs
// >= n_atoms, and the tail up to the stride.  Scalar heads pass n_atoms = np = 1.
__device__ __forceinline__ void noise_record_build(float* rec, const NoiseRec& R, int obs_dim, int n_actions, int n_atoms, int np,
                                                   uint64_t key, uint32_t t, int set) {
    for (int e = threadIdx.x; e < R.stride; e += blockDim.x) {
        int v = 0;
        while (v < 8 && e >= R.off[v + 1]) ++v;
        const int i = e - R.off[v];
        const bool valid = v == 0 ? i < obs_dim : v == 5 ? i / np < n_actions && i % np < n_atoms : v == 7 ? i < n_atoms : v < 8;
        rec[e] = valid ? noise_factor(key, (uint32_t)i, v, set, t) : 0.f;
    }
}

// The weight noise of the four floats at offset e (a multiple of 4) of a parameter block: f_in[i] * f_out[j] for a weight,
// f_out[j] for a bias, 0 on padding.  rec: the record of the set.  W3 / b3 take the head's output side at column
// (e - w3) % (4 * np); Wv / bv the value head's input side at row (e - wv) / np and its output side at atom (e - wv) % np.
// With np a multiple of 4 a float4 never straddles two rows; with np == 1 (the dueling value head wv[H] | bv | pad[3]) one
// float4 of wv spans four rows, so that case takes one input factor per element.
__device__ __forceinline__ float4 noise_eps4(const float* rec, const NoiseRec& R, const Layout& L, int H, int np, int64_t e) {
    const int nh = 4 * np;
    auto outer = [&](float fi, const float* fo) {
        return make_float4(__fmul_rn(fi, fo[0]), __fmul_rn(fi, fo[1]), __fmul_rn(fi, fo[2]), __fmul_rn(fi, fo[3]));
    };
    auto vec = [](const float* f) { return make_float4(f[0], f[1], f[2], f[3]); };
    if (e < L.b1) return outer(rec[R.off[0] + e / H], rec + R.off[1] + e % H);
    if (e < L.w2) return vec(rec + R.off[1] + (e - L.b1));
    if (e < L.b2) return outer(rec[R.off[2] + (e - L.w2) / H], rec + R.off[3] + (e - L.w2) % H);
    if (e < L.w3) return vec(rec + R.off[3] + (e - L.b2));
    if (e < L.b3) return outer(rec[R.off[4] + (e - L.w3) / nh], rec + R.off[5] + (e - L.w3) % nh);
    if (e < L.wv) return vec(rec + R.off[5] + (e - L.b3));
    if (e < L.bv) {
        if (np == 1) {
            const float fo = rec[R.off[7]];
            const float* fi = rec + R.off[6] + (e - L.wv);
            return make_float4(__fmul_rn(fi[0], fo), __fmul_rn(fi[1], fo), __fmul_rn(fi[2], fo), __fmul_rn(fi[3], fo));
        }
        return outer(rec[R.off[6] + (e - L.wv) / np], rec + R.off[7] + (e - L.wv) % np);
    }
    if (e < L.end) return vec(rec + R.off[7] + (e - L.bv));
    return make_float4(0.f, 0.f, 0.f, 0.f);
}

// mu + sigma * eps as the header states it: one rounded product, then one rounded sum
__device__ __forceinline__ float noisy_weight(float mu, float sigma, float eps) { return __fadd_rn(mu, __fmul_rn(sigma, eps)); }

// Distributional (C51) networks (include/dmdqn_b200.h dmdqn_dist).  The head is W3[H][4 * Np] | b3[4 * Np], Np = N rounded
// up to a multiple of 4, column a * Np + j = atom j of action a; the Adam range ends after b3.
constexpr int kDistMaxAtoms = 64;
// The caller-owned scratch of the distributional learn kernels, byte offsets (256-aligned): the projected target
// distribution m [n_nets][B][Np], h2 [n_nets][B][H] and the logit gradient dX [n_nets][B][4 * Np].
struct DistScratch {
    size_t m, h2, dx, total;
};
inline DistScratch make_dist_scratch(const dmdqn_dims& d, int np) {
    DistScratch s;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t nb = (size_t)d.n_nets * d.batch;
    s.m = take(nb * np * 4);
    s.h2 = take(nb * d.hidden * 4);
    s.dx = take(nb * 4 * np * 4);
    s.total = off;
    return s;
}
// What the distributional kernels take beyond LearnArgs: the support and the scratch pointers.
struct DistArgs {
    int n_atoms, np, nh;              // N, Np, 4 * Np
    float lo, hi, dz;                 // (float)v_min, (float)v_max, (float)dz64
    double v_min, dz64;               // dz64 = (v_max - v_min) / (N - 1) in float64
    float *m, *h2, *dx;
};
inline DistArgs make_dist_args(const dmdqn_dims& d, const dmdqn_dist& ds) {
    DistArgs D;
    D.n_atoms = ds.n_atoms;
    D.np = dist_np(ds.n_atoms);
    D.nh = 4 * D.np;
    D.v_min = ds.v_min;
    D.dz64 = (ds.v_max - ds.v_min) / (ds.n_atoms - 1);
    D.lo = (float)ds.v_min;
    D.hi = (float)ds.v_max;
    D.dz = (float)D.dz64;
    const DistScratch s = make_dist_scratch(d, D.np);
    char* p = static_cast<char*>(ds.scratch);
    D.m = p ? reinterpret_cast<float*>(p + s.m) : nullptr;
    D.h2 = p ? reinterpret_cast<float*>(p + s.h2) : nullptr;
    D.dx = p ? reinterpret_cast<float*>(p + s.dx) : nullptr;
    return D;
}
// z_j = (float)(v_min + j * dz64): one rounded float64 product, one rounded sum, then rounded to float
__device__ __forceinline__ float dist_z(double v_min, double dz64, int j) { return (float)__dadd_rn(v_min, __dmul_rn((double)j, dz64)); }
// Softmax statistics of one action's logits x[0..n): mx = max_j x_j, s = sum_j expf(x_j - mx) in j order
__device__ __forceinline__ void dist_stats(const float* x, int n, float& mx, float& s) {
    float m = x[0];
    for (int j = 1; j < n; ++j) m = fmaxf(m, x[j]);
    float t = 0.f;
    for (int j = 0; j < n; ++j) t = __fadd_rn(t, expf(__fsub_rn(x[j], m)));
    mx = m;
    s = t;
}
// The expected value Q = sum_j p_j z_j (fmaf in j order), p_j = expf(x_j - mx) / s
__device__ __forceinline__ float dist_expect(const float* x, int n, const float* z, float& mx, float& s) {
    dist_stats(x, n, mx, s);
    float q = 0.f;
    for (int j = 0; j < n; ++j) q = fmaf(__fdiv_rn(expf(__fsub_rn(x[j], mx)), s), z[j], q);
    return q;
}

// The Rainbow scratch: the C51 regions, then the folded heads W3e[H][4 * Np] | b3e[4 * Np] of the online (0) and the target
// (1) network, [2][n_nets][(H + 1) * 4 * Np] floats.
struct RainbowScratch {
    DistScratch dist;
    size_t head, total;
};
inline RainbowScratch make_rainbow_scratch(const dmdqn_dims& d, int np) {
    RainbowScratch s;
    s.dist = make_dist_scratch(d, np);
    s.head = s.dist.total;
    s.total = s.head + (2 * (size_t)d.n_nets * (d.hidden + 1) * 4 * np * 4 + 255) / 256 * 256;
    return s;
}
// Quantile (QR-DQN) networks (include/dmdqn_b200.h dmdqn_quantile): the C51 head layout, scratch and Adam range for
// N = n_quantiles atoms; the scratch's m region holds the target samples T.  What the kernels take beyond LearnArgs:
struct QuantArgs {
    int n_atoms, np, nh;              // N, Np, 4 * Np
    float kappa;                      // (float)kappa
    float *m, *h2, *dx;
};
inline QuantArgs make_quantile_args(const dmdqn_dims& d, const dmdqn_quantile& qs) {
    QuantArgs D;
    D.n_atoms = qs.n_quantiles;
    D.np = dist_np(qs.n_quantiles);
    D.nh = 4 * D.np;
    D.kappa = (float)qs.kappa;
    const DistScratch s = make_dist_scratch(d, D.np);
    char* p = static_cast<char*>(qs.scratch);
    D.m = p ? reinterpret_cast<float*>(p + s.m) : nullptr;
    D.h2 = p ? reinterpret_cast<float*>(p + s.h2) : nullptr;
    D.dx = p ? reinterpret_cast<float*>(p + s.dx) : nullptr;
    return D;
}
// The expected value Q = (sum_i x_i, fp32 adds in i order) / N
__device__ __forceinline__ float quantile_mean(const float* x, int n) {
    float s = 0.f;
    for (int i = 0; i < n; ++i) s = __fadd_rn(s, x[i]);
    return __fdiv_rn(s, (float)n);
}

// Fraction i of sampled row `row` (row_base + r), set 0 (tau) or 1 (tau') at step t: the top 23 bits of the first Philox
// word, ((x >> 9) + 0.5) * 2^-23, exact in fp32 and strictly inside (0, 1).
__host__ __device__ __forceinline__ float iqn_tau(uint64_t key, uint32_t row, uint32_t i, uint32_t t, int set) {
    const uint4 w = philox4x32_10(make_uint4(row, i, t, 0x69716e00u | (uint32_t)set), make_uint2((uint32_t)key, (uint32_t)(key >> 32)));
    return ((float)(w.x >> 9) + 0.5f) * 0x1p-23f;
}
// Midpoint k of K: (float)((2k + 1) / (2.0 K)), as QR-DQN forms its quantile fractions
__host__ __device__ __forceinline__ float iqn_midpoint(int k, int K) { return (float)((2.0 * k + 1.0) / (2.0 * K)); }
// Cosine feature m of fraction tau: cos(pi * m * tau) in float64, rounded to float
__device__ __forceinline__ float iqn_cos(int m, float tau) { return (float)cos(3.141592653589793 * (double)m * (double)tau); }

// The quantile Huber pair term of one (i, j) pair (include/dmdqn_b200.h dmdqn_quantile): u = T_j - theta_i, fraction tau_i
// with omt = 1 - tau_i, k = (float)kappa.  rho -> the loss term, dr -> its derivative in theta_i.
__device__ __forceinline__ void quantile_pair(float u, float tau, float omt, float k, float& rho, float& dr) {
    const float w = u < 0.f ? omt : tau;
    if (k > 0.f) {
        const float au = fabsf(u);
        rho = __fmul_rn(w, au <= k ? __fdiv_rn(__fmul_rn(0.5f, __fmul_rn(u, u)), k) : __fsub_rn(au, __fmul_rn(0.5f, k)));
        dr = __fdiv_rn(__fmul_rn(-w, fminf(fmaxf(u, -k), k)), k);
    } else {
        rho = __fmul_rn(w, fabsf(u));
        dr = u > 0.f ? -w : (u < 0.f ? w : 0.f);
    }
}

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

// The caller-owned scratch of the IQN learn kernels, byte offsets (256-aligned).  Debug views are [n_nets][B][count]; the
// per-(row, fraction) buffers are fraction-major per network, [n_nets][N][B][width], so that one pass of a row tile writes
// rows of stride width and the weight-gradient GEMMs of network g run over its N * B consecutive rows.
struct IqnScratch {
    size_t tau, tau_p, t, theta, grad;    // [nb][N], [nb][N'], [nb][N'], [nb][N], [nb][N]
    size_t h1n;                           // [2][nb][H]: h1 at s' of the online and the target network
    size_t c;                             // [n_nets][N][B][n_cos]: cosine features of the sampled fractions at s
    size_t z, h2, phi;                    // [n_nets][N][B][H]: z, h2 (then dh2), phi (then dphi) at s
    size_t part_bphi;                     // [n_nets][T][H]: dbphi partials of the online kernel's row tiles
    size_t total;
};
inline IqnScratch make_iqn_scratch(const dmdqn_dims& d, int n, int n_p, int n_cos) {
    IqnScratch s;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t nb = (size_t)d.n_nets * d.batch, h = d.hidden;
    const int tiles = row_tiles(d.batch, tile_bm(d.hidden));        // Workspace::tiles: part_bphi is indexed as part_b1
    s.tau = take(nb * n * 4);
    s.tau_p = take(nb * n_p * 4);
    s.t = take(nb * n_p * 4);
    s.theta = take(nb * n * 4);
    s.grad = take(nb * n * 4);
    s.h1n = take(2 * nb * h * 4);
    s.c = take(nb * n * n_cos * 4);
    s.z = take(nb * n * h * 4);
    s.h2 = take(nb * n * h * 4);
    s.phi = take(nb * n * h * 4);
    s.part_bphi = take((size_t)d.n_nets * tiles * h * 4);
    s.total = off;
    return s;
}
// What the IQN kernels take beyond LearnArgs
struct IqnArgs {
    int n, n_p, k, n_cos, ncp;        // N, N', K, n_cos, n_cos rounded up to 16 (the cosine tile's used width)
    float kappa;
    int64_t row_base;
    const uint64_t* key;
    int64_t wphi, bphi;
    float *tau, *tau_p, *t, *theta, *grad, *h1n, *c, *z, *h2, *phi, *part_bphi;
};
inline IqnArgs make_iqn_args(const dmdqn_dims& d, const dmdqn_iqn& q) {
    IqnArgs Q;
    Q.n = q.n_tau; Q.n_p = q.n_tau_prime; Q.k = q.n_policy; Q.n_cos = q.n_cos;
    Q.ncp = (q.n_cos + 15) / 16 * 16;
    Q.kappa = (float)q.kappa;
    Q.row_base = q.row_base;
    Q.key = q.key;
    const Layout L = make_layout(d.obs_stride, d.hidden, {1, 1, false, q.n_cos});
    Q.wphi = L.wphi; Q.bphi = L.bphi;
    const IqnScratch s = make_iqn_scratch(d, q.n_tau, q.n_tau_prime, q.n_cos);
    char* p = static_cast<char*>(q.scratch);
    auto at = [&](size_t o) { return p ? reinterpret_cast<float*>(p + o) : nullptr; };
    Q.tau = at(s.tau); Q.tau_p = at(s.tau_p); Q.t = at(s.t); Q.theta = at(s.theta); Q.grad = at(s.grad);
    Q.h1n = at(s.h1n); Q.c = at(s.c); Q.z = at(s.z); Q.h2 = at(s.h2); Q.phi = at(s.phi); Q.part_bphi = at(s.part_bphi);
    return Q;
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
LearnArgs make_learn_args(const dmdqn_dims& d, const dmdqn_hparams& hp, HeadShape hs, const dmdqn_replay& rp,
                          const dmdqn_nets& nets, char* ws, const Workspace& w, float* metrics, float* grads, int loss_batch);

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
int launch_noisy_fold(const dmdqn_dims& d, HeadShape hs, const dmdqn_nets& nets, const dmdqn_noisy& nz, cudaStream_t s);
int launch_noisy_adam_apply(const dmdqn_dims& d, const dmdqn_hparams& hp, HeadShape hs, const dmdqn_nets& nets,
                            const dmdqn_noisy& nz, const float* grads, char* ws, const Workspace& w, cudaStream_t s);
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
// Adam over [0, A.L.end) of every active block: plain (clipnorm == 0) or after global-norm clipping
int launch_adam(const LearnArgs& A, const float* grads, double clipnorm, float* norms_out, cudaStream_t s);
int launch_sync_target(const dmdqn_dims& d, int64_t stride, float* theta, float* theta_tgt, const uint8_t* mask, double tau,
                       cudaStream_t s);
// W3e | b3e of the online and the target block of every network into head[2][n_nets][(H + 1) * 4 * np] (hs.value blocks)
int launch_head_fold(const dmdqn_dims& d, HeadShape hs, const float* theta, const float* theta_tgt, float* head, cudaStream_t s);
int launch_peer_adam(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const dmdqn_peers& peers,
                     const float* my_loss_src, float* loss_out, char* ws, const Workspace& w, cudaStream_t s);
int launch_learn_dist(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                      const dmdqn_dist& ds, float* metrics, char* ws, const Workspace& w, float* grads, int loss_batch,
                      cudaStream_t s);
int launch_act_dist(const dmdqn_dims& d, const dmdqn_nets& nets, const dmdqn_dist& ds, const float* obs, int32_t stride,
                    const double* eps, const uint32_t* w1, const uint32_t* w2, int32_t* actions, float* q_out, cudaStream_t s);
int launch_learn_quantile(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                          const dmdqn_quantile& qs, float* metrics, char* ws, const Workspace& w, float* grads, int loss_batch,
                          cudaStream_t s);
int launch_act_quantile(const dmdqn_dims& d, const dmdqn_nets& nets, const dmdqn_quantile& qs, const float* obs, int32_t stride,
                        const double* eps, const uint32_t* w1, const uint32_t* w2, int32_t* actions, float* q_out,
                        cudaStream_t s);
int launch_learn_iqn(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                     const dmdqn_iqn& q, float* metrics, char* ws, const Workspace& w, float* grads, int loss_batch, cudaStream_t s);
int launch_act_iqn(const dmdqn_dims& d, const dmdqn_nets& nets, const dmdqn_iqn& q, const float* obs, int32_t stride,
                   const double* eps, const uint32_t* w1, const uint32_t* w2, int32_t* actions, float* q_out, cudaStream_t s);
int launch_rainbow_fold(const dmdqn_dims& d, const dmdqn_dist& ds, const dmdqn_nets& nets, const dmdqn_noisy& nz, cudaStream_t s);
int launch_learn_rainbow(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& eff,
                         const dmdqn_dist& ds, float* metrics, char* ws, const Workspace& w, float* grads, int loss_batch,
                         cudaStream_t s);
int launch_act_rainbow(const dmdqn_dims& d, const dmdqn_nets& nets, const dmdqn_noisy* noisy, const dmdqn_dist& ds,
                       const float* obs, int32_t stride, const double* eps, const uint32_t* w1, const uint32_t* w2,
                       int32_t* actions, float* q_out, cudaStream_t s);

}  // namespace dmdqn
