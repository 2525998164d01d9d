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

// Float offsets of W1|b1|W2|b2|W3|b3 inside one parameter block (include/dmdqn_b200.h).
struct Layout {
    int64_t w1, b1, w2, b2, w3, b3, stride;
};
__host__ __device__ inline Layout make_layout(int dp, int h) {
    Layout l;
    l.w1 = 0;
    l.b1 = (int64_t)dp * h;
    l.w2 = l.b1 + h;
    l.b2 = l.w2 + (int64_t)h * h;
    l.w3 = l.b2 + h;
    l.b3 = l.w3 + (int64_t)h * 4;
    l.stride = (l.b3 + 4 + 31) / 32 * 32;  // blocks start on 128-byte lines
    return l;
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
               const double* eps, const uint32_t* w1, const uint32_t* w2, int32_t* actions, float* q_out,
               cudaStream_t s);
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
int launch_sync_target(const dmdqn_dims& d, const dmdqn_nets& nets, const uint8_t* mask, double tau,
                       cudaStream_t s);
int launch_peer_adam(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const dmdqn_peers& peers,
                     const float* my_loss_src, float* loss_out, char* ws, const Workspace& w, cudaStream_t s);

}  // namespace dmdqn
