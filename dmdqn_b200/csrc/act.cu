// K2 -- batched epsilon-greedy action selection: a cluster of four CTAs per agent runs the batch-1
// MLP (89 -> H -> H -> 4) as a GEMV chain with argmax and the epsilon mask fused in.
//
// Replaces DQNAgent.select_action (reference src/agents/dqn_agent.py:263-274) and
// select_greedy_action (reference src/experimental/agent.py:148-152).
// HBM bound: every action reads the agent's 4*P weight bytes once (AI 0.5 flop/B).  The layer outputs
// are split by columns over the four CTAs of a cluster (each streams a [K][H/4] slice of W1 and W2
// with 16-byte loads, every load of a layer in flight at once), the activation slices are exchanged
// through distributed shared memory, and the K split over thread groups is combined in a fixed order
// (deterministic Q-values).  Four CTAs per agent give 1024 CTAs at 256 agents; the launch bound asks for four
// resident CTAs per SM (64 registers: measured best -- 2 / 3 / 4 / 5 / 6 per SM give 24 / 21 / 20 / 27 / 33 us at 256
// agents): an agent is a chain of two HBM latencies, three cluster barriers and serial reductions, so the number of
// agents in flight matters more than the number of loads each thread keeps in flight.
// Exploring agents skip the forward pass, as the reference does.
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace dmdqn {

namespace {

constexpr int kActThreads = 256;
constexpr int kActCluster = 4;

// This CTA's column slice of a layer, in two steps so that the weight loads of BOTH hidden layers are in flight
// before the first FMA (they do not depend on the activations): load_slice issues every 16-byte load of the
// [K][H/4] slice, gemv_slice consumes them: out[c0 .. c0 + Hs) = relu(bias + x[0..K) . W) written into the `out`
// buffer of every CTA of the cluster.  x, part in (local) shared memory.  MAXIT = ceil(K / groups).
template <int MAXIT>
__device__ __forceinline__ void load_slice(float4 (&w)[MAXIT], const float* __restrict__ W, int K, int H, int rank) {
    const int Hs = H / kActCluster, c4 = Hs >> 2;        // threads covering one row slice with float4
    const int groups = kActThreads / c4;                 // K is split over this many thread groups
    const int col4 = threadIdx.x % c4, grp = threadIdx.x / c4;
    const float4* Wv = reinterpret_cast<const float4*>(W + rank * Hs) + col4;
#pragma unroll
    for (int i = 0; i < MAXIT; ++i) {
        const int k = grp + i * groups;
        w[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k < K)                                       // volatile: ptxas would otherwise sink the loads to their uses
            asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(w[i].x), "=f"(w[i].y), "=f"(w[i].z), "=f"(w[i].w)
                         : "l"(Wv + (size_t)k * (H >> 2)));
    }
}

template <int MAXIT>
__device__ __forceinline__ void gemv_slice(cg::cluster_group& cluster, const float4 (&w)[MAXIT], const float* __restrict__ bias,
                                           const float* x, float* out, float* part, int K, int H, int rank) {
    const int Hs = H / kActCluster, c4 = Hs >> 2;
    const int groups = kActThreads / c4;
    const int col4 = threadIdx.x % c4, grp = threadIdx.x / c4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < MAXIT; ++i) {
        const int k = grp + i * groups;
        float xv = 0.f;                                  // volatile too: keeps every FMA behind the last global load
        if (k < K) asm volatile("ld.shared.f32 %0, [%1];" : "=f"(xv) : "r"((uint32_t)__cvta_generic_to_shared(x + k)));
        acc.x = fmaf(xv, w[i].x, acc.x);
        acc.y = fmaf(xv, w[i].y, acc.y);
        acc.z = fmaf(xv, w[i].z, acc.z);
        acc.w = fmaf(xv, w[i].w, acc.w);
    }
    reinterpret_cast<float4*>(part)[grp * c4 + col4] = acc;
    __syncthreads();
    if (threadIdx.x < Hs) {
        const int j = threadIdx.x;
        float s = bias[rank * Hs + j];
        for (int g = 0; g < groups; ++g) s += part[g * Hs + j];
        s = fmaxf(s, 0.f);
#pragma unroll
        for (int r = 0; r < kActCluster; ++r) cluster.map_shared_rank(out, r)[rank * Hs + j] = s;
    }
    cluster.sync();
}

// Same layer slice with the weight rows streamed 8 at a time (wide layers)
__device__ __forceinline__ void gemv_slice_loop(cg::cluster_group& cluster, const float* __restrict__ W, const float* __restrict__ bias,
                                                const float* x, float* out, float* part, int K, int H, int rank) {
    const int Hs = H / kActCluster, c4 = Hs >> 2;
    const int groups = kActThreads / c4;
    const int col4 = threadIdx.x % c4, grp = threadIdx.x / c4;
    const float4* Wv = reinterpret_cast<const float4*>(W + rank * Hs) + col4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
    for (int k = grp; k < K; k += groups) {
        const float4 w = __ldg(Wv + (size_t)k * (H >> 2));
        const float xv = x[k];
        acc.x = fmaf(xv, w.x, acc.x); acc.y = fmaf(xv, w.y, acc.y);
        acc.z = fmaf(xv, w.z, acc.z); acc.w = fmaf(xv, w.w, acc.w);
    }
    reinterpret_cast<float4*>(part)[grp * c4 + col4] = acc;
    __syncthreads();
    if (threadIdx.x < Hs) {
        const int j = threadIdx.x;
        float s = bias[rank * Hs + j];
        for (int g = 0; g < groups; ++g) s += part[g * Hs + j];
        s = fmaxf(s, 0.f);
#pragma unroll
        for (int r = 0; r < kActCluster; ++r) cluster.map_shared_rank(out, r)[rank * Hs + j] = s;
    }
    cluster.sync();
}

// Noisy networks: sigma, key and step counters of the blocks act_kernel<H, DUELING, true> reads (include/dmdqn_b200.h).
struct ActNoise {
    const float* sigma;
    const uint64_t* key;
    const int32_t* learn_step;
    NoiseRec R;
};

// gemv_slice_loop on noisy parameters: each weight is mu + sigma * (fin[k] * fout[col]) and each bias mu + sigma * fout[col],
// formed in registers with the arithmetic of the fold kernel, so the sums are those of the loop above on the folded block.
// fin, fout: this layer's factor vectors in (local) shared memory.
__device__ __forceinline__ void gemv_slice_noisy(cg::cluster_group& cluster, const float* __restrict__ W, const float* __restrict__ Ws,
                                                 const float* __restrict__ bias, const float* __restrict__ bias_s,
                                                 const float* fin, const float* fout, const float* x, float* out, float* part,
                                                 int K, int H, int rank) {
    const int Hs = H / kActCluster, c4 = Hs >> 2;
    const int groups = kActThreads / c4;
    const int col4 = threadIdx.x % c4, grp = threadIdx.x / c4;
    const size_t c0 = (size_t)rank * Hs + 4 * col4;
    const float4* Wv = reinterpret_cast<const float4*>(W + c0);
    const float4* Sv = reinterpret_cast<const float4*>(Ws + c0);
    const float4 fo = *reinterpret_cast<const float4*>(fout + c0);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int k = grp; k < K; k += groups) {
        const float4 m = __ldg(Wv + (size_t)k * (H >> 2)), s = __ldg(Sv + (size_t)k * (H >> 2));
        const float fi = fin[k], xv = x[k];
        acc.x = fmaf(xv, noisy_weight(m.x, s.x, __fmul_rn(fi, fo.x)), acc.x);
        acc.y = fmaf(xv, noisy_weight(m.y, s.y, __fmul_rn(fi, fo.y)), acc.y);
        acc.z = fmaf(xv, noisy_weight(m.z, s.z, __fmul_rn(fi, fo.z)), acc.z);
        acc.w = fmaf(xv, noisy_weight(m.w, s.w, __fmul_rn(fi, fo.w)), acc.w);
    }
    reinterpret_cast<float4*>(part)[grp * c4 + col4] = acc;
    __syncthreads();
    if (threadIdx.x < Hs) {
        const int j = rank * Hs + threadIdx.x;
        float s = noisy_weight(bias[j], bias_s[j], fout[j]);
        for (int g = 0; g < groups; ++g) s += part[g * Hs + threadIdx.x];
        s = fmaxf(s, 0.f);
#pragma unroll
        for (int r = 0; r < kActCluster; ++r) cluster.map_shared_rank(out, r)[j] = s;
    }
    cluster.sync();
}

// DUELING: the block is in the dueling layout and the head is folded (include/dmdqn_b200.h) in registers: every CTA folds
// its W3 rows with their wv weights, rank 0 folds the bias.
// NOISY: the parameters are mu (theta) + sigma * eps with the online noise at the network's learn_step; every CTA builds
// the network's noise record in shared memory with the fold kernel's function and streams mu and sigma (8P bytes per
// action) row by row.
template <int H_, bool DUELING, bool NOISY>
__global__ void __cluster_dims__(kActCluster, 1, 1) __launch_bounds__(kActThreads, 4)
act_kernel(dmdqn_dims d, Layout L, const float* __restrict__ theta, const float* __restrict__ obs, int stride,
           const double* __restrict__ eps, const uint32_t* __restrict__ w_explore,
           const uint32_t* __restrict__ w_action, int32_t* __restrict__ actions, float* __restrict__ q_out, ActNoise nz) {
    extern __shared__ __align__(16) float smem[];
    cg::cluster_group cluster = cg::this_cluster();
    const int a = blockIdx.x / kActCluster, rank = (int)cluster.block_rank();
    constexpr int H = H_;
    const int Dp = d.obs_stride;
    // explore iff u < eps with u = w / 2^32 (dqn_agent.py:263), exact in float64; the same for the four CTAs
    const bool explore = (double)w_explore[a] < eps[a] * 4294967296.0;
    if (explore) {
        if (threadIdx.x == 0 && rank == 0) actions[a] = (int32_t)__umulhi(w_action[a], (uint32_t)d.n_actions);
        return;  // dqn_agent.py:265: no forward pass
    }
    float* xs = smem;            // [Dp]
    float* h1 = xs + Dp;         // [H]
    float* h2 = h1 + H;          // [H]
    float* part = h2 + H;        // [groups][H/4] = [256*4]; later [4 ranks][4] head partials on rank 0
    const int net = d.n_nets == 1 ? 0 : a;
    const float* P = theta + (size_t)net * L.stride;
    const float* S = nullptr;                            // NOISY: sigma's block
    float* rec = part + kActThreads * 4;                 // NOISY: the online noise record
    if constexpr (NOISY) {
        S = nz.sigma + (size_t)net * L.stride;
        noise_record_build(rec, nz.R, d.obs_dim, d.n_actions, __ldg(nz.key + net), (uint32_t)__ldg(nz.learn_step + net), 0);
        for (int c = threadIdx.x; c < Dp; c += kActThreads)
            xs[c] = c < d.obs_dim ? obs[(size_t)a * stride + c] : 0.f;
        __syncthreads();
        gemv_slice_noisy(cluster, P + L.w1, S + L.w1, P + L.b1, S + L.b1, rec + nz.R.off[0], rec + nz.R.off[1], xs, h1, part,
                         Dp, H, rank);
        gemv_slice_noisy(cluster, P + L.w2, S + L.w2, P + L.b2, S + L.b2, rec + nz.R.off[2], rec + nz.R.off[3], h1, h2, part,
                         H, H, rank);
    } else {
        constexpr int C4 = H / kActCluster / 4, GROUPS = kActThreads / C4;
        // The register-resident W1 slice is sized for the yaml observation (89 -> stride 96); wider observations
        // (stride 112 / 128, accepted by validate_dims and by the learn kernels) stream layer 1 row by row instead.
        constexpr int kRegRows = 96;
        if constexpr (H <= 256) {
            if (Dp <= kRegRows) {
                float4 w1[(kRegRows + GROUPS - 1) / GROUPS], w2[(H + GROUPS - 1) / GROUPS];
                load_slice(w1, P + L.w1, Dp, H, rank);       // 4P bytes per action: all of this CTA's share is requested here
                load_slice(w2, P + L.w2, H, H, rank);
                for (int c = threadIdx.x; c < Dp; c += kActThreads)
                    xs[c] = c < d.obs_dim ? obs[(size_t)a * stride + c] : 0.f;
                __syncthreads();
                gemv_slice(cluster, w1, P + L.b1, xs, h1, part, Dp, H, rank);
                gemv_slice(cluster, w2, P + L.b2, h1, h2, part, H, H, rank);
            } else {
                float4 w2[(H + GROUPS - 1) / GROUPS];
                load_slice(w2, P + L.w2, H, H, rank);
                for (int c = threadIdx.x; c < Dp; c += kActThreads)
                    xs[c] = c < d.obs_dim ? obs[(size_t)a * stride + c] : 0.f;
                __syncthreads();
                gemv_slice_loop(cluster, P + L.w1, P + L.b1, xs, h1, part, Dp, H, rank);
                gemv_slice(cluster, w2, P + L.b2, h1, h2, part, H, H, rank);
            }
        } else {                                             // H = 512: a layer's slice does not fit the register file at once
            for (int c = threadIdx.x; c < Dp; c += kActThreads)
                xs[c] = c < d.obs_dim ? obs[(size_t)a * stride + c] : 0.f;
            __syncthreads();
            if (Dp <= kRegRows) {
                float4 w1[(kRegRows + GROUPS - 1) / GROUPS];
                load_slice(w1, P + L.w1, Dp, H, rank);
                gemv_slice(cluster, w1, P + L.b1, xs, h1, part, Dp, H, rank);
            } else {
                gemv_slice_loop(cluster, P + L.w1, P + L.b1, xs, h1, part, Dp, H, rank);
            }
            gemv_slice_loop(cluster, P + L.w2, P + L.b2, h1, h2, part, H, H, rank);
        }
    }

    // layer 3: q[a] = b3[a] + sum_j h2[j] * W3[j][a]: every CTA sums its H/4 rows (warp butterfly, warps in
    // order), rank 0 adds the four partials in rank order
    constexpr int Hs = H / kActCluster;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (threadIdx.x < Hs) {
        const int j = rank * Hs + threadIdx.x;
        float4 w = __ldg(reinterpret_cast<const float4*>(P + L.w3) + j);
        float v = 0.f;
        if constexpr (DUELING) v = __ldg(P + layout_wv(L) + j);
        if constexpr (NOISY) {
            const float4 s = __ldg(reinterpret_cast<const float4*>(S + L.w3) + j);
            const float fi = rec[nz.R.off[4] + j], *fo = rec + nz.R.off[5];
            w = make_float4(noisy_weight(w.x, s.x, __fmul_rn(fi, fo[0])), noisy_weight(w.y, s.y, __fmul_rn(fi, fo[1])),
                            noisy_weight(w.z, s.z, __fmul_rn(fi, fo[2])), noisy_weight(w.w, s.w, __fmul_rn(fi, fo[3])));
            if constexpr (DUELING)
                v = noisy_weight(v, __ldg(S + layout_wv(L) + j), __fmul_rn(rec[nz.R.off[6] + j], rec[nz.R.off[7]]));
        }
        if constexpr (DUELING) {
            float x[4] = {w.x, w.y, w.z, w.w};
            head_fold(x, v, d.n_actions);
            w = make_float4(x[0], x[1], x[2], x[3]);
        }
        const float hv = h2[j];
        p = make_float4(hv * w.x, hv * w.y, hv * w.z, hv * w.w);
    }
    for (int off = 16; off; off >>= 1) {
        p.x += __shfl_xor_sync(0xffffffffu, p.x, off);
        p.y += __shfl_xor_sync(0xffffffffu, p.y, off);
        p.z += __shfl_xor_sync(0xffffffffu, p.z, off);
        p.w += __shfl_xor_sync(0xffffffffu, p.w, off);
    }
    __syncthreads();             // part is reused
    float4* wsum = reinterpret_cast<float4*>(part);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = p;
    __syncthreads();
    if (threadIdx.x == 0) {
        float4 t = wsum[0];
        for (int w = 1; w < (Hs + 31) / 32; ++w) { t.x += wsum[w].x; t.y += wsum[w].y; t.z += wsum[w].z; t.w += wsum[w].w; }
        reinterpret_cast<float4*>(cluster.map_shared_rank(part, 0))[16 + rank] = t;
    }
    cluster.sync();
    if (threadIdx.x == 0 && rank == 0) {
        float q[4] = {P[L.b3 + 0], P[L.b3 + 1], P[L.b3 + 2], P[L.b3 + 3]};
        float bv = 0.f;
        if constexpr (DUELING) bv = P[layout_bv(L, H)];
        if constexpr (NOISY) {
            const float* fo = rec + nz.R.off[5];
            for (int k = 0; k < 4; ++k) q[k] = noisy_weight(q[k], S[L.b3 + k], fo[k]);
            if constexpr (DUELING) bv = noisy_weight(bv, S[layout_bv(L, H)], rec[nz.R.off[7]]);
        }
        if constexpr (DUELING) head_fold(q, bv, d.n_actions);
        for (int r = 0; r < kActCluster; ++r) {
            const float4 t = reinterpret_cast<const float4*>(part)[16 + r];
            q[0] += t.x; q[1] += t.y; q[2] += t.z; q[3] += t.w;
        }
        int best = 0;                                   // ties -> lowest index (torch.argmax)
        for (int k = 1; k < d.n_actions; ++k) if (q[k] > q[best]) best = k;
        actions[a] = best;
        if (q_out) {
            for (int k = 0; k < 4; ++k) q_out[(size_t)a * 4 + k] = q[k];
        }
    }
}

}  // namespace

int launch_act(const dmdqn_dims& d, const dmdqn_nets& nets, const float* obs, int32_t stride,
               const double* eps, const uint32_t* w1, const uint32_t* w2, int32_t* actions, float* q_out, bool dueling,
               cudaStream_t s, const dmdqn_noisy* noisy) {
    const Layout L = make_layout(d.obs_stride, d.hidden, dueling);
    ActNoise nz = {};
    nz.R = make_noise_rec(d.obs_stride, d.hidden);
    size_t smem = (size_t)(d.obs_stride + 2 * d.hidden + kActThreads * 4) * sizeof(float);
    if (noisy) {
        nz.sigma = noisy->sigma; nz.key = noisy->key; nz.learn_step = nets.learn_step;
        smem += (size_t)nz.R.stride * sizeof(float);
    }
    const dim3 grid(d.n_agents * kActCluster);
    auto run = [&](auto kernel) {
        kernel<<<grid, kActThreads, smem, s>>>(d, L, nets.theta, obs, stride, eps, w1, w2, actions, q_out, nz);
    };
    switch (d.hidden * 4 + (dueling ? 1 : 0) + (noisy ? 2 : 0)) {
        case 256: run(act_kernel<64, false, false>); break;
        case 257: run(act_kernel<64, true, false>); break;
        case 258: run(act_kernel<64, false, true>); break;
        case 259: run(act_kernel<64, true, true>); break;
        case 512: run(act_kernel<128, false, false>); break;
        case 513: run(act_kernel<128, true, false>); break;
        case 514: run(act_kernel<128, false, true>); break;
        case 515: run(act_kernel<128, true, true>); break;
        case 1024: run(act_kernel<256, false, false>); break;
        case 1025: run(act_kernel<256, true, false>); break;
        case 1026: run(act_kernel<256, false, true>); break;
        case 1027: run(act_kernel<256, true, true>); break;
        case 2048: run(act_kernel<512, false, false>); break;
        case 2049: run(act_kernel<512, true, false>); break;
        case 2050: run(act_kernel<512, false, true>); break;
        case 2051: run(act_kernel<512, true, true>); break;
        default: DMDQN_CHECK_ARG(false, "hidden=%d: the act kernel is built for 64, 128, 256, 512", d.hidden);
    }
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

}  // namespace dmdqn
