// K1 -- device-resident ring replay buffer: push, sample (index draw + reward z-score), gather.
//
// Replaces ReplayBuffer.add / sample / __len__ and DQNAgent.remember / store_experience
// (reference src/agents/dqn_agent.py:27-89,306-325).  The ring keeps deque(maxlen=C)
// semantics: logical index j (0 = oldest) lives in slot (n_written - size + j) mod C.
// Rows are padded to obs_stride floats (89 -> 96: three whole 128-byte lines) so that every
// gather in K3/K4 is made of aligned 16-byte accesses.
#include "common.cuh"

namespace dmdqn {

namespace {

// ---------------------------------------------------------------- push ------------------
__global__ void __launch_bounds__(64)
push_kernel(dmdqn_dims d, dmdqn_replay rp, const float* __restrict__ obs, const int32_t* __restrict__ act,
            const double* __restrict__ rew, const float* __restrict__ next_obs,
            const uint8_t* __restrict__ done, int in_stride, const uint8_t* __restrict__ mask) {
    const int a = blockIdx.x;
    if (mask && !mask[a]) return;
    const long long nw = rp.n_written[a];
    const size_t row = (size_t)a * d.capacity + (size_t)(nw % d.capacity);  // overwrite the oldest
    float* dst_s = rp.obs + row * d.obs_stride;
    float* dst_n = rp.next_obs + row * d.obs_stride;
    for (int c = threadIdx.x; c < d.obs_stride; c += blockDim.x) {
        const bool in = c < d.obs_dim;
        dst_s[c] = in ? obs[(size_t)a * in_stride + c] : 0.f;
        dst_n[c] = in ? next_obs[(size_t)a * in_stride + c] : 0.f;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        rp.act[row] = act[a];
        rp.rew[row] = rew[a];
        rp.done[row] = done[a] ? 1 : 0;
        rp.n_written[a] = nw + 1;
        if (rp.priority) rp.priority[row] = rp.priority_max[a];   // a new transition gets the ring's largest priority
    }
}

// ---------------------------------------------------------------- sample ----------------
constexpr int kSampleThreads = 256;
constexpr int kPerChunk = 128;                 // prioritized replay: slots per chunk of the canonical priority sum
constexpr int kPerScan = 8;                    // chunks a warp loads before it adds (32 loads in flight per lane)

// Canonical float64 tree sum over a batch held in shared memory: lane l adds elements
// l, l+32, ... in order, then an xor butterfly (16,8,4,2,1).  oracle/replay.py
// zscore_canonical restates exactly this, so the z-score is bit-comparable.
template <typename F>
__device__ __forceinline__ double tree_sum(int n, int lane, F elem) {
    double acc = 0.0;
    for (int i = lane; i < n; i += 32) acc = __dadd_rn(acc, elem(i));
    for (int off = 16; off; off >>= 1) acc = __dadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
    return acc;
}

// n-step return of a row whose first-step term is z0: the later rewards of rows j+1 .. j+m-1 (ring row `row` = row j)
// are read again here, L1/L2-hot since the lookahead read their done flags; every load is issued before the sum.
// R = z0; g = 1; for k = 1..m-1: g = g * gamma; R = R + g * z_k, float64 with separate multiply and add.
__device__ __forceinline__ double nstep_return(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, int row,
                                               int m, double z0, double mean, double denom, bool normalize) {
    if (m <= 1) return z0;
    const int C = d.capacity, agent = row / C, slot = row - agent * C;
    const double* rw = rp.rew + (size_t)agent * C;
    double r[DMDQN_MAX_NSTEP - 1];
#pragma unroll
    for (int k = 1; k < DMDQN_MAX_NSTEP; ++k) r[k - 1] = k < m ? rw[slot + k < C ? slot + k : slot + k - C] : 0.0;
    double ret = z0, gk = 1.0;
#pragma unroll
    for (int k = 1; k < DMDQN_MAX_NSTEP; ++k) {
        if (k < m) {
            gk = __dmul_rn(gk, hp.gamma);
            const double z = normalize ? __ddiv_rn(__dsub_rn(r[k - 1], mean), denom) : r[k - 1];
            ret = __dadd_rn(ret, __dmul_rn(gk, z));
        }
    }
    return ret;
}

// One CTA per network.  smem: js[B] (draws in, then j_i), pt[B], words[B] (logical indices out), rs[B].
//
// Draw without replacement = CPython random.sample's pool path with randbelow(m) := (w*m) >> 32
// (reference dqn_agent.py:63):   for i in 0..B-1:  j_i = randbelow(n-i); result[i] = pool[j_i];
// pool[j_i] = pool[t_i], t_i = n-i-1, pool = identity at the start.  The loop is sequential only through
// the <= B displaced pool entries, so it is resolved in parallel instead of replayed:
//   W_k := the value step k writes to pool[j_k] = pool_k[t_k] = W_{pt[k]} if pt[k] >= 0 else t_k,
//          pt[k] = latest k' < k with j_k' == t_k  (the only way position t_k was displaced before step k)
//   result[i] = W_{pj[i]} if pj[i] >= 0 else j_i,   pj[i] = latest k < i with j_k == j_i.
// pj / pt come from a B x B compare (thread i scans k < i; every read is a shared-memory broadcast) and
// the W chains (almost always of length 0 or 1) are chased read-only.  Same integers as the sequential
// loop for every input (oracle/replay.py fisher_yates_indices replays the loop itself).
// PER: DMDQN_SAMPLE_PRIORITIZED (its own instantiation, so the uniform modes compile to the same code as without it).
// NSTEP: hp.n_step > 1, n-step returns (include/dmdqn_b200.h dmdqn_sample; tests/replay_oracle.py restates every step).  The
// one-step instantiation writes the drawn row as the bootstrap row and gamma * (1 - done) as the discount.
// (Running n_step 1 through the n-step path instead was measured slower at n_step 1: DESIGN.md section 8.)
template <bool PER, bool NSTEP>
__global__ void __launch_bounds__(kSampleThreads)
sample_kernel(dmdqn_dims d, dmdqn_hparams hp, dmdqn_replay rp, int32_t* __restrict__ learn_step,
              const uint32_t* __restrict__ draws, const uint8_t* __restrict__ learn_mask, int advance,
              int32_t* __restrict__ rows, float* __restrict__ r_hat, int32_t* __restrict__ act_b,
              float* __restrict__ done_b, int32_t* __restrict__ active, float4* __restrict__ adam_sc,
              int32_t* __restrict__ sync, int tiles, float* __restrict__ is_w, int32_t* __restrict__ nrows,
              float* __restrict__ disc_b) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int B = d.batch, Bp = (B + 1) & ~1;
    int* js = reinterpret_cast<int*>(smem_raw);
    int* pt = js + Bp;
    int* words = pt + Bp;
    double* rs = reinterpret_cast<double*>(words + Bp);
    __shared__ double stat[2];
    __shared__ int per_last, per_pmin;         // prioritized replay: last slot with a non-zero priority, min drawn priority (bits)
    __shared__ double per_beta;
    const int g = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const bool per = hp.sample_mode == DMDQN_SAMPLE_PRIORITIZED;
    const bool shared_net = d.n_nets == 1 && d.n_agents > 1;
    // dataflow flags of the tcgen05 learn kernels (learn_tc.cu): this launch is ordered after every kernel of the previous
    // step, so it is the one place where they can be reset without a race
    // K3 of the same call is a programmatic dependent launch: its CTAs may set up (barriers, TMEM) while this grid runs; they
    // read nothing of this kernel's before their griddepcontrol.wait, which returns when this grid has completed
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tid < 4 && g == 0) sync[tid] = 0;
    if (tid == 4) sync[4 + g] = 0;
    if (tid >= 32 && tid < 32 + tiles) sync[4 + d.n_nets + g * tiles + (tid - 32)] = 0;

    // Population: this agent's ring, or (shared parameters) all rings of this GPU, which the
    // host keeps equally filled, concatenated agent-major.
    const long long nw0 = rp.n_written[shared_net ? 0 : g];
    const int size0 = (int)(nw0 < d.capacity ? nw0 : d.capacity);
    const long long pop = shared_net ? (long long)size0 * d.n_agents : size0;
    const bool on = (learn_mask == nullptr || learn_mask[g]) && pop >= B;  // dqn_agent.py:61-62
    int t_step = 0;
    if (tid == 0) {
        active[g] = on ? 1 : 0;
        int t = learn_step[g];
        if (on && advance) learn_step[g] = ++t;    // dqn_agent.py:359
        t_step = t;
    }
    if (!on) return;
    // Adam scalars of this step, the only place they are evaluated (every Adam kernel loads them with adam_step, common.cuh):
    // alpha_t = lr * sqrt(1 - b2^t) / (1 - b1^t) in float64, then rounded (oracle/dqn.py adam_scalars).  Two double-precision
    // pow() calls (~2 us) by ONE thread: thread 0 runs them while the other warps are still in their index scan (warp 0's is
    // the shortest), not in front of a barrier every thread waits at.
    auto adam_scalars = [&]() {
        const int t = t_step;
        const double bc1 = 1.0 - pow(hp.beta1, (double)t), bc2 = 1.0 - pow(hp.beta2, (double)t);
        const int freq = hp.target_update_frequency > 0 ? hp.target_update_frequency : 1;
        const int sync_mode = hp.tau >= 0.0 ? 2 : (t % freq == 0 ? 1 : 0);          // counter already incremented (:359,376)
        adam_sc[g] = make_float4((float)(hp.learning_rate * sqrt(bc2) / bc1),
                                 (float)(hp.adam_form == DMDQN_ADAM_KERAS ? hp.adam_eps : hp.adam_eps * sqrt(bc2)),
                                 __int_as_float(sync_mode), 0.f);
    };

    if constexpr (PER) {
        // Proportional prioritized replay (include/dmdqn_b200.h; tests/replay_oracle.py restates every step): words[i] is
        // the drawn PHYSICAL slot here, not a logical index.
        const int C = d.capacity, nch = (C + kPerChunk - 1) / kPerChunk, warp = tid >> 5;
        const float* __restrict__ pr = rp.priority + (size_t)g * C;
        double* prefix = rs + Bp;                       // [nch + 1]: chunk totals, then their exclusive prefixes
        if (tid == 0) { per_last = -1; per_pmin = 0x7f800000; }
        int last = -1;
        for (int c0 = warp * kPerScan; c0 < nch; c0 += (kSampleThreads / 32) * kPerScan) {
            float v[kPerScan][4];
#pragma unroll
            for (int u = 0; u < kPerScan; ++u)          // every load of the group is issued before the first add
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int sl = (c0 + u) * kPerChunk + 32 * k + lane;
                    v[u][k] = sl < C ? __ldg(pr + sl) : 0.f;
                }
#pragma unroll
            for (int u = 0; u < kPerScan; ++u) {        // chunk total: lane l adds slots l, l+32, l+64, l+96, then the butterfly
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    acc = __dadd_rn(acc, (double)v[u][k]);
                    if (v[u][k] > 0.f) last = (c0 + u) * kPerChunk + 32 * k + lane;
                }
                for (int off = 16; off; off >>= 1) acc = __dadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, off));
                if (lane == 0 && c0 + u < nch) prefix[c0 + u + 1] = acc;
            }
        }
        last = __reduce_max_sync(0xffffffffu, last);
        __syncthreads();                                // per_last / per_pmin initialised, chunk totals in place
        if (lane == 0 && last >= 0) atomicMax(&per_last, last);
        if (tid == 32) {                                // chunk totals -> exclusive prefixes, in chunk order
            double run = 0.0;
            prefix[0] = 0.0;
            for (int c = 1; c <= nch; ++c) {
                run = __dadd_rn(run, prefix[c]);
                prefix[c] = run;
            }
        }
        if (tid == 0) {
            adam_scalars();
            double beta = hp.per_beta0;                 // beta_t of this step, t = learn_step after the increment
            if (hp.per_beta_steps > 0)
                beta = fmin(1.0, __dadd_rn(hp.per_beta0, __ddiv_rn(__dmul_rn(__dsub_rn(1.0, hp.per_beta0), (double)t_step),
                                                                   (double)hp.per_beta_steps)));
            per_beta = beta;
        }
        __syncthreads();
        const double S = prefix[nch];
        for (int i = tid; i < B; i += kSampleThreads) {
            const double w = (double)draws[(size_t)g * B + i];
            const double u = __ddiv_rn(__dmul_rn(__dadd_rn((double)i, __dmul_rn(w, 0x1p-32)), S), (double)B);
            int lo = 0, hi = nch - 1;                   // the last chunk whose exclusive prefix is <= u
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (prefix[mid] <= u) lo = mid; else hi = mid - 1;
            }
            const int base = lo * kPerChunk;
            double run = prefix[lo];
            int slot = -1;
            for (int s0 = 0; s0 < kPerChunk && slot < 0; s0 += 32) {   // walk the chunk in slot order, 32 loads ahead of the adds
                float v[32];
#pragma unroll
                for (int k = 0; k < 32; ++k) v[k] = base + s0 + k < C ? __ldg(pr + base + s0 + k) : 0.f;
#pragma unroll
                for (int k = 0; k < 32; ++k) {
                    run = __dadd_rn(run, (double)v[k]);
                    if (slot < 0 && run > u) slot = base + s0 + k;
                }
            }
            if (slot < 0) slot = per_last >= 0 ? per_last : 0;         // rounding carried the walk past the chunk
            words[i] = slot;
            atomicMin(&per_pmin, __float_as_int(__ldg(pr + slot)));
        }
    } else if (hp.sample_mode == DMDQN_SAMPLE_FISHER_YATES) {
        const int n = (int)pop;
        for (int i = tid; i < B; i += kSampleThreads)
            js[i] = (int)__umulhi(draws[(size_t)g * B + i], (unsigned)(n - i));
        __syncthreads();
        for (int i0 = 0; i0 < B; i0 += kSampleThreads) {   // the warp's trip count is its largest i: keep the loop warp-uniform
            const int i = i0 + tid;
            const int ji = i < B ? js[i] : -1, ti = i < B ? n - i - 1 : -1;
            int pj = -1, ptk = -1;
            const int kend = min(B, i0 + (tid | 31));       // every lane of the warp scans up to the warp's last i (extra k >= i are masked)
#pragma unroll 4
            for (int k = 0; k < kend; ++k) {
                const int jk = js[k];
                const bool before = k < i;
                pj = (before && jk == ji) ? k : pj;
                ptk = (before && jk == ti) ? k : ptk;
            }
            if (i < B) { pt[i] = ptk; words[i] = pj; }
        }
        if (tid == 0) adam_scalars();
        __syncthreads();
        for (int i = tid; i < B; i += kSampleThreads) {    // words[i] is read and rewritten by its own thread only
            int k = words[i];
            int v = js[i];
            if (k >= 0) {
                while (pt[k] >= 0) k = pt[k];
                v = n - k - 1;
            }
            words[i] = v;
        }
    } else if (hp.sample_mode == DMDQN_SAMPLE_REPLACEMENT) {
        for (int i = tid; i < B; i += kSampleThreads) words[i] = (int)__umulhi(draws[(size_t)g * B + i], (unsigned)pop);
        if (tid == 0) adam_scalars();
    } else {                                            // explicit logical indices, clamped
        for (int i = tid; i < B; i += kSampleThreads) {
            const int v = (int)draws[(size_t)g * B + i];
            words[i] = v < 0 ? 0 : (v >= pop ? (int)pop - 1 : v);
        }
        if (tid == 0) adam_scalars();
    }
    __syncthreads();

    for (int i = tid; i < B; i += kSampleThreads) {
        const int logical = words[i];
        const int agent = shared_net ? logical / size0 : g;
        const int lj = shared_net ? logical % size0 : logical;
        const long long nw = shared_net ? rp.n_written[agent] : nw0;
        const long long sz = nw < d.capacity ? nw : d.capacity;
        const int slot = per ? words[i] : (int)((nw - sz + lj) % d.capacity);
        const int row = agent * d.capacity + slot;
        if constexpr (PER) {                            // importance weight (p_min / p_i)^beta_t in float64
            const float p = rp.priority[row];
            is_w[(size_t)g * B + i] = p > 0.f ? (float)pow(__ddiv_rn((double)__int_as_float(per_pmin), (double)p), per_beta) : 1.f;
        }
        rows[(size_t)g * B + i] = row;
        // (an L2 prefetch of the two sampled rows was measured here: +6 us in this kernel, nothing gained in K3 / K4a)
        act_b[(size_t)g * B + i] = rp.act[row];
        if constexpr (!NSTEP) {
            const bool dn = rp.done[row];
            done_b[(size_t)g * B + i] = dn ? 1.f : 0.f;
            js[i] = row;                                // the draw's scratch is free now: row and done for the pass below
            pt[i] = dn;
        }
        rs[i] = rp.rew[row];
        if constexpr (NSTEP) {
            // the return covers rows j .. j+m-1 of this agent's ring: up to n_step, the first done, the newest row
            const int C = d.capacity;
            const int j = per ? (int)(((long long)slot - (nw - sz) % C + C) % C) : lj;
            const int lim = min(hp.n_step, (int)sz - j);
            const uint8_t* dn = rp.done + (size_t)agent * C;
            unsigned bits = 0;                          // bit k: row j+k is done; every load is issued before the scan
#pragma unroll
            for (int k = 0; k < DMDQN_MAX_NSTEP; ++k)
                if (k < lim && dn[slot + k < C ? slot + k : slot + k - C]) bits |= 1u << k;
            const int m = bits ? __ffs(bits) : lim;
            double gm = hp.gamma;                       // gamma^m, float64, left to right
            for (int k = 1; k < m; ++k) gm = __dmul_rn(gm, hp.gamma);
            const int last = slot + m - 1;
            nrows[(size_t)g * B + i] = agent * C + (last < C ? last : last - C);
            done_b[(size_t)g * B + i] = bits ? 1.f : 0.f;      // the return ends on its first done, if any
            disc_b[(size_t)g * B + i] = bits ? 0.f : (float)gm;
            js[i] = row;                                // the draw's scratch is free now: row and m for the reward pass
            pt[i] = m;
        }
    }
    __syncthreads();
    if constexpr (!NSTEP) {     // one-step targets bootstrap from the drawn row: warps 1.. write them while warp 0 sums
        for (int i = tid - 32; tid >= 32 && i < B; i += kSampleThreads - 32) {
            nrows[(size_t)g * B + i] = js[i];
            disc_b[(size_t)g * B + i] = (float)hp.gamma * (1.0f - (pt[i] ? 1.f : 0.f));
        }
    }
    if (hp.normalize_rewards) {                         // dqn_agent.py:66-69, float64; warp 0 keeps the canonical tree
        if (tid < 32) {
            const double mean = __ddiv_rn(tree_sum(B, lane, [&](int i) { return rs[i]; }), (double)B);
            const double var = __ddiv_rn(tree_sum(B, lane, [&](int i) {
                                             const double dv = __dsub_rn(rs[i], mean);
                                             return __dmul_rn(dv, dv);
                                         }), (double)B);
            if (lane == 0) { stat[0] = mean; stat[1] = __dadd_rn(__dsqrt_rn(var), 1e-8); }
        }
        __syncthreads();
        const double mean = stat[0], denom = stat[1];
        for (int i = tid; i < B; i += kSampleThreads) {
            const double z = __ddiv_rn(__dsub_rn(rs[i], mean), denom);
            r_hat[(size_t)g * B + i] = (float)(NSTEP ? nstep_return(d, hp, rp, js[i], pt[i], z, mean, denom, true) : z);
        }
    } else {
        for (int i = tid; i < B; i += kSampleThreads)
            r_hat[(size_t)g * B + i] = (float)(NSTEP ? nstep_return(d, hp, rp, js[i], pt[i], rs[i], 0.0, 1.0, false) : rs[i]);
    }
}

// ---------------------------------------------------------------- gather ----------------
// One warp per sampled transition.  The ring rows are obs_stride floats (whole 128-byte lines, 16-byte aligned), so the
// read side is one 16-byte load per lane and tensor (24 of the 32 lanes at obs_stride = 96); the dense output rows are
// obs_dim = 89 floats, i.e. not 16-byte aligned from row to row, so the write side stays 4-byte but fully coalesced:
// the pieces are exchanged through shuffles so that lane l writes columns l, l + 32, l + 64 (consecutive lanes ->
// consecutive addresses, whole 128-byte segments).
__global__ void __launch_bounds__(128)
gather_kernel(dmdqn_dims d, dmdqn_replay rp, const int32_t* __restrict__ rows, const int32_t* __restrict__ nrows,
              const float* __restrict__ r_hat,
              const int32_t* __restrict__ act_b, const float* __restrict__ done_b,
              const int32_t* __restrict__ active, float* __restrict__ states, int32_t* __restrict__ actions,
              float* __restrict__ rewards, float* __restrict__ next_states, float* __restrict__ dones,
              int32_t* __restrict__ active_out) {
    const int lane = threadIdx.x & 31;
    const long long r = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
    const long long total = (long long)d.n_nets * d.batch;
    if (r >= total) return;
    const int g = (int)(r / d.batch);
    if (active_out && (r % d.batch) == 0 && lane == 0) active_out[g] = active[g];
    if (!active[g]) return;
    const size_t src = (size_t)rows[r] * d.obs_stride;             // s of the drawn row
    const size_t nsrc = (size_t)nrows[r] * d.obs_stride;           // s' of its bootstrap row (n-step returns)
    const int q = d.obs_stride >> 2;                               // 16-byte pieces per row (<= 32: obs_stride <= 128)
    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), n4 = s4;
    if (lane < q) {
        s4 = __ldg(reinterpret_cast<const float4*>(rp.obs + src) + lane);
        n4 = __ldg(reinterpret_cast<const float4*>(rp.next_obs + nsrc) + lane);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {                                   // column c = 32 k + lane lives in piece c / 4 = 8 k + lane / 4, component lane % 4
        const int c = 32 * k + lane, from = 8 * k + (lane >> 2);
        const float sx = __shfl_sync(0xffffffffu, s4.x, from), sy = __shfl_sync(0xffffffffu, s4.y, from);
        const float sz = __shfl_sync(0xffffffffu, s4.z, from), sw = __shfl_sync(0xffffffffu, s4.w, from);
        const float nx = __shfl_sync(0xffffffffu, n4.x, from), ny = __shfl_sync(0xffffffffu, n4.y, from);
        const float nz = __shfl_sync(0xffffffffu, n4.z, from), nw = __shfl_sync(0xffffffffu, n4.w, from);
        const int comp = lane & 3;
        if (c < d.obs_dim) {
            states[r * d.obs_dim + c] = comp == 0 ? sx : comp == 1 ? sy : comp == 2 ? sz : sw;
            next_states[r * d.obs_dim + c] = comp == 0 ? nx : comp == 1 ? ny : comp == 2 ? nz : nw;
        }
    }
    if (lane == 0) {
        actions[r] = act_b[r];
        rewards[r] = r_hat[r];
        dones[r] = done_b[r];
    }
}

}  // namespace

int launch_push(const dmdqn_dims& d, const dmdqn_replay& rp, const float* obs, const int32_t* act,
                const double* rew, const float* next_obs, const uint8_t* done, int32_t in_stride,
                const uint8_t* mask, cudaStream_t s) {
    push_kernel<<<d.n_agents, 64, 0, s>>>(d, rp, obs, act, rew, next_obs, done, in_stride, mask);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_sample(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                  const void* draws, const uint8_t* learn_mask, int advance, char* ws, const Workspace& w,
                  cudaStream_t s) {
    DMDQN_CHECK_ARG(d.batch <= 4096, "batch %d: the sample kernel serves batches up to 4096", d.batch);
    const bool per = hp.sample_mode == DMDQN_SAMPLE_PRIORITIZED;
    // prioritized replay keeps the chunk prefixes of the ring in shared memory (8 bytes per 128 slots)
    DMDQN_CHECK_ARG(!per || d.capacity <= DMDQN_PER_MAX_CAPACITY,
                    "capacity=%d: prioritized replay serves rings of up to %d slots", d.capacity, DMDQN_PER_MAX_CAPACITY);
    const size_t smem = (size_t)((d.batch + 1) & ~1) * (3 * 4 + 8) +
                        (per ? (size_t)((d.capacity + kPerChunk - 1) / kPerChunk + 1) * 8 : 0);
    const bool nstep = hp.n_step > 1;
    static size_t configured[4][kMaxDevices] = {};
    const auto kernel = per ? (nstep ? sample_kernel<true, true> : sample_kernel<true, false>)
                            : (nstep ? sample_kernel<false, true> : sample_kernel<false, false>);
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(kernel), smem, configured[2 * per + nstep])) return rc;
    kernel<<<d.n_nets, kSampleThreads, smem, s>>>(
        d, hp, rp, nets.learn_step, static_cast<const uint32_t*>(draws), learn_mask, advance,
        reinterpret_cast<int32_t*>(ws + w.rows), reinterpret_cast<float*>(ws + w.r_hat),
        reinterpret_cast<int32_t*>(ws + w.act_b), reinterpret_cast<float*>(ws + w.done_b),
        reinterpret_cast<int32_t*>(ws + w.active), reinterpret_cast<float4*>(ws + w.adam_sc),
        reinterpret_cast<int32_t*>(ws + w.sync), w.tiles, reinterpret_cast<float*>(ws + w.is_w),
        reinterpret_cast<int32_t*>(ws + w.nrows), reinterpret_cast<float*>(ws + w.disc_b));
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_gather(const dmdqn_dims& d, const dmdqn_replay& rp, const char* ws, const Workspace& w,
                  float* states, int32_t* actions, float* rewards, float* next_states, float* dones,
                  int32_t* active_out, cudaStream_t s) {
    const long long total = (long long)d.n_nets * d.batch;
    gather_kernel<<<(unsigned)((total + 3) / 4), 128, 0, s>>>(
        d, rp, reinterpret_cast<const int32_t*>(ws + w.rows), reinterpret_cast<const int32_t*>(ws + w.nrows),
        reinterpret_cast<const float*>(ws + w.r_hat),
        reinterpret_cast<const int32_t*>(ws + w.act_b), reinterpret_cast<const float*>(ws + w.done_b),
        reinterpret_cast<const int32_t*>(ws + w.active), states, actions, rewards, next_states, dones,
        active_out);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

}  // namespace dmdqn
