// K3 / K4 -- the Double-DQN learn step, fp32 (FFMA) path.
//
// Replaces DQNAgent.learn (reference src/agents/dqn_agent.py:328-380):
//   K3  target_kernel      gather s' -> online(s') -> argmax, target(s') -> TD target y   (:342-347)
//   K4a online_kernel      gather s  -> online(s) keeping h1,h2 -> loss, dL/dq -> dh2, dh1  (:349-356)
//   K4b wgrad_adam_kernel  dW = A^T * D per layer, Adam in the epilogue, hard/Polyak sync  (:357,372-377)
//
// Tiling (Tile<H>, common.cuh): a CTA owns BM batch rows of one network and ALL H output
// columns of a layer, so activations never leave shared memory between layers; weights are
// streamed through shared memory in KC-row chunks (register-staged double buffer); each
// thread owns an 8x8 register tile (rows split 4+4, columns split 4+4 so that every
// 16-byte shared-memory access of a quarter-warp is conflict-free).  All sums run in a
// fixed order: results are deterministic run to run.
#include "common.cuh"

namespace dmdqn {

namespace {

// ------------------------------------------------------------------------------------------
// Thread coordinates inside a CTA tile.
// ------------------------------------------------------------------------------------------
template <int H>
struct Coord {
    int wn, wm, lm, ln;
    __device__ __forceinline__ Coord() {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        wn = warp % Tile<H>::WN;
        wm = warp / Tile<H>::WN;
        lm = lane >> 3;
        ln = lane & 7;
    }
    // i in 0..7 -> tile row; rows 0..3 and 16..19 (+4*lm) of the warp's 32 rows
    __device__ __forceinline__ int row(int i) const { return wm * 32 + (i >> 2) * 16 + lm * 4 + (i & 3); }
    // half in {0,1} -> first of 4 consecutive columns
    __device__ __forceinline__ int col0(int half) const { return wn * 64 + half * 32 + ln * 4; }
};

// ------------------------------------------------------------------------------------------
// Streaming a KC x H chunk of the weight operand global -> shared with cp.async (LDGSTS): no
// register staging, so the copy of chunk c+1 is in flight for the whole FFMA block of chunk c.
//   direct     : chunk[kk][n] = W[(k0+kk)*ldw + n]   16-byte copies   (forward:  x . W)
//   transposed : chunk[kk][n] = W[n*ldw + k0 + kk]    4-byte copies, transposing on the fly
//                                                                      (backward: d . W^T)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, bool valid = true) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int src_bytes = valid ? 16 : 0;            // 0 -> the 16 destination bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

template <int H, bool TRANS>
__device__ __forceinline__ void chunk_issue(float* Ws, const float* __restrict__ W, int ldw, int k0) {
    using T = Tile<H>;
    if (!TRANS) {
#pragma unroll
        for (int r = 0; r < T::KC * H / 4 / T::NT; ++r) {
            const int f = threadIdx.x + r * T::NT;
            const int kk = f / (H / 4), n4 = f % (H / 4);
            cp_async16(Ws + kk * T::LDW + n4 * 4, W + (size_t)(k0 + kk) * ldw + n4 * 4);
        }
    } else {
#pragma unroll
        for (int r = 0; r < T::KC * H / T::NT; ++r) {
            const int f = threadIdx.x + r * T::NT;
            const int n = f / T::KC, kk = f % T::KC;
            cp_async4(Ws + kk * T::LDW + n, W + (size_t)n * ldw + k0 + kk);
        }
    }
    cp_async_commit();
}

__device__ __forceinline__ void fma8(float (&acc)[8], float a, const float4& b0, const float4& b1) {
    acc[0] = fmaf(a, b0.x, acc[0]); acc[1] = fmaf(a, b0.y, acc[1]);
    acc[2] = fmaf(a, b0.z, acc[2]); acc[3] = fmaf(a, b0.w, acc[3]);
    acc[4] = fmaf(a, b1.x, acc[4]); acc[5] = fmaf(a, b1.y, acc[5]);
    acc[6] = fmaf(a, b1.z, acc[6]); acc[7] = fmaf(a, b1.w, acc[7]);
}

// acc[BM x H tile] = As[BM][K] (shared, row-major, stride lda) * op(W)[K][H] (global, streamed).
// Ends with a __syncthreads(): As and Ws may be overwritten right after it returns.
template <int H, bool TRANS>
__device__ __forceinline__ void gemm_rowA(float (&acc)[8][8], const Coord<H>& c, const float* As, int lda,
                                          const float* __restrict__ W, int ldw, int K, float* Ws) {
    using T = Tile<H>;
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    chunk_issue<H, TRANS>(Ws, W, ldw, 0);
    cp_async_wait_all();
    __syncthreads();
    int buf = 0;
    for (int k0 = 0; k0 < K; k0 += T::KC) {
        const bool more = k0 + T::KC < K;
        if (more) chunk_issue<H, TRANS>(Ws + (buf ^ 1) * (T::KC * T::LDW), W, ldw, k0 + T::KC);
        const float* Wb = Ws + buf * (T::KC * T::LDW);
#pragma unroll
        for (int kk = 0; kk < T::KC; kk += 4) {
            float4 a[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
                a[i] = *reinterpret_cast<const float4*>(As + c.row(i) * lda + k0 + kk);
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const float4 b0 = *reinterpret_cast<const float4*>(Wb + (kk + s) * T::LDW + c.col0(0));
                const float4 b1 = *reinterpret_cast<const float4*>(Wb + (kk + s) * T::LDW + c.col0(1));
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float av = s == 0 ? a[i].x : s == 1 ? a[i].y : s == 2 ? a[i].z : a[i].w;
                    fma8(acc[i], av, b0, b1);
                }
            }
        }
        if (more) cp_async_wait_all();
        __syncthreads();
        buf ^= 1;
    }
}

// Hs[row][col] = relu(acc + bias[col]); optionally also to global `gout` (row-major [B][H]).
template <int H>
__device__ __forceinline__ void store_relu(const float (&acc)[8][8], const Coord<H>& c,
                                           const float* __restrict__ bias, float* Hs,
                                           float* __restrict__ gout, int r0, int B) {
    using T = Tile<H>;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int col = c.col0(half);
        const float4 b = __ldg(reinterpret_cast<const float4*>(bias + col));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 v;
            v.x = fmaxf(acc[i][half * 4 + 0] + b.x, 0.f);
            v.y = fmaxf(acc[i][half * 4 + 1] + b.y, 0.f);
            v.z = fmaxf(acc[i][half * 4 + 2] + b.z, 0.f);
            v.w = fmaxf(acc[i][half * 4 + 3] + b.w, 0.f);
            const int row = c.row(i);
            *reinterpret_cast<float4*>(Hs + row * T::LDH + col) = v;
            if (gout && r0 + row < B) *reinterpret_cast<float4*>(gout + (size_t)(r0 + row) * H + col) = v;
        }
    }
}

// Gather BM observation rows (obs_stride floats each, whole 16-byte pieces) into Xs; rows
// past the batch are zero.
template <int H>
__device__ __forceinline__ void gather_tile(float* Xs, int ldx, const float* __restrict__ ring,
                                            const int32_t* __restrict__ rows, int r0, int B, int Dp) {
    using T = Tile<H>;
    const int q = Dp >> 2;
    for (int f = threadIdx.x; f < T::BM * q; f += T::NT) {
        const int i = f / q, c4 = f % q;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r0 + i < B) v = __ldg(reinterpret_cast<const float4*>(ring + (size_t)rows[r0 + i] * Dp) + c4);
        *reinterpret_cast<float4*>(Xs + i * ldx + c4 * 4) = v;
    }
}

// qs[i][a] = b3[a] + sum_j Hs2[i][j] * W3[j][a].  W3 (H x 4) is staged in shared memory (w3s,
// reusing the idle weight-chunk buffer); a row is split over 4 adjacent lanes (j = q, q+4, ...)
// whose partial sums are combined by a fixed xor butterfly.  Caller syncs before; ends synced.
template <int H>
__device__ __forceinline__ void layer3(const float* Hs2, const float* __restrict__ W3,
                                       const float* __restrict__ b3, float* qs, float* w3s) {
    using T = Tile<H>;
    for (int f = threadIdx.x; f < H; f += T::NT)
        reinterpret_cast<float4*>(w3s)[f] = __ldg(reinterpret_cast<const float4*>(W3) + f);
    __syncthreads();
    for (int o = threadIdx.x; o < T::BM * 4; o += T::NT) {
        const int i = o >> 2, q = o & 3;
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
        for (int j = q; j < H; j += 4) {
            const float h = Hs2[i * T::LDH + j];
            const float4 w = reinterpret_cast<const float4*>(w3s)[j];
            s.x = fmaf(h, w.x, s.x); s.y = fmaf(h, w.y, s.y);
            s.z = fmaf(h, w.z, s.z); s.w = fmaf(h, w.w, s.w);
        }
#pragma unroll
        for (int off = 1; off < 4; off <<= 1) {
            s.x += __shfl_xor_sync(0xffffffffu, s.x, off); s.y += __shfl_xor_sync(0xffffffffu, s.y, off);
            s.z += __shfl_xor_sync(0xffffffffu, s.z, off); s.w += __shfl_xor_sync(0xffffffffu, s.w, off);
        }
        const float v = q == 0 ? s.x : q == 1 ? s.y : q == 2 ? s.z : s.w;
        qs[o] = v + __ldg(b3 + q);
    }
    __syncthreads();
}

template <int H>
struct Smem {
    using T = Tile<H>;
    float *Xs, *Hs1, *Hs2, *Ws, *qs0, *qs1, *gs;
    int* as;
    int ldx;
    __device__ __forceinline__ Smem(float* base, int Dp) {
        ldx = Dp + 4;
        Xs = base;
        Hs1 = Xs + T::BM * ldx;
        Hs2 = Hs1 + T::BM * T::LDH;
        Ws = Hs2 + T::BM * T::LDH;
        qs0 = Ws + 2 * T::KC * T::LDW;
        qs1 = qs0 + T::BM * 4;
        gs = qs1 + T::BM * 4;
        as = reinterpret_cast<int*>(gs + T::BM);
    }
    static size_t bytes(int Dp) {
        return sizeof(float) * ((size_t)T::BM * (Dp + 4) + 2 * (size_t)T::BM * T::LDH + 2 * (size_t)T::KC * T::LDW +
                                10 * (size_t)T::BM);
    }
};

// The head W3 | b3 of network g's parameter set `tgt` (P: that set's block): the plain instantiations of K3 / K4a read it
// from P, the same code as before dueling heads existed; the dueling ones read the fold kernel's W3e | b3e.
template <bool DUELING>
__device__ __forceinline__ const float* head_w3(const LearnArgs& A, const float* P, int tgt, int g) {
    if constexpr (DUELING) return (tgt ? A.head[1] : A.head[0]) + (size_t)g * A.head_stride;
    else return P + A.L.w3;
}

// ------------------------------------------------------------------------------------------
// K3: TD targets.
// ------------------------------------------------------------------------------------------
template <int H, bool DUELING>
__global__ void __launch_bounds__(Tile<H>::NT, 1) target_kernel(const LearnArgs A) {
    using T = Tile<H>;
    extern __shared__ __align__(16) float smem[];
    const int g = blockIdx.x / A.ws_tiles, rt = blockIdx.x % A.ws_tiles;
    if (!A.active[g]) return;
    const int B = A.d.batch, Dp = A.d.obs_stride, r0 = rt * T::BM;
    Smem<H> S(smem, Dp);
    const Coord<H> c;
    const int32_t* nrows = A.nrows + (size_t)g * B;
    gather_tile<H>(S.Xs, S.ldx, A.rp.next_obs, nrows, r0, B, Dp);

    float acc[8][8];
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {          // 0: online(s')  1: target(s')
        const float* P = (pass == 0 ? A.nets.theta : A.nets.theta_tgt) + (size_t)g * A.L.stride;
        const float* W3 = head_w3<DUELING>(A, P, pass, g);
        gemm_rowA<H, false>(acc, c, S.Xs, S.ldx, P + A.L.w1, H, Dp, S.Ws);
        store_relu<H>(acc, c, P + A.L.b1, S.Hs1, nullptr, r0, B);
        gemm_rowA<H, false>(acc, c, S.Hs1, T::LDH, P + A.L.w2, H, H, S.Ws);
        store_relu<H>(acc, c, P + A.L.b2, S.Hs2, nullptr, r0, B);
        __syncthreads();
        layer3<H>(S.Hs2, W3, DUELING ? W3 + 4 * H : P + A.L.b3, pass == 0 ? S.qs0 : S.qs1, S.Ws);
    }
    for (int i = threadIdx.x; i < T::BM; i += T::NT) {
        const int gr = r0 + i;
        if (gr >= B) continue;
        const float* qo = S.qs0 + i * 4;
        const float* qt = S.qs1 + i * 4;
        int best = 0;                               // argmax online(s'), ties -> lowest (:342)
        float tmax = qt[0];
        for (int k = 1; k < A.d.n_actions; ++k) {
            if (qo[k] > qo[best]) best = k;
            tmax = fmaxf(tmax, qt[k]);
        }
        const float tq = A.double_dqn ? qt[best] : tmax;
        const size_t o = (size_t)g * B + gr;
        // targets = r + gamma * (1 - done) * target_q, left to right (:347); the sample kernel formed the discount
        A.y[o] = A.r_hat[o] + A.disc_b[o] * tq;
        for (int k = 0; k < 4; ++k) {
            A.q_next[o * 4 + k] = qo[k];
            A.tq_all[o * 4 + k] = qt[k];
        }
    }
}

// ------------------------------------------------------------------------------------------
// K4a: online forward on s, loss gradient, activation gradients.
// ------------------------------------------------------------------------------------------
template <int H, bool DUELING>
__global__ void __launch_bounds__(Tile<H>::NT, 1) online_kernel(const LearnArgs A) {
    using T = Tile<H>;
    extern __shared__ __align__(16) float smem[];
    const int g = blockIdx.x / A.ws_tiles, rt = blockIdx.x % A.ws_tiles;
    if (!A.active[g]) return;
    const int B = A.d.batch, Dp = A.d.obs_stride, r0 = rt * T::BM;
    Smem<H> S(smem, Dp);
    const Coord<H> c;
    const int32_t* rows = A.rows + (size_t)g * B;
    const float* P = A.nets.theta + (size_t)g * A.L.stride;
    const float* W3 = head_w3<DUELING>(A, P, 0, g);
    const size_t sb = (size_t)g * B;                 // this network's rows in [n_nets][B][...]
    gather_tile<H>(S.Xs, S.ldx, A.rp.obs, rows, r0, B, Dp);

    float acc[8][8];
    gemm_rowA<H, false>(acc, c, S.Xs, S.ldx, P + A.L.w1, H, Dp, S.Ws);
    store_relu<H>(acc, c, P + A.L.b1, S.Hs1, A.h1 + sb * H, r0, B);
    gemm_rowA<H, false>(acc, c, S.Hs1, T::LDH, P + A.L.w2, H, H, S.Ws);
    store_relu<H>(acc, c, P + A.L.b2, S.Hs2, nullptr, r0, B);
    __syncthreads();
    layer3<H>(S.Hs2, W3, DUELING ? W3 + 4 * H : P + A.L.b3, S.qs0, S.Ws);

    // loss terms and dL/dpred per row (:349-352; SURVEY App. A.8)
    float* terms = S.qs1;                            // [BM] loss terms
    for (int i = threadIdx.x; i < T::BM; i += T::NT) {
        const int gr = r0 + i;
        float gi = 0.f, term = 0.f;
        int ai = 0;
        if (gr < B) {
            ai = A.act_b[sb + gr];
            const float e = S.qs0[i * 4 + ai] - A.y[sb + gr];
            if (A.loss == DMDQN_LOSS_MSE) {
                term = e * e;
                gi = (2.0f * e) / (float)A.loss_batch;
            } else {
                const float ae = fabsf(e);
                term = ae <= 1.0f ? 0.5f * e * e : ae - 0.5f;
                gi = fminf(fmaxf(e, -1.0f), 1.0f) / (float)A.loss_batch;
            }
            if (A.per) {                             // prioritized replay: importance weight, then the new priority
                const float wi = A.is_w[sb + gr];
                term = wi * term;
                gi = wi * gi;
                per_store_priority(A, rows[gr], e);
            }
            for (int k = 0; k < 4; ++k) A.q_all[(sb + gr) * 4 + k] = S.qs0[i * 4 + k];
        }
        S.gs[i] = gi;
        S.as[i] = ai;
        terms[i] = term;
    }
    __syncthreads();
    const size_t pt = (size_t)g * A.ws_tiles + rt;   // partial slot of this (network, row tile)
    if (threadIdx.x == 0) {                          // per-tile loss / metric / db3 partials, rows in order
        float ls = 0.f, qsum = 0.f, qsq = 0.f, hist[4] = {0.f, 0.f, 0.f, 0.f}, db3[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = 0; i < T::BM && r0 + i < B; ++i) {
            ls += terms[i];
            for (int k = 0; k < A.d.n_actions; ++k) {
                const float q = S.qs0[i * 4 + k];
                qsum += q;
                qsq = fmaf(q, q, qsq);
            }
            hist[S.as[i]] += 1.f;
            db3[S.as[i]] += S.gs[i];
        }
        float* pl = A.part_loss + pt * 8;
        pl[0] = ls; pl[1] = qsum; pl[2] = qsq;
        pl[3] = hist[0]; pl[4] = hist[1]; pl[5] = hist[2]; pl[6] = hist[3]; pl[7] = 0.f;
        for (int k = 0; k < 4; ++k) A.part_b3[pt * 4 + k] = db3[k];
    }
    // dW3 partial, dh2 = (dq W3^T) * relu'(h2) in place, db2 partial: one thread per column
    for (int j = threadIdx.x; j < H; j += T::NT) {
        const float4 w3 = __ldg(reinterpret_cast<const float4*>(W3) + j);
        float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f, sb2 = 0.f;
        for (int i = 0; i < T::BM; ++i) {
            const float h = S.Hs2[i * T::LDH + j];
            const float gi = S.gs[i];
            const int ai = S.as[i];
            const float t = h * gi;
            d0 += ai == 0 ? t : 0.f; d1 += ai == 1 ? t : 0.f;
            d2 += ai == 2 ? t : 0.f; d3 += ai == 3 ? t : 0.f;
            const float w = ai == 0 ? w3.x : ai == 1 ? w3.y : ai == 2 ? w3.z : w3.w;
            const float dh = h > 0.f ? gi * w : 0.f;
            S.Hs2[i * T::LDH + j] = dh;
            sb2 += dh;
        }
        reinterpret_cast<float4*>(A.part_w3 + pt * H * 4)[j] = make_float4(d0, d1, d2, d3);
        A.part_b2[pt * H + j] = sb2;
    }
    __syncthreads();
    for (int f = threadIdx.x; f < T::BM * (H / 4); f += T::NT) {   // dh2 tile -> scratch, coalesced
        const int i = f / (H / 4), c4 = f % (H / 4);
        if (r0 + i < B)
            reinterpret_cast<float4*>(A.dh2 + (sb + r0 + i) * H)[c4] =
                *reinterpret_cast<const float4*>(S.Hs2 + i * T::LDH + c4 * 4);
    }
    // dh1 = (dh2 W2^T) * relu'(h1), in place over h1
    gemm_rowA<H, true>(acc, c, S.Hs2, T::LDH, P + A.L.w2, H, H, S.Ws);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int col = c.col0(half);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int row = c.row(i);
            float4* hp = reinterpret_cast<float4*>(S.Hs1 + row * T::LDH + col);
            const float4 h = *hp;
            float4 v;
            v.x = h.x > 0.f ? acc[i][half * 4 + 0] : 0.f;
            v.y = h.y > 0.f ? acc[i][half * 4 + 1] : 0.f;
            v.z = h.z > 0.f ? acc[i][half * 4 + 2] : 0.f;
            v.w = h.w > 0.f ? acc[i][half * 4 + 3] : 0.f;
            *hp = v;
            if (r0 + row < B) *reinterpret_cast<float4*>(A.dh1 + (sb + r0 + row) * H + col) = v;
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < H; j += T::NT) {   // db1 partial
        float s = 0.f;
        for (int i = 0; i < T::BM; ++i) s += S.Hs1[i * T::LDH + j];
        A.part_b1[pt * H + j] = s;
    }
}

// ------------------------------------------------------------------------------------------
// K4b: weight gradients with Adam + target sync in the epilogue.
// ------------------------------------------------------------------------------------------
// keras 3.9.2 Adam.update_step op order: m += (g-m)(1-b1); v += (g*g-v)(1-b2);
// theta -= (m*alpha)/(sqrt(v)+eps); then theta_tgt per the sync mode.
__device__ __forceinline__ void adam_elem(const AdamStep& k, float g, float& th, float& m, float& v, float& tg) {
    m = m + (g - m) * k.one_m_b1;
    v = v + (g * g - v) * k.one_m_b2;
    th = th - (m * k.alpha) / (sqrtf(v) + k.eps);
    if (k.sync == 1) tg = th;
    else if (k.sync == 2) tg = k.tau * th + (1.0f - k.tau) * tg;
}

__device__ __forceinline__ void adam_vec4(const AdamStep& k, const float* g, float* th, float* m, float* v,
                                          float* tg) {
    float4 t4 = *reinterpret_cast<float4*>(th), m4 = *reinterpret_cast<float4*>(m);
    float4 v4 = *reinterpret_cast<float4*>(v);
    float4 tg4 = k.sync == 2 ? *reinterpret_cast<float4*>(tg) : make_float4(0.f, 0.f, 0.f, 0.f);
    adam_elem(k, g[0], t4.x, m4.x, v4.x, tg4.x);
    adam_elem(k, g[1], t4.y, m4.y, v4.y, tg4.y);
    adam_elem(k, g[2], t4.z, m4.z, v4.z, tg4.z);
    adam_elem(k, g[3], t4.w, m4.w, v4.w, tg4.w);
    *reinterpret_cast<float4*>(th) = t4;
    *reinterpret_cast<float4*>(m) = m4;
    *reinterpret_cast<float4*>(v) = v4;
    if (k.sync) *reinterpret_cast<float4*>(tg) = tg4;
}

template <int H>
__global__ void __launch_bounds__(Tile<H>::NT) wgrad_adam_kernel(const LearnArgs A) {
    using T = Tile<H>;
    constexpr int LDA = T::BM + 4;
    extern __shared__ __align__(16) float smem[];
    float (*As)[T::KC * LDA] = reinterpret_cast<float (*)[T::KC * LDA]>(smem);
    float (*Bs)[T::KC * T::LDW] = reinterpret_cast<float (*)[T::KC * T::LDW]>(smem + 2 * T::KC * LDA);
    const int B = A.d.batch, Dp = A.d.obs_stride;
    const int tiles_w2 = H / T::BM, tiles_w1 = (Dp + T::BM - 1) / T::BM;
    const int per_net = tiles_w2 + tiles_w1 + 1;
    const int g = blockIdx.x / per_net, t = blockIdx.x % per_net;
    const size_t sb = (size_t)g * B;
    float* th = A.nets.theta + (size_t)g * A.L.stride;
    float* tg = A.nets.theta_tgt + (size_t)g * A.L.stride;
    float* am = A.nets.adam_m + (size_t)g * A.L.stride;
    float* av = A.nets.adam_v + (size_t)g * A.L.stride;

    if (t == per_net - 1) {
        // misc tile: biases and the H x 4 head from the per-row-tile partials (summed in tile
        // order), plus the step's metrics (:359-370).
        if (!A.active[g]) {
            if (threadIdx.x < DMDQN_METRICS_STRIDE && A.metrics) A.metrics[g * DMDQN_METRICS_STRIDE + threadIdx.x] = 0.f;
            return;
        }
        const AdamStep k = adam_step(A, g);
        const size_t p0 = (size_t)g * A.ws_tiles;
        auto upd = [&](int64_t off, float gsum) {
            if (A.grads) {
                A.grads[(size_t)g * A.L.stride + off] = gsum;
                return;
            }
            float tgv = k.sync == 2 ? tg[off] : 0.f;
            adam_elem(k, gsum, th[off], am[off], av[off], tgv);
            if (k.sync) tg[off] = tgv;
        };
        for (int e = threadIdx.x; e < 3 * H + 1; e += T::NT) {
            if (e < 2 * H) {                               // b1, b2
                const float* part = e < H ? A.part_b1 : A.part_b2;
                const int j = e < H ? e : e - H;
                float gsum = 0.f;
                for (int r = 0; r < A.ws_tiles; ++r) gsum += part[(p0 + r) * H + j];
                upd((e < H ? A.L.b1 : A.L.b2) + j, gsum);
                continue;
            }
            // one head row: W3[j][0..3] (j < H) or b3 (j == H); dueling: projected, with its value weight wv[j] / bv
            const int j = e - 2 * H;
            float w[4] = {0.f, 0.f, 0.f, 0.f};
            for (int r = 0; r < A.ws_tiles; ++r) {
                const float4 pw = j < H ? *reinterpret_cast<const float4*>(A.part_w3 + ((p0 + r) * H + j) * 4)
                                        : *reinterpret_cast<const float4*>(A.part_b3 + (p0 + r) * 4);
                w[0] += pw.x; w[1] += pw.y; w[2] += pw.z; w[3] += pw.w;
            }
            if (A.dueling) {
                upd(j < H ? layout_wv(A.L) + j : layout_bv(A.L, H), head_project(w, A.d.n_actions));
                if (j == H && A.grads)                     // the pad after bv is inside the Adam range: its gradient is 0
                    for (int p = 1; p < 4; ++p) A.grads[(size_t)g * A.L.stride + layout_bv(A.L, H) + p] = 0.f;
            }
            const int64_t off = j < H ? A.L.w3 + (int64_t)j * 4 : A.L.b3;
            for (int a = 0; a < 4; ++a) upd(off + a, w[a]);
        }
        if (threadIdx.x == 0 && A.metrics) finish_metrics(A, g, A.ws_tiles, [](const float* p) { return *p; });
        return;
    }
    if (!A.active[g]) return;

    // dW tile: rows m0..m0+BM of W2 (A = h1, D = dh2) or W1 (A = gathered s, D = dh1); K = batch.
    const bool is_w2 = t < tiles_w2;
    const int m0 = (is_w2 ? t : t - tiles_w2) * T::BM;
    const int m_valid = is_w2 ? H : Dp;
    const float* Asrc = is_w2 ? A.h1 + sb * H : A.rp.obs;
    const float* Dsrc = (is_w2 ? A.dh2 : A.dh1) + sb * H;
    const int32_t* rows = A.rows + sb;
    const int lda_src = is_w2 ? H : Dp;
    const Coord<H> c;

    constexpr int A4 = T::KC * T::BM / 4;            // 16-byte pieces in an A chunk
    constexpr int NA = (A4 + T::NT - 1) / T::NT;
    auto issue = [&](int k0, int buf) {
#pragma unroll
        for (int r = 0; r < NA; ++r) {
            const int f = threadIdx.x + r * T::NT;
            if (f < A4) {
                const int kk = f / (T::BM / 4), m4 = f % (T::BM / 4);
                const int kr = k0 + kk, m = m0 + m4 * 4;
                const bool ok = kr < B && m < m_valid;
                const size_t src_row = ok ? (is_w2 ? (size_t)kr : (size_t)rows[kr]) : 0;
                cp_async16(&As[buf][kk * LDA + m4 * 4], Asrc + src_row * lda_src + (ok ? m : 0), ok);
            }
        }
#pragma unroll
        for (int r = 0; r < T::KC * H / 4 / T::NT; ++r) {
            const int f = threadIdx.x + r * T::NT;
            const int kk = f / (H / 4), n4 = f % (H / 4);
            const bool ok = k0 + kk < B;
            cp_async16(&Bs[buf][kk * T::LDW + n4 * 4], Dsrc + (size_t)(ok ? k0 + kk : 0) * H + n4 * 4, ok);
        }
        cp_async_commit();
    };

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    issue(0, 0);
    cp_async_wait_all();
    __syncthreads();
    int buf = 0;
    for (int k0 = 0; k0 < B; k0 += T::KC) {
        const bool more = k0 + T::KC < B;
        if (more) issue(k0 + T::KC, buf ^ 1);
#pragma unroll
        for (int kk = 0; kk < T::KC; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk * LDA + c.wm * 32 + c.lm * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk * LDA + c.wm * 32 + 16 + c.lm * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk * T::LDW + c.col0(0)]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk * T::LDW + c.col0(1)]);
            fma8(acc[0], a0.x, b0, b1); fma8(acc[1], a0.y, b0, b1);
            fma8(acc[2], a0.z, b0, b1); fma8(acc[3], a0.w, b0, b1);
            fma8(acc[4], a1.x, b0, b1); fma8(acc[5], a1.y, b0, b1);
            fma8(acc[6], a1.z, b0, b1); fma8(acc[7], a1.w, b0, b1);
        }
        if (more) cp_async_wait_all();
        __syncthreads();
        buf ^= 1;
    }

    const AdamStep k = adam_step(A, g);
    const int64_t wbase = is_w2 ? A.L.w2 : A.L.w1;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + c.row(i);
        if (m >= m_valid) continue;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int64_t off = wbase + (int64_t)m * H + c.col0(half);
            if (A.grads)
                *reinterpret_cast<float4*>(A.grads + (size_t)g * A.L.stride + off) =
                    make_float4(acc[i][half * 4], acc[i][half * 4 + 1], acc[i][half * 4 + 2], acc[i][half * 4 + 3]);
            else
                adam_vec4(k, &acc[i][half * 4], th + off, am + off, av + off, tg + off);
        }
    }
}

// Dueling fold (include/dmdqn_b200.h): W3e | b3e of network blockIdx.x's online (blockIdx.y = 0) or target (1) block into
// head[blockIdx.y][blockIdx.x], one thread per W3 row and one more for the bias.
__global__ void __launch_bounds__(256) fold_kernel(Layout L, int H, int n_actions, const float* __restrict__ theta,
                                                   const float* __restrict__ theta_tgt, float* __restrict__ head) {
    const int g = blockIdx.x, n_nets = gridDim.x;
    const float* P = (blockIdx.y ? theta_tgt : theta) + (size_t)g * L.stride;
    float* out = head + ((size_t)blockIdx.y * n_nets + g) * (4 * H + 4);
    for (int j = threadIdx.x; j <= H; j += blockDim.x) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(P + (j < H ? L.w3 + 4 * j : L.b3)));
        float x[4] = {w.x, w.y, w.z, w.w};
        head_fold(x, __ldg(P + (j < H ? layout_wv(L) + j : layout_bv(L, H))), n_actions);
        reinterpret_cast<float4*>(out)[j] = make_float4(x[0], x[1], x[2], x[3]);
    }
}

// theta_tgt <- theta (tau < 0) or Polyak (tau >= 0) for the masked networks.
__global__ void sync_target_kernel(int64_t stride, const float* __restrict__ theta, float* __restrict__ tgt,
                                   const uint8_t* __restrict__ mask, float tau) {
    const int g = blockIdx.y;
    if (mask && !mask[g]) return;
    const float4* src = reinterpret_cast<const float4*>(theta + (size_t)g * stride);
    float4* dst = reinterpret_cast<float4*>(tgt + (size_t)g * stride);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < stride / 4;
         i += (int64_t)gridDim.x * blockDim.x) {
        float4 s = src[i];
        if (tau >= 0.f) {
            const float4 o = dst[i];
            s.x = tau * s.x + (1.f - tau) * o.x; s.y = tau * s.y + (1.f - tau) * o.y;
            s.z = tau * s.z + (1.f - tau) * o.z; s.w = tau * s.w + (1.f - tau) * o.w;
        }
        dst[i] = s;
    }
}

// Adam + target sync from an explicit (all-reduced) gradient block: the tail of K4b when the
// gradient had to leave the kernel for the NCCL all-reduce.
__global__ void adam_apply_kernel(const LearnArgs A, const float* __restrict__ grads) {
    const int g = blockIdx.y;
    if (!A.active[g]) return;
    const AdamStep k = adam_step(A, g);
    const size_t base = (size_t)g * A.L.stride;
    const int64_t n4 = A.L.end / 4;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 g4 = *reinterpret_cast<const float4*>(grads + base + i * 4);
        const float gv[4] = {g4.x, g4.y, g4.z, g4.w};
        adam_vec4(k, gv, A.nets.theta + base + i * 4, A.nets.adam_m + base + i * 4, A.nets.adam_v + base + i * 4,
                  A.nets.theta_tgt + base + i * 4);
    }
}

// Noisy networks (include/dmdqn_b200.h dmdqn_noisy).  Fold: CTA (c, g, s) builds the noise record of network g and set s in
// shared memory (every CTA of the pair builds it: a few thousand Philox draws against the ~MB it streams), CTA c == 0
// stores it, and every CTA writes eff = mu + sigma * eps over its share of the stride.  HBM bound: 8 bytes read and 4
// written per float.
constexpr int kNoisyThreads = 256;

__global__ void __launch_bounds__(kNoisyThreads)
noisy_fold_kernel(Layout L, NoiseRec R, int H, int obs_dim, int n_actions, int dueling, const dmdqn_nets nets,
                  const dmdqn_noisy nz, int64_t per) {
    extern __shared__ __align__(16) float rec[];
    const int g = blockIdx.y, set = blockIdx.z;
    noise_record_build(rec, R, obs_dim, n_actions, __ldg(nz.key + g), (uint32_t)__ldg(nets.learn_step + g), set);
    __syncthreads();
    if (blockIdx.x == 0)
        for (int e = threadIdx.x; e < R.stride; e += blockDim.x) nz.noise[((size_t)g * 2 + set) * R.stride + e] = rec[e];
    const size_t base = (size_t)g * L.stride;
    const float4* mu = reinterpret_cast<const float4*>((set ? nets.theta_tgt : nets.theta) + base);
    const float4* sg = reinterpret_cast<const float4*>((set ? nz.sigma_tgt : nz.sigma) + base);
    float4* out = reinterpret_cast<float4*>((set ? nz.eff_tgt : nz.eff) + base);
    const int64_t i0 = blockIdx.x * per, i1 = min(i0 + per, L.stride / 4);
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const float4 m = __ldg(mu + i), s = __ldg(sg + i), e = noise_eps4(rec, R, L, H, dueling, i * 4);
        out[i] = make_float4(noisy_weight(m.x, s.x, e.x), noisy_weight(m.y, s.y, e.y), noisy_weight(m.z, s.z, e.z),
                             noisy_weight(m.w, s.w, e.w));
    }
}

// Adam on mu and sigma from the effective-weight gradient g: g_mu = g, g_sigma = g * eps with set 0's record, each through
// adam_vec4 as adam_apply_kernel applies it.  HBM bound: g once, and theta / m / v (+ target) of mu and of sigma.
__global__ void __launch_bounds__(kNoisyThreads)
noisy_adam_apply_kernel(const LearnArgs A, const dmdqn_noisy nz, NoiseRec R, const float* __restrict__ grads, int64_t per) {
    extern __shared__ __align__(16) float rec[];
    const int g = blockIdx.y;
    if (!A.active[g] || *reinterpret_cast<volatile int*>(A.error) != 0) return;
    const float* src = nz.noise + (size_t)g * 2 * R.stride;
    for (int e = threadIdx.x; e < R.stride; e += blockDim.x) rec[e] = src[e];
    __syncthreads();
    const AdamStep k = adam_step(A, g);
    const int H = A.d.hidden;
    const size_t base = (size_t)g * A.L.stride;
    const int64_t i0 = blockIdx.x * per, i1 = min(i0 + per, A.L.end / 4);
    for (int64_t i = i0 + threadIdx.x; i < i1; i += blockDim.x) {
        const float4 g4 = *reinterpret_cast<const float4*>(grads + base + i * 4);
        const float4 e = noise_eps4(rec, R, A.L, H, A.dueling, i * 4);
        const float gm[4] = {g4.x, g4.y, g4.z, g4.w};
        const float gs[4] = {__fmul_rn(g4.x, e.x), __fmul_rn(g4.y, e.y), __fmul_rn(g4.z, e.z), __fmul_rn(g4.w, e.w)};
        const size_t o = base + i * 4;
        adam_vec4(k, gm, A.nets.theta + o, A.nets.adam_m + o, A.nets.adam_v + o, A.nets.theta_tgt + o);
        adam_vec4(k, gs, nz.sigma + o, nz.sigma_m + o, nz.sigma_v + o, nz.sigma_tgt + o);
    }
}

// CTAs per network (fold: per network and set) of the two noisy kernels: enough for two waves over the SMs, each CTA
// streaming at least 2048 float4s.
inline int noisy_chunks(int n_sm, int64_t pairs, int64_t n4) {
    const int64_t want = (2 * (int64_t)n_sm + pairs - 1) / pairs;
    return (int)max((int64_t)1, min(want, (n4 + 2047) / 2048));
}

// Global-norm clipping in front of the same Adam + target sync (dmdqn_clip_adam_apply, include/dmdqn_b200.h): one
// cluster of kClipCtas CTAs per network.  CTA r of the cluster owns float4s [r * per, (r + 1) * per) of the block
// [0, b3 + 4): it brings them into shared memory with one bulk copy, forms their float64 sum of squares in a fixed
// order, and after a cluster barrier every CTA adds the kClipCtas partials over DSMEM in rank order, so all of them
// hold the same norm n.  The gradient is then read from shared memory, scaled by s = c / max(n, c) and applied by
// adam_vec4 exactly as adam_apply_kernel applies it; the block is read from HBM once.
constexpr int kClipCtas = 8;            // the portable cluster size
constexpr int kClipThreads = 256;

inline int64_t clip_per_cta(const Layout& L) { return (L.end / 4 + kClipCtas - 1) / kClipCtas; }   // float4s

__device__ __forceinline__ void clip_mbar_wait(uint32_t bar, bool& ok) {
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        uint32_t done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(bar) : "memory");
        if (done) return;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > 2000000000ull) { ok = false; return; }     // ~2 s: a copy that never lands is an error, not a hang
    }
}

__global__ void __cluster_dims__(kClipCtas, 1, 1) __launch_bounds__(kClipThreads)
clip_adam_apply_kernel(const LearnArgs A, const float* __restrict__ grads, int64_t per, double clipnorm,
                       float* __restrict__ norms_out) {
    extern __shared__ __align__(16) float4 gsm[];       // this CTA's slice of the gradient block
    __shared__ __align__(8) uint64_t bar;
    __shared__ double warp_sum[kClipThreads / 32];
    __shared__ double part;                             // this CTA's sum of squares: read by every CTA of the cluster
    __shared__ int part_ok;                             // 0: the copy timed out or the step was poisoned
    __shared__ float scale_sh;
    __shared__ int apply_sh;
    const int g = blockIdx.y, tid = threadIdx.x;
    const uint32_t rank = blockIdx.x;                   // == %cluster_ctarank: the cluster spans gridDim.x
    if (!A.active[g]) {                                 // the same for every CTA of the cluster: no barrier is pending
        if (rank == 0 && tid == 0 && norms_out) norms_out[g] = 0.f;
        return;
    }
    const int64_t n4 = A.L.end / 4, i0 = (int64_t)rank * per;
    const int cnt = (int)max((int64_t)0, min(per, n4 - i0));
    const size_t base = (size_t)g * A.L.stride + (size_t)i0 * 4;
    const uint32_t sbar = (uint32_t)__cvta_generic_to_shared(&bar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(sbar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (cnt > 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sbar), "r"((uint32_t)cnt * 16u) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"((uint32_t)__cvta_generic_to_shared(gsm)), "l"(grads + base), "r"((uint32_t)cnt * 16u), "r"(sbar)
                         : "memory");
        }
    }
    __syncthreads();
    bool ok = true;
    if (cnt > 0) clip_mbar_wait(sbar, ok);
    double ss = 0.0;                                    // float squares are exact in float64
    for (int i = tid; i < cnt; i += kClipThreads) {
        const float4 v = gsm[i];
        ss = fma((double)v.x, (double)v.x, ss); ss = fma((double)v.y, (double)v.y, ss);
        ss = fma((double)v.z, (double)v.z, ss); ss = fma((double)v.w, (double)v.w, ss);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    const int any_bad = __syncthreads_or(!ok);
    if ((tid & 31) == 0) warp_sum[tid >> 5] = ss;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int w = 0; w < kClipThreads / 32; ++w) s += warp_sum[w];
        part = s;
        // a tcgen05 K4b whose bounded waits expired wrote no gradient for this step and set the error flag
        part_ok = !any_bad && *reinterpret_cast<volatile int*>(A.error) == 0;
    }
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (tid == 0) {
        double total = 0.0;
        int all_ok = 1;
        const uint32_t mine = (uint32_t)__cvta_generic_to_shared(&part), mine_ok = (uint32_t)__cvta_generic_to_shared(&part_ok);
        for (uint32_t r = 0; r < kClipCtas; ++r) {       // rank order on every CTA: one n per cluster
            uint32_t pa, po;
            double p;
            int o;
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(pa) : "r"(mine), "r"(r));
            asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(po) : "r"(mine_ok), "r"(r));
            asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(p) : "r"(pa) : "memory");
            asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(o) : "r"(po) : "memory");
            total += p;
            all_ok &= o;
        }
        const double n = sqrt(total);
        scale_sh = isfinite(n) ? (float)(clipnorm / fmax(n, clipnorm)) : 1.f;
        apply_sh = all_ok;
        if (rank == 0 && norms_out) norms_out[g] = all_ok ? (float)n : 0.f;
    }
    __syncthreads();
    const float s = scale_sh;
    const bool scaled = s != 1.f;                       // s == 1: the unscaled gradient, as dmdqn_adam_apply reads it
    if (apply_sh) {                                     // adam_apply_kernel's loop, the gradient from shared memory
        const AdamStep k = adam_step(A, g);
#pragma unroll 4
        for (int i = tid; i < cnt; i += kClipThreads) {
            float4 g4 = gsm[i];
            if (scaled) { g4.x *= s; g4.y *= s; g4.z *= s; g4.w *= s; }
            const float gv[4] = {g4.x, g4.y, g4.z, g4.w};
            adam_vec4(k, gv, A.nets.theta + base + i * 4, A.nets.adam_m + base + i * 4, A.nets.adam_v + base + i * 4,
                      A.nets.theta_tgt + base + i * 4);
        }
    }
    // no CTA may leave while a peer can still read its partial
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// K5: all-reduce of the shared network's gradient block over NVLink peer memory fused with Adam + target sync
// (include/dmdqn_b200.h dmdqn_allreduce_adam).  Block b of every rank exchanges its own flag with block b of every
// peer, so there is no grid-wide dependency inside a GPU and no co-residency requirement; the gradient blocks were
// completed by the previous kernel of each rank's stream, the flag only says "that kernel is done".
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__global__ void __launch_bounds__(256)
peer_reduce_adam_kernel(const LearnArgs A, const dmdqn_peers P, const float* __restrict__ my_loss_src,
                        float* __restrict__ loss_out) {
    __shared__ int timed_out;
    const int b = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) timed_out = 0;
    if (b == 0 && tid == 0) {                       // this rank's share of the loss travels with block 0's flag
        *P.loss[P.rank] = *my_loss_src;
        __threadfence_system();
    }
    __syncthreads();
    if (tid < P.world) st_release_sys(P.flags[tid] + P.rank * DMDQN_PEER_BLOCKS + b, P.epoch);
    if (tid < P.world) {
        const uint32_t* f = P.flags[P.rank] + tid * DMDQN_PEER_BLOCKS + b;
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        while ((int32_t)(ld_acquire_sys(f) - P.epoch) < 0) {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > 2000000000ull) { timed_out = 1; break; }    // ~2 s: a missing peer is an error, not a hang
            __nanosleep(200);
        }
    }
    __syncthreads();
    if (timed_out) {
        if (tid == 0) atomicExch(A.error, DMDQN_PEER_TIMEOUT);
        return;
    }
    if (!A.active[0]) return;                       // (the learn decision is collective: every rank or none)
    const AdamStep k = adam_step(A, 0);
    const int64_t n4 = A.L.end / 4;
    for (int64_t i = b * (int64_t)blockDim.x + tid; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v[DMDQN_MAX_PEERS];
#pragma unroll
        for (int p = 0; p < DMDQN_MAX_PEERS; ++p)   // every peer's piece in flight before the first add
            if (p < P.world) v[p] = __ldcv(reinterpret_cast<const float4*>(P.grads[p]) + i);
        float4 sum = v[0];
#pragma unroll
        for (int p = 1; p < DMDQN_MAX_PEERS; ++p)   // rank order on every rank: bit-identical replicas
            if (p < P.world) { sum.x += v[p].x; sum.y += v[p].y; sum.z += v[p].z; sum.w += v[p].w; }
        const float gv[4] = {sum.x, sum.y, sum.z, sum.w};
        adam_vec4(k, gv, A.nets.theta + i * 4, A.nets.adam_m + i * 4, A.nets.adam_v + i * 4, A.nets.theta_tgt + i * 4);
    }
    if (b == 0 && tid == 0 && loss_out) {
        float ls = 0.f;
        for (int p = 0; p < P.world; ++p) ls += __ldcv(P.loss[p]);
        *loss_out = ls;
    }
}

template <int H, bool DUELING>
int launch_learn_h(const LearnArgs& A, int stages, cudaStream_t s) {
    using T = Tile<H>;
    const size_t smem = Smem<H>::bytes(A.d.obs_stride);
    const size_t smem_w = sizeof(float) * 2 * T::KC * ((T::BM + 4) + T::LDW);
    static size_t cfg_t[kMaxDevices] = {}, cfg_o[kMaxDevices] = {}, cfg_w[kMaxDevices] = {};    // per device, not per process
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(target_kernel<H, DUELING>), smem, cfg_t)) return rc;
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(online_kernel<H, DUELING>), smem, cfg_o)) return rc;
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(wgrad_adam_kernel<H>), smem_w, cfg_w)) return rc;
    const int grid = A.d.n_nets * A.ws_tiles;
    if (stages & DMDQN_STAGE_TARGET) {
        target_kernel<H, DUELING><<<grid, T::NT, smem, s>>>(A);
        DMDQN_CUDA(cudaGetLastError());
    }
    if (stages & DMDQN_STAGE_ONLINE) {
        online_kernel<H, DUELING><<<grid, T::NT, smem, s>>>(A);
        DMDQN_CUDA(cudaGetLastError());
    }
    if (stages & DMDQN_STAGE_WGRAD) {
        const int per_net = H / T::BM + (A.d.obs_stride + T::BM - 1) / T::BM + 1;
        wgrad_adam_kernel<H><<<A.d.n_nets * per_net, T::NT, smem_w, s>>>(A);
        DMDQN_CUDA(cudaGetLastError());
    }
    return DMDQN_OK;
}

}  // namespace

LearnArgs make_learn_args(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                          char* ws, const Workspace& w, float* metrics, float* grads, int loss_batch) {
    LearnArgs A = {};
    A.d = d;
    A.L = make_layout(d.obs_stride, d.hidden, hp.dueling == 1);
    A.rp = rp;
    A.nets = nets;
    A.loss = hp.loss;
    A.double_dqn = hp.double_dqn;
    A.loss_batch = loss_batch > 0 ? loss_batch : d.batch;
    A.one_m_b1 = (float)(1.0 - hp.beta1);
    A.one_m_b2 = (float)(1.0 - hp.beta2);
    A.tau = (float)hp.tau;
    A.ws_tiles = w.tiles;
    A.rows = reinterpret_cast<const int32_t*>(ws + w.rows);
    A.nrows = reinterpret_cast<const int32_t*>(ws + w.nrows);
    A.act_b = reinterpret_cast<const int32_t*>(ws + w.act_b);
    A.active = reinterpret_cast<const int32_t*>(ws + w.active);
    A.r_hat = reinterpret_cast<const float*>(ws + w.r_hat);
    A.disc_b = reinterpret_cast<const float*>(ws + w.disc_b);
    A.adam_sc = reinterpret_cast<const float4*>(ws + w.adam_sc);
    A.y = reinterpret_cast<float*>(ws + w.y);
    A.q_all = reinterpret_cast<float*>(ws + w.q_all);
    A.q_next = reinterpret_cast<float*>(ws + w.q_next);
    A.tq_all = reinterpret_cast<float*>(ws + w.tq_all);
    A.h1 = reinterpret_cast<float*>(ws + w.h1);
    A.dh1 = reinterpret_cast<float*>(ws + w.dh1);
    A.dh2 = reinterpret_cast<float*>(ws + w.dh2);
    A.part_loss = reinterpret_cast<float*>(ws + w.part_loss);
    A.part_b3 = reinterpret_cast<float*>(ws + w.part_b3);
    A.part_w3 = reinterpret_cast<float*>(ws + w.part_w3);
    A.part_b2 = reinterpret_cast<float*>(ws + w.part_b2);
    A.part_b1 = reinterpret_cast<float*>(ws + w.part_b1);
    A.mask2 = reinterpret_cast<uint32_t*>(ws + w.mask2);
    A.ga = reinterpret_cast<float2*>(ws + w.ga);
    A.w3_copy = reinterpret_cast<float*>(ws + w.w3_copy);
    A.error = reinterpret_cast<int*>(ws + w.tc_error);
    A.sched = reinterpret_cast<int*>(ws + w.sync);
    A.metrics = metrics;
    A.grads = grads;
    A.per = hp.sample_mode == DMDQN_SAMPLE_PRIORITIZED && rp.priority != nullptr;
    A.is_w = reinterpret_cast<const float*>(ws + w.is_w);
    A.per_alpha = hp.per_alpha;
    A.per_eps = hp.per_eps;
    A.dueling = hp.dueling == 1;
    if (A.dueling) {
        A.head_stride = 4 * (int64_t)d.hidden + 4;
        A.head[0] = reinterpret_cast<const float*>(ws + w.head);
        A.head[1] = A.head[0] + (size_t)d.n_nets * A.head_stride;
    } else {
        A.head_stride = A.L.stride;
        A.head[0] = nets.theta + A.L.w3;
        A.head[1] = nets.theta_tgt + A.L.w3;
    }
    return A;
}

int launch_learn(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_replay& rp, const dmdqn_nets& nets,
                 float* metrics, char* ws, const Workspace& w, int stages, float* grads, int loss_batch, cudaStream_t s) {
    const LearnArgs A = make_learn_args(d, hp, rp, nets, ws, w, metrics, grads, loss_batch);
    if (hp.precision != DMDQN_PRECISION_FP32) {
        if (!tc_supported(d)) {
            set_error("precision=%d (tcgen05) needs hidden=256 and obs_stride in {32,64,96}; got hidden=%d obs_stride=%d",
                      hp.precision, d.hidden, d.obs_stride);
            return DMDQN_ERR_ARG;
        }
        return launch_learn_tc(A, hp.precision, stages, s);
    }
    switch (d.hidden) {
        case 64: return A.dueling ? launch_learn_h<64, true>(A, stages, s) : launch_learn_h<64, false>(A, stages, s);
        case 128: return A.dueling ? launch_learn_h<128, true>(A, stages, s) : launch_learn_h<128, false>(A, stages, s);
        case 256: return A.dueling ? launch_learn_h<256, true>(A, stages, s) : launch_learn_h<256, false>(A, stages, s);
        case 512: return A.dueling ? launch_learn_h<512, true>(A, stages, s) : launch_learn_h<512, false>(A, stages, s);
    }
    set_error("unsupported hidden width %d", d.hidden);
    return DMDQN_ERR_ARG;
}

int launch_adam_apply(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const float* grads, char* ws,
                      const Workspace& w, cudaStream_t s) {
    const LearnArgs A = make_learn_args(d, hp, {}, nets, ws, w, nullptr, nullptr, 0);
    adam_apply_kernel<<<dim3(64, d.n_nets), 256, 0, s>>>(A, grads);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_clip_adam_apply(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const float* grads,
                           double clipnorm, float* norms_out, char* ws, const Workspace& w, cudaStream_t s) {
    const LearnArgs A = make_learn_args(d, hp, {}, nets, ws, w, nullptr, nullptr, 0);
    const int64_t per = clip_per_cta(A.L);
    const size_t smem = (size_t)per * 16;
    static size_t cfg[kMaxDevices] = {};
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(clip_adam_apply_kernel), smem, cfg)) return rc;
    clip_adam_apply_kernel<<<dim3(kClipCtas, d.n_nets), kClipThreads, smem, s>>>(A, grads, per, clipnorm, norms_out);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_peer_adam(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const dmdqn_peers& peers,
                     const float* my_loss_src, float* loss_out, char* ws, const Workspace& w, cudaStream_t s) {
    const LearnArgs A = make_learn_args(d, hp, {}, nets, ws, w, nullptr, nullptr, 0);
    peer_reduce_adam_kernel<<<DMDQN_PEER_BLOCKS, 256, 0, s>>>(A, peers, my_loss_src, loss_out);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_fold(const dmdqn_dims& d, const dmdqn_nets& nets, char* ws, const Workspace& w, cudaStream_t s) {
    const Layout L = make_layout(d.obs_stride, d.hidden, true);
    fold_kernel<<<dim3(d.n_nets, 2), 256, 0, s>>>(L, d.hidden, d.n_actions, nets.theta, nets.theta_tgt,
                                                  reinterpret_cast<float*>(ws + w.head));
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_noisy_fold(const dmdqn_dims& d, bool dueling, const dmdqn_nets& nets, const dmdqn_noisy& nz, cudaStream_t s) {
    const Layout L = make_layout(d.obs_stride, d.hidden, dueling);
    const NoiseRec R = make_noise_rec(d.obs_stride, d.hidden);
    int n_sm = 0;
    if (int rc = device_sm_count(&n_sm)) return rc;
    const int64_t n4 = L.stride / 4;
    const int chunks = noisy_chunks(n_sm, 2 * (int64_t)d.n_nets, n4);
    const int64_t per = (n4 + chunks - 1) / chunks;
    noisy_fold_kernel<<<dim3(chunks, d.n_nets, 2), kNoisyThreads, R.stride * sizeof(float), s>>>(
        L, R, d.hidden, d.obs_dim, d.n_actions, dueling ? 1 : 0, nets, nz, per);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_noisy_adam_apply(const dmdqn_dims& d, const dmdqn_hparams& hp, const dmdqn_nets& nets, const dmdqn_noisy& nz,
                            const float* grads, char* ws, const Workspace& w, cudaStream_t s) {
    const LearnArgs A = make_learn_args(d, hp, {}, nets, ws, w, nullptr, nullptr, 0);
    const NoiseRec R = make_noise_rec(d.obs_stride, d.hidden);
    int n_sm = 0;
    if (int rc = device_sm_count(&n_sm)) return rc;
    const int64_t n4 = A.L.end / 4;
    const int chunks = noisy_chunks(n_sm, d.n_nets, n4);
    const int64_t per = (n4 + chunks - 1) / chunks;
    noisy_adam_apply_kernel<<<dim3(chunks, d.n_nets), kNoisyThreads, R.stride * sizeof(float), s>>>(A, nz, R, grads, per);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

int launch_sync_target(const dmdqn_dims& d, const dmdqn_nets& nets, const uint8_t* mask, double tau, bool dueling,
                       cudaStream_t s) {
    const Layout L = make_layout(d.obs_stride, d.hidden, dueling);
    dim3 grid(32, d.n_nets);
    sync_target_kernel<<<grid, 256, 0, s>>>(L.stride, nets.theta, nets.theta_tgt, mask, (float)tau);
    DMDQN_CUDA(cudaGetLastError());
    return DMDQN_OK;
}

}  // namespace dmdqn
