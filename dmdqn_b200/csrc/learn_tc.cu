// K3 / K4 on the 5th-generation tensor cores (tcgen05, kind::tf32, accumulators in TMEM).
//
// Same arithmetic contract as learn.cu (reference src/agents/dqn_agent.py:328-380), H = 256:
//   tc_target_kernel   K3   s' -> online(s'), target(s') -> TD target
//   tc_online_kernel   K4a  s  -> online(s), loss gradient, dh2, dh1 = (dh2 W2^T) * relu'(h1)
//   tc_wgrad_kernel    K4b  dW2 = h1^T dh2, dW1 = s^T dh1 with Adam + target sync in the epilogue
//
// tcgen05 has no fp32 MMA kind, so every fp32 operand x is split as x = hi + lo with
// hi = x rounded to tf32 and lo = x - hi (exact), and a product A*B is issued as three MMAs
// A_lo*B_hi + A_hi*B_lo + A_hi*B_hi accumulated in fp32 in TMEM ("3xTF32"; measured 3e-7 relative
// on B200, tools/umma_probe.cu).  PASSES = 1 issues only A*B (plain TF32, ~1e-3, toleranced apart).
//
// K3 / K4a are PERSISTENT (one CTA per SM walks its (network, 128-row tile) items) and warp-specialised:
//   warps 0-15  gather / epilogue: thread = batch row of the tile (UMMA M = 128), four warps per TMEM
//               sub-partition splitting the 256 columns in quarters.  They gather the observation rows of the
//               NEXT item into registers while the tensor pipe works on the current one, read accumulators with
//               tcgen05.ld, and write the next layer's A operand: hi part to shared memory (K-major, 128-byte
//               swizzle), lo part to TMEM columns 256..511 (A-from-TMEM MMA) -- 128 KB each, so all 512 TMEM
//               columns are used: 256 accumulator + 256 operand;
//   warp 16     lane 0 issues every tcgen05.mma and commits stages / GEMMs to mbarriers;
//   warp 17     lane 0 is the TMA producer: every weight chunk (8 k x 256 weights, raw fp32) travels global -> shared memory
//               through a tensor map that lands it IN the UMMA canonical layout of its GEMM -- x.W: rank-5 view {32 columns,
//               4 k-rows, 8 column blocks, K / 4 k-groups, network}, box {32, 4, 8, 2, 1}, SWIZZLE_128B_ATOM_32B = the MN-major
//               "128B_BASE32B" layout; d.W^T: box {8 k-columns, 256 rows}, SWIZZLE_32B = K-major SW32 -- straight into the hi half
//               of a stage, completion on the stage's mbarrier (expect_tx); each chunk is also requested into L2 six chunks ahead;
//   warps 18-23 converters, three groups of two warps: split a landed chunk IN PLACE (a 16-byte piece is read, its tf32-rounded
//               hi part stays at the same address, the lo part goes 8 KB further -- the layout is whatever TMA produced), then
//               hand the stage to the MMA lane.  Nobody holds weights in registers across a latency, nobody transposes them in
//               shared memory, and the epilogue warps never touch a weight.
// One ring of five stages serves all GEMMs of a kernel: tma (landed) -> conv (split) -> empty (tcgen05.commit: MMAs retired).
#include <cuda.h>
#include <string.h>
#include "common.cuh"

namespace dmdqn {

namespace {

constexpr int H = 256;          // hidden width served by this path
constexpr int BM = 128;         // batch rows per CTA (UMMA M)
constexpr int EW = 16;          // gather / epilogue warps of K3 / K4a
constexpr int NT = EW * 32;     // 512 threads
constexpr int W_MMA = EW, W_TMA = EW + 1, W_CONV = EW + 2;   // warps 18..23: three converter groups of two warps
constexpr int CONV_WARPS = 6, CONV_GROUP_WARPS = 2;
constexpr int NT_F = (EW + 8) * 32;   // 768 threads per K3 / K4a CTA: six warpgroups (setmaxnreg is per warpgroup)
// Register split (setmaxnreg works per warpgroup, inside the pool the CTA was launched with: 768 x 80): the MMA / TMA
// warpgroup and the converter warpgroup shrink to 32 and release 2 x 128 x 48 registers, which is exactly what the
// four gather / epilogue warpgroups need to grow to 104 (4 x 128 x 24).
constexpr int REGS_EPI = 104, REGS_AUX = 32;
constexpr int KC = 16;          // k-rows of a K4b operand chunk
constexpr uint32_t ATOM = BM * 128;           // bytes of one K-major SW128 atom column (128 rows x 32 floats)
constexpr unsigned long long WAIT_LIMIT_NS = 2000000000ull;   // a wrong descriptor must end in an error flag, not in a hung GPU

// ------------------------------------------------------------------------------------------
// PTX wrappers (syntax as in the CUTLASS sm100 headers shipped with the image).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// layout: 2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B, 1 = SWIZZLE_128B_BASE32B (the only MN-major layout for tf32)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16 |
           (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32 | (uint64_t)1 << 46 | (uint64_t)layout << 61;
}
// kind::tf32, fp32 accumulate, M = 128, N = 256
__host__ __device__ constexpr uint32_t make_idesc(bool a_mn, bool b_mn) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(H >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
__device__ __forceinline__ void mma_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t accum) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d), "l"(a), "l"(b), "r"(idesc),
                 "r"(accum) : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t accum) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d), "r"(a_tmem), "l"(b),
                 "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity), "r"(1000000u) : "memory");   // suspend-time hint (ns): sleep instead of re-polling
    return done;
}
// Bounded wait (wall-clock bound, ~2 s): false = the phase never completed.
__device__ __forceinline__ bool mbar_wait_slow(uint32_t bar, uint32_t parity) {
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        if (mbar_try(bar, parity)) return true;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > WAIT_LIMIT_NS) return false;
    }
}
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try(bar, parity)) return true;
    if (mbar_try(bar, parity)) return true;
    return mbar_wait_slow(bar, parity);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// TMA, 1-D: `bytes` contiguous bytes global -> shared memory, completion counted on `bar`
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar) : "memory");
}
// TMA, tensor map: one box of a rank-3 tensor
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
                 "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, int c4, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(dst),
                 "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(bar) : "memory");
}
template <int N> __device__ __forceinline__ void regs_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void regs_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
__device__ __forceinline__ void epi_sync() { asm volatile("bar.sync 1, 512;" ::: "memory"); }    // the 16 gather / epilogue warps of K3 / K4a
__device__ __forceinline__ void l2_prefetch(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
        "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
        "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};\n" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])),
        "r"(__float_as_uint(v[16])), "r"(__float_as_uint(v[17])), "r"(__float_as_uint(v[18])), "r"(__float_as_uint(v[19])),
        "r"(__float_as_uint(v[20])), "r"(__float_as_uint(v[21])), "r"(__float_as_uint(v[22])), "r"(__float_as_uint(v[23])),
        "r"(__float_as_uint(v[24])), "r"(__float_as_uint(v[25])), "r"(__float_as_uint(v[26])), "r"(__float_as_uint(v[27])),
        "r"(__float_as_uint(v[28])), "r"(__float_as_uint(v[29])), "r"(__float_as_uint(v[30])), "r"(__float_as_uint(v[31]))
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// x = hi + lo, hi = x rounded to tf32 (nearest, ties away from zero), lo = x - hi exact in fp32.
// The rounding is an integer add on the bit pattern (the carry walks into the exponent like the magnitude
// does) followed by the mask: two instructions where cvt.rna.tf32 expands to four on sm_100a (its inf/nan
// guard is dropped: a non-finite activation poisons the step either way).  Plain truncation (one LOP3)
// was tried and rejected: |lo| doubles and, worse, every truncated lo errs toward zero, so the error of a
// K = 512 gradient sum grows linearly instead of as a random walk (1.1e-5 of the tensor scale at B = 512).
__device__ __forceinline__ float tf32_hi(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}
template <int PASSES>
__device__ __forceinline__ void split4(const float4& x, float4& hi, float4& lo) {
    if (PASSES == 1) { hi = x; lo = make_float4(0.f, 0.f, 0.f, 0.f); return; }   // the tensor core truncates itself
    hi = make_float4(tf32_hi(x.x), tf32_hi(x.y), tf32_hi(x.z), tf32_hi(x.w));
    lo = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
}

// Byte offsets inside UMMA canonical tiles (validated by tools/umma_probe.cu).
//   K-major, 128-byte swizzle: [k/32][row][128 B], 16-byte piece index ^= row % 8
__device__ __forceinline__ uint32_t off_k128(int rows, int r, int k) {
    return (uint32_t)((k >> 5) * rows * 128 + r * 128 + ((((k & 31) >> 2) ^ (r & 7)) << 4) + ((k & 3) << 2));
}
//   MN-major tf32 (128B_BASE32B): atoms of 4 k x 32 mn = 512 B, [k/4][mn/32][k%4][128 B], 32-byte piece ^= k % 4
__device__ __forceinline__ uint32_t off_mn(int mn_total, int k, int mn) {
    return (uint32_t)((k >> 2) * (mn_total >> 5) * 512 + (mn >> 5) * 512 + (k & 3) * 128 +
                      ((((mn & 31) >> 3) ^ (k & 3)) << 5) + ((mn & 7) << 2));
}

// Release / acquire on a global flag (gpu scope).  The producer calls flag_release after a CTA-wide barrier that follows
// its last global store of the item; the consumer's bounded spin ends in an error flag, never in a hung GPU.
__device__ __forceinline__ void flag_release_add(int* f) {
    asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(f) : "memory");
}
__device__ __forceinline__ bool flag_acquire_ge(const int* f, int want) {
    // bounded by an iteration count (one register) rather than by the global timer: 2^21 polls of a ~256 ns sleep + an L2 round
    // trip are 2-3 s, the same order as the mbarrier waits' bound
    for (int i = 0; i < (1 << 21); ++i) {
        int v;
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        if (v >= want) return true;
        __nanosleep(256);
    }
    return false;
}
#ifdef TC_TIMING
__device__ __forceinline__ unsigned smid_() { unsigned r; asm volatile("mov.u32 %0, %%smid;" : "=r"(r)); return r; }
#endif
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Phase stamps (build with -DTC_TIMING, tools/phase_timing.sh): a few threads print clock64 deltas.
#ifdef TC_TIMING
#define KT_BEGIN const long long kt0_ = clock64(); long long kt1_ = 0
#define KT_END(name) do { if (threadIdx.x == 0 && (blockIdx.x % 37 == 0 || blockIdx.x == gridDim.x - 1)) \
        printf("%s cta %d kernel total %lld cycles, first item at %lld\n", name, blockIdx.x, clock64() - kt0_, kt1_ - kt0_); } while (0)
#define KT_FIRST() do { if (!kt1_) kt1_ = clock64(); } while (0)
#define TS_DECL long long ts_[16]; int tsi_ = 0
#define TS() do { if (tsi_ < 16) ts_[tsi_++] = clock64(); } while (0)
#define TS_D(i) (i < tsi_ ? ts_[i] - ts_[i - 1] : 0LL)
#define TS_PRINT(name) do { if (TC_TIMING > 1 && threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == 77 || blockIdx.x == gridDim.x - 1)) \
        printf("%s cta %d: %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld | total %lld\n", name, blockIdx.x, TS_D(1), TS_D(2), TS_D(3), \
               TS_D(4), TS_D(5), TS_D(6), TS_D(7), TS_D(8), TS_D(9), TS_D(10), TS_D(11), TS_D(12), ts_[tsi_ - 1] - ts_[0]); tsi_ = 0; } while (0)
#define WG_TS_DECL long long wts_[20]; int wtsi_ = 0
#define WG_TS() do { if (wtsi_ < 20) wts_[wtsi_++] = clock64(); } while (0)
#define WG_D(i) ((i) < wtsi_ ? wts_[i] - wts_[(i) - 1] : 0LL)
#define WG_TS_PRINT(name, cond) do { if (TC_TIMING > 1 && (cond) && (blockIdx.x == 0 || blockIdx.x == 100)) \
        printf("%s cta %d: %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld %lld\n", name, blockIdx.x, WG_D(1), WG_D(2), WG_D(3), WG_D(4), \
               WG_D(5), WG_D(6), WG_D(7), WG_D(8), WG_D(9), WG_D(10), WG_D(11), WG_D(12), WG_D(13), WG_D(14)); } while (0)
#else
#define KT_FIRST()
#define KT_BEGIN
#define KT_END(name)
#define TS_DECL
#define TS()
#define TS_PRINT(name)
#define WG_TS_DECL
#define WG_TS()
#define WG_TS_PRINT(name, cond)
#endif

// Shared-memory carve-up of the K3 / K4a kernels (offsets from a 1024-byte aligned base).
struct Fwd {
    static constexpr uint32_t R = 0;                          // 128 KB: X hi|lo during layer 1, then activation hi
    static constexpr uint32_t XLO = 3 * ATOM;                 // X lo (K <= 96) inside R
    static constexpr uint32_t WB = 8 * ATOM;                  // 80 KB weight ring: five in-place stages of 16 KB (hi 8 KB | lo 8 KB), one k-step each,
                                                              // shared by the x.W chunks (MN-major) and the d.W^T chunks (K-major SW32)
    static constexpr uint32_t BIAS1 = WB + 81920;             // b1[256]
    static constexpr uint32_t BIAS2 = BIAS1 + 1024;           // b2[256]
    static constexpr uint32_t W3S = BIAS2 + 1024;             // W3[256][4]
    static constexpr uint32_t QP = W3S + 4096;                // q partials [4][128][4]; K4a: dW3 / db2 partials of the upper row half
    static constexpr uint32_t ROWF = QP + 8192;               // per-row words: [BM ..] dL/dq 4-vectors, [7 BM ..] warp partials (3760 bytes used)
    static constexpr uint32_t BARS = ROWF + 3840;             // mbarriers | tmem base: the last 256 bytes of the ROWF block
    static constexpr uint32_t TOTAL = ROWF + 4096;            // + 1 KB alignment slack = 232 448 bytes: all of the 227 KB a CTA can have
};
// Barrier block (byte offsets from Fwd::BARS).
struct Bar {
    static constexpr uint32_t TMA_B = 112, CONV_B = 152, EMPTY_B = 192;  // weight ring: TMA landed / converted / MMAs retired, per stage
    static constexpr uint32_t AREADY = 232, DONE = 240;                  // A operand published (16 warps) / GEMM retired (1 commit)
    static constexpr uint32_t TMEM = 248;                                // TMEM base address (written by tcgen05.alloc)
};
constexpr int NSB = 5;                                        // stages of the weight ring (x.W and d.W^T chunks alike)
constexpr uint32_t STG_B = 16384, RAW_B = 8192;               // a stage: hi 8 KB | lo 8 KB (8 k x 256 weights, one k-step)

// Chunk / GEMM counters.  Every role walks the same sequence of items, GEMMs and chunks, so each keeps its own copy:
// b = chunks that have gone through the weight ring so far (stage = count % stages, use = count / stages,
// mbarrier parity = use & 1), gemms = GEMMs retired (parity of AREADY / DONE).
struct Ring {
    uint32_t b = 0, gemms = 0;
};

__device__ __forceinline__ float4 ldg_stream(const float* p) {   // volatile: issue order = program order
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_plain(const float* p) {    // coherent (the same kernel writes these arrays), issue order kept
    float4 v;
    asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ void sts4(uint32_t a, const float4& v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}

// ------------------------------------------------------------------------------------------
// TMA producer (lane 0 of warp W_TMA).
// ------------------------------------------------------------------------------------------
// Under load a DRAM read takes ~2 000 cycles and the tensor pipe wants a chunk every ~470, which five stages cannot cover, so
// every x.W chunk (rows 8c .. 8c+7 of W: 8 KB contiguous) is also requested into L2 PF chunks ahead of its copy (of this
// matrix, then of `next`: the matrix the ring streams after this one), which turns the copies into L2 hits.
constexpr int PF = 6;
// x.W IN PLACE (the ring both directions share): W seen through a rank-5 tensor map {32 columns, 4 k-rows, 8 column blocks,
// K / 4 k-groups, network} with box {32, 4, 8, 2, 1} and the 32-byte-atom 128-byte swizzle -- one box is a chunk of 8 k-rows x 256
// columns landing as [k / 4][column / 32][k % 4][128 B] with the 32-byte piece xor-ed by k % 4: the UMMA MN-major
// "128B_BASE32B" layout itself.  The converters then split it where it lies (hi stays, lo 8 KB further), exactly as they do
// for d.W^T: no raw slots, five stages deep instead of three, one barrier hop less per chunk.
__device__ __forceinline__ bool tma_fwd(uint32_t sbase, const CUtensorMap* tm, int g, const float* __restrict__ W, int K, Ring& r,
                                            bool ok, const float* __restrict__ next) {
    const uint32_t bars = sbase + Fwd::BARS;
    const int nchunks = K >> 3;
    for (int c = 0; c < nchunks; ++c) {
        const uint32_t s = r.b % NSB, u = r.b / NSB;
        if (c + PF < nchunks) l2_prefetch(W + (size_t)(c + PF) * 8 * H, RAW_B);
        else if (next) l2_prefetch(next + (size_t)(c + PF - nchunks) * 8 * H, RAW_B);
        if (u && ok) ok = mbar_wait(bars + Bar::EMPTY_B + 8 * s, (u - 1) & 1);
        mbar_expect_tx(bars + Bar::TMA_B + 8 * s, RAW_B);
        tma_load_5d(sbase + Fwd::WB + s * STG_B, tm, 0, 0, 0, 2 * c, g, bars + Bar::TMA_B + 8 * s);
        ++r.b;
    }
    return ok;
}
// d.W^T: box {8 k-columns, 256 rows, network g} of W2 seen as a rank-3 tensor -> 256 rows of 32 B with the 32-byte swizzle of
// the UMMA K-major SW32 layout, straight into the hi half of a stage (five stages of 16 KB: one k-step each)
__device__ __forceinline__ bool tma_bwd(uint32_t sbase, const CUtensorMap* tm, int g, Ring& r, bool ok) {
    const uint32_t bars = sbase + Fwd::BARS;
    for (int c = 0; c < H / 8; ++c) {
        const uint32_t s = r.b % NSB, u = r.b / NSB;
        if (u && ok) ok = mbar_wait(bars + Bar::EMPTY_B + 8 * s, (u - 1) & 1);
        mbar_expect_tx(bars + Bar::TMA_B + 8 * s, RAW_B);
        tma_load_3d(sbase + Fwd::WB + s * STG_B, tm, c * 8, 0, g, bars + Bar::TMA_B + 8 * s);       // in place: the hi half of the stage
        ++r.b;
    }
    return ok;
}
// ------------------------------------------------------------------------------------------
// Converters (warps W_CONV .. W_CONV + 5): raw fp32 chunk -> hi | lo halves of its stage, in place.  Three groups of two warps;
// chunk c of the ring goes to group c % 3, so each group has three chunk times for its wait -> read -> split -> write -> fence
// -> arrive chain.
// ------------------------------------------------------------------------------------------
template <int PASSES>
__device__ __forceinline__ bool conv_ring(uint32_t sbase, int grp, int t, Ring& r, bool ok, int nchunks = H / 8) {
    // In place: the chunk landed in the hi half of its stage already in the UMMA layout (the tensor map's box order and swizzle
    // are the layout), so a thread reads a 16-byte piece, leaves its hi part at the same address and puts the lo part 8 KB
    // further.  Stages (5) and groups (3) do not line up, and an mbarrier parity wait cannot tell "two phases ahead" from
    // "done": a group first waits until the stage's previous chunk has been converted (by whichever group) before it trusts
    // the parity of the stage's TMA barrier.
    const uint32_t bars = sbase + Fwd::BARS;
    constexpr int NGRP = CONV_WARPS / CONV_GROUP_WARPS;
    for (int c = 0; c < nchunks; ++c) {
        const uint32_t b = r.b + (uint32_t)c;
        if ((int)(b % NGRP) != grp) continue;
        const uint32_t s = b % NSB, u = b / NSB;
        const uint32_t st = sbase + Fwd::WB + s * STG_B;
        if (u && ok) ok = mbar_wait(bars + Bar::CONV_B + 8 * s, (u - 1) & 1);
        if (ok) ok = mbar_wait(bars + Bar::TMA_B + 8 * s, u & 1);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            float4 x[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) x[i] = lds4(st + (uint32_t)(t + 64 * (4 * half + i)) * 16u);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float4 hi, lo;
                split4<PASSES>(x[i], hi, lo);
                const uint32_t o = st + (uint32_t)(t + 64 * (4 * half + i)) * 16u;
                if (PASSES == 3) { sts4(o, hi); sts4(o + RAW_B, lo); }      // (one pass: the tensor core truncates the raw words itself)
            }
        }
        fence_async_smem();
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(bars + Bar::CONV_B + 8 * s);
    }
    r.b += (uint32_t)nchunks;
    return ok;
}

// ------------------------------------------------------------------------------------------
// MMA lane (lane 0 of warp W_MMA): D[128 x 256] (TMEM columns 0..255) = A[128 x K] * op(W), fp32 via PASSES MMAs.
//   A hi: shared memory, K-major SW128 at a_hi; A lo: shared memory (a_lo_smem != 0) or TMEM columns.
//   BT = false: x.W, stages MN-major;  BT = true: d.W^T, stages K-major SW32.  One k-step (8 k) per chunk either way.
// ------------------------------------------------------------------------------------------
template <int PASSES, bool BT>
__device__ __forceinline__ bool mma_gemm(uint32_t sbase, uint32_t tmem, uint32_t a_hi, uint32_t a_lo_smem, uint32_t a_lo_tmem,
                                         int K, Ring& r, bool ok) {
    const uint32_t bars = sbase + Fwd::BARS;
    constexpr int KCX = 8;
    constexpr uint32_t idesc = make_idesc(false, !BT);
    // Descriptors differ only in their 14-bit start-address field: build each once, then add (bytes >> 4).
    const uint64_t a_hi0 = make_desc(a_hi, 16, 1024, 2);
    const uint64_t a_lo0 = make_desc(a_lo_smem, 16, 1024, 2);
    const uint64_t b0 = BT ? make_desc(sbase + Fwd::WB, 16, 256, 6) : make_desc(sbase + Fwd::WB, 512, 4096, 1);
    if (ok) ok = mbar_wait(bars + Bar::AREADY, r.gemms & 1);      // all 16 epilogue warps have published the A operand
    tc_fence_after();
    const int nchunks = K / KCX;
    for (int c = 0; c < nchunks; ++c) {
        const uint32_t s = r.b % NSB, u = r.b / NSB;
        if (ok) ok = mbar_wait(bars + Bar::CONV_B + 8 * s, u & 1);   // the converters have finished chunk c
        tc_fence_after();
#pragma unroll
        for (int ks = 0; ks < KCX / 8; ++ks) {
            const int kg = c * KCX + ks * 8;
            const uint32_t a_off = ((uint32_t)(kg >> 5) * ATOM + (uint32_t)((kg & 31) >> 3) * 32) >> 4;
            const uint32_t b_off = (s * STG_B) >> 4;
            const uint64_t a_hi_d = a_hi0 + a_off;
            const uint64_t b_hi = b0 + b_off, b_lo = b0 + b_off + (RAW_B >> 4);
            uint32_t acc = (c | ks) ? 1u : 0u;
            if (PASSES == 3) {                                // small terms first
                if (a_lo_smem) mma_ss(tmem, a_lo0 + a_off, b_hi, idesc, acc);
                else mma_ts(tmem, a_lo_tmem + (uint32_t)kg, b_hi, idesc, acc);
                mma_ss(tmem, a_hi_d, b_lo, idesc, 1u);
                acc = 1u;
            }
            mma_ss(tmem, a_hi_d, b_hi, idesc, acc);
        }
        umma_commit(bars + Bar::EMPTY_B + 8 * s);   // the stage is free once these MMAs retire
        ++r.b;
    }
    umma_commit(bars + Bar::DONE);
    r.gemms += 1;
    return ok;
}

// ------------------------------------------------------------------------------------------
// Gather / epilogue side.
// ------------------------------------------------------------------------------------------
// Every epilogue thread calls this once its part of the next GEMM's A operand (shared memory and / or TMEM) is
// written: generic-proxy writes -> async proxy, tcgen05.st -> tcgen05.mma, one arrival per warp.
__device__ __forceinline__ void a_ready(uint32_t sbase) {
    fence_async_smem();
    tc_fence_before();
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(sbase + Fwd::BARS + Bar::AREADY);
}
// ... and this to wait for the GEMM that consumes it (every MMA retired, accumulator readable)
__device__ __forceinline__ bool wait_gemm(uint32_t sbase, Ring& r, bool ok) {
    if (ok) ok = mbar_wait(sbase + Fwd::BARS + Bar::DONE, r.gemms & 1);
    tc_fence_after();
    r.gemms += 1;
    return ok;
}

// Gather 128 observation rows -> hi (R) and lo (R + XLO), K-major SW128; rows past the batch are zero.
// begin() issues every load of the thread (row ids first, then up to 6 independent 16-byte pieces, the
// pieces of a row on consecutive lanes) -- it is called one item AHEAD, while the tensor pipe works on the
// current tile; store() splits and writes them once R is free.
template <int PASSES>
struct XGather {
    static constexpr int MAXP = BM * 96 / 4 / NT;             // 6 pieces per thread at obs_stride = 96
    float4 x[MAXP];
    uint32_t off[MAXP];
    int n;
    float4 sp;                                                // this thread's share of the item's small parameters (b1 | b2 | W3)

    // (P: the parameter block the item uses, W3: its head (LearnArgs::head).  Its biases and head weights -- 6 KB that every
    // epilogue reads from shared memory -- travel with the rows, one item ahead, instead of being fetched at the top of the item
    // with the epilogue warps waiting.)
    __device__ __forceinline__ void begin(const float* __restrict__ ring, const int32_t* __restrict__ rows, int r0, int B, int Dp,
                                          const float* __restrict__ P, const float* __restrict__ W3, const Layout& L) {
        {
            const int j = threadIdx.x;
            if (j < H) { sp.x = __ldg(P + L.b1 + j); sp.y = __ldg(P + L.b2 + j); }
            else sp = __ldg(reinterpret_cast<const float4*>(W3) + (j - H));
        }
        const int q = Dp >> 2;                                // 16-byte pieces per row
        n = BM * q / NT;
        const int dr = NT / q, dp = NT % q;
        int r = threadIdx.x / q, pc = threadIdx.x % q;
        int32_t rid[MAXP], col[MAXP];
#pragma unroll
        for (int j = 0; j < MAXP; ++j) {
            rid[j] = -1;
            if (j < n) {
                if (r0 + r < B) rid[j] = __ldg(rows + r0 + r);
                off[j] = off_k128(BM, r, pc << 2);
                col[j] = pc << 2;
                r += dr; pc += dp;
                if (pc >= q) { pc -= q; r += 1; }
            }
        }
#pragma unroll
        for (int j = 0; j < MAXP; ++j) {
            x[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j < n && rid[j] >= 0) x[j] = ldg_stream(ring + (size_t)rid[j] * Dp + col[j]);
        }
    }
    __device__ __forceinline__ void store(uint32_t sbase) {
        {
            float* s = reinterpret_cast<float*>(__cvta_shared_to_generic((size_t)sbase));
            const int j = threadIdx.x;
            if (j < H) { s[Fwd::BIAS1 / 4 + j] = sp.x; s[Fwd::BIAS2 / 4 + j] = sp.y; }
            else reinterpret_cast<float4*>(s + Fwd::W3S / 4)[j - H] = sp;
        }
#pragma unroll
        for (int j = 0; j < MAXP; ++j) {
            if (j < n) {
                float4 hi, lo;
                split4<PASSES>(x[j], hi, lo);
                sts4(sbase + Fwd::R + off[j], hi);
                if (PASSES == 3) sts4(sbase + Fwd::XLO + off[j], lo);
            }
        }
    }
};

// Per-thread epilogue coordinates: thread = batch row of the tile, four warps share a TMEM
// sub-partition and split the 256 columns in quarters (two 32-column blocks each).
struct Epi {
    int row, part;
    uint32_t lane_addr;
    __device__ __forceinline__ Epi() {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        row = (warp & 3) * 32 + lane;
        part = warp >> 2;
        lane_addr = (uint32_t)((warp & 3) * 32) << 16;
    }
};

// Epilogue of a hidden layer feeding another GEMM: a = relu(D + bias); hi -> shared memory R (next A operand),
// lo -> TMEM columns 256.., raw -> global (optional), returns the relu mask bits of this thread's 64 columns.
// Scratch activations are stored TRANSPOSED, [feature][batch]: a warp's 32 lanes are 32 consecutive
// batch rows, so every store below is one full 128-byte line, and K4b can stream them K-major.
template <int PASSES>
__device__ __forceinline__ void epi_hidden(uint32_t sbase, uint32_t tmem, const Epi& e, uint32_t bias_off,
                                           float* __restrict__ gout_t, int ldt, uint32_t (&mask)[2]) {
#pragma unroll 1
    for (int cc = 0; cc < 2; ++cc) {
        const int c0 = e.part * 64 + cc * 32;
        float v[32], lo[32];
        float4 bq[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)       // every bias load of the block before the first (volatile) store below
            bq[j] = lds4(sbase + bias_off + (uint32_t)(c0 + 4 * j) * 4);
        tmem_ld32(tmem + e.lane_addr + (uint32_t)c0, v);
        uint32_t m = 0;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
            const float4 b = bq[j >> 2];
            float4 x = make_float4(fmaxf(v[j] + b.x, 0.f), fmaxf(v[j + 1] + b.y, 0.f), fmaxf(v[j + 2] + b.z, 0.f),
                                   fmaxf(v[j + 3] + b.w, 0.f));
            m |= (x.x > 0.f ? 1u : 0u) << j | (x.y > 0.f ? 1u : 0u) << (j + 1) | (x.z > 0.f ? 1u : 0u) << (j + 2) |
                 (x.w > 0.f ? 1u : 0u) << (j + 3);
            if (gout_t) {
                gout_t[(size_t)(c0 + j) * ldt] = x.x; gout_t[(size_t)(c0 + j + 1) * ldt] = x.y;
                gout_t[(size_t)(c0 + j + 2) * ldt] = x.z; gout_t[(size_t)(c0 + j + 3) * ldt] = x.w;
            }
            float4 hi, l4;
            split4<PASSES>(x, hi, l4);
            sts4(sbase + Fwd::R + off_k128(BM, e.row, c0 + j), hi);
            lo[j] = l4.x; lo[j + 1] = l4.y; lo[j + 2] = l4.z; lo[j + 3] = l4.w;
        }
        mask[cc] = m;
        if (PASSES == 3) tmem_st32(tmem + e.lane_addr + 256u + (uint32_t)c0, lo);
    }
    if (PASSES == 3) tmem_st_wait();
    // visibility to the MMA lane comes with this thread's a_ready()
}

// Epilogue of layer 2 feeding the 4-wide head: q[a] = b3[a] + sum_j relu(D[j] + b2[j]) * W3[j][a]; the four
// column quarters of a row are combined in fixed order through shared memory.  Optionally stores the raw
// h2 row (for dW3) and returns the relu mask.
__device__ __forceinline__ void epi_head(uint32_t sbase, uint32_t tmem, const Epi& e, bool keep_h2,
                                         uint32_t (&mask)[2], float (&q)[4], const float* __restrict__ b3) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
    for (int cc = 0; cc < 2; ++cc) {
        const int c0 = e.part * 64 + cc * 32;
        float v[32];
        tmem_ld32(tmem + e.lane_addr + (uint32_t)c0, v);
        uint32_t m = 0;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            float b;
            asm volatile("ld.shared.f32 %0, [%1];" : "=f"(b) : "r"(sbase + Fwd::BIAS2 + (uint32_t)(c0 + j) * 4));
            const float x = fmaxf(v[j] + b, 0.f);
            v[j] = x;
            m |= (x > 0.f ? 1u : 0u) << j;
            const float4 w = lds4(sbase + Fwd::W3S + (uint32_t)(c0 + j) * 16);
            acc.x = fmaf(x, w.x, acc.x); acc.y = fmaf(x, w.y, acc.y);
            acc.z = fmaf(x, w.z, acc.z); acc.w = fmaf(x, w.w, acc.w);
        }
        mask[cc] = m;
        if (keep_h2) {      // raw h2 tile -> R (free once layer 2 has run), read back column-wise for dW3 / db2
#pragma unroll
            for (int j = 0; j < 32; j += 4)
                sts4(sbase + Fwd::R + off_k128(BM, e.row, c0 + j), make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
        }
    }
    float4* qp = reinterpret_cast<float4*>(__cvta_shared_to_generic((size_t)(sbase + Fwd::QP)));
    qp[e.part * BM + e.row] = acc;
    epi_sync();
    const float4 p0 = qp[e.row], p1 = qp[BM + e.row], p2 = qp[2 * BM + e.row], p3 = qp[3 * BM + e.row];
    q[0] = ((p0.x + p1.x) + (p2.x + p3.x)) + __ldg(b3 + 0); q[1] = ((p0.y + p1.y) + (p2.y + p3.y)) + __ldg(b3 + 1);
    q[2] = ((p0.z + p1.z) + (p2.z + p3.z)) + __ldg(b3 + 2); q[3] = ((p0.w + p1.w) + (p2.w + p3.w)) + __ldg(b3 + 3);
}

__device__ __forceinline__ uint32_t tc_prologue(uint32_t sbase) {
    const int warp = threadIdx.x >> 5;
    const uint32_t bars = sbase + Fwd::BARS;
    if (threadIdx.x == 0) {
        for (int b = 0; b < NSB; ++b) {
            mbar_init(bars + Bar::TMA_B + 8 * b, 1);
            mbar_init(bars + Bar::CONV_B + 8 * b, CONV_GROUP_WARPS);
            mbar_init(bars + Bar::EMPTY_B + 8 * b, 1);
        }
        mbar_init(bars + Bar::AREADY, EW);
        mbar_init(bars + Bar::DONE, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bars + Bar::TMEM), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(bars + Bar::TMEM));
    return tmem;
}
__device__ __forceinline__ void tc_epilogue(uint32_t tmem) {
    tc_fence_before();
    __syncthreads();
    if ((threadIdx.x >> 5) == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// ------------------------------------------------------------------------------------------
// K3: item = (network, 128-row tile, which parameter set): Q(s') of the online net (-> q_next) or of the
// target net (-> tq_all).  The two halves are independent items (twice as many, half as long: less tail on
// 148 SMs); K4a combines them into the TD target of its rows (reference :342-347).  A CTA walks the items
// blockIdx.x, + gridDim.x, ... of active networks; every role runs the same walk.
// ------------------------------------------------------------------------------------------
// The head K3 / K4a read for network g's parameter set `tgt` (P: that set's block): the plain instantiation reads W3 | b3
// from P itself, the same code as before dueling heads existed; the dueling one reads the fold kernel's W3e | b3e
// (LearnArgs::head).  b3 follows W3 in both.
template <bool DUELING>
__device__ __forceinline__ const float* head_w3(const LearnArgs& A, const float* P, int tgt, int g) {
    if constexpr (DUELING) return (tgt ? A.head[1] : A.head[0]) + (size_t)g * A.head_stride;
    else return P + A.L.w3;
}
template <bool DUELING>
__device__ __forceinline__ const float* head_b3(const LearnArgs& A, const float* P, int tgt, int g) {
    if constexpr (DUELING) return head_w3<true>(A, P, tgt, g) + 4 * H;
    else return P + A.L.b3;
}

__device__ __forceinline__ int k3_next(const LearnArgs& A, int q, int n_items) {
    while (q < n_items && !A.active[(q >> 1) / A.tc_tiles]) q += gridDim.x;
    return q;
}

template <int PASSES, bool DUELING>
__global__ void __launch_bounds__(NT_F, 1) tc_target_kernel(const LearnArgs A, const __grid_constant__ CUtensorMap tm_w1,
                                                            const __grid_constant__ CUtensorMap tm_w2,
                                                            const __grid_constant__ CUtensorMap tm_w1t,
                                                            const __grid_constant__ CUtensorMap tm_w2t) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const int B = A.d.batch, Dp = A.d.obs_stride;
    const int n_items = 2 * A.d.n_nets * A.tc_tiles;
    const int warp = threadIdx.x >> 5;
    KT_BEGIN;
    const uint32_t tmem = tc_prologue(sbase);
    if (A.chain) {
        asm volatile("griddepcontrol.wait;" ::: "memory");   // the sample kernel (this launch may have started under its tail) is complete
        pdl_launch_dependents();               // K4a's CTAs may take an SM as soon as this kernel's CTA has left it
    }
    Ring ring;
    bool ok = true;
    if (warp >= EW) {
        regs_dec<REGS_AUX>();          // one instruction for both auxiliary warpgroups (.aligned)
      if (warp == W_MMA) {
        if ((threadIdx.x & 31) == 0) {
            // This lane also publishes the PREVIOUS item's outputs (release of the per-tile flag): it has just seen every
            // epilogue warp arrive for this item's layer 1 -- an arrival that follows that warp's last store of the previous
            // item -- and it is idle until the layer-1 epilogue is done, so the fence costs the epilogue warps nothing.
            int prev = -1;
            for (int q = k3_next(A, blockIdx.x, n_items); q < n_items; q = k3_next(A, q + gridDim.x, n_items)) {
                ok = mma_gemm<PASSES, false>(sbase, tmem, sbase + Fwd::R, sbase + Fwd::XLO, 0, Dp, ring, ok);
                if (prev >= 0) flag_release_add(A.k3_done + (size_t)((prev >> 1) / A.tc_tiles) * A.ws_tiles + (prev >> 1) % A.tc_tiles);
                prev = q;
                ok = mma_gemm<PASSES, false>(sbase, tmem, sbase + Fwd::R, 0, tmem + 256u, H, ring, ok);
            }
            if (!ok) atomicExch(A.error, 13);
        }
        __syncwarp();
      } else if (warp == W_TMA) {
        if ((threadIdx.x & 31) == 0) {
            for (int q = k3_next(A, blockIdx.x, n_items); q < n_items;) {
                const int g = (q >> 1) / A.tc_tiles;
                const float* P = ((q & 1) ? A.nets.theta_tgt : A.nets.theta) + (size_t)g * A.L.stride;
                const int qn = k3_next(A, q + gridDim.x, n_items);
                const float* Pn = qn < n_items ? ((qn & 1) ? A.nets.theta_tgt : A.nets.theta) + (size_t)((qn >> 1) / A.tc_tiles) * A.L.stride + A.L.w1 : nullptr;
                ok = tma_fwd(sbase, (q & 1) ? &tm_w1t : &tm_w1, g, P + A.L.w1, Dp, ring, ok, P + A.L.w2);
                ok = tma_fwd(sbase, (q & 1) ? &tm_w2t : &tm_w2, g, P + A.L.w2, H, ring, ok, Pn);
                q = qn;
            }
            if (!ok) atomicExch(A.error, 23);
        }
        __syncwarp();
      } else if (warp < W_CONV + CONV_WARPS) {   // converters (the last two warps only fill the warpgroup)
        const int tc = threadIdx.x - W_CONV * 32, cg = (warp - W_CONV) / CONV_GROUP_WARPS, t = tc % (CONV_GROUP_WARPS * 32);
        for (int q = k3_next(A, blockIdx.x, n_items); q < n_items; q = k3_next(A, q + gridDim.x, n_items)) {
            ok = conv_ring<PASSES>(sbase, cg, t, ring, ok, Dp / 8);
            ok = conv_ring<PASSES>(sbase, cg, t, ring, ok, H / 8);
        }
        if (!ok && tc == 0) atomicExch(A.error, 33);
      }
    } else {
        regs_inc<REGS_EPI>();
        const Epi e;
        XGather<PASSES> xg;
        int q = k3_next(A, blockIdx.x, n_items);
        if (q < n_items) {
            const int g = (q >> 1) / A.tc_tiles, rt = (q >> 1) % A.tc_tiles;
            const float* P = ((q & 1) ? A.nets.theta_tgt : A.nets.theta) + (size_t)g * A.L.stride;
            xg.begin(A.rp.next_obs, A.nrows + (size_t)g * B, rt * BM, B, Dp, P, head_w3<DUELING>(A, P, q & 1, g), A.L);
        }
        int q_last = -1;                                       // the last item is published here, the others by the MMA lane
        while (q < n_items) {
            const int item = q >> 1, pass = q & 1;            // 0: online(s')  1: target(s')
            const int g = item / A.tc_tiles, rt = item % A.tc_tiles, r0 = rt * BM;
            const float* P = (pass == 0 ? A.nets.theta : A.nets.theta_tgt) + (size_t)g * A.L.stride;
            TS_DECL;
            TS();
            KT_FIRST();
            xg.store(sbase);          // observation rows and b1 | b2 | W3 of this item: requested one item ago
            a_ready(sbase);
            epi_sync();        // biases / head weights visible to every epilogue thread
            TS();
            ok = wait_gemm(sbase, ring, ok);
            TS();
            uint32_t mask[2];
            epi_hidden<PASSES>(sbase, tmem, e, Fwd::BIAS1, nullptr, 0, mask);
            a_ready(sbase);
            TS();
            const int qn = k3_next(A, q + gridDim.x, n_items);
            if (qn < n_items) {                                // the next tile's rows travel while layer 2 runs
                const int gn = (qn >> 1) / A.tc_tiles, rtn = (qn >> 1) % A.tc_tiles;
                const float* Pn = ((qn & 1) ? A.nets.theta_tgt : A.nets.theta) + (size_t)gn * A.L.stride;
                xg.begin(A.rp.next_obs, A.nrows + (size_t)gn * B, rtn * BM, B, Dp, Pn, head_w3<DUELING>(A, Pn, qn & 1, gn), A.L);
            }
            ok = wait_gemm(sbase, ring, ok);
            TS();
            float qv[4];
            epi_head(sbase, tmem, e, false, mask, qv, head_b3<DUELING>(A, P, pass, g));
            TS();
            TS_PRINT("K3 store L1 epi1 L2 epi2");
            const int gr = r0 + e.row;
            if (e.part == 0 && gr < B) {
                float* out = (pass == 0 ? A.q_next : A.tq_all) + ((size_t)g * B + gr) * 4;
                *reinterpret_cast<float4*>(out) = make_float4(qv[0], qv[1], qv[2], qv[3]);
            }
            q_last = q;
            q = qn;
        }
        epi_sync();
        if (q_last >= 0 && threadIdx.x == 0) flag_release_add(A.k3_done + (size_t)((q_last >> 1) / A.tc_tiles) * A.ws_tiles + (q_last >> 1) % A.tc_tiles);
        if (!ok && threadIdx.x == 0) atomicExch(A.error, 3);
        KT_END("K3");
    }
    tc_epilogue(tmem);
}

// ------------------------------------------------------------------------------------------
// K4a: item = (network, 128-row tile).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int k4_next(const LearnArgs& A, int q, int n_items) {
    while (q < n_items && !A.active[q / A.tc_tiles]) q += gridDim.x;
    return q;
}

template <int PASSES, bool DUELING>
__global__ void __launch_bounds__(NT_F, 1) tc_online_kernel(const LearnArgs A, const __grid_constant__ CUtensorMap tmap_w2,
                                                            const __grid_constant__ CUtensorMap tm_w1,
                                                            const __grid_constant__ CUtensorMap tm_w2) {
    extern __shared__ uint8_t smem_raw[];
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    float* sf = reinterpret_cast<float*>(__cvta_shared_to_generic((size_t)sbase));
    const int B = A.d.batch, Dp = A.d.obs_stride;
    const int n_items = A.d.n_nets * A.tc_tiles;
    const int warp = threadIdx.x >> 5;
    KT_BEGIN;
    const uint32_t tmem = tc_prologue(sbase);
    if (A.chain) pdl_launch_dependents();      // K4b's CTAs may take an SM as soon as this kernel's CTA has left it
    Ring ring;
    bool ok = true;
    if (warp >= EW) {
        regs_dec<REGS_AUX>();          // one instruction for both auxiliary warpgroups (.aligned)
      if (warp == W_MMA) {
        if ((threadIdx.x & 31) == 0) {
            int prev = -1;                                     // as in K3: the previous item is published from this lane's idle window
            for (int q = k4_next(A, blockIdx.x, n_items); q < n_items; q = k4_next(A, q + gridDim.x, n_items)) {
                ok = mma_gemm<PASSES, false>(sbase, tmem, sbase + Fwd::R, sbase + Fwd::XLO, 0, Dp, ring, ok);
                ok = mma_gemm<PASSES, false>(sbase, tmem, sbase + Fwd::R, 0, tmem + 256u, H, ring, ok);
                // (the epilogue issues the second half of an item's dh1^T stores after it has published the NEXT item's layer-1
                // operand, so the previous item is complete only once this item's LAYER-2 operand has been published)
                if (prev >= 0) flag_release_add(A.k4a_done + prev / A.tc_tiles);
                prev = q;
                ok = mma_gemm<PASSES, true>(sbase, tmem, sbase + Fwd::R, 0, tmem + 256u, H, ring, ok);
            }
            if (!ok) atomicExch(A.error, 14);
        }
        __syncwarp();
      } else if (warp == W_TMA) {
        if ((threadIdx.x & 31) == 0) {
            for (int q = k4_next(A, blockIdx.x, n_items); q < n_items; q = k4_next(A, q + gridDim.x, n_items)) {
                const int g = q / A.tc_tiles;
                // K3 may still be running on other SMs: both halves of this tile's TD-target inputs must have been published
                if (A.chain && ok) ok = flag_acquire_ge(A.k3_done + (size_t)g * A.ws_tiles + q % A.tc_tiles, 2);
                const float* P = A.nets.theta + (size_t)g * A.L.stride;
                const int qn = k4_next(A, q + gridDim.x, n_items);
                const float* Pn = qn < n_items ? A.nets.theta + (size_t)(qn / A.tc_tiles) * A.L.stride + A.L.w1 : nullptr;
                // one ring for all three GEMMs: a stage is reused as soon as its MMAs have retired, whatever GEMM they belong to
                ok = tma_fwd(sbase, &tm_w1, g, P + A.L.w1, Dp, ring, ok, P + A.L.w2);
                ok = tma_fwd(sbase, &tm_w2, g, P + A.L.w2, H, ring, ok, Pn);
                ok = tma_bwd(sbase, &tmap_w2, g, ring, ok);
            }
            if (!ok) atomicExch(A.error, 24);
        }
        __syncwarp();
      } else if (warp < W_CONV + CONV_WARPS) {   // converters (the last two warps only fill the warpgroup)
        const int tc = threadIdx.x - W_CONV * 32, cg = (warp - W_CONV) / CONV_GROUP_WARPS, t = tc % (CONV_GROUP_WARPS * 32);
        for (int q = k4_next(A, blockIdx.x, n_items); q < n_items; q = k4_next(A, q + gridDim.x, n_items)) {
            ok = conv_ring<PASSES>(sbase, cg, t, ring, ok, Dp / 8);
            ok = conv_ring<PASSES>(sbase, cg, t, ring, ok, H / 8);
            ok = conv_ring<PASSES>(sbase, cg, t, ring, ok, H / 8);
        }
        if (!ok && tc == 0) atomicExch(A.error, 34);
      }
    } else {
        regs_inc<REGS_EPI>();
        const Epi e;
        XGather<PASSES> xg;
        int q = k4_next(A, blockIdx.x, n_items);
        if (q < n_items) {
            const float* P = A.nets.theta + (size_t)(q / A.tc_tiles) * A.L.stride;
            xg.begin(A.rp.obs, A.rows + (size_t)(q / A.tc_tiles) * B, (q % A.tc_tiles) * BM, B, Dp, P, head_w3<DUELING>(A, P, 0, q / A.tc_tiles), A.L);
        }
        int q_last = -1;                                       // the last item is published here, the others by the MMA lane
        while (q < n_items) {
            const int g = q / A.tc_tiles, rt = q % A.tc_tiles, r0 = rt * BM;
            const size_t sb = (size_t)g * B;
            const float* P = A.nets.theta + (size_t)g * A.L.stride;
            const int gr = r0 + e.row;
            const bool valid = gr < B;
            TS_DECL;
            TS();
            KT_FIRST();
            if (q_last < 0) {         // first item of the CTA; later items were published at the end of the previous one
                xg.store(sbase);      // observation rows and b1 | b2 | W3 of this item: requested one item ago
                a_ready(sbase);
            }
            epi_sync();        // biases / head weights visible to every epilogue thread
            TS();
            ok = wait_gemm(sbase, ring, ok);
            TS();
            uint32_t mask1[2], mask2[2];
            epi_hidden<PASSES>(sbase, tmem, e, Fwd::BIAS1, valid ? A.h1 + sb * H + gr : nullptr, B, mask1);
            a_ready(sbase);
            TS();
            // TD target of this row from the two halves of K3 (reference :342-347), ties -> lowest index
            // Computed while the layer-2 GEMM runs (the epilogue warps have nothing else to do).  In a chain the TMA lane has waited
            // for K3's flag of this tile before it sent the first weight chunk of the item, so both halves have long been in L2
            // (the loads bypass L1).
            float yi = 0.f;
            if (valid) {
                const float4 qo = ldg_plain(A.q_next + (sb + gr) * 4);
                const float4 qt = ldg_plain(A.tq_all + (sb + gr) * 4);
                const float q_on[4] = {qo.x, qo.y, qo.z, qo.w}, q_tg[4] = {qt.x, qt.y, qt.z, qt.w};
                float bmax = q_on[0], tq = q_tg[0], tmax = q_tg[0];
#pragma unroll
                for (int k = 1; k < 4; ++k) {
                    if (k < A.d.n_actions) {
                        if (q_on[k] > bmax) { bmax = q_on[k]; tq = q_tg[k]; }
                        tmax = fmaxf(tmax, q_tg[k]);
                    }
                }
                tq = A.double_dqn ? tq : tmax;
                yi = A.r_hat[sb + gr] + A.disc_b[sb + gr] * tq;
                if (e.part == 0) A.y[sb + gr] = yi;
            }
            const int ai_pre = valid ? A.act_b[sb + gr] : 0;
            ok = wait_gemm(sbase, ring, ok);
            TS();
            float qv[4];
            epi_head(sbase, tmem, e, true, mask2, qv, head_b3<DUELING>(A, P, 0, g));
            TS();

            // loss term and dL/dpred of this row (reference :349-352)
            float gi = 0.f, term = 0.f;
            int ai = 0;
            if (valid) {
                ai = ai_pre;
                const float qa = ai == 0 ? qv[0] : ai == 1 ? qv[1] : ai == 2 ? qv[2] : qv[3];
                const float err = qa - yi;
                if (A.loss == DMDQN_LOSS_MSE) {
                    term = err * err;
                    gi = (2.0f * err) / (float)A.loss_batch;
                } else {
                    const float ae = fabsf(err);
                    term = ae <= 1.0f ? 0.5f * err * err : ae - 0.5f;
                    gi = fminf(fmaxf(err, -1.0f), 1.0f) / (float)A.loss_batch;
                }
                if (A.per) {                                  // prioritized replay: importance weight, then the new priority
                    const float wi = A.is_w[sb + gr];
                    term = wi * term;
                    gi = wi * gi;
                    if (e.part == 0 && ok) per_store_priority(A, A.rows[sb + gr], err);
                }
                if (e.part == 0) {
                    A.ga[sb + gr] = make_float2(gi, __int_as_float(ai));
                    *reinterpret_cast<float4*>(A.q_all + (sb + gr) * 4) = make_float4(qv[0], qv[1], qv[2], qv[3]);
                }
            }
            float* rowf = sf + Fwd::ROWF / 4;                     // [BM ..]: per row float4 g * onehot(action), [7 BM ..]: warp partials
            if (e.part == 0) {
                // dL/dq of this row as a 4-vector (one non-zero): the column loop below then needs no selects
                reinterpret_cast<float4*>(rowf + BM)[e.row] = make_float4(ai == 0 ? gi : 0.f, ai == 1 ? gi : 0.f, ai == 2 ? gi : 0.f, ai == 3 ? gi : 0.f);
                // per-tile loss / metric / db3 partials: butterfly over the 32 rows of this warp (fixed order), then
                // the four warp partials are added in warp order by thread 0
                float red[11];
                red[0] = term;
                red[1] = 0.f; red[2] = 0.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float qq = (valid && k < A.d.n_actions) ? qv[k] : 0.f;
                    red[1] += qq;
                    red[2] = fmaf(qq, qq, red[2]);
                    red[3 + k] = (valid && ai == k) ? 1.f : 0.f;
                    red[7 + k] = (valid && ai == k) ? gi : 0.f;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                    for (int v = 0; v < 11; ++v) red[v] += __shfl_xor_sync(0xffffffffu, red[v], o);
                if ((threadIdx.x & 31) == 0)
#pragma unroll
                    for (int v = 0; v < 11; ++v) rowf[7 * BM + (threadIdx.x >> 5) * 11 + v] = red[v];
            }
            epi_sync();
            TS();
            if (threadIdx.x < 11) {
                const float* wp = rowf + 7 * BM + threadIdx.x;
                const float tot = ((wp[0] + wp[11]) + wp[22]) + wp[33];
                const size_t pt = (size_t)g * A.tc_tiles + rt;
                if (threadIdx.x < 7) A.part_loss[pt * 8 + threadIdx.x] = tot;      // loss, q sum, q^2 sum, action histogram
                else A.part_b3[pt * 4 + (threadIdx.x - 7)] = tot;
            }
            {   // dW3[j][a] = sum_i h2[i][j] g_i [a_i = a] and db2[j] = sum_i dh2[i][j] over this tile's rows, read back from the h2
                // tile epi_head left in R.  Thread = (four adjacent columns, 16 rows): warp w covers the 32 columns of block
                // w % 8 and the row half w / 8, lane = (column quad, row group).  One 16-byte load brings four columns of a row
                // (they are one swizzled piece of the K-major tile), one broadcast load the row's g * onehot(action): two
                // shared-memory loads per four elements (the previous column-per-thread loop needed eight and was bound by
                // them).  The four row groups of a warp are combined by a fixed xor butterfly, the two row halves through QP.
                const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
                const int j0 = ((w & 7) * 8 + (l & 7)) * 4, rh = w >> 3, rg = l >> 3;
                float4 w3c[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) w3c[c] = lds4(sbase + Fwd::W3S + (uint32_t)(j0 + c) * 16);
                float d[4][4], s2[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) { d[c][0] = d[c][1] = d[c][2] = d[c][3] = 0.f; s2[c] = 0.f; }
                const uint32_t hrow = sbase + Fwd::R + (uint32_t)(j0 >> 5) * ATOM;
                const uint32_t piece = (uint32_t)((j0 & 31) >> 2);
                const uint32_t gsel = sbase + Fwd::ROWF + BM * 4;
                const int i_begin = rh * (BM / 2) + rg * 16;
#pragma unroll 4
                for (int u = 0; u < 16; ++u) {
                    const int i = i_begin + u;
                    const float4 h4 = lds4(hrow + (uint32_t)i * 128u + ((piece ^ (uint32_t)(i & 7)) << 4));
                    const float4 gs = lds4(gsel + (uint32_t)i * 16u);
                    const float hv[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        d[c][0] = fmaf(hv[c], gs.x, d[c][0]); d[c][1] = fmaf(hv[c], gs.y, d[c][1]);
                        d[c][2] = fmaf(hv[c], gs.z, d[c][2]); d[c][3] = fmaf(hv[c], gs.w, d[c][3]);
                        const float gw = fmaf(gs.w, w3c[c].w, fmaf(gs.z, w3c[c].z, fmaf(gs.y, w3c[c].y, gs.x * w3c[c].x)));   // = g * W3[j][a]: the other terms are exact zeros
                        s2[c] += hv[c] > 0.f ? gw : 0.f;
                    }
                }
#pragma unroll
                for (int o = 8; o <= 16; o <<= 1) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
#pragma unroll
                        for (int a = 0; a < 4; ++a) d[c][a] += __shfl_xor_sync(0xffffffffu, d[c][a], o);
                        s2[c] += __shfl_xor_sync(0xffffffffu, s2[c], o);
                    }
                }
                TS();
                float* up = sf + Fwd::QP / 4;                     // [256][8] floats: partials of the upper row half
                if (rh == 1 && rg == 0) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        reinterpret_cast<float4*>(up)[(j0 + c) * 2] = make_float4(d[c][0], d[c][1], d[c][2], d[c][3]);
                        up[(j0 + c) * 8 + 4] = s2[c];
                    }
                }
                epi_sync();
                if (rh == 0 && rg == 0) {
                    const size_t pt = (size_t)g * A.tc_tiles + rt;
                    float sb2[4];
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float4 u4 = reinterpret_cast<const float4*>(up)[(j0 + c) * 2];
                        reinterpret_cast<float4*>(A.part_w3 + pt * H * 4)[j0 + c] = make_float4(d[c][0] + u4.x, d[c][1] + u4.y, d[c][2] + u4.z, d[c][3] + u4.w);
                        sb2[c] = s2[c] + up[(j0 + c) * 8 + 4];
                    }
                    *reinterpret_cast<float4*>(A.part_b2 + pt * H + j0) = make_float4(sb2[0], sb2[1], sb2[2], sb2[3]);
                }
            }
            epi_sync();          // R is rewritten with dh2 below
            TS();

            // dh2[j] = relu'(h2[j]) * g * W3[j][a]  (dq has one non-zero per row): hi -> R, lo -> TMEM.  It is not
            // written to global memory: K4b rebuilds its dh2^T operand from relu'(h2) bits, g, the action and W3.
            if (valid) reinterpret_cast<uint2*>(A.mask2)[(sb + gr) * 4 + e.part] = make_uint2(mask2[0], mask2[1]);
            if (rt == 0 && threadIdx.x < H)    // W3 as this step saw it (K4b updates W3 while other CTAs of the network still need the old values)
                reinterpret_cast<float4*>(A.w3_copy + (size_t)g * H * 4)[threadIdx.x] =
                    *reinterpret_cast<const float4*>(sf + Fwd::W3S / 4 + threadIdx.x * 4);
#pragma unroll 1
            for (int cc = 0; cc < 2; ++cc) {
                const int c0 = e.part * 64 + cc * 32;
                float lo[32], wv[32];
#pragma unroll
                for (int j = 0; j < 32; ++j)      // all 32 loads first: the volatile stores below would otherwise serialise load -> store chains
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(wv[j]) : "r"(sbase + Fwd::W3S + (uint32_t)(c0 + j) * 16 + (uint32_t)ai * 4));
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    float x[4];
#pragma unroll
                    for (int t = 0; t < 4; ++t) x[t] = ((mask2[cc] >> (j + t)) & 1u) ? gi * wv[j + t] : 0.f;
                    float4 hi, l4;
                    split4<PASSES>(make_float4(x[0], x[1], x[2], x[3]), hi, l4);
                    sts4(sbase + Fwd::R + off_k128(BM, e.row, c0 + j), hi);
                    lo[j] = l4.x; lo[j + 1] = l4.y; lo[j + 2] = l4.z; lo[j + 3] = l4.w;
                }
                if (PASSES == 3) tmem_st32(tmem + e.lane_addr + 256u + (uint32_t)c0, lo);
            }
            if (PASSES == 3) tmem_st_wait();
            a_ready(sbase);
            TS();
            const int qn = k4_next(A, q + gridDim.x, n_items);
            if (qn < n_items) {                                   // the next tile's rows travel while the backward GEMM runs
                const float* Pn = A.nets.theta + (size_t)(qn / A.tc_tiles) * A.L.stride;
                xg.begin(A.rp.obs, A.rows + (size_t)(qn / A.tc_tiles) * B, (qn % A.tc_tiles) * BM, B, Dp, Pn, head_w3<DUELING>(A, Pn, 0, qn / A.tc_tiles),
                         A.L);
            }
            // dh1 = (dh2 W2^T) * relu'(h1)
            ok = wait_gemm(sbase, ring, ok);
            TS();
            {   // The accumulator is read in two halves; as soon as the second half is in registers the TMEM columns and R are free,
                // so the NEXT item's layer-1 operand is published first (its GEMM starts, and the proxy fence inside a_ready() --
                // a MEMBAR.ALL.CTA -- does not wait for 32 fresh global stores per thread), and the second half of the dh1^T stores
                // goes out in that GEMM's shadow.
                float v[32];
                const int c0 = e.part * 64;
                tmem_ld32(tmem + e.lane_addr + (uint32_t)c0, v);
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        A.dh1[sb * H + (size_t)(c0 + j) * B + gr] = ((mask1[0] >> j) & 1u) ? v[j] : 0.f;
                }
                tmem_ld32(tmem + e.lane_addr + (uint32_t)(c0 + 32), v);
                if (qn < n_items) {
                    xg.store(sbase);
                    a_ready(sbase);
                }
                if (valid) {
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        A.dh1[sb * H + (size_t)(c0 + 32 + j) * B + gr] = ((mask1[1] >> j) & 1u) ? v[j] : 0.f;
                }
            }
            TS();
            TS_PRINT("K4a store L1 epi1 L2 epi2 loss dW3loop dW3out dh2 bwdGEMM dh1store");
            q_last = q;
            q = qn;
        }
        epi_sync();
        if (q_last >= 0 && threadIdx.x == 0) flag_release_add(A.k4a_done + q_last / A.tc_tiles);
        if (!ok && threadIdx.x == 0) atomicExch(A.error, 4);
        KT_END("K4a");
    }
    tc_epilogue(tmem);
}

// ------------------------------------------------------------------------------------------
// K4b
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void adam1(const AdamStep& k, float g, float& th, float& m, float& v, float& tg) {
    m = m + (g - m) * k.one_m_b1;
    v = v + (g * g - v) * k.one_m_b2;
    // MUFU square root and reciprocal (each within ~2 ulp): the quotient is a step of at most ~lr, so a few
    // ulp of it are far below one ulp of the weight it is subtracted from; the IEEE sequences cost ~60
    // dependent instructions per element and made the epilogue issue-bound
    float sq;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(v));
    th = th - __fdividef(m * k.alpha, sq + k.eps);
    if (k.sync == 1) tg = th;
    else if (k.sync == 2) tg = k.tau * th + (1.0f - k.tau) * tg;
}

// Adam on one element without the target sync (the caller applies it per 16-byte group)
__device__ __forceinline__ void adam_fast(const AdamStep& k, float g, float& th, float& m, float& v) {
    m = m + (g - m) * k.one_m_b1;
    v = v + (g * g - v) * k.one_m_b2;
    float sq;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(v));
    th = th - __fdividef(m * k.alpha, sq + k.eps);
}

struct Wg {     // persistent wgrad kernel, one CTA per SM
    static constexpr int STAGES = 3;
    static constexpr uint32_t A_BYTES = KC * BM * 4;          // 8 KB
    static constexpr uint32_t B_BYTES = KC * H * 4;           // 16 KB
    static constexpr uint32_t AUX = 2 * A_BYTES + 2 * B_BYTES;   // A hi|lo, B hi|lo: 48 KB, then the side area of the stage
    static constexpr uint32_t AUX_MASK = 128;                 // dW2: (g, action) pairs [16] at + 0, relu'(h2) words [16][8] at + 128
    static constexpr uint32_t AUX_BYTES = 6144;               // dW1: the 16 gathered observation rows of the chunk (<= 96 floats each)
    static constexpr uint32_t STG = AUX + AUX_BYTES;          // 54 KB (a multiple of 1 KB: every stage starts swizzle-aligned)
    static constexpr int TLD = 36;                            // floats per row of an epilogue transpose tile
    static constexpr uint32_t TILES = STAGES * STG;           // 8 epilogue warps x 32 x TLD floats
    static constexpr uint32_t W3T = TILES + 8 * 32 * TLD * 4; // W3^T [2 item parities][4 actions][256] floats
    static constexpr uint32_t BARS = W3T + 2 * 4 * H * 4;
    static constexpr uint32_t FULL = 0, CONV = 24, EMPTY = 48, ACC_FULL = 72, ACC_FREE = 88, TMEM = 104;   // byte offsets from BARS
    static constexpr int NQ = 8;                              // item queue: the TMA warp is never more than ~4 items ahead of the epilogue
    static constexpr uint32_t QFULL = 112, QITEM = QFULL + 8 * NQ;   // NQ mbarriers (item published) | NQ item numbers
    static constexpr uint32_t TOTAL = BARS + 256;
    static constexpr int EPI_WARPS = 8, CONV_WARPS = 8;       // warps 0-7 / 8-15; warp 16: MMA lane, warp 17: TMA, 18-19 fill the warpgroup
    static constexpr int NCONV = CONV_WARPS * 32;
    static constexpr int NTW = 20 * 32;                       // five warpgroups
    // setmaxnreg per warpgroup inside the pool the CTA was launched with (640 x 96): 2 x 128 x 160 + 2 x 128 x 64 + 128 x 32
    static constexpr int REGS_EPI = 160, REGS_CONV = 64, REGS_AUX = 32;
};
__device__ __forceinline__ void conv_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }   // the 8 converter warps of K4b

// Work items of K4b: per network two dW2 tiles (rows t*128..) and one dW1 tile.  The dW2 tiles come first in
// the item order (they are the longer ones), so a static round-robin over the CTAs ends on the short items.
__device__ __forceinline__ void wg_item(int q, int G, int& g, int& t) {
    if (q < 2 * G) { g = q >> 1; t = q & 1; }
    else { g = q - 2 * G; t = 2; }
}

// The item order is a QUEUE: the TMA warp decides which item comes next and publishes it through shared memory; the other
// roles pop the items in the same order.  In a chain (K4b is a programmatic dependent launch of K4a: its CTAs take over the
// SMs K4a's last partial wave leaves idle, at different times) the items are drawn from a global counter (reset by the sample
// kernel and by the last CTA to finish), so a CTA that starts early simply draws more; launched on its own the walk is the
// static round-robin.  Only items of active networks are published; -1 ends the walk.  No "slot free" barrier is needed:
// publishing item n comes after the TMA warp has issued every chunk of item n - 1, which needs the MMA lane inside item
// >= n - 4 (three stages, >= 1 chunk per item), which needs the epilogue to have released item n - 6: every role has
// popped item n - 8 long before its slot is reused.
__device__ __forceinline__ int wg_pop(uint32_t bars, int& nq, bool& ok) {
    const uint32_t slot = (uint32_t)nq & (Wg::NQ - 1);
    int q = -1;
    if ((threadIdx.x & 31) == 0) {
        if (ok) ok = mbar_wait(bars + Wg::QFULL + 8 * slot, (uint32_t)(nq >> 3) & 1u);
        if (ok) asm volatile("ld.shared.s32 %0, [%1];" : "=r"(q) : "r"(bars + Wg::QITEM + 4 * slot));
    }
    ++nq;
    q = __shfl_sync(0xffffffffu, q, 0);
    if (q < 0) ok = __shfl_sync(0xffffffffu, (int)ok, 0) != 0;
    return q;
}
__device__ __forceinline__ float ldcg_f(const float* p) {        // L2 loads: data another kernel's CTAs may have written while this CTA was resident
    float v;
    asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// dW tile: D[128 x 256] = A^T-operand * D-operand over K = batch, Adam in the epilogue.
//   t = 0,1: dW2 rows t*128.. : A = h1^T scratch [m][k] (K-major SW64), B = dh2 rebuilt [k][n] (MN-major)
//   t = 2  : dW1 rows 0..95   : A = s gathered from the ring [k][m] (MN-major),  B = dh1^T scratch (K-major SW64);
//            A column m = obs_stride is set to 1, so row obs_stride of the tile is db1 = sum_k dh1[k][:] for free;
//            the epilogue of this item also folds the per-row-tile partials of db2 / dW3 / db3 (from K4a) and
//            emits the metrics.
// Persistent and warp-specialised like K3 / K4a: a CTA walks its items q = blockIdx.x, + gridDim.x, ...; per 16-row chunk
//   warp 17    TMA producer: the K-major scratch operand (h1^T / dh1^T) lands IN PLACE in the hi half of its stage
//              through a tensor map with the 64-byte swizzle the UMMA layout uses (a box of {16 batch columns, 128 or 256
//              feature rows}; columns past the batch are zero-filled by the hardware); the small inputs of the other
//              operand travel with cp.async.bulk into the stage's side area -- (g, action) pairs + relu'(h2) words for
//              dW2, one copy per gathered observation row for dW1 (lane = row) -- all on the stage's mbarrier;
//   warps 8-15 converters: split the landed operand into hi | lo in place (same address: the swizzle is already
//              applied), and BUILD the other operand in the UMMA MN-major layout: dW2's dh2[k][n] = relu'(h2) ? g_k *
//              W3[n][a_k] : 0 from the side area and W3^T in shared memory, dW1's observation rows + ones column;
//   warp 16    lane 0 issues the chunk's six tcgen05.mma, alternating between two TMEM accumulators per item;
//   warps 0-7  read a finished accumulator and do the Adam read-modify-write of theta / m / v / theta_tgt.
// Stage ring: FULL (TMA landed) -> CONV (converted / built) -> EMPTY (tcgen05.commit).  Nobody waits on a global load
// with operands in registers any more (the previous version's producers spent ~3.3 k cycles per chunk on exactly that,
// against 768 cycles of tensor time).  The epilogue is pure HBM traffic (24 bytes per parameter) and the GEMM needs
// almost none, so running them concurrently on every SM keeps HBM busy for the whole kernel.
template <int PASSES>
__global__ void __launch_bounds__(Wg::NTW, 1) tc_wgrad_kernel(const LearnArgs A, const __grid_constant__ CUtensorMap tmap_h1,
                                                              const __grid_constant__ CUtensorMap tmap_dh1) {
    extern __shared__ uint8_t smem_raw[];
    const int B = A.d.batch, Dp = A.d.obs_stride, G = A.d.n_nets;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = sbase + Wg::BARS;
    const int n_items = 3 * G;
    const int nchunks = (B + KC - 1) / KC;

    if (tid == 0) {
        for (int s = 0; s < Wg::STAGES; ++s) {
            mbar_init(bars + Wg::FULL + 8 * s, 1);                    // one arrive.expect_tx + the bytes of the chunk
            mbar_init(bars + Wg::CONV + 8 * s, Wg::CONV_WARPS);       // one arrival per converter warp
            mbar_init(bars + Wg::EMPTY + 8 * s, 1);                   // one tcgen05.commit
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bars + Wg::ACC_FULL + 8 * b, 1);                // one tcgen05.commit
            mbar_init(bars + Wg::ACC_FREE + 8 * b, Wg::EPI_WARPS);    // one arrival per epilogue warp
        }
        for (int b = 0; b < Wg::NQ; ++b) mbar_init(bars + Wg::QFULL + 8 * b, 1);   // one arrival: the TMA warp's lane 0
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bars + Wg::TMEM), "r"(512));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem) : "r"(bars + Wg::TMEM));
    bool ok = true;

    if (warp >= Wg::EPI_WARPS + Wg::CONV_WARPS) {
        regs_dec<Wg::REGS_AUX>();
        if (warp == Wg::EPI_WARPS + Wg::CONV_WARPS) {
            // ------------------------------------------------------------------ MMA lane -------------------
            {
                uint32_t used = 0;
                int n = 0, nq = 0;
                for (;;) {
                    const int q = wg_pop(bars, nq, ok);
                    if (q < 0) break;
                    if (lane != 0) continue;
                    int g, t;
                    wg_item(q, G, g, t);
                    const bool is_w2 = t < 2;
                    const uint32_t acc_buf = (uint32_t)(n & 1);
                    const uint32_t d_tmem = tmem + acc_buf * 256u;
                    const uint32_t idesc = make_idesc(!is_w2, is_w2);
                    if (n >= 2 && ok)                                 // the epilogue has read item n - 2 out of this accumulator
                        ok = mbar_wait(bars + Wg::ACC_FREE + 8 * acc_buf, (uint32_t)((n >> 1) - 1) & 1u);
                    for (int c = 0; c < nchunks; ++c) {
                        const uint32_t s = used % Wg::STAGES, u = used / Wg::STAGES;
                        if (ok) ok = mbar_wait(bars + Wg::CONV + 8 * s, u & 1u);
                        tc_fence_after();
                        const uint32_t st = sbase + s * Wg::STG;
#pragma unroll
                        for (int ks = 0; ks < 2; ++ks) {
                            uint64_t a_hi, a_lo, b_hi, b_lo;
                            if (is_w2) {      // A K-major SW64; B MN-major: 8 n-groups per k-group -> k-group stride 4096 B, a k-step is two k-groups
                                a_hi = make_desc(st + ks * 32, 16, 512, 4);
                                a_lo = make_desc(st + Wg::A_BYTES + ks * 32, 16, 512, 4);
                                b_hi = make_desc(st + 2 * Wg::A_BYTES + ks * 2 * 4096, 512, 4096, 1);
                                b_lo = make_desc(st + 2 * Wg::A_BYTES + Wg::B_BYTES + ks * 2 * 4096, 512, 4096, 1);
                            } else {          // A MN-major: 4 m-groups per k-group -> k-group stride 2048 B; B K-major SW64
                                a_hi = make_desc(st + ks * 2 * 2048, 512, 2048, 1);
                                a_lo = make_desc(st + Wg::A_BYTES + ks * 2 * 2048, 512, 2048, 1);
                                b_hi = make_desc(st + 2 * Wg::A_BYTES + ks * 32, 16, 512, 4);
                                b_lo = make_desc(st + 2 * Wg::A_BYTES + Wg::B_BYTES + ks * 32, 16, 512, 4);
                            }
                            uint32_t acc = (c | ks) ? 1u : 0u;
                            if (PASSES == 3) {
                                mma_ss(d_tmem, a_lo, b_hi, idesc, acc);
                                mma_ss(d_tmem, a_hi, b_lo, idesc, 1u);
                                acc = 1u;
                            }
                            mma_ss(d_tmem, a_hi, b_hi, idesc, acc);
                        }
                        umma_commit(bars + Wg::EMPTY + 8 * s);
                        if (c == nchunks - 1) umma_commit(bars + Wg::ACC_FULL + 8 * acc_buf);
                        ++used;
                    }
                    ++n;
                }
                if (!ok && lane == 0) atomicExch(A.error, 15);
            }
            __syncwarp();
        } else if (warp == Wg::EPI_WARPS + Wg::CONV_WARPS + 1) {
            // ------------------------------------------------------------------ TMA producer ---------------
            uint32_t used = 0;
            int nq = 0;
            int draws = 0;
            for (;;) {
                // In a chain the CTAs of this kernel start at different times (whenever K4a leaves an SM), so the items are drawn
                // from the global counter; launched on its own every CTA starts at once and the static round-robin (long dW2 items
                // first) is already balanced -- and measurably faster (190 vs 195 us at cfg3).
                int q = (int)blockIdx.x + draws * (int)gridDim.x;
                ++draws;
                if (A.chain) {
                    if (lane == 0) q = atomicAdd(A.sched, 1);
                    q = __shfl_sync(0xffffffffu, q, 0);
                }
                if (q >= n_items || !ok) break;
                int g, t;
                wg_item(q, G, g, t);
                if (!A.active[g]) {                                   // nothing to compute: only the metrics row is cleared
                    if (t == 2 && lane < DMDQN_METRICS_STRIDE && A.metrics) A.metrics[g * DMDQN_METRICS_STRIDE + lane] = 0.f;
                    continue;
                }
                if (A.chain) {
                    // every K4a item of this network has published its scratch (h1^T, dh1^T, masks, (g, action), partials);
                    // the tensor-map / bulk reads below are async-proxy reads of data written through the generic proxy
                    int fine = 1;
                    if (lane == 0) {
                        fine = flag_acquire_ge(A.k4a_done + g, A.tc_tiles) ? 1 : 0;
                        asm volatile("fence.proxy.async;" ::: "memory");
                    }
                    ok = __shfl_sync(0xffffffffu, fine, 0) != 0;
                    if (!ok) break;
                }
                if (lane == 0) {
                    asm volatile("st.shared.s32 [%0], %1;" ::"r"(bars + Wg::QITEM + 4 * ((uint32_t)nq & (Wg::NQ - 1))), "r"(q) : "memory");
                    mbar_arrive(bars + Wg::QFULL + 8 * ((uint32_t)nq & (Wg::NQ - 1)));
                }
                ++nq;
                const size_t sb = (size_t)g * B;
                int32_t rid = 0;
                if (t == 2 && lane < KC && lane < B) rid = __ldg(A.rows + sb + lane);
                for (int c = 0; c < nchunks; ++c) {
                    const uint32_t s = used % Wg::STAGES, u = used / Wg::STAGES;
                    const uint32_t st = sbase + s * Wg::STG, full = bars + Wg::FULL + 8 * s;
                    const int nvalid = min(KC, B - c * KC);
                    int32_t rid_next = 0;
                    if (t == 2 && c + 1 < nchunks && (c + 1) * KC + lane < B && lane < KC) rid_next = __ldg(A.rows + sb + (c + 1) * KC + lane);
                    if (u && ok) ok = mbar_wait(bars + Wg::EMPTY + 8 * s, (u - 1) & 1u);     // the MMAs of the stage's previous chunk have retired
                    if (t < 2) {
                        if (lane == 0) {
                            mbar_expect_tx(full, Wg::A_BYTES + (uint32_t)nvalid * 40u);
                            tma_load_3d(st, &tmap_h1, c * KC, t * BM, g, full);
                            bulk_g2s(st + Wg::AUX, A.ga + sb + c * KC, (uint32_t)nvalid * 8u, full);
                            bulk_g2s(st + Wg::AUX + Wg::AUX_MASK, A.mask2 + (sb + c * KC) * 8, (uint32_t)nvalid * 32u, full);
                        }
                    } else {
                        if (lane == 0) {
                            mbar_expect_tx(full, Wg::B_BYTES + (uint32_t)(nvalid * Dp) * 4u);
                            tma_load_3d(st + 2 * Wg::A_BYTES, &tmap_dh1, c * KC, 0, g, full);
                        }
                        __syncwarp();                                 // expect_tx is posted before any row copy can complete
                        if (lane < nvalid) bulk_g2s(st + Wg::AUX + (uint32_t)(lane * Dp) * 4u, A.rp.obs + (size_t)rid * Dp, (uint32_t)Dp * 4u, full);
                    }
                    __syncwarp();
                    rid = rid_next;
                    ++used;
                }
            }
            if (lane == 0) {                                          // end of the walk
                asm volatile("st.shared.s32 [%0], %1;" ::"r"(bars + Wg::QITEM + 4 * ((uint32_t)nq & (Wg::NQ - 1))), "r"(-1) : "memory");
                mbar_arrive(bars + Wg::QFULL + 8 * ((uint32_t)nq & (Wg::NQ - 1)));
                // the last CTA to make its final draw leaves the counter at zero for the next launch (a stage launched on its
                // own has no sample kernel in front of it to do that)
                if (A.chain && atomicAdd(A.sched + 1, 1) == (int)gridDim.x - 1) {
                    atomicExch(A.sched + 1, 0);
                    atomicExch(A.sched, 0);
                }
            }
            if (!ok && lane == 0) atomicExch(A.error, 25);
        }
    } else if (warp >= Wg::EPI_WARPS) {
        // ------------------------------------------------------------------ converters ------------------
        regs_dec<Wg::REGS_CONV>();
        const int tc = tid - Wg::EPI_WARPS * 32;                      // 0..255
        uint32_t used = 0;
        int n = 0;
        auto put = [&](uint32_t o, uint32_t lo_off, const float4& x) {
            float4 hi, lo;
            split4<PASSES>(x, hi, lo);
            sts4(o, hi);
            if (PASSES == 3) sts4(o + lo_off, lo);
        };
        auto in_place = [&](uint32_t o, uint32_t lo_off) {            // landed raw piece -> hi at the same address, lo beside it
            const float4 x = lds4(o);
            put(o, lo_off, x);
        };
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        int nq = 0;
        WG_TS_DECL;
        for (;;) {
            const int q = wg_pop(bars, nq, ok);
            if (q < 0) break;
            int g, t;
            wg_item(q, G, g, t);
            WG_TS();
            if (t < 2) {
                // W3 as K4a saw it (the items are drawn dynamically, so it is fetched at the start of the item: an L2 hit that
                // elapses next to the first chunk's TMA)
                const float4 w3n = ldg_plain(A.w3_copy + (size_t)g * H * 4 + tc * 4);
                // ---- dW2: A in place; B = dh2 rebuilt, staged MN-major ([k][n], n contiguous): thread = (k-row bu of the chunk,
                // 16 columns n = 128 hh + 32 i + 4 l7 + 0..3, i = 0..3), so one (g, action) pair and four mask words serve 16
                // values, W3^T comes from shared memory as four conflict-free 16-byte loads, every store is a 16-byte piece.
                const int bu = tc >> 4, ng = tc & 15, hh = ng >> 3, l7 = ng & 7;
                const uint32_t w3t = sbase + Wg::W3T + (uint32_t)(n & 1) * (4 * H * 4);
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(w3t + (uint32_t)(0 * H + tc) * 4), "f"(w3n.x) : "memory");
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(w3t + (uint32_t)(1 * H + tc) * 4), "f"(w3n.y) : "memory");
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(w3t + (uint32_t)(2 * H + tc) * 4), "f"(w3n.z) : "memory");
                asm volatile("st.shared.f32 [%0], %1;" ::"r"(w3t + (uint32_t)(3 * H + tc) * 4), "f"(w3n.w) : "memory");
                conv_sync();      // every item: a warp two items ahead would overwrite the buffer a slower warp still reads
                const int mshift = l7 << 2;
                const uint32_t w3t_thr = w3t + (uint32_t)(128 * hh + 4 * l7) * 4;
                const uint32_t b_dst = 2 * Wg::A_BYTES + off_mn(H, bu, 128 * hh + 4 * l7);   // piece i: + i atoms of 512 B
                for (int c = 0; c < nchunks; ++c) {
                    const uint32_t s = used % Wg::STAGES, u = used / Wg::STAGES;
                    const uint32_t st = sbase + s * Wg::STG;
                    if (ok) ok = mbar_wait(bars + Wg::FULL + 8 * s, u & 1u);
                    in_place(st + (uint32_t)tc * 16u, Wg::A_BYTES);
                    in_place(st + (uint32_t)(tc + Wg::NCONV) * 16u, Wg::A_BYTES);
                    float gg = 0.f;
                    uint32_t wa = w3t_thr;
                    uint4 mq = make_uint4(0u, 0u, 0u, 0u);
                    if (c * KC + bu < B) {                            // rows past the batch: the side area holds stale bytes
                        float2 gq;
                        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(gq.x), "=f"(gq.y) : "r"(st + Wg::AUX + (uint32_t)bu * 8u));
                        asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(mq.x), "=r"(mq.y), "=r"(mq.z), "=r"(mq.w)
                                     : "r"(st + Wg::AUX + Wg::AUX_MASK + (uint32_t)bu * 32u + (uint32_t)hh * 16u));
                        gg = gq.x;
                        wa += (uint32_t)__float_as_int(gq.y) * (H * 4);
                    }
                    const uint32_t mw[4] = {mq.x, mq.y, mq.z, mq.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float4 w4 = lds4(wa + (uint32_t)i * 128u);
                        const uint32_t bits = mw[i] >> mshift;
                        const float4 x = make_float4((bits & 1u) ? gg * w4.x : 0.f, (bits & 2u) ? gg * w4.y : 0.f,
                                                     (bits & 4u) ? gg * w4.z : 0.f, (bits & 8u) ? gg * w4.w : 0.f);
                        put(st + b_dst + (uint32_t)i * 512u, Wg::B_BYTES, x);
                    }
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bars + Wg::CONV + 8 * s);
                    ++used;
                }
            } else {
                // ---- dW1 (+ db1): B in place; A = the chunk's observation rows [k][m] (MN-major; column m = Dp is the ones column)
                const int am = (tc & 31) << 2, ak = tc >> 5;          // pieces p = tc, tc + 256: k = ak, ak + 8
                const bool a_live = am < Dp, a_ones = am == Dp;
                const uint32_t a_dst = off_mn(BM, ak, am);            // k + 8: two k-groups further = + 2 * 2048 B
                for (int c = 0; c < nchunks; ++c) {
                    const uint32_t s = used % Wg::STAGES, u = used / Wg::STAGES;
                    const uint32_t st = sbase + s * Wg::STG;
                    if (ok) ok = mbar_wait(bars + Wg::FULL + 8 * s, u & 1u);
#pragma unroll
                    for (int r = 0; r < 4; ++r) in_place(st + 2 * Wg::A_BYTES + (uint32_t)(tc + Wg::NCONV * r) * 16u, Wg::B_BYTES);
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        const int kk = ak + 8 * r;
                        const bool in_batch = c * KC + kk < B;
                        float4 x = z4;
                        if (a_ones) x.x = in_batch ? 1.f : 0.f;
                        else if (a_live && in_batch) x = lds4(st + Wg::AUX + (uint32_t)(kk * Dp + am) * 4u);
                        put(st + a_dst + (uint32_t)r * 4096u, Wg::A_BYTES, x);
                    }
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bars + Wg::CONV + 8 * s);
                    ++used;
                }
            }
            ++n;
        }
        WG_TS();
        WG_TS_PRINT("K4b converters", tc == 0);
        if (!ok && tc == 0) atomicExch(A.error, 5);
    } else {
        regs_inc<Wg::REGS_EPI>();
        // ------------------------------------------------------------------ epilogue -------------------
        const int et = tid, ew = warp;                            // 0..255 / 0..7
        const int ehalf = ew >> 2;                                // TMEM lane = weight row (ew & 3) * 32 + lane of the tile; column half
        const uint32_t lane_addr = (uint32_t)((ew & 3) * 32) << 16;
        float* tile = reinterpret_cast<float*>(__cvta_shared_to_generic((size_t)(sbase + Wg::TILES))) + ew * (32 * Wg::TLD);
        const int rsub = lane >> 3, c4 = (lane & 7) << 2;
        int n = 0, nq = 0;
        WG_TS_DECL;
#ifdef TC_TIMING
        const long long wg_t0 = clock64();
        unsigned long long wg_g0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(wg_g0));
#endif
        for (;;) {
            const int q = wg_pop(bars, nq, ok);
            if (q < 0) break;
            int g, t;
            wg_item(q, G, g, t);
            // A bounded mbarrier wait that expired (here or in K3 / K4a of this step) means the accumulators are garbage:
            // leave theta / m / v alone and report it through the learned flag instead of applying the update.
            const int err_code = *reinterpret_cast<volatile int*>(A.error);
            const bool poisoned = __any_sync(0xffffffffu, err_code != 0 || !ok);   // warp-uniform
            const size_t pb = (size_t)g * A.L.stride;
            float* th = A.nets.theta + pb;
            float* tg = A.nets.theta_tgt + pb;
            float* am = A.nets.adam_m + pb;
            float* av = A.nets.adam_v + pb;
            const AdamStep k = adam_step(A, g);
            const bool is_w2 = t < 2;
            const int m0 = is_w2 ? t * BM : 0;
            if (t == 2 && poisoned) {
                if (et < DMDQN_METRICS_STRIDE && A.metrics) A.metrics[g * DMDQN_METRICS_STRIDE + et] = et == 7 ? -(float)(err_code ? err_code : 6) : 0.f;
            } else if (t == 2) {
                // head / bias gradients: per-row-tile partials from K4a summed in tile order, then Adam
                auto upd = [&](int64_t off, float grad) {
                    if (A.grads) { A.grads[pb + off] = grad; return; }
                    float tgv = k.sync == 2 ? tg[off] : 0.f;
                    adam1(k, grad, th[off], am[off], av[off], tgv);
                    if (k.sync) tg[off] = tgv;
                };
                const size_t p0 = (size_t)g * A.tc_tiles;
                float s2 = 0.f, w[4] = {0.f, 0.f, 0.f, 0.f};
                for (int r = 0; r < A.tc_tiles; ++r) {
                    s2 += ldcg_f(A.part_b2 + (p0 + r) * H + et);
                    const float4 pw = ldg_plain(A.part_w3 + ((p0 + r) * H + et) * 4);
                    w[0] += pw.x; w[1] += pw.y; w[2] += pw.z; w[3] += pw.w;
                }
                upd(A.L.b2 + et, s2);
                if (A.dueling) {          // the folded head's gradient projected onto W3[et][.] | wv[et], and b3 | bv by one thread
                    upd(A.L.wv + et, head_project(w, A.d.n_actions));
                    if (et == 0) {
                        float b[4] = {0.f, 0.f, 0.f, 0.f};
                        for (int r = 0; r < A.tc_tiles; ++r)
                            for (int a = 0; a < 4; ++a) b[a] += ldcg_f(A.part_b3 + (p0 + r) * 4 + a);
                        upd(A.L.bv, head_project(b, A.d.n_actions));
                        for (int a = 0; a < 4; ++a) upd(A.L.b3 + a, b[a]);
                        if (A.grads)              // the pad after bv is inside the Adam range: its gradient is 0
                            for (int p = 1; p < 4; ++p) A.grads[pb + A.L.bv + p] = 0.f;
                    }
                }
                for (int a = 0; a < 4; ++a) upd(A.L.w3 + (int64_t)et * 4 + a, w[a]);
                if (et < 4 && !A.dueling) {
                    float s3 = 0.f;
                    for (int r = 0; r < A.tc_tiles; ++r) s3 += ldcg_f(A.part_b3 + (p0 + r) * 4 + et);
                    upd(A.L.b3 + et, s3);
                }
                if (et == 0 && A.metrics) finish_metrics(A, g, A.tc_tiles, [](const float* p) { return ldcg_f(p); });
            }
            const uint32_t acc_buf = (uint32_t)(n & 1);
            WG_TS();
            if (ok) ok = mbar_wait(bars + Wg::ACC_FULL + 8 * acc_buf, (uint32_t)(n >> 1) & 1u);
            tc_fence_after();
            WG_TS();
            // TMEM (lane = weight row) -> per-warp smem tile -> 8 lanes per 128-byte row segment, so the
            // Adam read-modify-write of theta / m / v / theta_tgt is fully coalesced.  Offsets are 32-bit float
            // indices into the network's parameter block; all mode decisions are made per item, not per element.
            const int wbase = (int)(is_w2 ? A.L.w2 : A.L.w1) + (m0 + (ew & 3) * 32 + rsub) * H + c4;   // + 4 u' H + c0
            const int mrow0 = m0 + (ew & 3) * 32 + rsub;                                              // tile row of u' = 0
            const int sync = k.sync;
#pragma unroll 1
            for (int cc = 0; cc < 4; ++cc) {
                const int c0 = ehalf * 128 + cc * 32;
                float v[32];
                tmem_ld32(tmem + acc_buf * 256u + lane_addr + (uint32_t)c0, v);
                if (cc == 3) {                                    // this warp has read its whole part of the accumulator
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bars + Wg::ACC_FREE + 8 * acc_buf);
                }
                __syncwarp();
                if (poisoned) continue;                           // warp-uniform: the accumulator has been released above
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(tile + lane * Wg::TLD + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                __syncwarp();
                const float* trow = tile + rsub * Wg::TLD + c4;   // row 4 u' + rsub of the tile
                if (A.grads) {                                    // shared-parameter mode: raw gradients out, no update
#pragma unroll
                    for (int up = 0; up < 8; ++up) {
                        const int m = mrow0 + 4 * up;
                        const bool bias_row = !is_w2 && m == Dp;
                        if (is_w2 || m < Dp || bias_row)
                            *reinterpret_cast<float4*>(A.grads + pb + (bias_row ? (int)A.L.b1 + c0 + c4 : wbase + 4 * up * H + c0)) =
                                *reinterpret_cast<const float4*>(trow + 4 * up * Wg::TLD);
                    }
                } else {
                    // one batch of eight row groups: every theta / m / v load of the column block is issued before the first
                    // use, so twenty-four 16-byte loads per thread are in flight while the HBM latency elapses (the gradient
                    // comes from the tile at use; the Polyak target is read late: it is the rare mode)
                    int off[8];
                    float4 t4[8], m4[8], v4[8];
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int m = mrow0 + 4 * u;
                        off[u] = wbase + 4 * u * H + c0;
                        if (!is_w2) off[u] = m == Dp ? (int)A.L.b1 + c0 + c4 : (m < Dp ? off[u] : -1);   // db1 from the ones column
                        if (is_w2 || off[u] >= 0) {
                            t4[u] = ldg_plain(th + off[u]);
                            m4[u] = ldg_plain(am + off[u]);
                            v4[u] = ldg_plain(av + off[u]);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        if (!is_w2 && off[u] < 0) continue;
                        const float4 gr = *reinterpret_cast<const float4*>(trow + 4 * u * Wg::TLD);
                        adam_fast(k, gr.x, t4[u].x, m4[u].x, v4[u].x); adam_fast(k, gr.y, t4[u].y, m4[u].y, v4[u].y);
                        adam_fast(k, gr.z, t4[u].z, m4[u].z, v4[u].z); adam_fast(k, gr.w, t4[u].w, m4[u].w, v4[u].w);
                        *reinterpret_cast<float4*>(th + off[u]) = t4[u];
                        *reinterpret_cast<float4*>(am + off[u]) = m4[u];
                        *reinterpret_cast<float4*>(av + off[u]) = v4[u];
                        if (sync == 1) {
                            *reinterpret_cast<float4*>(tg + off[u]) = t4[u];
                        } else if (sync == 2) {
                            const float omt = 1.0f - k.tau;
                            const float4 g4 = ldg_plain(tg + off[u]);
                            *reinterpret_cast<float4*>(tg + off[u]) =
                                make_float4(k.tau * t4[u].x + omt * g4.x, k.tau * t4[u].y + omt * g4.y,
                                            k.tau * t4[u].z + omt * g4.z, k.tau * t4[u].w + omt * g4.w);
                        }
                    }
                }
                __syncwarp();                                     // the tile is rewritten by the next column block
            }
            ++n;
        }
        WG_TS();
        WG_TS_PRINT("K4b epilogue (wait, adam)*", et == 0);
#ifdef TC_TIMING
        if (et == 0) { unsigned long long gt; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
            printf("K4bsum cta %d sm %d items %d cycles %lld chain %d t0 %llu t1 %llu\n", blockIdx.x, (int)smid_(), n, clock64() - wg_t0, A.chain, wg_g0, gt); }
#endif
        if (!ok && lane == 0) atomicExch(A.error, 6);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// The rank-3 tensor map K4a's TMA lane uses for d.W^T: W2 of every network as {256 columns, 256 rows, n_nets}, box =
// {16 columns, 256 rows, 1} (dense 256 x 64 B in shared memory).  Encoded per launch (the library keeps no state
// and the caller's theta pointer may be a per-agent view); the driver entry point is looked up once.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// One encoder for every tensor map of this file.  The library keeps no state, so the maps are built per launch -- nine per learn
// step, ~1.3 us of host time each -- but a map is a pure function of (base address, shape, strides, box, swizzle): the last few
// results are memoised per host thread, which takes ~10 us off the host side of a step for a caller that passes the same buffers
// every step (the usual case) and changes nothing for one that does not.
struct MapKey {
    const void* base;
    cuuint64_t dims[5], strides[4];
    cuuint32_t box[5];
    int rank, swz;
};
int encode_tiled(CUtensorMap* out, const float* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides, const cuuint32_t* box,
                 CUtensorMapSwizzle swz) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        DMDQN_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn) {
            set_error("cuTensorMapEncodeTiled is not available from this driver");
            return DMDQN_ERR_CUDA;
        }
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    constexpr int kSlots = 32;
    static thread_local MapKey keys[kSlots];
    static thread_local CUtensorMap maps[kSlots];
    static thread_local int used = 0, next = 0;
    MapKey k = {};
    k.base = base; k.rank = rank; k.swz = (int)swz;
    for (int i = 0; i < rank; ++i) { k.dims[i] = dims[i]; k.box[i] = box[i]; }
    for (int i = 0; i + 1 < rank; ++i) k.strides[i] = strides[i];
    for (int i = 0; i < used; ++i)
        if (memcmp(&keys[i], &k, sizeof(MapKey)) == 0) { *out = maps[i]; return DMDQN_OK; }
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const CUresult rc = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, const_cast<float*>(base), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled (rank %d) failed with CUresult %d", rank, (int)rc);
        return DMDQN_ERR_CUDA;
    }
    keys[next] = k; maps[next] = *out;
    next = (next + 1) % kSlots;
    if (used < kSlots) ++used;
    return DMDQN_OK;
}
int encode_map3(CUtensorMap* out, const float* base, cuuint64_t d0, cuuint64_t d1, cuuint64_t d2, cuuint64_t stride1_bytes,
                cuuint64_t stride2_bytes, cuuint32_t box0, cuuint32_t box1, CUtensorMapSwizzle swz) {
    const cuuint64_t dims[3] = {d0, d1, d2};
    const cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    const cuuint32_t box[3] = {box0, box1, 1};
    return encode_tiled(out, base, 3, dims, strides, box, swz);
}
// x.W chunks in the UMMA MN-major layout straight from TMA (tma_fwd): the [K][256] matrix at float offset `woff` of every
// network's parameter block as {32 columns, 4 k-rows, 8 column blocks, K / 4 k-groups, network}.
int make_fwd_tensor_map(const LearnArgs& A, const float* theta, int64_t woff, int K, CUtensorMap* out) {
    const cuuint64_t dims[5] = {32, 4, (cuuint64_t)(H / 32), (cuuint64_t)(K / 4), (cuuint64_t)A.d.n_nets};
    const cuuint64_t strides[4] = {(cuuint64_t)H * 4, 128, (cuuint64_t)H * 16, (cuuint64_t)A.L.stride * 4};
    const cuuint32_t box[5] = {32, 4, (cuuint32_t)(H / 32), 2, 1};
    return encode_tiled(out, theta + woff, 5, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
}
int make_w2_tensor_map(const LearnArgs& A, CUtensorMap* out) {
    return encode_map3(out, A.nets.theta + A.L.w2, H, H, A.d.n_nets, (cuuint64_t)H * sizeof(float),
                       (cuuint64_t)A.L.stride * sizeof(float), 8, H, CU_TENSOR_MAP_SWIZZLE_32B);
}
// K4b's K-major operands: the transposed scratch [n_nets][H features][B batch] as {B, H, n_nets}, box = {16 batch columns,
// `rows` features}, landing with the 64-byte swizzle of the UMMA K-major SW64 layout (16-byte piece ^= (row / 2) % 4).
int make_scratch_tensor_map(const LearnArgs& A, const float* scratch, int rows, CUtensorMap* out) {
    return encode_map3(out, scratch, A.d.batch, H, A.d.n_nets, (cuuint64_t)A.d.batch * sizeof(float),
                       (cuuint64_t)A.d.batch * H * sizeof(float), KC, (cuuint32_t)rows, CU_TENSOR_MAP_SWIZZLE_64B);
}

template <int PASSES, bool DUELING>
int launch_tc(const LearnArgs& A, int stages, cudaStream_t s) {
    const size_t smem_f = Fwd::TOTAL + 1024, smem_w = Wg::TOTAL + 1024;
    int n_sm = 0;
    if (int rc = device_sm_count(&n_sm)) return rc;
    static size_t cfg_t[kMaxDevices] = {}, cfg_o[kMaxDevices] = {}, cfg_w[kMaxDevices] = {};    // per device, not per process
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(tc_target_kernel<PASSES, DUELING>), smem_f, cfg_t)) return rc;
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(tc_online_kernel<PASSES, DUELING>), smem_f, cfg_o)) return rc;
    if (int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(tc_wgrad_kernel<PASSES>), smem_w, cfg_w)) return rc;
    const int items = A.d.n_nets * A.tc_tiles;                    // persistent: one CTA per SM walks its items
    // In a chain (sample + K3 + K4a + K4b issued by one call) K4a and K4b are programmatic dependent launches: their CTAs
    // are scheduled as soon as every CTA of the previous kernel is resident, take over SMs as that kernel's CTAs leave, and
    // order themselves behind the data they need with the per-tile / per-network flags.  Every CTA of the producer is
    // resident (or finished) before a consumer CTA exists, so a waiting consumer can never starve its producer.
    cudaLaunchAttribute pdl[1];
    pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.stream = s;
    cfg.attrs = pdl;
    if (stages & DMDQN_STAGE_TARGET) {
        cfg.gridDim = dim3(2 * items < n_sm ? 2 * items : n_sm);
        cfg.blockDim = dim3(NT_F);
        cfg.dynamicSmemBytes = smem_f;
        cfg.numAttrs = A.chain ? 1 : 0;         // in a chain: launched under the tail of the sample kernel (griddepcontrol.wait inside)
        CUtensorMap m1, m2, m1t, m2t;
        if (int rc = make_fwd_tensor_map(A, A.nets.theta, A.L.w1, A.d.obs_stride, &m1)) return rc;
        if (int rc = make_fwd_tensor_map(A, A.nets.theta, A.L.w2, H, &m2)) return rc;
        if (int rc = make_fwd_tensor_map(A, A.nets.theta_tgt, A.L.w1, A.d.obs_stride, &m1t)) return rc;
        if (int rc = make_fwd_tensor_map(A, A.nets.theta_tgt, A.L.w2, H, &m2t)) return rc;
        DMDQN_CUDA(cudaLaunchKernelEx(&cfg, tc_target_kernel<PASSES, DUELING>, A, m1, m2, m1t, m2t));
    }
    if (stages & DMDQN_STAGE_ONLINE) {
        CUtensorMap tmap;
        if (int rc = make_w2_tensor_map(A, &tmap)) return rc;
        cfg.gridDim = dim3(items < n_sm ? items : n_sm);
        cfg.blockDim = dim3(NT_F);
        cfg.dynamicSmemBytes = smem_f;
        cfg.numAttrs = A.chain ? 1 : 0;
        CUtensorMap m1, m2;
        if (int rc = make_fwd_tensor_map(A, A.nets.theta, A.L.w1, A.d.obs_stride, &m1)) return rc;
        if (int rc = make_fwd_tensor_map(A, A.nets.theta, A.L.w2, H, &m2)) return rc;
        DMDQN_CUDA(cudaLaunchKernelEx(&cfg, tc_online_kernel<PASSES, DUELING>, A, tmap, m1, m2));
    }
    if (stages & DMDQN_STAGE_WGRAD) {
        const int items = A.d.n_nets * 3;
        CUtensorMap tmap_h1, tmap_dh1;
        if (int rc = make_scratch_tensor_map(A, A.h1, BM, &tmap_h1)) return rc;
        if (int rc = make_scratch_tensor_map(A, A.dh1, H, &tmap_dh1)) return rc;
        cfg.gridDim = dim3(items < n_sm ? items : n_sm);
        cfg.blockDim = dim3(Wg::NTW);
        cfg.dynamicSmemBytes = smem_w;
        cfg.numAttrs = A.chain ? 1 : 0;
        DMDQN_CUDA(cudaLaunchKernelEx(&cfg, tc_wgrad_kernel<PASSES>, A, tmap_h1, tmap_dh1));
    }
    return DMDQN_OK;
}

}  // namespace

bool tc_supported(const dmdqn_dims& d) {
    // batch % 4: the transposed scratch is streamed in 16-byte pieces along the batch axis
    return d.hidden == H && d.obs_stride % 32 == 0 && d.obs_stride <= 96 && d.batch % 4 == 0 && d.batch <= 4096;
}

int launch_learn_tc(const LearnArgs& args, int precision, int stages, cudaStream_t s) {
    LearnArgs A = args;
    A.tc_tiles = (A.d.batch + BM - 1) / BM;
    A.chain = (stages & kAllStages) == kAllStages ? 1 : 0;      // the sample kernel of this call has just reset the flags
    A.k4a_done = A.sched + 4;
    A.k3_done = A.k4a_done + A.d.n_nets;
    if (A.dueling) return precision == DMDQN_PRECISION_TF32 ? launch_tc<1, true>(A, stages, s) : launch_tc<3, true>(A, stages, s);
    return precision == DMDQN_PRECISION_TF32 ? launch_tc<1, false>(A, stages, s) : launch_tc<3, false>(A, stages, s);
}

}  // namespace dmdqn
