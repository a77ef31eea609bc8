// Tensor-core path of the batched RHS and of its VJP (ODENet.forward / prior_only_forward, odenet.py:85-98, and what
// torch.autograd computes through them) for every call beyond the resident solver kernels' capacity (B >= 5 rows):
// hand-written tcgen05.mma (kind::tf32, 3xTF32 split for fp32 parity) with accumulators in tensor memory, operands staged
// by 1-D TMA bulk copies and -- for everything derived from y or from the cotangent -- by producer warps that compute
// it on the fly.  Layouts: phx_tc.cuh.  Two MMA kernels, each in a few compile-time modes, plus small finishing passes:
//
//   tc_branch_kernel<MODE, TRANS, PAIR>   "A(src) x image^T", M = 128 rows per CTA, N = Hn columns of ONE half
//       (sums | prods) of the 2*Hn-wide result, K split over CTAs, accumulation in chunks of 16 k-blocks folded into a
//       tensor-memory running sum by drain warps (see "Accumulation chains" below).  704 threads: 16 producer warps,
//       1 bulk-copy warp, 1 MMA-issue warp (uniform control flow + elect.sync), 4 drain warps.
//         <0,0>  [S|P] partial  = act(y) W1          rows = batch, k = genes, A = soft-sign / log1p of y by half
//         <1,0>  gSP partial    = (g relu(m)) WA     rows = batch, k = genes, A = cotangent x per-gene factor
//         <1,1>  Wa_bar partial = (g relu(m))^T [S|P]   rows = genes, k = batch rows (transposed loads: lanes along genes)
//         <0,1>  Ws_bar | Wp_bar partial = act(y)^T gSP  rows = genes, k = batch rows
//       PAIR = 1 is the experimental cta_group::2 form (off by default, DESIGN.md section 7).
//   tc_spfinish_kernel    fixed-order sum of the K-split partials; mode 0: + bias, exp on the prods half -> [S|P];
//       mode 1: prods half x Pr -> gSP; writes the plain [B][K2] copy and the hi|lo operand images of the consumers.
//   tc_gradfinish_kernel  the same for the parameter cotangents, scattered into the flat gradient vector.
//   tc_joint_kernel<EMODE>   "image_A x image_B^T" with both operands by bulk copy: persistent, M = 128 genes,
//       N = 256 batch rows, 4-stage ring, double-buffered TMEM accumulators, 8 epilogue warps working straight out of
//       tensor memory (lanes are genes => every global access of the epilogue is a coalesced 128-byte row segment).
//         <0>  f = fscale * relu(m) * ([S|P] WA^T - y)   (or the un-decayed joint)        odenet.py:89-90
//         <1>  u = gS Ws                                    (k-blocks of the sums half)
//         <2>  ybar = (u + (gP Wp)/(1+s)) / (1+|y-.5|)^2 - g relu(m)    soft-sign / log1p backward in the epilogue
//
// Every accumulation order is fixed (MMA issue order, K-split reduction order) => results are run-to-run identical.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <mutex>
#include "phx_common.cuh"

namespace {

constexpr int BK = PHX_TC_BK;

// in-kernel cycle counters of the branch kernel (tools/tc_check.py with PHX_TC_PROF=1): compiled in only with
// -DPHX_TC_PROFILE=1 (PHX_TC_PROFILE_BUILD=1 python -m phoenix_b200.build --force) -- the producers are instruction-bound
#ifndef PHX_TC_PROFILE
#define PHX_TC_PROFILE 0
#endif
#define PROF(p) (PHX_TC_PROFILE ? (p).prof : (unsigned long long*)nullptr)

__device__ __forceinline__ unsigned smem_u32(const void* ptr) { return (unsigned)__cvta_generic_to_shared(ptr); }

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
            "selp.u32 %0, 1, 0, P1;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    }
}
// one non-blocking test of the phase with parity `parity` (1: that phase has completed)
__device__ __forceinline__ unsigned mbar_test(unsigned bar, unsigned parity) {
    unsigned done;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done;
}
__device__ __forceinline__ void mbar_arrive(unsigned bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// cluster-scope variants for the 2-CTA (cta_group::2) kernels
__device__ __forceinline__ void mbar_wait_cluster(unsigned bar, unsigned parity) {
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n"
            ".reg .pred P1;\n"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%1], %2;\n"
            "selp.u32 %0, 1, 0, P1;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
    }
}
__device__ __forceinline__ void mbar_arrive_remote(unsigned bar, unsigned cta) {   // same barrier offset in CTA `cta`
    unsigned r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(bar), "r"(cta));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mma_tf32_pair(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc,
                                              unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mma_commit_pair(unsigned bar) {   // arrives on `bar` in BOTH CTAs of the pair
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
        "h"((unsigned short)3)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc512_pair(unsigned slot_saddr) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_saddr), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free512_pair(unsigned base) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(512u) : "memory");
}

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// shared-memory matrix descriptor, K-major, no swizzle (cute::UMMA::SmemDescriptor bit layout; version 1 = sm_100)
__device__ __forceinline__ uint64_t smem_desc(unsigned saddr, unsigned lbo_bytes, unsigned sbo_bytes,
                                              unsigned layout_type = 0) {
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3fffu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(layout_type & 7u) << 61;   // 0 no swizzle, 2 SWIZZLE_128B, 4 SWIZZLE_64B, 6 SWIZZLE_32B
    return d;
}
// instruction descriptor: D fp32, A/B tf32, both K-major, M x N  (cute::UMMA::InstrDescriptor bit layout)
__host__ __device__ inline unsigned idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_tf32(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc,
                                         unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same with the A operand read from TENSOR memory (lane = row, 8 consecutive 32-bit columns = the K = 8 slice)
__device__ __forceinline__ void mma_tf32_ts(unsigned tmem_d, unsigned tmem_a, uint64_t bdesc, unsigned idesc,
                                            unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the mbarrier once every MMA issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void mma_commit(unsigned bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_alloc512(unsigned slot_saddr) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_saddr), "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free512(unsigned base) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(512u) : "memory");
}
__device__ __forceinline__ void tmem_ld16(unsigned taddr, float (&v)[16]) {
    unsigned u[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
          "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(u[i]);
}

__device__ __forceinline__ void tmem_ld8(unsigned taddr, float (&v)[8]) {
    unsigned u[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(u[i]);
}

__device__ __forceinline__ float tf32_rna(float x) {
    unsigned u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}
__device__ __forceinline__ void split_tf32(float x, float& hi, float& lo) {
    hi = tf32_rna(x);
    // rna_tf32(x - hi) on the bit pattern (add half an ulp of the 10-bit mantissa, clear the low 13 bits): the same value
    // as cvt.rna.tf32 for every finite input in two integer instructions instead of four (cvt.rna.tf32.f32 is expanded
    // into add / non-finite test / select / mask).  A non-finite x already makes hi non-finite, so the product stays so.
    lo = __uint_as_float((__float_as_uint(x - hi) + 0x1000u) & 0xffffe000u);
}

// ---- operand images of the weights -------------------------------------------------------------------------------------
__global__ void tc_pack_kernel(int G, int H, int Hp, int K2, int Hn, const float* __restrict__ W1,
                               const float* __restrict__ WA, float* __restrict__ w1img, float* __restrict__ waimg,
                               float* __restrict__ watimg, float* __restrict__ w1kimg) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    // w1img: one thread per (gene g, branch, hidden unit n): reads of W1 rows are coalesced over n
    const int KB1 = phx_tc_KB1(G);
    const size_t n1 = (size_t)KB1 * BK * 2 * Hn;
    for (size_t i = tid0; i < n1; i += stride) {
        const int n = (int)(i % Hn);
        const int br = (int)((i / Hn) & 1);
        const int g = (int)(i / (2 * (size_t)Hn));
        const bool ok = g < G && n < H;
        const float v = ok ? W1[(size_t)g * K2 + br * Hp + n] : 0.f;
        const float vt = ok ? WA[(size_t)g * K2 + br * Hp + n] : 0.f;
        float hi, lo;
        split_tf32(v, hi, lo);
        const int kb = g / BK, k = g % BK;
        const size_t co = (size_t)kb * 4 * Hn * BK + (size_t)br * 2 * Hn * BK;
        const int off = phx_tc_btile_off(Hn, n, k);
        w1img[co + off] = hi;
        w1img[co + Hn * BK + off] = lo;
        split_tf32(vt, hi, lo);
        watimg[co + off] = hi;
        watimg[co + Hn * BK + off] = lo;
    }
    // waimg: one thread per (gene g, column c of [S|P] in Hn-padded numbering): reads of WA rows coalesced over c
    const int KB2 = 2 * Hn / BK, GT = phx_tc_GT(G);
    const size_t n2 = (size_t)GT * 128 * 2 * Hn;
    for (size_t i = tid0; i < n2; i += stride) {
        const int c = (int)(i % (2 * Hn));
        const int g = (int)(i / (2 * (size_t)Hn));
        const int br = c / Hn, n = c % Hn;
        const bool ok = g < G && n < H;
        const float v = ok ? WA[(size_t)g * K2 + br * Hp + n] : 0.f;
        const float vk = ok ? W1[(size_t)g * K2 + br * Hp + n] : 0.f;
        float hi, lo;
        split_tf32(v, hi, lo);
        const int gt = g >> 7, r = g & 127, kb = c / BK, k = c % BK;
        const size_t co = ((size_t)gt * KB2 + kb) * 2 * 128 * BK;
        const int off = phx_tc_tile_off(128, r, k);
        waimg[co + off] = hi;
        waimg[co + 128 * BK + off] = lo;
        split_tf32(vk, hi, lo);
        w1kimg[co + off] = hi;
        w1kimg[co + 128 * BK + off] = lo;
    }
}

// hi / lo split of a FINITE value of moderate magnitude (|x| < 1e38): round-to-nearest on the bit pattern, no non-finite test
__device__ __forceinline__ void split_tf32_finite(float x, float& hi, float& lo) {
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
    lo = __uint_as_float((__float_as_uint(x - hi) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ float rcp_fast(float x) {   // MUFU.RCP, 1 ulp; callers pass 1 <= x <= 1 + HILL_RCP_MAX
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// rcp.approx.ftz flushes 1/x to 0 once it is subnormal (x > 2^126 ~ 8.5e37), which would give s = 0 for huge finite z.
// Beyond this |z| the exactly rounded z / (1 + |z|) of the fp32 path (phx_rhs.cu::hill) is +-1 (1 / (1 + |z|) is far
// below half an ulp of 1), and NaN for an infinite z: copysign(1, z) + (z - z) gives exactly that.
constexpr float HILL_RCP_MAX = 1e30f;
// soft-sign s = z / (1 + |z|), z = y - 0.5 (odenet.py:21-27): the denominator is >= 1, so the range handling of a generic
// fast division is dead weight in the producers, which are instruction-bound
__device__ __forceinline__ float softsign_z(float z, float az) {
    return az <= HILL_RCP_MAX ? z * rcp_fast(1.0f + az) : copysignf(1.0f, z) + (z - z);
}
__device__ __forceinline__ float hill_s(float y) {
    const float z = y - 0.5f;
    return softsign_z(z, fabsf(z));
}
// l = log1p(s) (odenet.py:29-35).  With s = z / (1 + |z|):  log1p(s) = 2 atanh(u), u = s / (2 + s) = z / (2 + 2|z| + z),
// so l needs ONE reciprocal and an odd series in u.  For |z| <= 0.65 (y in [-0.15, 1.15]: expression data live in [0, 1])
// |u| <= 0.246 and five series terms leave a truncation error below 5e-9; measured <= 2.5 ulp against float64 (log1pf:
// 1.9 ulp).  Anything outside takes the library log1pf.
constexpr float HILL_L_SERIES_MAX = 0.65f;
__device__ __forceinline__ float hill_l_series(float z, float az) {   // valid for az = |z| <= HILL_L_SERIES_MAX
    const float u = z * rcp_fast(fmaf(2.f, az, 2.f) + z);
    const float w = u * u;
    float p = fmaf(w, 0.09090909090909091f, 0.1111111111111111f);
    p = fmaf(w, p, 0.14285714285714285f);
    p = fmaf(w, p, 0.2f);
    p = fmaf(w, p, 0.3333333333333333f);
    const float u2 = u + u;
    return fmaf(u2, w * p, u2);
}
__device__ __forceinline__ float hill_l(float y) {
    const float z = y - 0.5f, az = fabsf(z);
    if (az <= HILL_L_SERIES_MAX) return hill_l_series(z, az);
    return log1pf(softsign_z(z, az));   // NaN lands here too
}
// The producers' conversion of four source values into hi / lo A-operand values.  The common case -- every value of the
// WARP finite and, for the log1p branch, inside the series range -- is decided with ONE vote and runs as straight-line
// code for the four elements (the producers are instruction-bound: 18 instructions per element on the log1p branch
// instead of ~30 with per-element range and non-finite tests); anything else takes the guarded per-element path.  Both
// paths give the same bits for the values the fast one accepts.
template <int MODE>
__device__ __forceinline__ void convert4(const float (&x)[4], const float (&sc)[4], int br, float (&hi)[4], float (&lo)[4]) {
    float v[4], m = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        v[j] = MODE ? x[j] * sc[j] : x[j] - 0.5f;
        m = fmaxf(m, fabsf(v[j]));   // fmaxf drops a NaN operand: tested separately below
    }
    const bool fin = (v[0] - v[0]) + (v[1] - v[1]) + (v[2] - v[2]) + (v[3] - v[3]) == 0.f;   // false with any NaN / inf
    const float lim = MODE ? 1e38f : (br ? HILL_L_SERIES_MAX : HILL_RCP_MAX);
    if (__all_sync(0xffffffffu, fin && m <= lim)) {
        if (MODE) {
#pragma unroll
            for (int j = 0; j < 4; ++j) split_tf32_finite(v[j], hi[j], lo[j]);
        } else if (br) {
#pragma unroll
            for (int j = 0; j < 4; ++j) split_tf32_finite(hill_l_series(v[j], fabsf(v[j])), hi[j], lo[j]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) split_tf32_finite(v[j] * rcp_fast(1.0f + fabsf(v[j])), hi[j], lo[j]);
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float a = MODE ? v[j] : (br ? hill_l(x[j]) : hill_s(x[j]));
        split_tf32(a, hi[j], lo[j]);
    }
}

// ---- kernel 1: branch contraction ----------------------------------------------------------------------------------------
// Accumulation chains.  The tensor core adds each MMA result into the fp32 accumulator with truncation, so the error of
// a long chain grows linearly with its length (measured: ~6e-8 per accumulating MMA, 1.5e-4 at 1 900 MMAs, against 1e-5
// for a plain fp32 FMA loop).  To keep fp32 parity a CTA accumulates at most `chunk` k-blocks (6 MMAs each) in one
// tensor-memory accumulator, then its warps add that chunk sum into a RUNNING SUM with round-to-nearest fp32 adds.  The
// running sum lives in tensor memory too (tcgen05.ld / add / tcgen05.st), which is why a CTA owns ONE branch: chunk
// accumulator (Hn columns) + running sum (Hn columns) fit the 512 columns for every Hn <= 256.  The soft-sign CTAs
// need ~1/2 the ALU work per k-block of the log1p CTAs, so they get K ranges twice as long (phx_tc_branch_plan).
struct BranchParams {
    int G, B, Bpad, Hn, KB1, chunk, stages, nterms;   // G = valid k, B = valid rows, Bpad = mtiles * 128
    int ld;               // leading dimension of the source matrix
    int mode;             // 0: A = Hill activation of y (soft-sign / log1p by branch); 1: A = y[b][g] * ascale[g] (cotangent)
    const float* ascale;  // mode 1: per-gene factor relu(m) (or NULL)
    int mtiles, ks_p, per_p, ks_s, per_s;   // work split: blocks [0, mtiles*ks_p) are prods-branch CTAs, the rest sums
    unsigned a_lbo, a_sbo, b_lbo, b_sbo;    // descriptor fields
    unsigned a_kadv, b_kadv;                // byte advance of the start address per K = 8 MMA (two core matrices)
    const float* y;       // [B][G]
    const float* y2;      // mode 1: source of the prods-branch CTAs when it differs from y (cached Hill activations), else NULL
    const float* w1img;
    float* spart;         // [slot][Bpad][2*Hn]; sums branch uses slots < ks_s, prods branch slots < ks_p
    unsigned long long* prof;   // optional cycle counters (PHX_TC_PROF): see tools/tc_check.py
    unsigned stg_bytes;         // bytes of the producers' staging area (the TS running sum sits behind it)
    int a_stages;               // TS = 1: depth of the A ring in tensor memory and the columns of its hi / lo tiles
    int a_hi_col[4], a_lo_col[4];
};
constexpr int K1_PWARPS = 16;                      // producer warps
constexpr int K1_DWARPS = 4;                       // drain warps (one per TMEM lane quarter)
constexpr int K1_W_BULK = K1_PWARPS;               // warp roles
constexpr int K1_W_MMA = K1_PWARPS + 1;
constexpr int K1_W_DRAIN = K1_PWARPS + 2;          // 18..21: (warp & 3) covers the four lane quarters
constexpr int K1_THREADS = (K1_PWARPS + 2 + K1_DWARPS) * 32;
constexpr int K1_PF = 4;                           // k-blocks of y in flight per thread (HBM latency)
constexpr unsigned K1_A_TILE = 128 * BK * 4;       // bytes of one 128 x 16 tile
constexpr unsigned K1_A_BYTES = 2 * K1_A_TILE;     // hi, lo

__device__ __forceinline__ void tmem_ld16_nowait(unsigned taddr, unsigned (&u)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
          "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(unsigned taddr, const unsigned (&u)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(
            taddr),
        "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
        "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15])
        : "memory");
}
__device__ __forceinline__ bool elect_one() {
    unsigned pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
// descriptor of the tile at shared address `saddr` given the constant high part (offsets, version)
__device__ __forceinline__ uint64_t desc_at(uint64_t hi_part, unsigned saddr) {
    return hi_part | (uint64_t)((saddr >> 4) & 0x3fffu);
}

// TRANS = 0: A(row, k) = src[row][k]  (rows = batch, k = genes).  TRANS = 1: A(row, k) = src[k][row] (rows = genes,
// k = batch rows: the K = B parameter-cotangent contractions); lanes then run along the genes, so every load is a
// coalesced 128-byte row segment and the transpose happens in registers (4 batch rows -> one 16-byte k chunk).
// PAIR = 1: two CTAs of a cluster (the two SMs of a TPC) work on adjacent 128-row tiles of the same (branch, K range) and
// their tensor cores execute ONE tcgen05.mma.cta_group::2 (M = 256) issued by the leader CTA: each CTA stages its own A
// tile and only HALF of the B operand (rows [rank*Hn/2, +Hn/2) of the image), which cuts the shared-memory traffic per
// k-block from ~107 KB to ~73 KB -- the bound of the single-CTA kernel.  Producer arrivals and the "B half landed"
// signal of the peer CTA reach the leader's full barrier as remote (cluster-scope) arrives; slot release and chunk
// completion come back to both CTAs by multicast tcgen05.commit.
//
// TS = 1 (single CTA only): the A tiles live in TENSOR memory instead of shared memory.  The producers tcgen05.st their
// hi / lo values straight into spare columns next to the two accumulators (thread = tile row = its TMEM lane, so the row a
// thread converts is fixed by its warp's lane quarter) and the MMAs take A as a tensor-memory operand.  Per k-block this
// removes the 16 KB of A-tile stores and the 24 KB of A-operand reads from the shared-memory pipe -- the bound of the
// TS = 0 kernel (123 KB per k-block against 128 B/clk) -- leaving the B operand: 40 KB of reads + 27 KB of bulk copy.
// The ring of B stages (shared memory) and the ring of A stages (tensor memory, 2-4 deep) run on separate barriers.
template <int MODE, int TRANS, int PAIR, int TS>
__global__ void __launch_bounds__(K1_THREADS, 1) tc_branch_kernel(BranchParams p) {
    static_assert(!(TS && PAIR), "the tensor-memory A operand is implemented for the single-CTA kernel");
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // work item: branch, 128-row tile (PAIR: tile pair), K range (a whole number of chunks)
    int blk = PAIR ? blockIdx.x >> 1 : blockIdx.x;
    const unsigned crank = PAIR ? (blockIdx.x & 1u) : 0u;   // rank in the (2,1,1) cluster
    const bool leader = crank == 0;
    const int mt = PAIR ? (p.mtiles + 1) / 2 : p.mtiles;
    const int np = mt * p.ks_p;
    const int br = blk < np ? 1 : 0;
    if (!br) blk -= np;
    const int ks = blk / mt, per = br ? p.per_p : p.per_s;
    const int m0 = (PAIR ? 2 * (blk % mt) + (int)crank : blk % mt) * 128;
    const int kb0 = ks * per;
    const int nkb = min(p.KB1, kb0 + per) - kb0;   // >= 1 by construction (phx_tc_branch_plan)
    const int nchunks = (nkb + p.chunk - 1) / p.chunk;
    const int S = p.stages, Hn = p.Hn;
    const int Hb = PAIR ? Hn >> 1 : Hn;                 // B rows staged by this CTA
    const unsigned b_tile = (unsigned)Hb * BK * 4;
    const unsigned b_bytes = 2 * b_tile;
    constexpr unsigned A_SMEM = TS ? 0u : K1_A_BYTES;   // bytes of the A tiles inside a shared-memory stage
    const unsigned stage_bytes = A_SMEM + b_bytes;
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + (size_t)S * stage_bytes);
    // done / drained: one barrier each, or (TS) one pair per chunk accumulator: chunk c lives in accumulator c & 1
    const unsigned full0 = smem_u32(bars), empty0 = smem_u32(bars + S), done = smem_u32(bars + 2 * S),
                   drained = smem_u32(bars + 2 * S + 2);
    const unsigned fullA0 = smem_u32(bars + 2 * S + 4), emptyA0 = smem_u32(bars + 2 * S + 8);   // TS: A ring, <= 4 stages
    unsigned* slot = reinterpret_cast<unsigned*>(bars + 2 * S + 12);
    const unsigned stage0 = smem_u32(smem);
    const int SA = TS ? p.a_stages : S;

    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            // single CTA: producer warps + the bulk-copy issuer (expect_tx).  Pair, leader: + the peer's producer warps
            // and its "B half landed" relay; pair, peer: the barrier only tracks the peer's own bulk copy.
            mbar_init(full0 + 8 * s, TS ? 1 : (!PAIR ? K1_PWARPS + 1 : (leader ? 2 * K1_PWARPS + 2 : 1)));
            mbar_init(empty0 + 8 * s, 1);              // tcgen05.commit (multicast to both CTAs of a pair)
        }
        if (TS)
            for (int s = 0; s < SA; ++s) {
                mbar_init(fullA0 + 8 * s, K1_PWARPS);  // every producer warp has stored its columns of the A tile
                mbar_init(emptyA0 + 8 * s, 1);         // tcgen05.commit
            }
        mbar_init(done, 1);
        mbar_init(drained, PAIR ? 2 * K1_DWARPS : K1_DWARPS);
        if (TS) {
            mbar_init(done + 8, 1);
            mbar_init(drained + 8, K1_DWARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == K1_W_BULK) {
        if (PAIR) tmem_alloc512_pair(smem_u32(slot));
        else tmem_alloc512(smem_u32(slot));
    }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();   // both CTAs' barriers exist before any remote arrive / multicast commit
    tc_fence_after();
    // TS = 0: chunk accumulator in columns [0, Hn), running sum in [256, 256 + Hn).  TS = 1: TWO chunk accumulators
    // (columns [0, Hn) and [256, 256 + Hn), chunk c in accumulator c & 1) and the running sum in shared memory, so the
    // fold of chunk c overlaps the MMAs of chunk c + 1.
    const unsigned tmem = *slot;

    if (warp < K1_PWARPS) {
        // ---- producers: Hill activation of this CTA's 128 x 16 slab of y, hi/lo split, core-matrix layout ----
        // row rl of the tile, k-chunk kc (4 floats).  TS: the row is the thread's tensor-memory lane
        const int rl = (TRANS || TS) ? (warp & 3) * 32 + lane : warp * 8 + (lane & 7);
        const int kc = (TRANS || TS) ? warp >> 2 : lane >> 3;
        const int row = m0 + rl;
        const float* ybase = (MODE && br && p.y2) ? p.y2 : p.y;   // uniform over the CTA
        const float* src = TRANS ? ybase + row : ybase + (size_t)row * p.ld;
        const bool rok = row < p.B;
        const float rscale = (MODE && TRANS && p.ascale && rok) ? __ldg(p.ascale + row) : 1.f;
        const bool asc_vec = (reinterpret_cast<uintptr_t>(p.ascale) & 15) == 0;
        const unsigned a_off = (unsigned)phx_tc_btile_off(128, rl, kc * 4) * 4u;
        // y is read in super-blocks of K1_PF k-blocks, the loads of the NEXT super-block in flight while the current one is
        // converted and handed to the MMAs.
        //   TRANS = 1: lanes run along the genes, each load instruction of a warp is one contiguous 128-byte piece.
        //   TRANS = 0: a thread's own elements (row lane%8, 4 floats of a 64-byte k-block piece) would make every load
        //   instruction touch 8 rows x 2 sectors -- measured, the L1 wavefronts of those loads were what the producers
        //   waited for.  Instead the warp loads its 8 rows COALESCED (lane = float index inside the row's 256-byte
        //   super-block piece, two instructions per row) and redistributes through a private shared-memory staging
        //   buffer (double buffered, rows padded to 68 floats: conflict-free 128-bit reads), __syncwarp only.
        float cur[K1_PF][4], nxt[K1_PF][4];
        constexpr int SBF = K1_PF * BK;          // floats of one row in a super-block (64)
        constexpr int SROW = SBF + 4;            // padded row stride of the staging buffer
        // TS = 0: a private buffer per warp (its 8 rows).  TS = 1: one buffer per lane quarter, shared by the four warps
        // (w & 3) == quarter: warp (quarter, j) loads rows 8j .. 8j+7 of the quarter and reads row `lane`, k-chunk j;
        // the hand-over is a 128-thread named barrier instead of __syncwarp.
        float* stg = reinterpret_cast<float*>(smem + (size_t)S * stage_bytes + 256) +
                     (TS ? (size_t)(warp & 3) * 32 * SROW : (size_t)warp * 2 * 8 * SROW);
        constexpr int SBUF = (TS ? 32 : 8) * SROW;                  // floats of one staging buffer
        constexpr int NSBUF = TS ? 1 : 2;                           // TS: single-buffered (the running sum needs the room)
        const int srow0 = TS ? (warp >> 2) * 8 : 0;                 // first staging row this warp fills
        const int srd = TS ? lane : (lane & 7);                     // staging row this thread reads
        auto stage_sync = [&]() {
            if (TS) asm volatile("bar.sync %0, 128;" ::"r"(1 + (warp & 3)) : "memory");
            else __syncwarp();
        };
        const float padv = MODE ? 0.f : 0.5f;    // pads contribute zero: s(0.5) = l(0.5) = 0
        // rows whose stride and base are multiples of 16 bytes (e.g. 20 000 genes): interior super-blocks are fetched with
        // four 16-byte loads per thread (lane = 16-byte piece of one of two rows) instead of sixteen 4-byte ones
        const bool vec_rows = !TRANS && (p.ld & 3) == 0 && (reinterpret_cast<uintptr_t>(ybase) & 15) == 0;
        bool nxt_vec = false;                    // register layout of `nxt` (set by load, used by stage_put)
        auto load = [&](int i, float (&v)[K1_PF][4]) {   // k-blocks kb0 + i .. kb0 + i + K1_PF - 1
            if (TRANS) {
                if (i + K1_PF <= nkb && (kb0 + i + K1_PF) * BK <= p.G) {   // interior super-block: only the row test
                    const float* q = src + (size_t)((kb0 + i) * BK + kc * 4) * p.ld;
#pragma unroll
                    for (int u = 0; u < K1_PF; ++u)
#pragma unroll
                        for (int j = 0; j < 4; ++j) v[u][j] = rok ? __ldg(q + (size_t)(u * BK + j) * p.ld) : padv;
                    return;
                }
#pragma unroll
                for (int u = 0; u < K1_PF; ++u) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int g = (kb0 + i + u) * BK + kc * 4 + j;
                        v[u][j] = (rok && i + u < nkb && g < p.G) ? __ldg(src + (size_t)g * p.ld) : padv;
                    }
                }
            } else {
                // v[rr/2][(rr%2)*2 + h] = element (lane + 32 h) of row rr of this warp
                const int kvalid = min(p.G - (kb0 + i) * BK, (nkb - i) * BK);   // valid floats of the piece
                const int rbase = m0 + (TS ? (warp & 3) * 32 + srow0 : warp * 8);
                nxt_vec = false;
                if (vec_rows && kvalid >= SBF && rbase + 8 <= p.B) {
                    nxt_vec = true;
                    const float* rp = ybase + (size_t)(rbase + (lane >> 4)) * p.ld + (size_t)(kb0 + i) * BK + 4 * (lane & 15);
#pragma unroll
                    for (int q2 = 0; q2 < 4; ++q2)   // rows rbase + 2 q2 + (lane >> 4)
                        asm volatile("ld.global.nc.L2::256B.v4.f32 {%0,%1,%2,%3}, [%4];"
                                     : "=f"(v[q2][0]), "=f"(v[q2][1]), "=f"(v[q2][2]), "=f"(v[q2][3])
                                     : "l"(rp + (size_t)(2 * q2) * p.ld));
                    return;
                }
                if (kvalid >= SBF && rbase + 8 <= p.B) {   // interior: no predicates
                    const float* rp = ybase + (size_t)rbase * p.ld + (size_t)(kb0 + i) * BK + lane;
#pragma unroll
                    for (int rr = 0; rr < 8; ++rr)
#pragma unroll
                        for (int h = 0; h < 2; ++h)
                            asm volatile("ld.global.nc.L2::256B.f32 %0, [%1];"
                                         : "=f"(v[rr >> 1][(rr & 1) * 2 + h])
                                         : "l"(rp + (size_t)rr * p.ld + 32 * h));
                    return;
                }
#pragma unroll
                for (int rr = 0; rr < 8; ++rr) {
                    const int row8 = m0 + (TS ? (warp & 3) * 32 + srow0 : warp * 8) + rr;
                    const float* rp = ybase + (size_t)row8 * p.ld + (size_t)(kb0 + i) * BK;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int e = lane + 32 * h;
                        float t = padv;
                        if (row8 < p.B && e < kvalid)
                            asm volatile("ld.global.nc.L2::256B.f32 %0, [%1];" : "=f"(t) : "l"(rp + e));
                        v[rr >> 1][(rr & 1) * 2 + h] = t;
                    }
                }
            }
        };
        auto stage_put = [&](int buf, const float (&v)[K1_PF][4]) {   // TRANS = 0: registers -> staging buffer
            float* d = stg + buf * SBUF + srow0 * SROW;
            if (nxt_vec) {
#pragma unroll
                for (int q2 = 0; q2 < 4; ++q2)
                    *reinterpret_cast<float4*>(d + (2 * q2 + (lane >> 4)) * SROW + 4 * (lane & 15)) =
                        make_float4(v[q2][0], v[q2][1], v[q2][2], v[q2][3]);
                return;
            }
#pragma unroll
            for (int rr = 0; rr < 8; ++rr)
#pragma unroll
                for (int h = 0; h < 2; ++h) d[rr * SROW + lane + 32 * h] = v[rr >> 1][(rr & 1) * 2 + h];
        };
        long long t_empty = 0, t_load = 0, t_conv = 0, t_store = 0, t0 = clock64();
        int s = 0;           // ring slot of k-block i
        unsigned ph = 0;     // its phase parity
        int sbuf = 0;
        if (TRANS) {
            load(0, cur);
        } else {
            load(0, nxt);
            stage_put(0, nxt);
            stage_sync();
        }
        int sa = 0;          // TS: A-ring slot of k-block i and its phase parity
        unsigned pha = 0;
        const unsigned tq = TS ? tmem + ((unsigned)((warp & 3) * 32) << 16) + 4u * (unsigned)kc : 0u;
        for (int i0 = 0; i0 < nkb; i0 += K1_PF) {
            const long long tl0 = PROF(p) ? clock64() : 0;
            if (i0 + K1_PF < nkb) load(i0 + K1_PF, nxt);
            if (PROF(p)) t_load += clock64() - tl0;
#pragma unroll
            for (int u = 0; u < K1_PF; ++u) {
                const int i = i0 + u;
                if (i < nkb) {
                    const long long tc0 = PROF(p) ? clock64() : 0;
                    // TS: test the A slot of this k-block NOW, so that the barrier round trip hides behind the conversion
                    unsigned slot_free = 0;
                    if (TS && lane == 0) slot_free = mbar_test(emptyA0 + 8 * sa, pha ^ 1u);
                    float xin[4];
                    if (TRANS) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) xin[j] = cur[u][j];
                    } else {
                        const float4 t =
                            *reinterpret_cast<const float4*>(stg + sbuf * SBUF + srd * SROW + u * BK + kc * 4);
                        xin[0] = t.x; xin[1] = t.y; xin[2] = t.z; xin[3] = t.w;
                    }
                    float hi[4], lo[4];
                    float sc4[4] = {rscale, rscale, rscale, rscale};
                    if (MODE && !TRANS && p.ascale) {   // per-gene factors of this thread's k-chunk: one 16-byte load
                        const int g0 = (kb0 + i) * BK + kc * 4;
                        if (asc_vec && g0 + 3 < p.G) {
                            const float4 t = __ldg(reinterpret_cast<const float4*>(p.ascale + g0));
                            sc4[0] = t.x; sc4[1] = t.y; sc4[2] = t.z; sc4[3] = t.w;
                        } else {
#pragma unroll
                            for (int j = 0; j < 4; ++j) sc4[j] = g0 + j < p.G ? __ldg(p.ascale + g0 + j) : 0.f;
                        }
                    }
                    // (MODE 1: the per-gene factor is applied here, NOT where the load of y is issued: a use right behind
                    // the load would wait for it and serialise the prefetch)
                    convert4<MODE>(xin, sc4, br, hi, lo);
                    const long long tw = PROF(p) ? clock64() : 0;
                    if (PROF(p)) t_conv += tw - tc0 + (long long)(__float_as_uint(hi[0]) & 0u);
                    if (TS) {
                        if (lane == 0 && !slot_free) mbar_wait(emptyA0 + 8 * sa, pha ^ 1u);   // the MMAs of this slot are done
                        __syncwarp();
                        tc_fence_after();
                        const long long ts0 = PROF(p) ? clock64() : 0;
                        if (PROF(p)) t_empty += ts0 - tw;
                        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(
                                         tq + (unsigned)p.a_hi_col[sa]),
                                     "r"(__float_as_uint(hi[0])), "r"(__float_as_uint(hi[1])), "r"(__float_as_uint(hi[2])),
                                     "r"(__float_as_uint(hi[3]))
                                     : "memory");
                        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(
                                         tq + (unsigned)p.a_lo_col[sa]),
                                     "r"(__float_as_uint(lo[0])), "r"(__float_as_uint(lo[1])), "r"(__float_as_uint(lo[2])),
                                     "r"(__float_as_uint(lo[3]))
                                     : "memory");
                        // (deferring this hand-over behind the next k-block's conversion was tried: the MMAs starve, 3 % slower)
                        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(fullA0 + 8 * sa);
                        if (PROF(p)) t_store += clock64() - ts0;
                        if (++sa == SA) {
                            sa = 0;
                            pha ^= 1u;
                        }
                        continue;
                    }
                    if (lane == 0) mbar_wait(empty0 + 8 * s, ph ^ 1u);   // one poller per warp
                    __syncwarp();
                    if (PROF(p)) t_empty += clock64() - tw;
                    unsigned char* a = smem + (size_t)s * stage_bytes + a_off;
                    *reinterpret_cast<float4*>(a) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<float4*>(a + K1_A_TILE) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                    fence_async_smem();   // generic-proxy writes -> visible to the tensor core's async-proxy reads
                    __syncwarp();
                    if (lane == 0) {
                        if (PAIR && !leader) mbar_arrive_remote(full0 + 8 * s, 0u);
                        else mbar_arrive(full0 + 8 * s);
                    }
                    if (++s == S) {
                        s = 0;
                        ph ^= 1u;
                    }
                }
            }
            if (TRANS) {
#pragma unroll
                for (int u = 0; u < K1_PF; ++u)
#pragma unroll
                    for (int j = 0; j < 4; ++j) cur[u][j] = nxt[u][j];
            } else if (i0 + K1_PF < nkb) {
                const long long tl1 = PROF(p) ? clock64() : 0;
                if (NSBUF == 2) sbuf ^= 1;   // the other buffer: last read one super-block ago (ordered by the hand-over sync)
                else stage_sync();           // single buffer: every warp of the group has read this super-block
                stage_put(sbuf, nxt);
                stage_sync();
                if (PROF(p)) t_load += clock64() - tl1;
            }
        }
        if (PROF(p) && tid == 0) {
            unsigned long long* q = PROF(p) + 8 * br + 4;
            atomicAdd(q + 0, (unsigned long long)(clock64() - t0));
            atomicAdd(q + 1, (unsigned long long)t_empty);
            atomicAdd(PROF(p) + 16 + 8 * br + 0, (unsigned long long)t_load);
            atomicAdd(PROF(p) + 16 + 8 * br + 1, (unsigned long long)t_conv);
            atomicAdd(PROF(p) + 16 + 8 * br + 2, (unsigned long long)t_store);
        }
    } else if (warp == K1_W_BULK) {
        if (lane == 0) {
            int s = 0;
            unsigned ph = 0;
            for (int i = 0; i < nkb; ++i) {
                mbar_wait(empty0 + 8 * s, ph ^ 1u);
                if (!PAIR) {
                    mbar_expect_tx(full0 + 8 * s, b_bytes);
                    bulk_g2s(stage0 + s * stage_bytes + A_SMEM,
                             p.w1img + ((size_t)(kb0 + i) * 4 + 2 * br) * Hn * BK, b_bytes, full0 + 8 * s);
                } else {
                    // this CTA's half of the rows: in the image the rows of one k-chunk are contiguous, so the half
                    // tile is 2 (hi|lo) x 4 (k-chunks) pieces of Hn/16 core matrices
                    mbar_expect_tx(full0 + 8 * s, b_bytes);
                    const float* chunk = p.w1img + ((size_t)(kb0 + i) * 4 + 2 * br) * Hn * BK;
                    const unsigned dst0 = stage0 + s * stage_bytes + K1_A_BYTES;
#if PHX_TC_BRANCH_SW64
                    // rows are 64 contiguous bytes: this CTA's half of a tile is one contiguous piece
#pragma unroll
                    for (int hl = 0; hl < 2; ++hl)
                        bulk_g2s(dst0 + hl * b_tile, chunk + (size_t)hl * Hn * BK + (size_t)crank * Hb * BK, b_tile,
                                 full0 + 8 * s);
#else
                    const unsigned piece = (unsigned)(Hn >> 4) * 128u;
#pragma unroll
                    for (int hl = 0; hl < 2; ++hl)
#pragma unroll
                        for (int kc4 = 0; kc4 < 4; ++kc4)
                            bulk_g2s(dst0 + hl * b_tile + kc4 * piece,
                                     chunk + (size_t)hl * Hn * BK + ((size_t)kc4 * (Hn >> 3) + crank * (Hn >> 4)) * 32,
                                     piece, full0 + 8 * s);
#endif
                }
                if (++s == S) {
                    s = 0;
                    ph ^= 1u;
                }
            }
        }
    } else if (warp == K1_W_MMA) {
        // ---- MMA issuer: the whole warp runs the loop (uniform control flow, descriptors in uniform registers); one
        // elected lane issues the tcgen05 instructions.  In a pair only the leader issues; the peer's warp relays
        // "my half of B has landed" to the leader's full barrier. ----
        const unsigned idesc = idesc_tf32(PAIR ? 256 : 128, Hn);
        const unsigned lt = PHX_TC_BRANCH_SW64 ? 4u : 0u;
        const uint64_t a_hi_part = smem_desc(0, p.a_lbo, p.a_sbo, lt), b_hi_part = smem_desc(0, p.b_lbo, p.b_sbo, lt);
        int s = 0, c = 0, ic = 0, sa = 0;
        unsigned ph = 0, pha = 0;
        long long t_full = 0, t_drained = 0, t0 = clock64();
        if (PAIR && !leader) {
            for (int i = 0; i < nkb; ++i) {
                if (lane == 0) {
                    mbar_wait(full0 + 8 * s, ph);
                    mbar_arrive_remote(full0 + 8 * s, 0u);
                }
                __syncwarp();
                if (++s == S) {
                    s = 0;
                    ph ^= 1u;
                }
            }
        } else
        for (int i = 0; i < nkb; ++i) {
            if (TS) {
                if (ic == 0 && c >= 2) {   // chunk c - 2 must have left this accumulator
                    const long long tw = PROF(p) ? clock64() : 0;
                    mbar_wait(drained + 8 * (c & 1), (unsigned)((c >> 1) - 1) & 1u);
                    if (PROF(p)) t_drained += clock64() - tw;
                }
            } else if (ic == 0 && c > 0) {   // the previous chunk's sum must have left the chunk accumulator (both CTAs)
                const long long tw = PROF(p) ? clock64() : 0;
                if (PAIR) mbar_wait_cluster(drained, (unsigned)(c - 1) & 1u);
                else mbar_wait(drained, (unsigned)(c - 1) & 1u);
                if (PROF(p)) t_drained += clock64() - tw;
            }
            const long long tw = PROF(p) ? clock64() : 0;
            if (PAIR) mbar_wait_cluster(full0 + 8 * s, ph);
            else mbar_wait(full0 + 8 * s, ph);
            if (TS) mbar_wait(fullA0 + 8 * sa, pha);
            if (PROF(p)) t_full += clock64() - tw;
            tc_fence_after();
            const unsigned a_base = stage0 + s * stage_bytes, b_base = a_base + A_SMEM;
            if (TS) {
                if (elect_one()) {
                    const unsigned ta_hi = tmem + (unsigned)p.a_hi_col[sa], ta_lo = tmem + (unsigned)p.a_lo_col[sa];
                    const unsigned tacc = tmem + ((c & 1) ? 256u : 0u);
#pragma unroll
                    for (int k8 = 0; k8 < BK / 8; ++k8) {
                        const uint64_t b_hi = desc_at(b_hi_part, b_base + k8 * p.b_kadv);
                        const uint64_t b_lo = desc_at(b_hi_part, b_base + b_tile + k8 * p.b_kadv);
                        const unsigned acc = (ic > 0 || k8 > 0) ? 1u : 0u;
                        if (p.nterms == 3) {
                            mma_tf32_ts(tacc, ta_lo + 8u * k8, b_hi, idesc, acc);
                            mma_tf32_ts(tacc, ta_hi + 8u * k8, b_lo, idesc, 1u);
                            mma_tf32_ts(tacc, ta_hi + 8u * k8, b_hi, idesc, 1u);
                        } else {
                            mma_tf32_ts(tacc, ta_hi + 8u * k8, b_hi, idesc, acc);
                        }
                    }
                    mma_commit(emptyA0 + 8 * sa);
                    mma_commit(empty0 + 8 * s);
                    if (ic == p.chunk - 1 || i == nkb - 1) mma_commit(done + 8 * (c & 1));
                }
                if (++sa == SA) {
                    sa = 0;
                    pha ^= 1u;
                }
            } else if (elect_one()) {
#pragma unroll
                for (int k8 = 0; k8 < BK / 8; ++k8) {
                    const uint64_t a_hi = desc_at(a_hi_part, a_base + k8 * p.a_kadv);
                    const uint64_t a_lo = desc_at(a_hi_part, a_base + K1_A_TILE + k8 * p.a_kadv);
                    const uint64_t b_hi = desc_at(b_hi_part, b_base + k8 * p.b_kadv);
                    const uint64_t b_lo = desc_at(b_hi_part, b_base + b_tile + k8 * p.b_kadv);
                    const unsigned acc = (ic > 0 || k8 > 0) ? 1u : 0u;
                    if (PAIR) {
                        if (p.nterms == 3) {
                            mma_tf32_pair(tmem, a_lo, b_hi, idesc, acc);
                            mma_tf32_pair(tmem, a_hi, b_lo, idesc, 1u);
                            mma_tf32_pair(tmem, a_hi, b_hi, idesc, 1u);
                        } else {
                            mma_tf32_pair(tmem, a_hi, b_hi, idesc, acc);
                        }
                    } else if (p.nterms == 3) {
                        mma_tf32(tmem, a_lo, b_hi, idesc, acc);
                        mma_tf32(tmem, a_hi, b_lo, idesc, 1u);
                        mma_tf32(tmem, a_hi, b_hi, idesc, 1u);
                    } else {
                        mma_tf32(tmem, a_hi, b_hi, idesc, acc);
                    }
                }
                if (PAIR) {
                    mma_commit_pair(empty0 + 8 * s);
                    if (ic == p.chunk - 1 || i == nkb - 1) mma_commit_pair(done);
                } else {
                    mma_commit(empty0 + 8 * s);
                    if (ic == p.chunk - 1 || i == nkb - 1) mma_commit(done);
                }
            }
            __syncwarp();
            if (++s == S) {
                s = 0;
                ph ^= 1u;
            }
            if (++ic == p.chunk) {
                ic = 0;
                ++c;
            }
        }
        if (PROF(p) && lane == 0) {
            unsigned long long* q = PROF(p) + 8 * br;
            atomicAdd(q + 0, (unsigned long long)(clock64() - t0));
            atomicAdd(q + 1, (unsigned long long)t_full);
            atomicAdd(q + 2, (unsigned long long)t_drained);
            atomicAdd(q + 3, (unsigned long long)nkb);
        }
    } else {
        // ---- drain warps: running sum += chunk sum (round-to-nearest fp32 adds), all inside tensor memory; the last
        // chunk's result goes to this CTA's partial-sum slot ----
        const int q = warp & 3;
        const unsigned trow = tmem + ((unsigned)(q * 32) << 16);
        float* dst = p.spart + ((size_t)ks * p.Bpad + (m0 + q * 32 + lane)) * (2 * Hn) + br * Hn;
        long long t_drain = 0;
        // TS: running sum in shared memory as [column quad][row] float4 (consecutive lanes -> consecutive 16 bytes)
        float4* rs = reinterpret_cast<float4*>(smem + (size_t)S * stage_bytes + 256 + p.stg_bytes) + (q * 32 + lane);
        if (TS) {
            for (int c = 0; c < nchunks; ++c) {
                if (lane == 0) mbar_wait(done + 8 * (c & 1), (unsigned)(c >> 1) & 1u);
                __syncwarp();
                const long long tw = PROF(p) ? clock64() : 0;
                tc_fence_after();
                const bool last = c == nchunks - 1;
                const unsigned tacc = trow + ((c & 1) ? 256u : 0u);
                for (int c0 = 0; c0 < Hn; c0 += 32) {
                    const bool two = c0 + 16 < Hn;
                    unsigned v0[16], v1[16];
                    tmem_ld16_nowait(tacc + c0, v0);
                    if (two) tmem_ld16_nowait(tacc + c0 + 16, v1);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        float4 a = make_float4(__uint_as_float(v0[j]), __uint_as_float(v0[j + 1]), __uint_as_float(v0[j + 2]),
                                               __uint_as_float(v0[j + 3]));
                        float4* r = rs + (size_t)((c0 + j) >> 2) * 128;
                        if (c > 0) {
                            const float4 o = *r;
                            a.x = o.x + a.x; a.y = o.y + a.y; a.z = o.z + a.z; a.w = o.w + a.w;
                        }
                        if (last) *reinterpret_cast<float4*>(dst + c0 + j) = a;
                        else *r = a;
                        if (two) {
                            float4 b = make_float4(__uint_as_float(v1[j]), __uint_as_float(v1[j + 1]),
                                                   __uint_as_float(v1[j + 2]), __uint_as_float(v1[j + 3]));
                            float4* r1 = rs + (size_t)((c0 + 16 + j) >> 2) * 128;
                            if (c > 0) {
                                const float4 o = *r1;
                                b.x = o.x + b.x; b.y = o.y + b.y; b.z = o.z + b.z; b.w = o.w + b.w;
                            }
                            if (last) *reinterpret_cast<float4*>(dst + c0 + 16 + j) = b;
                            else *r1 = b;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(drained + 8 * (c & 1));
                if (PROF(p)) t_drain += clock64() - tw;
            }
        } else
        for (int c = 0; c < nchunks; ++c) {
            if (lane == 0) mbar_wait(done, (unsigned)c & 1u);
            __syncwarp();
            const long long tw = PROF(p) ? clock64() : 0;
            tc_fence_after();
            const bool last = c == nchunks - 1;
            for (int c0 = 0; c0 < Hn; c0 += 32) {
                // two 16-column groups in flight per round trip to tensor memory
                const bool two = c0 + 16 < Hn;
                unsigned v0[16], v1[16], r0[16], r1[16];
                tmem_ld16_nowait(trow + c0, v0);
                if (two) tmem_ld16_nowait(trow + c0 + 16, v1);
                if (c > 0) {
                    tmem_ld16_nowait(trow + 256 + c0, r0);
                    if (two) tmem_ld16_nowait(trow + 256 + c0 + 16, r1);
                }
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if (c > 0) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        v0[j] = __float_as_uint(__uint_as_float(r0[j]) + __uint_as_float(v0[j]));
                        if (two) v1[j] = __float_as_uint(__uint_as_float(r1[j]) + __uint_as_float(v1[j]));
                    }
                }
                if (last) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        *reinterpret_cast<uint4*>(dst + c0 + j) = make_uint4(v0[j], v0[j + 1], v0[j + 2], v0[j + 3]);
                        if (two)
                            *reinterpret_cast<uint4*>(dst + c0 + 16 + j) =
                                make_uint4(v1[j], v1[j + 1], v1[j + 2], v1[j + 3]);
                    }
                } else {
                    tmem_st16(trow + 256 + c0, v0);
                    if (two) tmem_st16(trow + 256 + c0 + 16, v1);
                }
            }
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (PAIR && !leader) mbar_arrive_remote(drained, 0u);
                else mbar_arrive(drained);
            }
            if (PROF(p)) t_drain += clock64() - tw;
        }
        if (PROF(p) && warp == K1_W_DRAIN && lane == 0) atomicAdd(PROF(p) + 8 * br + 6, (unsigned long long)t_drain);
    }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();   // the peer's shared memory and barriers stay alive until the leader is done
    if (warp == K1_W_BULK) {
        if (PAIR) tmem_free512_pair(tmem);
        else tmem_free512(tmem);
    }
}

// ---- K-split reduction + bias + exp + operand image of [S|P] ------------------------------------------------------------
// one thread per (batch row b in [0, BT*256), 4 consecutive Hn-numbered columns)
__global__ void tc_spfinish_kernel(int B, int Bpad, int H, int Hp, int Hn, int K2, int ks_s, int ks_p, int mode, const float* __restrict__ spart,
                                   const float* __restrict__ bias, float* __restrict__ SP, float* __restrict__ spimg,
                                   float* __restrict__ timg) {
    const int BT = phx_tc_BT(B), KB2 = 2 * Hn / BK, C4 = 2 * Hn / 4;
    const size_t total = (size_t)BT * 256 * C4;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int b = (int)(i % ((size_t)BT * 256));   // rows fastest: image stores of a warp are contiguous
        const int c4 = (int)(i / ((size_t)BT * 256));
        const int c = c4 * 4, br = c / Hn, n0 = c % Hn;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (b < B) {
            const int nslots = br ? ks_p : ks_s;
            for (int s = 0; s < nslots; ++s) {
                const float4 t = *reinterpret_cast<const float4*>(spart + ((size_t)s * Bpad + b) * (2 * Hn) + c);
                v[0] += t.x; v[1] += t.y; v[2] += t.z; v[3] += t.w;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = n0 + j;
                if (n < H) {
                    if (mode == 0) {          // [S|P]: bias, exp on the prods half
                        float x = v[j] + bias[br * Hp + n];
                        v[j] = br ? expf(x) : x;
                    } else if (br) {          // gSP: prods half scaled by Pr (bias = the plain [S|P] of this batch)
                        v[j] = v[j] * bias[(size_t)b * K2 + Hp + n];
                    }
                } else {
                    v[j] = 0.f;
                }
                if (n < Hp) SP[(size_t)b * K2 + br * Hp + n] = v[j];
            }
        }
        float hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) split_tf32(v[j], hi[j], lo[j]);
        const int bt = b >> 8, r = b & 255, kb = c / BK, k = c % BK;
        float* chunk = spimg + ((size_t)bt * KB2 + kb) * 2 * 256 * BK;
        const int off = phx_tc_tile_off(256, r, k);
        *reinterpret_cast<float4*>(chunk + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<float4*>(chunk + 256 * BK + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        if (timg && b < ((B + BK - 1) / BK) * BK) {
            // the same values as the B operand of the K = batch contractions: [b / 16][branch][hi|lo][Hn x 16]
            float* tch = timg + ((size_t)(b / BK) * 4 + 2 * br) * Hn * BK;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int o = phx_tc_btile_off(Hn, n0 + j, b % BK);
                tch[o] = hi[j];
                tch[Hn * BK + o] = lo[j];
            }
        }
    }
}

// parameter cotangents from the K-split partial sums part[slot][Gpad][2*Hn] of the K = batch contractions
//   which = 0: Ws_bar[n][g] / Wp_bar[n][g]  <- part[.][g][br*Hn + n]      which = 1: Wa_bar[g][br*H + n]
__global__ void tc_gradfinish_kernel(int which, int G, int Gpad, int H, int Hn, int ks_s, int ks_p,
                                     const float* __restrict__ part, float* __restrict__ d0, float* __restrict__ d1,
                                     int accumulate) {
    const size_t total = (size_t)G * 2 * H;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        int g, br, n;
        if (which == 0) {   // g fastest: coalesced stores into [H][G]
            g = (int)(i % G);
            const int c = (int)(i / G);
            br = c / H; n = c % H;
        } else {            // column fastest: coalesced loads and stores of [G][2H]
            const int c = (int)(i % (2 * H));
            g = (int)(i / (2 * H));
            br = c / H; n = c % H;
        }
        const int nslots = br ? ks_p : ks_s;
        if (which == 0 && !(br ? d1 : d0)) continue;   // that half is not wanted
        float v = 0.f;
        for (int s = 0; s < nslots; ++s) v += part[((size_t)s * Gpad + g) * (2 * Hn) + br * Hn + n];
        float* dst = which == 0 ? (br ? d1 : d0) + (size_t)n * G + g : d0 + (size_t)g * 2 * H + br * H + n;
        *dst = accumulate ? *dst + v : v;
    }
}

// ---- kernel 2: joint contraction + decay epilogue -------------------------------------------------------------------------
struct JointParams {
    int G, B, KB2, GT, BT, nterms, decay;
    unsigned a_lbo, a_sbo, b_lbo, b_sbo;   // descriptor fields
    unsigned a_kadv, b_kadv;               // byte advance of the start address per K = 8 MMA (two core matrices)
    int kb_lo, kb_hi;     // k-blocks of the images used by this launch
    int emode;            // epilogue: 0 f = fscale*(decay ? relu(m)*(acc - y) : acc); 1 f = acc; 2 state cotangent:
                          //   f = (f + acc/(1+s(y))) / (1+|y-.5|)^2 - (decay ? g*relu(m) : 0)   (f holds u on entry);
                          // 3 the same with u and v accumulated side by side (k-blocks below / above the middle)
                          // 4 prior loss (train_insilico.py:134-135): f = fscale * (acc - g) with g = prior_grad, and the
                          //   sum of (acc - g)^2 per epilogue warp -> part (the joint itself is never written)
                          // 5 = 0, then `post`: the next stage input / the step's end value from f, x0 and the older
                          //   stage derivatives, in the same pass (no separate elementwise kernel over the state)
    float fscale;
    const float* waimg;   // A image: [GT][KB2][hi|lo][128 x 16]
    const float* spimg;   // B image: [BT][KB2][hi|lo][256 x 16]
    const float* y;       // [B][G]
    const float* g;       // [B][G] cotangent (emode 2 with decay)
    const float* relum;   // [G]
    float* f;             // [B][G]
    double* part;         // emode 4: [gridDim.x][8] per-epilogue-warp sums of (acc - g)^2
    PhxRhsPost post;      // emode 5 = emode 0 followed by the RK stage algebra of the streaming solvers (phx_common.cuh)
};
constexpr int K2_THREADS = 320;   // bulk-copy issuer, MMA issuer, 8 epilogue warps
constexpr int K2_STAGES = 4;
constexpr unsigned K2_A_TILE = 128 * BK * 4, K2_B_TILE = 256 * BK * 4;
constexpr unsigned K2_STAGE_BYTES = 2 * K2_A_TILE + 2 * K2_B_TILE;   // 48 KB

template <int EMODE>
__global__ void __launch_bounds__(K2_THREADS, 1) tc_joint_kernel(JointParams p) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int S = K2_STAGES;
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + (size_t)S * K2_STAGE_BYTES);
    const unsigned full0 = smem_u32(bars), empty0 = smem_u32(bars + S), tfull0 = smem_u32(bars + 2 * S),
                   tempty0 = smem_u32(bars + 2 * S + 2);
    unsigned* slot = reinterpret_cast<unsigned*>(bars + 2 * S + 4);
    const unsigned stage0 = smem_u32(smem);
    const int ntiles = p.GT * p.BT;

    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(tfull0 + 8 * b, 1);
            mbar_init(tempty0 + 8 * b, 8);   // one arrive per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc512(smem_u32(slot));
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem = *slot;

    if (warp == 0) {
        if (lane == 0) {
            int it = 0;
            for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
                const int gt = t / p.BT, bt = t % p.BT;
                for (int kb = p.kb_lo; kb < p.kb_hi; ++kb, ++it) {
                    const int s = it % S;
                    const unsigned ph = (unsigned)(it / S) & 1u;
                    mbar_wait(empty0 + 8 * s, ph ^ 1u);
                    mbar_expect_tx(full0 + 8 * s, K2_STAGE_BYTES);
                    const unsigned dst = stage0 + s * K2_STAGE_BYTES;
                    bulk_g2s(dst, p.waimg + ((size_t)gt * p.KB2 + kb) * 2 * 128 * BK, 2 * K2_A_TILE, full0 + 8 * s);
                    bulk_g2s(dst + 2 * K2_A_TILE, p.spimg + ((size_t)bt * p.KB2 + kb) * 2 * 256 * BK, 2 * K2_B_TILE,
                             full0 + 8 * s);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const unsigned idesc = idesc_tf32(128, 256);
            int it = 0, j = 0;
            for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
                // EMODE 3 (fused u|v pass): both halves of tensor memory hold ONE tile (u in columns 0..255, v in
                // 256..511), so there is no second buffer and the MMAs of a tile wait for the previous epilogue
                const int buf = EMODE == 3 ? 0 : (j & 1);
                const unsigned tph = EMODE == 3 ? (unsigned)j & 1u : (unsigned)(j >> 1) & 1u;
                mbar_wait(tempty0 + 8 * buf, tph ^ 1u);   // epilogue has drained this accumulator
                tc_fence_after();
                const int kb_mid = (p.kb_lo + p.kb_hi) >> 1;
                for (int kb = p.kb_lo; kb < p.kb_hi; ++kb, ++it) {
                    const bool second = EMODE == 3 && kb >= kb_mid;
                    const unsigned d = tmem + (unsigned)(EMODE == 3 ? (second ? 256 : 0) : buf * 256);
                    const int kb_first = second ? kb_mid : p.kb_lo;
                    const int s = it % S;
                    const unsigned ph = (unsigned)(it / S) & 1u;
                    mbar_wait(full0 + 8 * s, ph);
                    tc_fence_after();
                    const unsigned a_base = stage0 + s * K2_STAGE_BYTES, b_base = a_base + 2 * K2_A_TILE;
#pragma unroll
                    for (int k8 = 0; k8 < BK / 8; ++k8) {
                        const uint64_t a_hi = smem_desc(a_base + k8 * p.a_kadv, p.a_lbo, p.a_sbo);
                        const uint64_t a_lo = smem_desc(a_base + K2_A_TILE + k8 * p.a_kadv, p.a_lbo, p.a_sbo);
                        const uint64_t b_hi = smem_desc(b_base + k8 * p.b_kadv, p.b_lbo, p.b_sbo);
                        const uint64_t b_lo = smem_desc(b_base + K2_B_TILE + k8 * p.b_kadv, p.b_lbo, p.b_sbo);
                        const unsigned acc = (kb > kb_first || k8 > 0) ? 1u : 0u;
                        if (p.nterms == 3) {
                            mma_tf32(d, a_lo, b_hi, idesc, acc);
                            mma_tf32(d, a_hi, b_lo, idesc, 1u);
                            mma_tf32(d, a_hi, b_hi, idesc, 1u);
                        } else {
                            mma_tf32(d, a_hi, b_hi, idesc, acc);
                        }
                    }
                    mma_commit(empty0 + 8 * s);
                }
                mma_commit(tfull0 + 8 * buf);
            }
        }
    } else {
        // ---- epilogue warps 2..9: lane quarter q = warp % 4 of the accumulator = 32 consecutive genes; the two warps
        // of a quarter take 128 batch rows (accumulator columns) each.  y does not depend on the MMAs, so the loads of
        // the next 16 columns are always in flight while the current 16 are combined and stored.
        const int q = warp & 3, half = (warp - 2) >> 2;
        int j = 0;
        double sq = 0.0;   // EMODE 4
        for (int t = blockIdx.x; t < ntiles; t += gridDim.x, ++j) {
            const int gt = t / p.BT, bt = t % p.BT;
            const int buf = EMODE == 3 ? 0 : (j & 1);
            const unsigned tph = EMODE == 3 ? (unsigned)j & 1u : (unsigned)(j >> 1) & 1u;
            const int g = gt * 128 + q * 32 + lane;
            const bool gok = g < p.G;
            const float rm = (gok && p.decay) ? p.relum[g] : 1.f;
            const int b0 = bt * 256 + half * 128;
            const int ncol = min(128, p.B - b0);   // valid batch rows of this warp's half (may be <= 0)
            const bool need_y = (EMODE >= 2 && EMODE < 4) || ((EMODE == 0 || EMODE == 5) && p.decay);
            constexpr bool need_u = EMODE == 2;
            const bool need_g = EMODE == 4 || (EMODE >= 2 && EMODE < 4 && p.decay);
            float yv[16], yn[16], uv[16], un[16], gv[16], gn[16];
            auto loadin = [&](int c0, float (&dy)[16], float (&du)[16], float (&dg)[16]) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                    const bool ok = gok && c0 + jj < ncol;
                    const size_t idx = (size_t)(b0 + c0 + jj) * p.G + g;
                    // EMODE 5 may write the next stage input over the state it reads (same thread, same element): no
                    // non-coherent loads from that buffer
                    dy[jj] = (need_y && ok) ? (EMODE == 5 ? p.y[idx] : __ldg(p.y + idx)) : 0.f;
                    du[jj] = (need_u && ok) ? p.f[idx] : 0.f;
                    dg[jj] = (need_g && ok) ? __ldg(p.g + idx) : 0.f;
                }
            };
            loadin(0, yn, un, gn);
            mbar_wait(tfull0 + 8 * buf, tph);
            tc_fence_after();
            for (int c0 = 0; c0 < ncol; c0 += 16) {
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                    yv[jj] = yn[jj];
                    uv[jj] = un[jj];
                    gv[jj] = gn[jj];
                }
                if (c0 + 16 < ncol) loadin(c0 + 16, yn, un, gn);
                if (EMODE == 5) {
                    // f as in EMODE 0, then the RK stage algebra that follows it (PhxRhsPost).  The loads do not depend on
                    // the MMAs: x0 and the two oldest derivatives are in flight before the accumulator is read, the
                    // others follow two arrays (32 loads per thread) at a time -- what fits the 168 registers of a
                    // 320-thread CTA without spilling loaded values (a spilled load serialises on its latency).
                    const PhxRhsPost& po = p.post;
                    const int nk = po.nk;
                    float xv[16], ka[16], kb[16], r[16], o[16];
                    auto ld16 = [&](const float* src, float (&d)[16], bool use) {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) {
                            const bool ok = use && gok && c0 + jj < ncol;
                            d[jj] = ok ? __ldg(src + (size_t)(b0 + c0 + jj) * p.G + g) : 0.f;
                        }
                    };
                    ld16(po.x0, xv, true);
                    ld16(po.k[0], ka, nk > 0);
                    ld16(po.k[1], kb, nk > 1);
                    float v[16];
                    tmem_ld16(tmem + ((unsigned)(q * 32) << 16) + (unsigned)(buf * 256 + half * 128 + c0), v);
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) r[jj] = p.fscale * (p.decay ? rm * (v[jj] - yv[jj]) : v[jj]);
                    if (po.mode == PHX_POST_CHAIN) {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) {
                            o[jj] = ka[jj] * po.c[0];
                            if (nk > 1) o[jj] = fmaf(kb[jj], po.c[1], o[jj]);
                        }
                        if (nk > 2) {
                            ld16(po.k[2], ka, true);
                            ld16(po.k[3], kb, nk > 3);
#pragma unroll
                            for (int jj = 0; jj < 16; ++jj) {
                                o[jj] = fmaf(ka[jj], po.c[2], o[jj]);
                                if (nk > 3) o[jj] = fmaf(kb[jj], po.c[3], o[jj]);
                            }
                        }
                        if (nk > 4) {
                            ld16(po.k[4], ka, true);
                            ld16(po.k[5], kb, nk > 5);
#pragma unroll
                            for (int jj = 0; jj < 16; ++jj) {
                                o[jj] = fmaf(ka[jj], po.c[4], o[jj]);
                                if (nk > 5) o[jj] = fmaf(kb[jj], po.c[5], o[jj]);
                            }
                        }
                        const float cl = po.cr;
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) {
                            o[jj] = nk == 0 ? r[jj] * cl : fmaf(r[jj], cl, o[jj]);
                            o[jj] = xv[jj] + o[jj];
                        }
                    } else {
                        // the newest derivative is r, the older ones a1.. = k[0..nk-1] (at most three)
                        const int fx = po.mode - PHX_POST_FX;
                        if (nk > 2) ld16(po.k[2], o, true);
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj) {
                            const float a1 = nk > 0 ? ka[jj] : r[jj];
                            const float a2 = nk > 1 ? kb[jj] : (nk == 1 ? r[jj] : 0.f);
                            const float a3 = nk > 2 ? o[jj] : (nk == 2 ? r[jj] : 0.f);
                            const float a4 = nk == 3 ? r[jj] : 0.f;
                            o[jj] = phx_fixed_formula(fx, xv[jj], a1, a2, a3, a4, po.dt);
                        }
                    }
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) {
                        if (gok && c0 + jj < ncol) {
                            const size_t idx = (size_t)(b0 + c0 + jj) * p.G + g;
                            po.out[idx] = o[jj];
                            if (po.store_f) p.f[idx] = r[jj];
                        }
                    }
                    continue;
                }
                float v[16];
                tmem_ld16(tmem + ((unsigned)(q * 32) << 16) + (unsigned)(buf * 256 + half * 128 + c0), v);
                if (EMODE == 3) {   // u from the first half of tensor memory, v from the second
#pragma unroll
                    for (int jj = 0; jj < 16; ++jj) uv[jj] = v[jj];
                    tmem_ld16(tmem + ((unsigned)(q * 32) << 16) + (unsigned)(256 + half * 128 + c0), v);
                }
#pragma unroll
                for (int jj = 0; jj < 16; ++jj) {
                    if (gok && c0 + jj < ncol) {
                        float r;
                        if (EMODE == 0) {
                            r = p.fscale * (p.decay ? rm * (v[jj] - yv[jj]) : v[jj]);
                        } else if (EMODE == 1) {
                            r = v[jj];
                        } else if (EMODE == 4) {
                            const float d = v[jj] - gv[jj];
                            sq += (double)(d * d);
                            r = p.fscale * d;
                        } else {
                            const float z = yv[jj] - 0.5f;
                            const float den = 1.0f + fabsf(z);
                            const float sv = z / den;
                            r = (uv[jj] + v[jj] / (1.0f + sv)) / (den * den);
                            if (p.decay) r = r - gv[jj] * rm;
                        }
                        p.f[(size_t)(b0 + c0 + jj) * p.G + g] = r;
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8 * buf);
        }
        if (EMODE == 4) {   // fixed-order butterfly over the lanes, one slot per (CTA, epilogue warp)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
            if (lane == 0) p.part[blockIdx.x * 8 + (warp - 2)] = sq;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_free512(tmem);
}

// loss = (sum of the per-warp partial sums, fixed order) * inv_n
__global__ void prior_loss_finish_kernel(const double* __restrict__ part, int n, double inv_n, float* __restrict__ loss) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < n; ++i) t += part[i];
        *loss = (float)(t * inv_n);
    }
}

// PHX_TC_PROF=1: 16 device counters, printed (and reset) by phx_tc_prof_dump()
unsigned long long* g_prof = nullptr;
unsigned long long* phx_tc_prof_buffer() {
    static int on = -1;
    if (on < 0) {
        const char* e = getenv("PHX_TC_PROF");
        on = (e && atoi(e)) ? 1 : 0;
        if (on) {
            cudaMalloc((void**)&g_prof, 32 * sizeof(unsigned long long));
            cudaMemset(g_prof, 0, 32 * sizeof(unsigned long long));
        }
    }
    return g_prof;
}

// ---- cached Hill activations of a CONSTANT input ------------------------------------------------------------------------
// The prior batch of training_step (train_insilico.py:134, 208: batch_for_prior, drawn once before the epoch loop) is the
// same [10 000, G] matrix at every optimiser step, yet the branch contraction of the forward and the Ws_bar | Wp_bar
// contraction of the backward each re-evaluate soft-sign / log1p of all its elements -- and those kernels are bound by
// exactly that producer work.  phx_hill_planes evaluates s(x) and l(x) ONCE (the producers' own device functions: the
// same bits); while a cache entry is set (phx_hill_cache_set, scoped by the caller around its launches) a mode-0 branch
// launch whose source is that x runs as a mode-1 launch over the planes (sums CTAs read s, prods CTAs read l).
__global__ void hill_planes_kernel(size_t n, const float* __restrict__ x, float* __restrict__ sp, float* __restrict__ lp) {
    const size_t step = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const float y = x[i];
        sp[i] = hill_s(y);
        lp[i] = hill_l(y);
    }
}
struct HillCache {
    const float* x;
    size_t n;
    const float* s;
    const float* l;
};
HillCache g_hill = {nullptr, 0, nullptr, nullptr};
std::mutex g_hill_mu;

// PHX_TC_UV_FUSED=0 selects the two-pass form of the state cotangent (u stored, then v + epilogue)
int uv_fused() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("PHX_TC_UV_FUSED");
        v = e ? atoi(e) : 0;
    }
    return v;
}

// EXPERIMENTAL, off by default (PHX_TC_PAIR=1 or phx_tc_set_pair): the branch-type contractions as CTA pairs (tcgen05
// cta_group::2).  Bit-identical results; measured SLOWER on B200 than the single-CTA kernel (DESIGN.md section 7).
// A operand of the branch-type contractions in tensor memory (tc_branch_kernel<.., TS = 1>): default on, PHX_TC_TS=0 keeps
// the shared-memory A tiles (bit-identical results either way: same operands, same MMA order).
int ts_mode() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("PHX_TC_TS");
        v = e ? atoi(e) : 1;
    }
    return v;
}
// columns of the A ring in tensor memory: the spare columns behind the chunk accumulator [0, Hn) and behind the running sum
// [256, 256 + Hn); a stage is 16 (hi) + 16 (lo) columns.  Returns the ring depth (0: no room, use the TS = 0 kernel).
int ts_plan(int Hn, int (&hi)[4], int (&lo)[4]) {
    const int W = 256 - Hn, n1 = W / 32;
    int n = 0;
    for (int r = 0; r < 2; ++r)
        for (int i = 0; i < n1 && n < 4; ++i) {
            hi[n] = r * 256 + Hn + 32 * i;
            lo[n] = hi[n] + 16;
            ++n;
        }
    if (W % 32 >= 16 && n < 4) {
        hi[n] = Hn + 32 * n1;
        lo[n] = 256 + Hn + 32 * n1;
        ++n;
    }
    return n >= 2 ? n : 0;
}

int g_pair = -1;
int pair_mode() {
    if (g_pair < 0) {
        const char* e = getenv("PHX_TC_PAIR");
        g_pair = e ? atoi(e) : 0;
    }
    return g_pair;
}

}  // namespace

int phx_tc_pack_launch(int G, int H, const PhxPacked& w, cudaStream_t st) {
    const int Hp = phx_Hp(H), Hn = phx_tc_Hn(H);
    tc_pack_kernel<<<PHX_TC_SMS * 8, 256, 0, st>>>(G, H, Hp, 2 * Hp, Hn, reinterpret_cast<const float*>(w.W1),
                                                    reinterpret_cast<const float*>(w.WA), const_cast<float*>(w.w1img),
                                                    const_cast<float*>(w.waimg), const_cast<float*>(w.watimg),
                                                    const_cast<float*>(w.w1kimg));
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("tc_pack launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

namespace {

struct TcScratch {
    float* spart;    // partial-sum slots of the branch-type contraction
    float* spimg;    // operand image of [S|P]
    float* gsimg;    // operand image of gSP
    float* sptimg;   // [S|P] as the B operand of the K = batch contractions
    float* gstimg;   // gSP likewise
    float* gslots;   // partial-sum slots of the K = batch contractions
};
TcScratch carve(int G, int H, int B, float* tcws) {
    const int Hn = phx_tc_Hn(H), Bpad = phx_round_up(B, 256);
    const PhxTcBranchPlan pl = phx_tc_branch_plan(G, B);
    TcScratch sc;
    sc.spart = reinterpret_cast<float*>(((uintptr_t)tcws + 127) & ~(uintptr_t)127);
    sc.spimg = sc.spart + (size_t)pl.slots * Bpad * 2 * Hn;
    sc.gsimg = sc.spimg + phx_tc_spimg_floats(H, B);
    sc.sptimg = sc.gsimg + phx_tc_spimg_floats(H, B);
    sc.gstimg = sc.sptimg + phx_tc_timg_floats(H, B);
    sc.gslots = sc.gstimg + phx_tc_timg_floats(H, B);
    return sc;
}

void set_attrs() {
    static bool done = false;
    if (done) return;
    cudaFuncSetAttribute(tc_branch_kernel<0, 0, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<1, 0, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<0, 1, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<1, 1, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<0, 0, 1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<1, 0, 1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<0, 1, 1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<1, 1, 1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<0, 0, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<1, 0, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<0, 1, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_branch_kernel<1, 1, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_joint_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_joint_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_joint_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_joint_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_joint_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    cudaFuncSetAttribute(tc_joint_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, PHX_SMEM_LIMIT);
    done = true;
}

// Launch configuration of one branch-type contraction, decided on the host: the K split (with the equal-cost split of
// mode 1), the substitution of cached Hill planes, where the A operand lives (a ring of `a_stages` stages in tensor memory,
// 0: shared-memory tiles) and the depth S1 of the shared-memory pipeline.  launch_branch_mma and phx_tc_launch_describe
// both take it from here, so what the library reports is what it launches.
struct BranchConfig {
    PhxTcBranchPlan pl;
    int mode;                   // after the cached-Hill substitution (mode 0 over cached planes runs as mode 1)
    bool hill_cached;
    int pair, a_stages, a_hi_col[4], a_lo_col[4];
    size_t stage1, staging, running;
    int S1;
};
int branch_config(int mode, int trans, int G, int H, int B, bool hill_cached, BranchConfig& c) {
    const int Hn = phx_tc_Hn(H);
    const int Kdim = trans ? B : G, Mdim = trans ? G : B;
    PhxTcBranchPlan pl = phx_tc_branch_plan(Kdim, Mdim);
    if (mode == 1) {   // both halves cost the same: equal K ranges (the planner's equal-cost split)
        pl.per_p = pl.per_s = pl.per_e;
        pl.ks_p = pl.ks_s = pl.ks_e;
    }
    c.hill_cached = mode == 0 && hill_cached;
    if (c.hill_cached) {   // cached Hill activations: a mode-1 launch over the two planes
        mode = 1;
        pl.per_p = pl.per_s = pl.per_e;
        pl.ks_p = pl.ks_s = pl.ks_e;
    }
    c.pl = pl;
    c.mode = mode;
    c.pair = pair_mode();
    for (int i = 0; i < 4; ++i) c.a_hi_col[i] = c.a_lo_col[i] = 0;
    const int chunk = phx_tc_chunk();
    const int Hb = c.pair ? Hn / 2 : Hn;   // B rows staged per CTA
    c.a_stages = (!c.pair && ts_mode()) ? ts_plan(Hn, c.a_hi_col, c.a_lo_col) : 0;
    int ts = c.a_stages > 0;
    size_t stage1 = (size_t)2 * Hb * BK * 4;
    // TS: single-buffered staging (4 lane quarters x 32 rows) and the running sum [Hn / 4][128] float4 behind it
    size_t staging = trans ? 0 : (size_t)4 * 32 * (K1_PF * BK + 4) * sizeof(float);
    size_t running = (size_t)Hn * 128 * sizeof(float);
    if (ts && (PHX_SMEM_LIMIT - 256 - staging - running) / stage1 < 2) ts = 0;   // no room for a B ring: shared-memory A
    // the tensor-memory form pays off through the overlapped chunk folds: a CTA needs at least two chunks of K (measured:
    // 3 551 x 120 x 1 024, one chunk per CTA, is 3-15 % slower with it; 20 000 x 200 x 4 096 is 8 % faster)
    if (ts && (pl.per_p > pl.per_s ? pl.per_p : pl.per_s) < 2 * chunk && !getenv("PHX_TC_TS_FORCE")) ts = 0;
    if (!ts) {
        c.a_stages = 0;
        stage1 += K1_A_BYTES;
        staging = trans ? 0 : (size_t)K1_PWARPS * 2 * 8 * (K1_PF * BK + 4) * sizeof(float);
        running = 0;
    }
    int S1 = (int)((PHX_SMEM_LIMIT - 256 - staging - running) / stage1);
    if (S1 > 6) S1 = 6;
    if (const char* e = getenv("PHX_TC_STAGES")) {   // experiment
        int v = atoi(e);
        if (v >= 1 && v < S1) S1 = v;
    }
    c.stage1 = stage1; c.staging = staging; c.running = running; c.S1 = S1;
    if (S1 < 1) {
        phx_set_error("tc branch kernel: stage of %zu bytes does not fit", stage1);
        return PHX_ERR_UNSUPPORTED;
    }
    return PHX_OK;
}

// the branch-type contraction itself: part[slot][Mpad][2*Hn] = A(src) x image^T.  trans = 0: M = batch rows, K = genes;
// trans = 1: M = genes, K = batch rows.  Returns the plan used (slot counts per half) through *plan.
int launch_branch_mma(int mode, int trans, int G, int H, int B, int nterms, const float* src, const float* ascale,
                      const float* bimg, float* spart, PhxTcBranchPlan* plan, cudaStream_t st) {
    const int Hn = phx_tc_Hn(H);
    const int Kdim = trans ? B : G, Mdim = trans ? G : B;
    const float* src2 = nullptr;
    bool hill_cached = false;
    if (mode == 0) {   // cached Hill activations of this very matrix
        std::lock_guard<std::mutex> lk(g_hill_mu);
        if (g_hill.x == src && g_hill.n == (size_t)G * B && g_hill.s && g_hill.l) {
            hill_cached = true;
            src = g_hill.s;
            src2 = g_hill.l;
            ascale = nullptr;
        }
    }
    BranchConfig cf;
    const int rc = branch_config(mode, trans, G, H, B, hill_cached, cf);
    const PhxTcBranchPlan& pl = cf.pl;
    *plan = pl;
    if (rc != PHX_OK) return rc;
    mode = cf.mode;
    BranchParams bp;
    const int pair = cf.pair;
    bp.G = Kdim; bp.B = Mdim; bp.Bpad = phx_round_up(pl.mtiles, 2) * 128; bp.Hn = Hn; bp.KB1 = phx_tc_KB1(Kdim); bp.chunk = phx_tc_chunk();
    bp.ld = G;
    bp.nterms = nterms; bp.mode = mode; bp.ascale = ascale;
    bp.mtiles = pl.mtiles; bp.ks_p = pl.ks_p; bp.per_p = pl.per_p; bp.ks_s = pl.ks_s; bp.per_s = pl.per_s;
    const int Hb = pair ? Hn / 2 : Hn;   // B rows staged per CTA
#if PHX_TC_BRANCH_SW64
    bp.a_lbo = 16; bp.a_sbo = 512; bp.b_lbo = 16; bp.b_sbo = 512;   // 8-row x 64-byte atoms; LBO unused when swizzled
    bp.a_kadv = 32; bp.b_kadv = 32;                                  // K = 8 floats further inside the 64-byte row
#else
    bp.a_lbo = 16 * 128; bp.a_sbo = 128; bp.b_lbo = (unsigned)(Hb / 8) * 128; bp.b_sbo = 128;
    bp.a_kadv = 2 * bp.a_lbo; bp.b_kadv = 2 * bp.b_lbo;
#endif
    bp.y = src; bp.y2 = src2; bp.w1img = bimg; bp.spart = spart;
    bp.prof = phx_tc_prof_buffer();
    bp.a_stages = cf.a_stages;
    for (int i = 0; i < 4; ++i) {
        bp.a_hi_col[i] = cf.a_hi_col[i];
        bp.a_lo_col[i] = cf.a_lo_col[i];
    }
    const int ts = cf.a_stages > 0;
    const size_t stage1 = cf.stage1, staging = cf.staging, running = cf.running;
    bp.stg_bytes = (unsigned)staging;
    const int S1 = cf.S1;
    bp.stages = S1;
    set_attrs();
    const size_t smem1 = (size_t)S1 * stage1 + 256 + staging + running;
    if (!pair) {
        const dim3 grid1(pl.mtiles * (pl.ks_p + pl.ks_s));
        if (ts) {
            if (!trans) {
                if (mode == 0) tc_branch_kernel<0, 0, 0, 1><<<grid1, K1_THREADS, smem1, st>>>(bp);
                else tc_branch_kernel<1, 0, 0, 1><<<grid1, K1_THREADS, smem1, st>>>(bp);
            } else {
                if (mode == 0) tc_branch_kernel<0, 1, 0, 1><<<grid1, K1_THREADS, smem1, st>>>(bp);
                else tc_branch_kernel<1, 1, 0, 1><<<grid1, K1_THREADS, smem1, st>>>(bp);
            }
        } else if (!trans) {
            if (mode == 0) tc_branch_kernel<0, 0, 0, 0><<<grid1, K1_THREADS, smem1, st>>>(bp);
            else tc_branch_kernel<1, 0, 0, 0><<<grid1, K1_THREADS, smem1, st>>>(bp);
        } else {
            if (mode == 0) tc_branch_kernel<0, 1, 0, 0><<<grid1, K1_THREADS, smem1, st>>>(bp);
            else tc_branch_kernel<1, 1, 0, 0><<<grid1, K1_THREADS, smem1, st>>>(bp);
        }
        return PHX_OK;
    }
    // CTA pairs: clusters of two along x
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * ((pl.mtiles + 1) / 2) * (pl.ks_p + pl.ks_s));
    cfg.blockDim = dim3(K1_THREADS);
    cfg.dynamicSmemBytes = smem1;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t e;
    if (!trans) {
        e = mode == 0 ? cudaLaunchKernelEx(&cfg, tc_branch_kernel<0, 0, 1, 0>, bp)
                      : cudaLaunchKernelEx(&cfg, tc_branch_kernel<1, 0, 1, 0>, bp);
    } else {
        e = mode == 0 ? cudaLaunchKernelEx(&cfg, tc_branch_kernel<0, 1, 1, 0>, bp)
                      : cudaLaunchKernelEx(&cfg, tc_branch_kernel<1, 1, 1, 0>, bp);
    }
    if (e != cudaSuccess) {
        phx_set_error("tc branch pair launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

// partial[B x 2Hn] = A(src) x image^T, then the finishing pass (mode 0: bias/exp -> [S|P]; mode 1: * Pr -> gSP)
int launch_branch(int mode, int G, int H, int B, int nterms, const float* src, const float* ascale, const float* bimg,
                  const float* fin_aux, float* out_plain, float* out_img, float* out_timg, float* spart,
                  cudaStream_t st) {
    const int Hp = phx_Hp(H), K2 = 2 * Hp, Hn = phx_tc_Hn(H), Bpad = phx_round_up(B, 256);
    PhxTcBranchPlan pl;
    int rc = launch_branch_mma(mode, 0, G, H, B, nterms, src, ascale, bimg, spart, &pl, st);
    if (rc != PHX_OK) return rc;
    const size_t total = (size_t)phx_tc_BT(B) * 256 * (2 * Hn / 4);
    int blocks = (int)((total + 255) / 256);
    if (blocks > PHX_TC_SMS * 16) blocks = PHX_TC_SMS * 16;
    tc_spfinish_kernel<<<blocks, 256, 0, st>>>(B, Bpad, H, Hp, Hn, K2, pl.ks_s, pl.ks_p, mode, spart, fin_aux, out_plain,
                                               out_img, out_timg);
    return PHX_OK;
}

// out^T tiles = Aimg[genes x k-blocks kb_lo..kb_hi) x Bimg[batch rows]^T with the epilogue `emode`
int launch_joint(int G, int H, int B, int nterms, const float* aimg, const float* bimg, int kb_lo, int kb_hi, int emode,
                 int decay, float fscale, const float* y, const float* g, const float* relum, float* out,
                 cudaStream_t st, double* part = nullptr, const PhxRhsPost* post = nullptr) {
    JointParams jp;
    memset(&jp.post, 0, sizeof(jp.post));
    if (post) jp.post = *post;
    jp.G = G; jp.B = B; jp.KB2 = phx_tc_KB2(H); jp.GT = phx_tc_GT(G); jp.BT = phx_tc_BT(B); jp.nterms = nterms;
    jp.decay = decay; jp.fscale = fscale; jp.kb_lo = kb_lo; jp.kb_hi = kb_hi; jp.emode = emode;
    jp.a_lbo = 16 * 128; jp.a_sbo = 128; jp.b_lbo = 32 * 128; jp.b_sbo = 128;
    jp.a_kadv = 2 * jp.a_lbo; jp.b_kadv = 2 * jp.b_lbo;
    jp.waimg = aimg; jp.spimg = bimg; jp.y = y; jp.g = g; jp.relum = relum; jp.f = out; jp.part = part;
    const int ntiles = jp.GT * jp.BT;
    const int grid = ntiles < PHX_TC_SMS ? ntiles : PHX_TC_SMS;
    set_attrs();
    const size_t smem2 = (size_t)K2_STAGES * K2_STAGE_BYTES + 256;
    if (emode == 0) tc_joint_kernel<0><<<grid, K2_THREADS, smem2, st>>>(jp);
    else if (emode == 1) tc_joint_kernel<1><<<grid, K2_THREADS, smem2, st>>>(jp);
    else if (emode == 2) tc_joint_kernel<2><<<grid, K2_THREADS, smem2, st>>>(jp);
    else if (emode == 3) tc_joint_kernel<3><<<grid, K2_THREADS, smem2, st>>>(jp);
    else if (emode == 5) tc_joint_kernel<5><<<grid, K2_THREADS, smem2, st>>>(jp);
    else tc_joint_kernel<4><<<grid, K2_THREADS, smem2, st>>>(jp);
    return grid;
}

int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("%s launch: %s", what, cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

}  // namespace

// SP (plain [B][K2], bias/exp applied) and, if f != 0, f; tcws = scratch of phx_tc_scratch_floats(G, H, B) floats
int phx_tc_rhs_forward_launch(int G, int H, int B, const PhxPacked& w, const float* y, float* f, int decay,
                              float fscale, float* SP, float* tcws, cudaStream_t st, const PhxRhsPost* post) {
    const TcScratch sc = carve(G, H, B, tcws);
    const int nterms = (w.tc == 1) ? 1 : 3;
    const bool fused = post && post->mode != PHX_POST_NONE;
    if (fused && (!post->x0 || !post->out || post->nk < 0 || post->nk > 6 || (post->mode == PHX_POST_CHAIN && post->nk > 6) || (post->store_f && !f) ||
                  (post->mode >= PHX_POST_FX && post->nk > 3))) {
        phx_set_error("tc rhs_forward: malformed stage-algebra record");
        return PHX_ERR_INVALID;
    }
    int rc = launch_branch(0, G, H, B, nterms, y, nullptr, w.w1img, w.bias, SP, sc.spimg, sc.sptimg, sc.spart, st);
    if (rc != PHX_OK) return rc;
    if (fused)
        launch_joint(G, H, B, nterms, w.waimg, sc.spimg, 0, phx_tc_KB2(H), 5, decay, fscale, y, nullptr, w.relum, f, st,
                     nullptr, post);
    else if (f)
        launch_joint(G, H, B, nterms, w.waimg, sc.spimg, 0, phx_tc_KB2(H), 0, decay, fscale, y, nullptr, w.relum, f, st);
    return check_launch("tc rhs_forward");
}

int phx_tc_vjp_state_launch(int G, int H, int B, const PhxPacked& w, const float* y, const float* g, int decay,
                            float* ybar, const float* SP, float* GS, float* J, float* tcws, cudaStream_t st) {
    const TcScratch sc = carve(G, H, B, tcws);
    const int nterms = (w.tc == 1) ? 1 : 3, KB2 = phx_tc_KB2(H);
    // gSP = (g relu(m)) WA over the genes, prods half scaled by Pr  (exp / Linear backward, odenet.py:86-89)
    int rc = launch_branch(1, G, H, B, nterms, g, decay ? w.relum : nullptr, w.watimg, SP, GS, sc.gsimg, sc.gstimg,
                           sc.spart, st);
    if (rc != PHX_OK) return rc;
    if (ybar) {
        // u = gS Ws (k-blocks of the sums half) and v = gP Wp (prods half) in the two halves of tensor memory, the
        // soft-sign / log1p backward in the epilogue.  (Two-pass form: EMODE 1 stores u, EMODE 2 finishes.)
        if (uv_fused()) {
            launch_joint(G, H, B, nterms, w.w1kimg, sc.gsimg, 0, KB2, 3, decay, 1.f, y, g, w.relum, ybar, st);
        } else {
            launch_joint(G, H, B, nterms, w.w1kimg, sc.gsimg, 0, KB2 / 2, 1, 0, 1.f, nullptr, nullptr, w.relum, ybar, st);
            launch_joint(G, H, B, nterms, w.w1kimg, sc.gsimg, KB2 / 2, KB2, 2, decay, 1.f, y, g, w.relum, ybar, st);
        }
    }
    if (J) launch_joint(G, H, B, nterms, w.waimg, sc.spimg, 0, KB2, 0, 0, 1.f, y, nullptr, w.relum, J, st);
    return check_launch("tc vjp_state");
}

// after phx_tc_rhs_forward_launch on the same scratch: f = fscale * (decay ? relu(m) * (J - y) : J) from the [S|P] image
int phx_tc_joint_launch(int G, int H, int B, const PhxPacked& w, const float* y, float* f, int decay, float fscale,
                        float* tcws, cudaStream_t st) {
    const TcScratch sc = carve(G, H, B, tcws);
    launch_joint(G, H, B, (w.tc == 1) ? 1 : 3, w.waimg, sc.spimg, 0, phx_tc_KB2(H), 0, decay, fscale, y, nullptr, w.relum,
                 f, st);
    return check_launch("tc joint");
}

// after phx_tc_rhs_forward_launch and phx_tc_vjp_state_launch on the same scratch: the K = batch contractions
//   Wa_bar[g][k] = sum_b (g relu(m))[b][g] [S|P][b][k],  Ws_bar[h][g] = sum_b gS[b][h] s[b][g],  Wp_bar likewise with l
// (Linear backward, odenet.py:86-89), written / accumulated into the flat gradient vector.
int phx_tc_vjp_params_launch(int G, int H, int B, const PhxPacked& w, const float* y, const float* g, int decay,
                             float* grads, int accumulate, float* tcws, cudaStream_t st, int pmask,
                             const PhxGradOff* goff) {
    const TcScratch sc = carve(G, H, B, tcws);
    const int nterms = (w.tc == 1) ? 1 : 3, Hn = phx_tc_Hn(H);
    const PhxGradOff off = goff ? *goff : phx_grad_offsets(G, H);
    const size_t total = (size_t)G * 2 * H;
    int blocks = (int)((total + 255) / 256);
    if (blocks > PHX_TC_SMS * 16) blocks = PHX_TC_SMS * 16;
    PhxTcBranchPlan pl;
    int rc;
    if (pmask & PHX_P_WA) {
        rc = launch_branch_mma(1, 1, G, H, B, nterms, g, decay ? w.relum : nullptr, sc.sptimg, sc.gslots, &pl, st);
        if (rc != PHX_OK) return rc;
        tc_gradfinish_kernel<<<blocks, 256, 0, st>>>(1, G, phx_round_up(pl.mtiles, 2) * 128, H, Hn, pl.ks_s, pl.ks_p,
                                                     sc.gslots, grads + off.Wa, nullptr, accumulate);
    }
    // Ws and Wp come out of one launch with one K split (phx_tc_branch_plan): with one of them frozen the launch and
    // its split stay as they are and only the kept half is written, so the kept half is bit-identical to the
    // all-parameter call
    if (pmask & (PHX_P_WS | PHX_P_WP)) {
        rc = launch_branch_mma(0, 1, G, H, B, nterms, y, nullptr, sc.gstimg, sc.gslots, &pl, st);
        if (rc != PHX_OK) return rc;
        tc_gradfinish_kernel<<<blocks, 256, 0, st>>>(0, G, phx_round_up(pl.mtiles, 2) * 128, H, Hn, pl.ks_s, pl.ks_p,
                                                     sc.gslots, (pmask & PHX_P_WS) ? grads + off.Ws : nullptr,
                                                     (pmask & PHX_P_WP) ? grads + off.Wp : nullptr, accumulate);
    }
    return check_launch("tc vjp_params");
}

// Prior-constrained loss term of training_step (train_insilico.py:134-135) on the tensor cores, fused: [S|P] from x, then
// the joint contraction whose epilogue compares with prior_grad on the fly -- gcot = scale * (J - prior_grad) is the
// cotangent the backward needs, loss = mean((J - prior_grad)^2); J itself never goes to memory.  The scratch keeps
// [S|P] and its images for the parameter contractions of the backward (phx_rhs_vjp with PHX_VJP_REUSE_FORWARD).
// part: >= 8 * PHX_TC_SMS doubles.
int phx_tc_prior_loss_launch(int G, int H, int B, const PhxPacked& w, const float* x, const float* prior_grad, float scale,
                             float* gcot, float* loss, float* SP, double* part, float* tcws, cudaStream_t st) {
    const TcScratch sc = carve(G, H, B, tcws);
    const int nterms = (w.tc == 1) ? 1 : 3;
    int rc = launch_branch(0, G, H, B, nterms, x, nullptr, w.w1img, w.bias, SP, sc.spimg, sc.sptimg, sc.spart, st);
    if (rc != PHX_OK) return rc;
    const int grid = launch_joint(G, H, B, nterms, w.waimg, sc.spimg, 0, phx_tc_KB2(H), 4, 0, scale, nullptr, prior_grad,
                                  w.relum, gcot, st, part);
    prior_loss_finish_kernel<<<1, 32, 0, st>>>(part, grid * 8, 1.0 / ((double)B * (double)G), loss);
    return check_launch("tc prior_loss");
}

extern "C" void phx_tc_set_pair(int on) { g_pair = on ? 1 : 0; }

// contraction (bits 0-1): 0 forward [S|P], 1 gSP, 2 Ws_bar | Wp_bar, 3 Wa_bar; bit 2: the activation operand is a pair of
// cached Hill planes (contractions 0 and 2 only).  Same decision as the launch, under the same environment and pair mode.
extern "C" int phx_tc_launch_describe(int contraction, int G, int H, int B, int32_t out[8]) {
    const int c = contraction & 3;
    const bool cached = (contraction & 4) != 0;
    if (!out || contraction < 0 || contraction > 7 || (cached && (c & 1)) || G < 1 || H < 1 || B < 1 ||
        phx_tc_Hn(H) > PHX_TC_MAX_HN) {
        phx_set_error("tc_launch_describe: invalid argument");
        return PHX_ERR_INVALID;
    }
    BranchConfig cf;
    const int rc = branch_config(c & 1, c >> 1, G, H, B, cached, cf);
    if (rc != PHX_OK) return rc;
    out[0] = cf.pl.mtiles; out[1] = cf.pl.ks_p; out[2] = cf.pl.per_p; out[3] = cf.pl.ks_s; out[4] = cf.pl.per_s;
    out[5] = cf.pl.slots; out[6] = cf.a_stages; out[7] = cf.S1;
    return PHX_OK;
}

extern "C" void phx_tc_prof_dump(void) {
    if (!g_prof) return;
    unsigned long long h[32];
    cudaMemcpy(h, g_prof, sizeof(h), cudaMemcpyDeviceToHost);
    cudaMemset(g_prof, 0, sizeof(h));
    for (int br = 0; br < 2; ++br) {
        const unsigned long long* q = h + 8 * br;
        const double n = q[3] ? (double)q[3] : 1.0;
        printf("tc_branch %s: k-blocks %llu | MMA thread cycles/k-block: total %.0f wait_full %.0f wait_drained %.0f | "
               "producer warp 0: total %.0f wait_empty %.0f drain %.0f\n",
               br ? "prods" : "sums", q[3], q[0] / n, q[1] / n, q[2] / n, q[4] / n, q[5] / n, q[6] / n);
        const unsigned long long* r = h + 16 + 8 * br;
        printf("          producer warp 0 phases / k-block: load+stage %.0f  convert %.0f  store+signal %.0f\n", r[0] / n,
               r[1] / n, r[2] / n);
    }
}

extern "C" int phx_hill_planes(phx_ctx* ctx, size_t n, const float* x, float* s_plane, float* l_plane, void* stream) {
    if (!ctx || !x || !s_plane || !l_plane || n == 0) {
        phx_set_error("hill_planes: invalid argument");
        return PHX_ERR_INVALID;
    }
    PhxDevGuard dev_guard(ctx);
    size_t blocks = (n + 255) / 256;
    if (blocks > (size_t)PHX_TC_SMS * 16) blocks = (size_t)PHX_TC_SMS * 16;
    hill_planes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(n, x, s_plane, l_plane);
    return check_launch("hill_planes");
}
extern "C" int phx_hill_cache_set(phx_ctx* ctx, const float* x, size_t n, const float* s_plane, const float* l_plane) {
    (void)ctx;
    std::lock_guard<std::mutex> lk(g_hill_mu);
    g_hill.x = (s_plane && l_plane) ? x : nullptr;
    g_hill.n = n;
    g_hill.s = s_plane;
    g_hill.l = l_plane;
    return PHX_OK;
}
