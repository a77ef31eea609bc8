// "Rows" solver kernels for sm_100a: up to PHX_ROWS_MAX INDEPENDENT one-row odeint problems (the samples of a
// training step, train_insilico.py:128-130) advance in lock-step as the rows of ONE persistent cooperative launch, every
// row with its own times, its own dopri5 step controller, its own status record and its own parameter cotangents.
//
// Why: the RHS is autonomous, so a stage evaluation of row b only needs row b's state -- but every row needs the same
// weights.  One pass over the CTA's weight slices (W1 in shared memory, WA in shared or TENSOR memory) and one
// inter-CTA exchange therefore serve all rows; rows that finish early are masked.  The arithmetic of a row does not
// depend on which row it is or on how many rows run beside it, so a row's results are bit-identical to a launch holding
// that problem alone (tests/test_gpu_rows.py).
//
// Thread mappings (512 threads = 16 warps = nqw quad-warps x ngg gene groups; a "quad" is one float4 of the K2-long rows):
//   pass 1  (WA)  thread = (quad q, gene group): J partials for the group's genes (reduced over the quads by a
//                 register-transposing butterfly: 16 shuffles per 4 genes x 4 rows) and, in the adjoint, the column sums
//                 gSP[q] += gj[g] * WA[g][q] in registers -- both from ONE read of the slice;
//   pass A  (W1)  thread = (quad q, gene group): branch pre-activations of the NEXT stage input;
//   pass 2  (W1)  thread = (gene, k-chunk c of 4): u = W1[g][:Hp].gS, v = W1[g][Hp:].gLP, two shuffle steps; lane c then
//                 owns row b = c of that gene;
//   theta   the parameter cotangents live in the PACKED layout (W1bar[G][K2], WAbar[G][K2]: every element of a CTA's
//           slice is (per-gene factor) x (per-quad factor)); thread = (quad, gene group) holds the quad factors of the six
//           stage slots in registers (read from tensor memory) and streams 16-byte stores.
// Per-stage factor tables: per-gene ones in shared memory, K2-long ones (S|Pr and gS|gLP per stage and row) in tensor
// memory next to the WA slice (lane = quad).
#pragma once
#include "phx_resident.cuh"

namespace {

constexpr int RM = PHX_ROWS_MAX;
constexpr int NFS = PHX_ROWS_NFS;
static_assert(RM == 4, "lane c <-> row b pairing of pass 2 and the [gene][4] float4 layouts assume 4 rows");

struct RowCtl {
    double tcur, tprev, dt, t_end;
    float cb[6][6];
    float cerr[7], cmid[7], xs[4];
    float dtf, h0, d1;
    int valid, done, accept, last, nonfinite_prev, code;
    int n_acc, n_rej, n_rhs, n_log, n_steps_interval, next_out;
    int slot[7];    // physical state slot (K / KY / KA) of logical stage q; FSAL swaps 0 <-> 6
    int fslot[7];   // physical factor slot of logical stage q (-1: the stage keeps no factors)
    int cur, theta_zero, pend, spec_done;
    int stepping;   // fixed grid: the row takes the current step (0: past its last step -- or its interval's last)
    int gj0, gj1;   // fixed grid, forward: the output times [gj0, gj1) the current step writes
};
struct RowsCtl {
    RowCtl r[RM];
    int all_done, any_pending, spec_valid, spec_pass, redo;
};
static_assert(sizeof(RowsCtl) <= PHX_RCTL_BYTES, "PHX_RCTL_BYTES too small");

__device__ __forceinline__ double tget_rows(const ResParams& p, int q, int i) {
    return (p.T * p.ntot <= PHX_T_INLINE) ? p.t_small[q * p.T + i] : p.t[q * p.T + i];
}

__device__ __forceinline__ float4 fma4s(const float4& w, float c, float4 a) {
    a.x = fmaf(w.x, c, a.x);
    a.y = fmaf(w.y, c, a.y);
    a.z = fmaf(w.z, c, a.z);
    a.w = fmaf(w.w, c, a.w);
    return a;
}
__device__ __forceinline__ float4 mul4(const float4& a, const float4& b) {
    return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w);
}
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float comp4(const float4& v, int e) { return e == 0 ? v.x : (e == 1 ? v.y : (e == 2 ? v.z : v.w)); }

// ---- tensor memory: 32x32b accesses of 4 / 16 / 24 consecutive columns (load + wait in one statement) --------------------
__device__ __forceinline__ uint32_t tm_quarter(uint32_t base) { return base + ((uint32_t)(32 * ((threadIdx.x >> 5) & 3)) << 16); }
__device__ __forceinline__ void tm_st4(uint32_t taddr, const float4& v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(__float_as_uint(v.x)),
                 "r"(__float_as_uint(v.y)), "r"(__float_as_uint(v.z)), "r"(__float_as_uint(v.w))
                 : "memory");
}
__device__ __forceinline__ void tm_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tm_ld4(uint32_t taddr, float4& v) {
    uint32_t a, b, c, d;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];\n\ttcgen05.wait::ld.sync.aligned;"
                 : "=r"(a), "=r"(b), "=r"(c), "=r"(d)
                 : "r"(taddr)
                 : "memory");
    v = make_float4(__uint_as_float(a), __uint_as_float(b), __uint_as_float(c), __uint_as_float(d));
}
__device__ __forceinline__ void tm_ld16(uint32_t taddr, float4 (&w)[4]) {
    uint32_t u[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
          "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
        : "r"(taddr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 4; ++i)
        w[i] = make_float4(__uint_as_float(u[4 * i]), __uint_as_float(u[4 * i + 1]), __uint_as_float(u[4 * i + 2]),
                           __uint_as_float(u[4 * i + 3]));
}
__device__ __forceinline__ void tm_st16(uint32_t taddr, const float4 (&w)[4]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(__float_as_uint(w[0].x)), "r"(__float_as_uint(w[0].y)), "r"(__float_as_uint(w[0].z)), "r"(__float_as_uint(w[0].w)),
        "r"(__float_as_uint(w[1].x)), "r"(__float_as_uint(w[1].y)), "r"(__float_as_uint(w[1].z)), "r"(__float_as_uint(w[1].w)),
        "r"(__float_as_uint(w[2].x)), "r"(__float_as_uint(w[2].y)), "r"(__float_as_uint(w[2].z)), "r"(__float_as_uint(w[2].w)),
        "r"(__float_as_uint(w[3].x)), "r"(__float_as_uint(w[3].y)), "r"(__float_as_uint(w[3].z)), "r"(__float_as_uint(w[3].w))
        : "memory");
}

// ---- the kernel context ---------------------------------------------------------------------------------------------------
struct RowsView {
    const ResParams& p;
    Smem& s;
    int warp, lane, qw, gg, q;
    bool qok;
    uint32_t tq;   // tensor-memory base address of this warp's lane quarter
    __device__ __forceinline__ RowsView(const ResParams& pp, Smem& ss) : p(pp), s(ss) {
        warp = threadIdx.x >> 5;
        lane = threadIdx.x & 31;
        qw = warp % p.nqw;
        gg = warp / p.nqw;
        q = 32 * qw + lane;
        qok = q < p.K2q;
        tq = 0u;
    }
    __device__ __forceinline__ RowsCtl* rc() const { return s.at<RowsCtl>(p.so.rctl); }
    __device__ __forceinline__ float* st(int i) const { return s.at<float>(p.so.st) + (size_t)i * RM * p.gpc; }
    __device__ __forceinline__ float* jred() const { return s.at<float>(p.so.jred); }
    __device__ __forceinline__ float* actL() const { return s.at<float>(p.so.actL); }
    __device__ __forceinline__ float* ysf() const { return s.at<float>(p.so.ysf); }       // [gpc][RM][NFS] (fgj, fm too)
    __device__ __forceinline__ float* fgj() const { return s.at<float>(p.so.FGJ); }
    __device__ __forceinline__ float* fm() const { return s.at<float>(p.so.FM); }
    __device__ __forceinline__ const float4* w1() const { return s.at<float4>(p.so.w1r); }
    // K2-long factor tables in tensor memory, row by row: row b (b < p.rows) owns 2 x NFS slots of 4 columns, so the
    // rows of a pass take the 2 * NFS * 4 * rows columns phx_rows_plan budgets beside the WA slice
    __device__ __forceinline__ uint32_t col_fsp(int fs, int b) const { return tq + (uint32_t)(p.tm_fac + (b * 2 * NFS + fs) * 4); }
    __device__ __forceinline__ uint32_t col_fg(int fs, int b) const { return tq + (uint32_t)(p.tm_fac + (b * 2 * NFS + NFS + fs) * 4); }
};

// one-time staging: constants, the W1 slice (rows padded to w1_stride float4), the WA slice (shared or tensor memory)
__device__ __forceinline__ void rows_prologue(const ResParams& p, Smem& s, RowsView& v, int w1_stride_q) {
    Xchg& x = s.x;
    s.pf.init(p.prof, reinterpret_cast<long long*>(smem_raw + p.so.ctrl + 512));
    x.ep = __ldcg(p.ll.epoch);
    x.ny = x.nd = 0;
    s.rg.par = 0;
    s.rg.pre = -1;
    const int n_loc = s.n_loc, g_lo = s.g_lo;
    for (int k = threadIdx.x; k < p.K2; k += THREADS) s.bias()[k] = p.w.bias[k];
    for (int j = threadIdx.x; j < p.gpc; j += THREADS) {
        s.relum()[j] = j < n_loc ? p.w.relum[g_lo + j] : 0.f;
        s.maskm()[j] = j < n_loc ? p.w.maskm[g_lo + j] : 0.f;
    }
    const unsigned bar = smem_u32(s.at<unsigned long long>(p.so.resbar));
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const unsigned row_bytes = (unsigned)p.K2q * 16u;
        const unsigned bytes = (unsigned)n_loc * row_bytes;
        if (bytes) {
            const unsigned nres = 1u + (p.so.war != PHX_NONE ? 1u : 0u);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * nres) : "memory");
            if (w1_stride_q == p.K2q) {
                bulk_g2s(smem_u32(smem_raw + p.so.w1r), s.w1g(), bytes, bar);
            } else {
                for (int j = 0; j < n_loc; ++j)
                    bulk_g2s(smem_u32(smem_raw + p.so.w1r) + (unsigned)j * w1_stride_q * 16u, s.w1g() + (size_t)j * p.K2q,
                             row_bytes, bar);
            }
            if (p.so.war != PHX_NONE) bulk_g2s(smem_u32(smem_raw + p.so.war), s.wag(), bytes, bar);
        }
    }
    // tensor memory: all 512 columns (one CTA per SM)
    uint32_t* slot = s.at<uint32_t>(p.so.watm);
    if (v.warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    s.tmem = *slot;
    v.tq = tm_quarter(s.tmem);
    if (p.tm_wa > 0) {
        // WA slice -> tensor memory, lane = quad, column = 4 * local gene + element; pad genes / pad quads hold zeros.
        // nqw == 4 here: warp (qw, gg) fills the columns of its own gene group in its own lane quarter.
        const int j0 = v.gg * p.gpg;
        for (int jc = j0; jc < j0 + p.gpg; jc += 4) {
            float4 w[4];
#pragma unroll
            for (int gi = 0; gi < 4; ++gi)
                w[gi] = (v.qok && jc + gi < n_loc) ? __ldg(s.wag() + (size_t)(jc + gi) * p.K2q + v.q) : zero4();
            tm_st16(v.tq + (uint32_t)(4 * jc), w);
        }
        tm_wait_st();
    }
    if (n_loc > 0) mbar_wait(bar, 0u);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

__device__ __forceinline__ void rows_release(const ResParams& p, Smem& s) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if ((threadIdx.x >> 5) == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s.tmem), "r"(512u) : "memory");
}

// sum of the 16 per-lane values a[v] over the 32 lanes of the warp with a register-transposing butterfly: after the four
// halving rounds lane l holds value index (l >> 1) & 15 summed over 16 lanes, the last round completes it.  The
// summation tree of every index is the same balanced tree over the lanes (a + b == b + a bit for bit).
__device__ __forceinline__ float transpose_reduce16(float (&a)[16]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int h = 8, m = 16; h >= 1; h >>= 1, m >>= 1) {
        const bool up = (lane & m) != 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (i < h) {
                const float keep = up ? a[i + h] : a[i];
                const float send = up ? a[i] : a[i + h];
                a[i] = keep + __shfl_xor_sync(0xffffffffu, send, m);
            }
        }
    }
    return a[0] + __shfl_xor_sync(0xffffffffu, a[0], 1);
}

// out[b][K2] = sum over the gene groups of acc[b] (this thread's quad), fixed order: groups g and g + ngg/2 first, then
// 0 .. ngg/2 - 1.  Ends with a block barrier.
__device__ __forceinline__ void xgroup_reduce(const RowsView& v, float4 (&acc)[RM], float* out) {
    const ResParams& p = v.p;
    float4* red4 = v.s.at<float4>(p.so.red);
    float4* out4 = reinterpret_cast<float4*>(out);
    const int half = p.ngg >> 1, K2q = p.K2q;
    if (v.gg >= half && v.qok) {
#pragma unroll
        for (int b = 0; b < RM; ++b) red4[((v.gg - half) * RM + b) * K2q + v.q] = acc[b];
    }
    __syncthreads();
    if (v.gg < half && v.qok) {
#pragma unroll
        for (int b = 0; b < RM; ++b) {
            float4& r = red4[(v.gg * RM + b) * K2q + v.q];
            r = add4(acc[b], r);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < RM * K2q; i += THREADS) {
        float4 t = red4[i];
        for (int g = 1; g < half; ++g) t = add4(t, red4[g * RM * K2q + i]);
        out4[i] = t;
    }
    __syncthreads();
}

// Pass 1 over the WA slice at the current branch vector s.sp(): J partials of every (gene, row) -> jred[qw][gene][row]
// and (adjoint) gSP partial sums of this CTA -> gsp_out[row][K2].  Ends with a block barrier.
template <bool ADJ>
__device__ __forceinline__ void rows_pass1(const RowsView& v, float* gsp_out) {
    const ResParams& p = v.p;
    const Smem& s = v.s;
    const int K2q = p.K2q, n_loc = s.n_loc;
    const float4* sp4 = reinterpret_cast<const float4*>(s.sp());
    const float4* war4 = s.at<float4>(p.so.war);
    const float4* gj4 = s.at<float4>(p.so.gjb);
    float4 SPq[RM], accG[RM];
#pragma unroll
    for (int b = 0; b < RM; ++b) {
        SPq[b] = v.qok ? sp4[b * K2q + v.q] : zero4();
        accG[b] = zero4();
    }
    float* jr = v.jred() + (size_t)v.qw * RM * p.gpc;
    const int j0 = v.gg * p.gpg;
    const int jend = min(j0 + p.gpg, (n_loc + 3) & ~3);
    for (int jc = j0; jc < jend; jc += 4) {
        float4 w[4];
        if (p.tm_wa > 0) {
            tm_ld16(v.tq + (uint32_t)(4 * jc), w);
        } else {
#pragma unroll
            for (int gi = 0; gi < 4; ++gi) w[gi] = (v.qok && jc + gi < n_loc) ? war4[(size_t)(jc + gi) * K2q + v.q] : zero4();
        }
        float pj[16];
#pragma unroll
        for (int gi = 0; gi < 4; ++gi) {
#pragma unroll
            for (int b = 0; b < RM; ++b) pj[gi * RM + b] = dot4(w[gi], SPq[b]);
            if (ADJ) {
                const float4 gj = (jc + gi < p.gpc) ? gj4[jc + gi] : zero4();
                accG[0] = fma4s(w[gi], gj.x, accG[0]);
                accG[1] = fma4s(w[gi], gj.y, accG[1]);
                accG[2] = fma4s(w[gi], gj.z, accG[2]);
                accG[3] = fma4s(w[gi], gj.w, accG[3]);
            }
        }
        const float r = transpose_reduce16(pj);
        const int idx = (v.lane >> 1) & 15;   // = gi * RM + b
        if ((v.lane & 1) == 0 && jc + (idx >> 2) < p.gpc) jr[(jc + (idx >> 2)) * RM + (idx & 3)] = r;
    }
    if (ADJ) xgroup_reduce(v, accG, gsp_out);
    else __syncthreads();
}

// Pass A over the W1 slice: out[row][K2] (this CTA's partial) = sum_g act[row][g] * W1[g][:], act = s on the sums half,
// l on the prods half.  Ends with a block barrier.
__device__ __forceinline__ void rows_passA(const RowsView& v, const float* as, const float* al, float* out) {
    const ResParams& p = v.p;
    const int n_loc = v.s.n_loc, Hq = p.Hp >> 2;
    const float4* w1 = v.w1();
    const int ws = p.ring_rows;   // W1 row stride in float4 (rows kernels reuse this field)
    const float4* as4 = reinterpret_cast<const float4*>(as);
    const float4* al4 = reinterpret_cast<const float4*>(al);
    float4 acc[RM];
#pragma unroll
    for (int b = 0; b < RM; ++b) acc[b] = zero4();
    const int j0 = v.gg * p.gpg, jend = min(j0 + p.gpg, n_loc);
    if (v.qok) {
        const bool prods = v.q >= Hq;
#pragma unroll 4
        for (int j = j0; j < jend; ++j) {
            const float4 w = w1[(size_t)j * ws + v.q];
            const float4 a = prods ? al4[j] : as4[j];
            acc[0] = fma4s(w, a.x, acc[0]);
            acc[1] = fma4s(w, a.y, acc[1]);
            acc[2] = fma4s(w, a.z, acc[2]);
            acc[3] = fma4s(w, a.w, acc[3]);
        }
    }
    xgroup_reduce(v, acc, out);
}

// branch vector after the all-reduce: add bias, exponentiate the prods half (odenet.py:86-87); padded columns -> 0
__device__ __forceinline__ void rows_finalize_sp(const RowsView& v, const float* src, float* dst) {
    const ResParams& p = v.p;
    for (int i = threadIdx.x; i < RM * p.K2; i += THREADS) {
        const int k = i % p.K2;
        float x = src[i] + v.s.bias()[k];
        if (k >= p.Hp) x = (k - p.Hp < p.H) ? expf(x) : 0.f;
        dst[i] = x;
    }
    __syncthreads();
}

// per-row block sums: every thread carries N partials of ITS row (row = threadIdx.x & 3 in the element loops);
// out[row * N + i] (shared memory, doubles) receives the block totals.  Ends with a block barrier.
template <int N>
__device__ __forceinline__ void block_sum_rows(const RowsView& v, double (&val)[N], double* out) {
    double* rs = v.s.at<double>(v.p.so.rsum);   // [WARPS][RM][8]
#pragma unroll
    for (int i = 0; i < N; ++i) {
        double t = val[i];
        t += __shfl_xor_sync(0xffffffffu, t, 4);
        t += __shfl_xor_sync(0xffffffffu, t, 8);
        t += __shfl_xor_sync(0xffffffffu, t, 16);
        if (v.lane < RM) rs[(v.warp * RM + v.lane) * 8 + i] = t;
    }
    __syncthreads();
    if (threadIdx.x < RM * N) {
        const int b = threadIdx.x / N, i = threadIdx.x - b * N;
        double t = 0;
        for (int w = 0; w < WARPS; ++w) t += rs[(w * RM + b) * 8 + i];
        out[threadIdx.x] = t;
    }
    __syncthreads();
}

__device__ __forceinline__ void row_set_coeffs(RowCtl& c) {
    const float dtf = (float)c.dt;
    c.dtf = dtf;
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) c.cb[i][j] = (float)c_beta[i][j] * dtf;
    for (int j = 0; j < 7; ++j) {
        c.cerr[j] = dtf * (float)c_err[j];
        c.cmid[j] = dtf * (float)c_mid[j];
    }
}
__device__ __forceinline__ void row_set_interp_x(RowCtl& c, double t, double t0, double t1) {
    const double x = (t - t0) / (t1 - t0);
    double xp = x;
    c.xs[0] = (float)xp;
    xp = xp * x;
    c.xs[1] = (float)xp;
    xp = xp * x;
    c.xs[2] = (float)xp;
    xp = xp * x;
    c.xs[3] = (float)xp;
}
__device__ __forceinline__ void row_init(RowCtl& c, bool valid) {
    c.valid = valid;
    c.done = !valid;
    c.accept = c.last = c.nonfinite_prev = 0;
    c.code = PHX_ST_OK;
    c.n_acc = c.n_rej = c.n_rhs = c.n_log = c.n_steps_interval = 0;
    c.next_out = 1;
    c.tcur = c.tprev = c.dt = c.t_end = 0;
    for (int i = 0; i < 7; ++i) c.slot[i] = i;
    c.fslot[0] = 0;
    c.fslot[1] = -1;
    for (int i = 2; i < 7; ++i) c.fslot[i] = i - 1;
    c.cur = 0;
    c.theta_zero = 1;
    c.pend = 0;
    c.spec_done = 0;
}
__device__ __forceinline__ void row_log_step(const ResParams& p, RowCtl& c, int q, double t0, double dt, int accepted) {
    if (blockIdx.x == 0 && p.steplog && c.n_log < p.steplog_cap) {
        double* lg = p.steplog + ((size_t)q * p.steplog_cap + c.n_log) * 3;
        lg[0] = t0;
        lg[1] = dt;
        lg[2] = (double)accepted;
    }
    c.n_log++;
}
__device__ __forceinline__ void row_write_status(const ResParams& p, int q, const RowCtl& c) {
    if (blockIdx.x == 0 && p.status) {
        phx_status* st = p.status + q;
        st->n_accepted = c.n_acc;
        st->n_rejected = c.n_rej;
        st->n_rhs = c.n_rhs;
        st->n_logged = min(c.n_log, p.steplog_cap);
        st->reserved = 0;
        st->t_fail = c.tcur;
        st->dt_fail = c.dt;
        __threadfence_system();
        st->code = c.code;
    }
}
// rk_common.py:154,175-176 before an attempted step; returns true when the row may step
__device__ __forceinline__ bool row_prestep(const ResParams& p, RowCtl& c) {
    int st = 0;
    if ((long long)c.n_steps_interval >= p.max_steps) st = PHX_ST_MAX_STEPS;
    else if (!(c.tcur + c.dt > c.tcur)) st = PHX_ST_DT_UNDERFLOW;
    else if (c.nonfinite_prev) st = PHX_ST_NONFINITE;
    if (st) {
        c.code = st;
        c.done = 1;
        return false;
    }
    row_set_coeffs(c);
    return true;
}

// =====================================================================================================================
// Forward solves
// =====================================================================================================================
// One RHS evaluation for all rows at the current branch vector: f = fsign relu(m) (J - y); yn = post(b, j, li, f); with
// do_next the Hill activations of yn become the next stage input and its branch vector is completed (pass A, all-reduce,
// bias / exp).
template <typename Post>
__device__ __forceinline__ void rows_fwd_eval(const ResParams& __restrict__ p, Smem& __restrict__ s, const RowsView& v,
                                              bool do_next, Post post) {
    Prof& pf = s.pf;
    rows_pass1<false>(v, nullptr);
    pf.tick(PT_PHASE_B);
    const float* jr = v.jred();
    const int tot = s.n_loc * RM;
    for (int e = threadIdx.x; e < tot; e += THREADS) {
        const int j = e >> 2, b = e & 3;
        float J = jr[e];
        for (int w = 1; w < p.nqw; ++w) J += jr[w * RM * p.gpc + e];
        const float f = p.fsign * (s.relum()[j] * (J - s.ysb()[e]));
        const float yn = post(b, j, e, f);
        if (do_next) {
            float sv, lv, den;
            hill(yn, sv, lv, den);
            s.ysb()[e] = yn;
            s.acts()[e] = sv;
            v.actL()[e] = lv;
        }
    }
    __syncthreads();
    pf.tick(PT_COMBINE);
    if (do_next) {
        rows_passA(v, s.acts(), v.actL(), s.sp());
        pf.tick(PT_PHASE_A);
        grid_allreduce_f(p, s, s.sp(), RM * p.K2);
        pf.tick(PT_ALLRED1);
        rows_finalize_sp(v, s.sp(), s.sp());
        pf.tick(PT_FINALIZE);
    }
}
// stand-alone pass A at the current stage input + its exchange
__device__ __forceinline__ void rows_eval_A(const ResParams& __restrict__ p, Smem& __restrict__ s, const RowsView& v) {
    Prof& pf = s.pf;
    rows_passA(v, s.acts(), v.actL(), s.sp());
    pf.tick(PT_PHASE_A);
    grid_allreduce_f(p, s, s.sp(), RM * p.K2);
    pf.tick(PT_ALLRED1);
    rows_finalize_sp(v, s.sp(), s.sp());
    pf.tick(PT_FINALIZE);
}

__global__ void __launch_bounds__(PHX_THREADS, 1) phx_rows_fwd_kernel(const __grid_constant__ ResParams p) {
    Smem s(p);
    RowsView v(p, s);
    rows_prologue(p, s, v, p.ring_rows);
    Prof& pf = s.pf;
    RowsCtl* rc = v.rc();
    const int g_lo = s.g_lo, n_loc = s.n_loc;
    const int tot = n_loc * RM;
    const double Nel = (double)p.G;
    float* Y = v.st(0);
    float* Y1 = v.st(1);
    auto K = [&](int i) { return v.st(2 + i); };
    double* dsum = s.at<double>(p.so.dred);   // [RM * 8] block / grid totals

    for (int q0 = 0; q0 < p.ntot; q0 += p.rows) {
        const int nr = min(p.rows, p.ntot - q0);
        if (threadIdx.x < RM) {
            RowCtl& c = rc->r[threadIdx.x];
            row_init(c, (int)threadIdx.x < nr);
            if (c.valid) c.tcur = tget_rows(p, q0 + threadIdx.x, 0);
        }
        __syncthreads();
        auto set_input = [&](int e, float ys) {
            s.ysb()[e] = ys;
            float sv, lv, den;
            hill(ys, sv, lv, den);
            s.acts()[e] = sv;
            v.actL()[e] = lv;
        };
        for (int e = threadIdx.x; e < p.gpc * RM; e += THREADS) {
            const int j = e >> 2, b = e & 3;
            float y = 0.5f;
            if (b < nr && j < n_loc) {
                y = p.y0[(size_t)(q0 + b) * p.y0_stride + g_lo + j];
                p.yout[(size_t)(q0 + b) * p.yout_stride + g_lo + j] = y;
            }
            Y[e] = y;
            set_input(e, y);
        }
        __syncthreads();

        if (p.method != PHX_DOPRI5) {
            // ---- fixed grid (solvers.py:48-50, 77-103): one step per output interval, or the steps of each row's own
            // grid (p.gdt); a row past its last step is left as it is while the others go on ----
            const float third = (float)(1.0 / 3.0);
            const int nst = (p.method == PHX_EULER) ? 1 : (p.method == PHX_MIDPOINT ? 2 : 4);
            int nk = p.T - 1;
            if (p.gdt) {
                nk = 0;
                for (int b = 0; b < nr; ++b) nk = max(nk, p.goff[q0 + b + 1] - p.goff[q0 + b]);
            }
            if (threadIdx.x < RM) {
                RowCtl& c = rc->r[threadIdx.x];
                c.gj0 = c.gj1 = 1;
                c.stepping = 1;
            }
            rows_eval_A(p, s, v);
            for (int i = 0; i < nk; ++i) {
                if (threadIdx.x < RM) {
                    RowCtl& c = rc->r[threadIdx.x];
                    const int q = q0 + threadIdx.x;
                    if (!c.valid) {
                        c.dtf = 0.f;
                    } else if (p.gdt) {
                        c.stepping = i < p.goff[q + 1] - p.goff[q];
                        c.dtf = c.stepping ? p.gdt[p.goff[q] + i] : 0.f;
                        int je = c.gj1;
                        while (je < p.T && p.gout[q * (p.T - 1) + je - 1] == i) ++je;
                        c.gj0 = c.gj1;
                        c.gj1 = je;
                    } else {
                        const double ta = tget_rows(p, q, i), tb = tget_rows(p, q, i + 1);
                        c.dtf = p.t_is_f32 ? ((float)tb - (float)ta) : (float)(tb - ta);
                    }
                }
                __syncthreads();
                const bool more = i + 1 < nk;
                for (int st = 0; st < nst; ++st) {
                    const bool last = st + 1 == nst;
                    rows_fwd_eval(p, s, v, !last || more, [&](int b, int j, int li, float f) {
                        const RowCtl& c = rc->r[b];
                        if (!c.stepping) return Y[li];   // (its stage input stays its state)
                        const float dtf = c.dtf;
                        float yn;
                        if (p.method == PHX_EULER) {
                            yn = Y[li] + dtf * f;
                        } else if (p.method == PHX_MIDPOINT) {
                            yn = (st == 0) ? Y[li] + f * (0.5f * dtf) : Y[li] + dtf * f;
                        } else {  // 3/8-rule RK4 (rk_common.py:96-103)
                            if (st == 0) yn = Y[li] + dtf * f * third;
                            else if (st == 1) yn = Y[li] + dtf * (f - K(0)[li] * third);
                            else if (st == 2) yn = Y[li] + dtf * (K(0)[li] - K(1)[li] + f);
                            else yn = Y[li] + (K(0)[li] + 3.f * (K(1)[li] + K(2)[li]) + f) * dtf * 0.125f;
                            if (!last) K(st)[li] = f;
                        }
                        if (last) {
                            if (b < nr) {
                                float* yo = p.yout + (size_t)(q0 + b) * p.yout_stride + g_lo + j;
                                if (p.gdt) {
                                    for (int jj = c.gj0; jj < c.gj1; ++jj) {
                                        const float sl = p.gsl[(q0 + b) * (p.T - 1) + jj - 1];
                                        yo[(size_t)jj * p.G] = sl < 0.f ? yn : Y[li] + sl * (yn - Y[li]);
                                    }
                                } else {
                                    yo[(size_t)(i + 1) * p.G] = yn;
                                }
                            }
                            Y[li] = yn;
                        }
                        return yn;
                    });
                }
            }
            if (threadIdx.x < nr) {
                RowCtl& c = rc->r[threadIdx.x];
                c.n_rhs = nst * (p.gdt ? p.goff[q0 + threadIdx.x + 1] - p.goff[q0 + threadIdx.x] : p.T - 1);
                c.tcur = tget_rows(p, q0 + threadIdx.x, p.T - 1);
                row_write_status(p, q0 + threadIdx.x, c);
            }
            __syncthreads();
            continue;
        }

        // ---- dopri5 (rk_common.py:111-228), one controller per row ----
        for (int which = 0; which < 2; ++which) {
            double acc[3] = {0, 0, 0};
            rows_eval_A(p, s, v);
            rows_fwd_eval(p, s, v, false, [&](int b, int j, int li, float f) {
                const float y = Y[li];
                const float scale = p.atol_f + fabsf(y) * p.rtol_f;
                if (which == 0) {
                    K(0)[li] = f;
                    const float r0 = y / scale, r1 = f / scale;
                    acc[0] += (double)(r0 * r0);
                    acc[1] += (double)(r1 * r1);
                    if (!isfinite(y)) acc[2] += 1.0;
                } else {
                    const float r = (f - K(0)[li]) / scale;
                    acc[0] += (double)(r * r);
                }
                return 0.f;
            });
            block_sum_rows<3>(v, acc, dsum);
            grid_sum_d(p, s, dsum, 3 * RM);
            pf.tick(PT_NORMS);
            if (threadIdx.x < RM) {
                RowCtl& c = rc->r[threadIdx.x];
                const double* d = dsum + threadIdx.x * 3;
                if (which == 0) {
                    const float d0 = sqrtf((float)(d[0] / Nel));
                    const float d1 = sqrtf((float)(d[1] / Nel));
                    c.d1 = d1;
                    c.h0 = init_h0(d0, d1);
                    c.nonfinite_prev = d[2] > 0.0;
                    if (p.first_step > 0) {
                        c.dt = p.first_step;
                        c.tprev = c.tcur;
                        c.n_rhs = 1;
                        c.n_steps_interval = 0;
                    }
                } else {
                    const float d2 = sqrtf((float)(d[0] / Nel)) / c.h0;
                    c.dt = init_dt(c.h0, c.d1, d2);
                    c.tprev = c.tcur;
                    c.n_rhs = 2;
                    c.n_steps_interval = 0;
                }
            }
            __syncthreads();
            if (p.first_step > 0) break;   // the caller's first step (every row's): no second evaluation
            if (which == 0) {
                for (int e = threadIdx.x; e < tot; e += THREADS) set_input(e, Y[e] + rc->r[e & 3].h0 * K(0)[e]);
                __syncthreads();
            }
        }

        while (true) {
            if (threadIdx.x < RM) {
                RowCtl& c = rc->r[threadIdx.x];
                if (!c.done) row_prestep(p, c);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                int all = 1;
                for (int b = 0; b < RM; ++b) all &= rc->r[b].done;
                rc->all_done = all;
            }
            __syncthreads();
            if (rc->all_done) break;
            for (int e = threadIdx.x; e < tot; e += THREADS) {
                const RowCtl& c = rc->r[e & 3];
                set_input(e, Y[e] + K(c.slot[0])[e] * c.cb[0][0]);
            }
            __syncthreads();
            rows_eval_A(p, s, v);
            double acc[2] = {0, 0};
            for (int st = 1; st <= 6; ++st) {
                rows_fwd_eval(p, s, v, st < 6, [&](int b, int j, int li, float f) {
                    const RowCtl& c = rc->r[b];
                    const int* sl = c.slot;
                    K(sl[st])[li] = f;
                    if (st < 6) {
                        float a = K(sl[0])[li] * c.cb[st][0];
                        for (int qq = 1; qq < st; ++qq) a = fmaf(K(sl[qq])[li], c.cb[st][qq], a);
                        a = fmaf(f, c.cb[st][st], a);
                        const float yn = Y[li] + a;
                        if (st == 5) Y1[li] = yn;
                        return yn;
                    }
                    const float ys = s.ysb()[li];
                    float er = K(sl[0])[li] * c.cerr[0];
                    for (int qq = 1; qq < 6; ++qq) er = fmaf(K(sl[qq])[li], c.cerr[qq], er);
                    er = fmaf(f, c.cerr[6], er);
                    const float tol = p.atol_f + p.rtol_f * fmaxf(fabsf(Y[li]), fabsf(ys));
                    const float r = er / tol;
                    acc[0] += (double)(r * r);
                    if (!isfinite(ys)) acc[1] += 1.0;
                    return 0.f;
                });
            }
            block_sum_rows<2>(v, acc, dsum);
            grid_sum_d(p, s, dsum, 2 * RM);
            pf.tick(PT_NORMS);
            if (threadIdx.x < RM) {
                RowCtl& c = rc->r[threadIdx.x];
                c.accept = 0;
                c.pend = 0;
                if (!c.done) {
                    const double* d = dsum + threadIdx.x * 2;
                    const float ratio = sqrtf((float)(d[0] / Nel));
                    const int accept = ratio <= 1.f;
                    row_log_step(p, c, q0 + threadIdx.x, c.tcur, c.dt, accept);
                    c.tprev = c.tcur;
                    if (accept) {
                        c.tcur = c.tcur + c.dt;
                        c.n_acc++;
                        c.nonfinite_prev = d[1] > 0.0;
                    } else {
                        c.n_rej++;
                    }
                    c.dt = next_dt(p, c.dt, ratio);
                    c.accept = accept;
                    c.n_rhs += 6;
                    c.n_steps_interval++;
                }
            }
            __syncthreads();
            // emit every pending output inside (tprev, tcur] from the quartic interpolant (rk_common.py:157): one output
            // per row and round
            while (true) {
                if (threadIdx.x < RM) {
                    RowCtl& c = rc->r[threadIdx.x];
                    c.pend = 0;
                    if (c.accept && !c.done && c.next_out < p.T) {
                        const double to = tget_rows(p, q0 + threadIdx.x, c.next_out);
                        if (to <= c.tcur) {
                            row_set_interp_x(c, to, c.tprev, c.tcur);
                            c.pend = 1;
                        }
                    }
                }
                __syncthreads();
                if (threadIdx.x == 0) {
                    int any = 0;
                    for (int b = 0; b < RM; ++b) any |= rc->r[b].pend;
                    rc->any_pending = any;
                }
                __syncthreads();
                if (!rc->any_pending) break;
                for (int e = threadIdx.x; e < tot; e += THREADS) {
                    const int j = e >> 2, b = e & 3;
                    const RowCtl& c = rc->r[b];
                    if (!c.pend) continue;
                    const int* sl = c.slot;
                    const float y0 = Y[e], y1 = Y1[e];
                    float m = K(sl[0])[e] * c.cmid[0];
                    for (int qq = 1; qq < 7; ++qq) m = fmaf(K(sl[qq])[e], c.cmid[qq], m);
                    const float ymid = y0 + m;
                    p.yout[(size_t)(q0 + b) * p.yout_stride + (size_t)c.next_out * p.G + g_lo + j] =
                        interp_eval(y0, y1, ymid, K(sl[0])[e], K(sl[6])[e], c.dtf, c.xs);
                }
                __syncthreads();
                if (threadIdx.x < RM) {
                    RowCtl& c = rc->r[threadIdx.x];
                    if (c.pend) {
                        c.next_out++;
                        c.n_steps_interval = 0;
                        if (c.next_out >= p.T) c.done = 1;
                    }
                }
                __syncthreads();
            }
            for (int e = threadIdx.x; e < tot; e += THREADS)
                if (rc->r[e & 3].accept) Y[e] = Y1[e];
            __syncthreads();
            if (threadIdx.x < RM) {
                RowCtl& c = rc->r[threadIdx.x];
                if (c.accept) {
                    const int t0 = c.slot[0];
                    c.slot[0] = c.slot[6];
                    c.slot[6] = t0;
                }
            }
            __syncthreads();
            pf.tick(PT_CTRL);
        }
        // a row stopped by a solver assertion never reached its remaining output times: they read NaN, not garbage
        for (int e = threadIdx.x; e < tot; e += THREADS) {
            const int j = e >> 2, b = e & 3;
            const RowCtl& c = rc->r[b];
            if (b < nr && c.code != PHX_ST_OK)
                for (int i = c.next_out; i < p.T; ++i)
                    p.yout[(size_t)(q0 + b) * p.yout_stride + (size_t)i * p.G + g_lo + j] = nanf("");
        }
        if (threadIdx.x < nr) row_write_status(p, q0 + threadIdx.x, rc->r[threadIdx.x]);
        __syncthreads();
    }
    pf.finish();
    rows_release(p, s);
    epilogue_epoch(p, s);
}


// =====================================================================================================================
// Adjoint sweeps
// =====================================================================================================================
// One RHS + VJP evaluation for all rows at the current stage input (ysb / acts, cotangent asb / gjb).  `sid` is the
// LOGICAL stage whose per-row slots receive the results (KY / KA in rc.slot[sid], theta factors in rc.fslot[sid]);
// `sid_next` the logical stage of the next input (for its stage-input record).
//   sp_ready: the branch vector of this input is already in s.sp(); otherwise a stand-alone pass A + exchange runs first.
//   has_next: ynext(b, j, li, ky) returns the next stage's y input per element; its pass A shares this evaluation's single
//             all-reduce.  anext(b, j, li, ka) returns the next stage's cotangent input (caller's per-element algebra).
template <typename YNext, typename ANext>
__device__ __forceinline__ void rows_adj_eval(const ResParams& __restrict__ p, Smem& __restrict__ s, const RowsView& v,
                                              int sid, int sid_next, bool sp_ready, bool has_next, YNext ynext,
                                              ANext anext) {
    Prof& pf = s.pf;
    RowsCtl* rc = v.rc();
    const int BL = RM * p.gpc, n = RM * p.K2, K2q = p.K2q, Hq = p.Hp >> 2;
    const int tot = s.n_loc * RM;
    if (!sp_ready) rows_eval_A(p, s, v);
    pf.tick(PT_COMBINE);
    // ---- pass 1: J partials + gSP partial sums --------------------------------------------------------------------------
    rows_pass1<true>(v, s.xv());
    pf.tick(PT_PHASE_B);
    {
        const float* jr = v.jred();
        for (int e = threadIdx.x; e < tot; e += THREADS) {
            const int j = e >> 2, b = e & 3;
            const RowCtl& c = rc->r[b];
            float J = jr[e];
            for (int w = 1; w < p.nqw; ++w) J += jr[w * BL + e];
            const float jm = J - s.ysb()[e];
            const float ky = -(s.relum()[j] * jm);
            v.st(4 + c.slot[sid])[e] = ky;
            const int fs = c.fslot[sid];
            if (fs >= 0) {
                v.fm()[e * NFS + fs] = (s.asb()[e] * jm) * s.maskm()[j];
                v.fgj()[e * NFS + fs] = s.gjb()[e];
            }
            if (has_next) {
                const float yn = ynext(b, j, e, ky);
                float sv, lv, den;
                hill(yn, sv, lv, den);
                s.ysb2()[e] = yn;
                s.acts2()[e] = sv;
                v.actL()[e] = lv;
                const int fsn = c.fslot[sid_next];
                if (fsn >= 0) v.ysf()[e * NFS + fsn] = yn;
            }
        }
    }
    __syncthreads();
    pf.tick(PT_EPILOGUE);
    if (has_next) {
        rows_passA(v, s.acts2(), v.actL(), s.xv() + n);
        pf.tick(PT_PHASE_A);
    }
    grid_allreduce_f(p, s, s.xv(), has_next ? 2 * n : n);
    pf.tick(PT_ALLRED2);
    // ---- finalize: gLP = gPr * Pr (exp backward), next stage's branch vector (bias, exp) -- every quad by ONE thread --
    // then the stage's K2-long theta factors go to tensor memory: warps 0..3 (one per lane quarter) each store the quad
    // block their quarter serves (S|Pr staged through the idle fold buffer, gS|gLP read back from xv).
    {
        float4* sp4 = reinterpret_cast<float4*>(s.sp());
        float4* xv4 = reinterpret_cast<float4*>(s.xv());
        float4* stage4 = s.at<float4>(p.so.red);
        const float4* bias4 = reinterpret_cast<const float4*>(s.bias());
        if (v.gg < RM && v.qok) {   // warp (quad block, gene group g) finalises row g
            const int fq = v.q;
            {
                const int b = v.gg;
                const float4 spv = sp4[b * K2q + fq];
                float4 gv = xv4[b * K2q + fq];
                if (fq >= Hq) gv = mul4(gv, spv);
                xv4[b * K2q + fq] = gv;
                stage4[b * K2q + fq] = spv;
                if (has_next) {
                    const float4 t = xv4[(RM + b) * K2q + fq], bq = bias4[fq];
                    float x[4] = {t.x + bq.x, t.y + bq.y, t.z + bq.z, t.w + bq.w};
                    if (fq >= Hq) {
#pragma unroll
                        for (int e4 = 0; e4 < 4; ++e4) x[e4] = (4 * fq + e4 - p.Hp < p.H) ? expf(x[e4]) : 0.f;
                    }
                    sp4[b * K2q + fq] = make_float4(x[0], x[1], x[2], x[3]);
                }
            }
        }
        __syncthreads();
        if (v.warp < 4) {
            const int fq = 32 * (v.warp % p.nqw) + v.lane;   // warp % nqw: the quad block this lane quarter serves
            const bool fok = fq < K2q;
#pragma unroll
            for (int b = 0; b < RM; ++b) {
                const int fs = rc->r[b].fslot[sid];
                if (b < p.rows && fs >= 0) {   // uniform over the warp
                    tm_st4(v.col_fsp(fs, b), fok ? stage4[b * K2q + fq] : zero4());
                    tm_st4(v.col_fg(fs, b), fok ? xv4[b * K2q + fq] : zero4());
                }
            }
            tm_wait_st();
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    pf.tick(PT_FINALIZE);
    // ---- pass 2 over W1: u = W1[g][:Hp] . gS, v = W1[g][Hp:] . gLP.  Same mapping as pass 1 (thread = quad x gene group,
    // the lane's gS|gLP quad in registers, one 16-byte shared-memory read per gene): a warp whose quads all lie in one half
    // contributes to u or to v only; the warp straddling Hp runs the transposing butterfly twice.
    {
        const float4* g4 = reinterpret_cast<const float4*>(s.xv());
        const float4* w1 = v.w1();
        const int ws = p.ring_rows;
        float4 gq[RM];
#pragma unroll
        for (int b = 0; b < RM; ++b) gq[b] = v.qok ? g4[b * K2q + v.q] : zero4();
        const int qlo = 32 * v.qw, qhi = min(qlo + 31, K2q - 1);
        const bool has_u = qlo < Hq, has_v = qhi >= Hq;     // warp-uniform
        const bool mine_u = v.q < Hq;
        float* ur = v.jred() + (size_t)v.qw * RM * p.gpc;                 // u partials [qw][gene][row]
        float* vr = s.at<float>(p.so.red) + (size_t)v.qw * RM * p.gpc;    // v partials (fold buffer is idle here)
        const int j0 = v.gg * p.gpg;
        const int jend = min(j0 + p.gpg, (s.n_loc + 3) & ~3);
        for (int jc = j0; jc < jend; jc += 4) {
            float pu[16], pv[16];
#pragma unroll
            for (int gi = 0; gi < 4; ++gi) {
                const float4 w = (v.qok && jc + gi < s.n_loc) ? w1[(size_t)(jc + gi) * ws + v.q] : zero4();
#pragma unroll
                for (int b = 0; b < RM; ++b) {
                    const float d = dot4(w, gq[b]);
                    pu[gi * RM + b] = mine_u ? d : 0.f;
                    pv[gi * RM + b] = mine_u ? 0.f : d;
                }
            }
            const int idx = (v.lane >> 1) & 15;
            const bool wr = (v.lane & 1) == 0 && jc + (idx >> 2) < p.gpc;
            const int o = (jc + (idx >> 2)) * RM + (idx & 3);
            if (has_u) {
                const float r = transpose_reduce16(pu);
                if (wr) ur[o] = r;
            } else if (wr) {
                ur[o] = 0.f;
            }
            if (has_v) {
                const float r = transpose_reduce16(pv);
                if (wr) vr[o] = r;
            } else if (wr) {
                vr[o] = 0.f;
            }
        }
        __syncthreads();
        for (int e = threadIdx.x; e < tot; e += THREADS) {
            const int j = e >> 2, b = e & 3;
            float uu = v.jred()[e], vw = s.at<float>(p.so.red)[e];
            for (int w = 1; w < p.nqw; ++w) {
                uu += v.jred()[w * BL + e];
                vw += s.at<float>(p.so.red)[w * BL + e];
            }
            const float z = s.ysb()[e] - 0.5f;
            const float den = 1.0f + fabsf(z);
            const float yb = (uu + vw / (1.0f + s.acts()[e])) / (den * den);
            const float ka = yb - s.gjb()[e];
            v.st(11 + rc->r[b].slot[sid])[e] = ka;
            const float an = anext(b, j, e, ka);
            if (has_next) {
                s.asb()[e] = an;
                s.gjb()[e] = an * s.relum()[j];
            }
        }
    }
    __syncthreads();
    if (has_next) s.swap_stage_buffers();
    pf.tick(PT_PHASE_C);
}

// ---- parameter-cotangent ("theta") passes, PACKED layout -------------------------------------------------------------------
// theta element (gene j, column k) of W1bar / WAbar in factor slot fs has the stage derivative U[fs][j] * V[fs][k]:
//   WAbar: U = gJ (FGJ), V = S|Pr (FSP);  W1bar: U = s (k < Hp) or l (k >= Hp), V = gS|gLP (FG);
//   biasbar[k] = V = gS|gLP (CTA 0);  mbar[j] = FM.
enum { TP_D01 = 0, TP_D2 = 1, TP_STEP = 2, TP_FIXED = 3 };
// Per-row arguments of a theta pass.  Weights are indexed by PHYSICAL factor slot.  The value written by a step / fixed
// pass is  th0 + sum_f wo[f] k[f]:  for an ordinary step wo == cs (the solution weights dt * beta_6); for the step that
// ends the interval it is the quartic dense output at t_end (interp.py:1-47) written as ONE linear combination -- the
// interpolant is linear in (y0, y1, y_mid, f0, f1), y1 and y_mid are th0 + linear combinations of the stage derivatives,
// and the coefficient of th0 collapses to exactly 1 (rows_interp_weights); euler / midpoint / rk4: wo = dt * b.
struct RowPP {
    float* src;   // theta at step start; nullptr while it is identically zero
    float* dst;   // may alias src
    float cs[NFS], ce[NFS], wo[NFS];
    int active, last, s0, s1;
    // speculative final step (see phx_rows_adj_kernel): the written value is ADDED to the group's packed sum `acc` instead
    // of stored in the row's own buffer: 1 = first such row of the pass (plain store), 2 = read-modify-write
    int spec;
    float* acc;
};
static_assert(sizeof(RowPP) * RM <= 1024, "RowPP block must fit its shared-memory slot");

// weights of the dense output at x = (t_end - t0) / dt as a linear combination of the stage derivatives (see RowPP)
__device__ __forceinline__ void rows_interp_weights(const RowCtl& c, RowPP& a) {
    const double x = c.xs[0], x2 = c.xs[1], x3 = c.xs[2], x4 = c.xs[3], dt = c.dtf;
    const double wy1 = -5.0 * x2 + 14.0 * x3 - 8.0 * x4;        // coefficient of (y1 - y0)
    const double wym = 16.0 * x2 - 32.0 * x3 + 16.0 * x4;       // coefficient of (y_mid - y0)
    const double wf0 = dt * (x - 4.0 * x2 + 5.0 * x3 - 2.0 * x4);
    const double wf1 = dt * (x2 - 3.0 * x3 + 2.0 * x4);
    for (int qq = 0; qq < 7; ++qq) {
        const int fs = c.fslot[qq];
        if (fs < 0) continue;
        double w = wy1 * (double)((qq < 6) ? c.cb[5][qq] : 0.f) + wym * (double)c.cmid[qq];
        if (qq == 0) w += wf0;
        if (qq == 6) w += wf1;
        a.wo[fs] = (float)w;
    }
}

__device__ __forceinline__ float rcp_approx(float x) {   // MUFU.RCP, 1 ulp; callers pass normal-range values (>= atol)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float2 bc2(float x) { return make_float2(x, x); }

// One pass over this CTA's share of every ACTIVE row's packed cotangent vector.  out[b * 2 + {0,1}] (shared memory, doubles)
// receives this CTA's partial sums per row: STEP (sum (err/tol)^2, non-finite count), D01 (sum (th/scale)^2,
// sum (k/scale)^2), D2 (sum ((k1-k0)/scale)^2, -).  Ends with a block barrier.
// The step / fixed passes are instruction-bound (8.9 M elements x rows at the headline shape): the three 6-term
// combinations of an element pair run as packed fp32x2 FMAs (FFMA2), the tolerance division is MUFU.RCP + FMUL (the error
// ratio only feeds the accept test and the step-size law), a non-finite theta is caught by a NaN-propagating FMA.
// ALL: every parameter is an adjoint parameter (p.pmask == PHX_P_ALL), so the mask tests fold away and the pass is the
// code it was before masks existed -- it is the instruction-bound part of the kernel (see rows_theta_pass)
template <int MODE, bool ALL>
__device__ __noinline__ void rows_theta_pass_impl(const ResParams& __restrict__ p, int g_lo, int n_loc, uint32_t tmem,
                                                  double* out) {
    Smem s(p);
    s.tmem = tmem;
    RowsView v(p, s);
    v.tq = tm_quarter(tmem);
    const int Hq = p.Hp >> 2;
    const int tot = n_loc * RM;
    const PhxPackedGradOff off = phx_packed_grad_offsets(p.G, p.H);
    const float atol_f = p.atol_f, rtol_f = p.rtol_f;
    const RowPP* pp = s.at<RowPP>(p.so.ppa);
    constexpr bool WRITES = MODE == TP_STEP || MODE == TP_FIXED;
    constexpr int NV = (MODE == TP_D01) ? 1 : (MODE == TP_D2 ? 2 : NFS);   // factor slots the mode touches
    // activation tables of the stored stage inputs, [gene][row][slot] like the other per-gene factor tables (the scratch
    // aliases the fold / J-partial buffers, idle here)
    float* US = s.at<float>(p.so.red);
    float* UL = US + NFS * RM * p.gpc;
    for (int i = threadIdx.x; i < NFS * tot; i += THREADS) {
        float sv, lv, den;
        hill(v.ysf()[i], sv, lv, den);
        US[i] = sv;
        UL[i] = lv;
    }
    double* dred = s.dred();
    if (threadIdx.x < WARPS * 8) dred[threadIdx.x] = 0.0;
    __syncthreads();
    const int j0 = v.gg * p.gpg, jend = min(j0 + p.gpg, n_loc);
    // only the adjoint parameters' parts of the packed slice are read or written (p.pmask): WAbar, the Ws (q < Hq) or Wp
    // half of a W1bar row and of the bias, mbar
    const int pm = ALL ? (int)PHX_P_ALL : p.pmask;
    const bool keep_wa = pm & PHX_P_WA, keep_w1 = pm & (v.q >= Hq ? PHX_P_WP : PHX_P_WS);
    const bool keep_b = pm & (v.q >= Hq ? PHX_P_BP : PHX_P_BS), keep_m = pm & PHX_P_M;
#pragma unroll 1
    for (int b = 0; b < RM; ++b) {
        if (!pp[b].active) continue;
        float* const src = pp[b].src;
        const int spec = WRITES ? pp[b].spec : 0;
        float* const dst = spec ? pp[b].acc : pp[b].dst;
        float a0 = 0.f, a1 = 0.f;
        int sl[NV];
        float cs[NV], ce[NV], wo[NV];
#pragma unroll
        for (int f = 0; f < NV; ++f) {
            sl[f] = (MODE == TP_D01) ? pp[b].s0 : (MODE == TP_D2 ? (f == 0 ? pp[b].s0 : pp[b].s1) : f);
            cs[f] = pp[b].cs[f];
            ce[f] = pp[b].ce[f];
            wo[f] = pp[b].wo[f];
        }
        const bool sep = MODE == TP_STEP && pp[b].last;    // the written value is not th1: a third combination
        // scalar tail of a step element: error-ratio term, non-finite flag
        auto tail = [&](const float th0, const float inc, const float er) {
            const float th1 = th0 + inc;
            const float tol = atol_f + rtol_f * fmaxf(fabsf(th0), fabsf(th1));
            const float r = er * rcp_approx(tol);
            a0 = fmaf(r, r, a0);
            a1 = fmaf(th1, 0.f, a1);      // 0 while finite, NaN once th1 is inf / NaN
            return th1;
        };
        // two theta elements (k = u * V) at once
        auto pair = [&](const float2 th0, const float (&u)[NV], const float2 (&Vp)[NV], float2& o) {
            float2 k[NV];
#pragma unroll
            for (int f = 0; f < NV; ++f) k[f] = __fmul2_rn(bc2(u[f]), Vp[f]);
            if (MODE == TP_D01) {
                const float sx = atol_f + fabsf(th0.x) * rtol_f, sy = atol_f + fabsf(th0.y) * rtol_f;
                const float ix = rcp_approx(sx), iy = rcp_approx(sy);
                a0 = fmaf(th0.x * ix, th0.x * ix, a0);
                a0 = fmaf(th0.y * iy, th0.y * iy, a0);
                a1 = fmaf(k[0].x * ix, k[0].x * ix, a1);
                a1 = fmaf(k[0].y * iy, k[0].y * iy, a1);
            } else if (MODE == TP_D2) {
                const float sx = atol_f + fabsf(th0.x) * rtol_f, sy = atol_f + fabsf(th0.y) * rtol_f;
                const float rx = (k[1].x - k[0].x) * rcp_approx(sx), ry = (k[1].y - k[0].y) * rcp_approx(sy);
                a0 = fmaf(rx, rx, a0);
                a0 = fmaf(ry, ry, a0);
            } else if (MODE == TP_FIXED) {
                float2 acc = __fmul2_rn(k[0], bc2(wo[0]));
#pragma unroll
                for (int f = 1; f < NV; ++f) acc = __ffma2_rn(k[f], bc2(wo[f]), acc);
                o = __fadd2_rn(th0, acc);
            } else {
                float2 inc = __fmul2_rn(k[0], bc2(cs[0])), er = __fmul2_rn(k[0], bc2(ce[0]));
#pragma unroll
                for (int f = 1; f < NV; ++f) {
                    inc = __ffma2_rn(k[f], bc2(cs[f]), inc);
                    er = __ffma2_rn(k[f], bc2(ce[f]), er);
                }
                o.x = tail(th0.x, inc.x, er.x);
                o.y = tail(th0.y, inc.y, er.y);
                if (sep) {
                    float2 acc = __fmul2_rn(k[0], bc2(wo[0]));
#pragma unroll
                    for (int f = 1; f < NV; ++f) acc = __ffma2_rn(k[f], bc2(wo[f]), acc);
                    o = __fadd2_rn(th0, acc);
                }
            }
        };
        auto quad = [&](const float (&u)[NV], const float4 (&V)[NV], const size_t idx) {
            const float4 th4 = src ? *reinterpret_cast<const float4*>(src + idx) : zero4();
            float2 lo[NV], hi[NV], o0 = make_float2(0.f, 0.f), o1 = make_float2(0.f, 0.f);
#pragma unroll
            for (int f = 0; f < NV; ++f) {
                lo[f] = make_float2(V[f].x, V[f].y);
                hi[f] = make_float2(V[f].z, V[f].w);
            }
            pair(make_float2(th4.x, th4.y), u, lo, o0);
            pair(make_float2(th4.z, th4.w), u, hi, o1);
            if (WRITES) {
                float4 o4 = make_float4(o0.x, o0.y, o1.x, o1.y);
                if (spec == 2) o4 = add4(*reinterpret_cast<const float4*>(dst + idx), o4);
                *reinterpret_cast<float4*>(dst + idx) = o4;
            }
        };
#pragma unroll 1
        for (int blk = 0; blk < 2; ++blk) {   // 0: WAbar (V = S|Pr, U = gJ), 1: W1bar (V = gS|gLP, U = s | l)
            float4 V[NV];
#pragma unroll
            for (int f = 0; f < NV; ++f) tm_ld4(blk == 0 ? v.col_fsp(sl[f], b) : v.col_fg(sl[f], b), V[f]);
            if (!v.qok) continue;
            const float* U = (blk == 0 ? v.fgj() : (v.q >= Hq ? UL : US)) + b * NFS;
            const size_t base = (blk == 0 ? off.WA : off.W1) + (size_t)g_lo * p.K2 + 4 * (size_t)v.q;
#pragma unroll 1
            for (int j = j0; (blk == 0 ? keep_wa : keep_w1) && j < jend; ++j) {
                float u[NV];
                if (NV == NFS) {
                    const float2* u2 = reinterpret_cast<const float2*>(U + j * (RM * NFS));
#pragma unroll
                    for (int f = 0; f < NFS / 2; ++f) {
                        const float2 t = u2[f];
                        u[(2 * f) % NV] = t.x;
                        u[(2 * f + 1) % NV] = t.y;
                    }
                } else {
#pragma unroll
                    for (int f = 0; f < NV; ++f) u[f] = U[j * (RM * NFS) + sl[f]];
                }
                quad(u, V, base + (size_t)j * p.K2);
            }
            if (blk == 1 && blockIdx.x == 0 && v.gg == 0 && keep_b) {   // biases: stage derivative = gS | gLP itself
                float u[NV];
#pragma unroll
                for (int f = 0; f < NV; ++f) u[f] = 1.f;
                quad(u, V, off.bias + 4 * (size_t)v.q);
            }
        }
        // gene multipliers: two genes per thread (elements e = (gene, row b)); an odd tail pairs with an all-zero element,
        // which adds exactly 0 to every sum
        for (int jp = 2 * (int)threadIdx.x; keep_m && jp < n_loc; jp += 2 * THREADS) {
            const bool two = jp + 1 < n_loc;
            const int e0 = jp * RM + b, e1 = (two ? jp + 1 : jp) * RM + b;
            float u[NV];
            float2 Vp[NV], o = make_float2(0.f, 0.f);
#pragma unroll
            for (int f = 0; f < NV; ++f) {
                u[f] = 1.f;
                Vp[f] = make_float2(v.fm()[e0 * NFS + sl[f]], two ? v.fm()[e1 * NFS + sl[f]] : 0.f);
            }
            const size_t idx = off.m + g_lo + jp;
            pair(make_float2(src ? src[idx] : 0.f, (src && two) ? src[idx + 1] : 0.f), u, Vp, o);
            if (WRITES) {
                dst[idx] = (spec == 2) ? dst[idx] + o.x : o.x;
                if (two) dst[idx + 1] = (spec == 2) ? dst[idx + 1] + o.y : o.y;
            }
        }
        const double t0 = warp_sum_d((double)a0);
        const double t1 = (MODE == TP_STEP) ? warp_sum_d(isfinite(a1) ? 0.0 : 1.0) : warp_sum_d((double)a1);
        if (v.lane == 0) {
            dred[v.warp * 8 + 2 * b] = t0;
            dred[v.warp * 8 + 2 * b + 1] = t1;
        }
    }
    __syncthreads();
    if (threadIdx.x < 2 * RM) {
        double t = 0;
        for (int w = 0; w < WARPS; ++w) t += dred[w * 8 + threadIdx.x];
        out[threadIdx.x] = t;
    }
    __syncthreads();
}

// SEMI: p.pmask may carry PHX_NORM_SEMINORM above the six parameter bits
template <int MODE, bool SEMI>
__device__ __forceinline__ void rows_theta_pass(const ResParams& __restrict__ p, int g_lo, int n_loc, uint32_t tmem, double* out) {
    if ((SEMI ? (p.pmask & PHX_P_ALL) : p.pmask) == PHX_P_ALL) rows_theta_pass_impl<MODE, true>(p, g_lo, n_loc, tmem, out);
    else rows_theta_pass_impl<MODE, false>(p, g_lo, n_loc, tmem, out);
}

// gsum (+)= sum over the valid rows of their final packed cotangents; every element is read by the thread that wrote it
__device__ __noinline__ void rows_theta_sum(const ResParams& __restrict__ p, int g_lo, int n_loc, float* gsum,
                                            bool accumulate) {
    Smem s(p);
    RowsView v(p, s);
    const RowsCtl* rc = v.rc();
    const PhxPackedGradOff off = phx_packed_grad_offsets(p.G, p.H);
    const float* src[RM];
    bool any = false;
#pragma unroll
    for (int b = 0; b < RM; ++b) {
        const RowCtl& c = rc->r[b];
        src[b] = (c.valid && !c.theta_zero && !c.spec_done) ? p.theta_ws + (size_t)(2 * b + c.cur) * p.ppk : nullptr;
        any |= src[b] != nullptr;
    }
    if (!any && accumulate) return;   // everything is already in the group's sum
    auto quad = [&](size_t idx) {
        float4 t = accumulate ? *reinterpret_cast<const float4*>(gsum + idx) : zero4();
#pragma unroll
        for (int b = 0; b < RM; ++b)
            if (src[b]) t = add4(t, *reinterpret_cast<const float4*>(src[b] + idx));
        *reinterpret_cast<float4*>(gsum + idx) = t;
    };
    const int j0 = v.gg * p.gpg, jend = min(j0 + p.gpg, n_loc);
    const int pm = p.pmask, Hq = p.Hp >> 2;   // the adjoint parameters' parts only (rows_theta_pass)
    if (v.qok) {
        for (int blk = 0; blk < 2; ++blk) {
            if (!(pm & (blk == 0 ? PHX_P_WA : (v.q >= Hq ? PHX_P_WP : PHX_P_WS)))) continue;
            const size_t base = (blk == 0 ? off.WA : off.W1) + (size_t)g_lo * p.K2 + 4 * (size_t)v.q;
            for (int j = j0; j < jend; ++j) quad(base + (size_t)j * p.K2);
        }
        if (blockIdx.x == 0 && v.gg == 0 && (pm & (v.q >= Hq ? PHX_P_BP : PHX_P_BS))) quad(off.bias + 4 * (size_t)v.q);
    }
    // multipliers: thread (gene j, row b) of the passes wrote element j of row b; lane b == 0 of every gene sums the rows
    // after the warp's writes are visible to it (same warp: the four row-threads of a gene are adjacent lanes)
    __syncwarp();
    for (int e = threadIdx.x; (pm & PHX_P_M) && e < n_loc * RM; e += THREADS) {
        if ((e & 3) != 0) continue;
        const size_t idx = off.m + g_lo + (e >> 2);
        float t = accumulate ? gsum[idx] : 0.f;
#pragma unroll
        for (int b = 0; b < RM; ++b)
            if (src[b]) t += src[b][idx];
        gsum[idx] = t;
    }
}

// Per-row sum over ALL theta elements of (k / atol)^2, k = k[fs1] - k[fs0] (fs0 < 0: k = k[fs1]), valid while the row's
// theta is identically zero (scale = atol, misc.py:63): no pass over memory, only Gram sums of the factors.  Returns this
// CTA's contribution for row threadIdx.x (threads 0..RM-1; other threads get 0).  zmask: rows to evaluate.
__device__ __noinline__ double rows_theta_zero_norm(const ResParams& __restrict__ p, int n_loc, uint32_t tmem, int sid1,
                                                    int sid0) {
    Smem s(p);
    s.tmem = tmem;
    RowsView v(p, s);
    v.tq = tm_quarter(tmem);
    const RowsCtl* rc = v.rc();
    const int BL = RM * p.gpc, Hq = p.Hp >> 2;
    double* gram = s.gram();   // [4 quad-warps][RM][12]
    // K2-long factors: warp (qw, gg) takes row gg
    if (v.gg < RM) {
        const RowCtl& c = rc->r[v.gg];
        const int f1 = c.fslot[sid1], f0 = sid0 >= 0 ? c.fslot[sid0] : c.fslot[sid1];
        float4 sp1, sp0, g1, g0;
        const int bt = v.gg < p.rows ? v.gg : 0;   // the rows a pass does not hold have no factor columns (val stays 0)
        tm_ld4(v.col_fsp(f1, bt), sp1);
        tm_ld4(v.col_fsp(f0, bt), sp0);
        tm_ld4(v.col_fg(f1, bt), g1);
        tm_ld4(v.col_fg(f0, bt), g0);
        double val[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // sp11 sp10 sp00 | gs11 gs10 gs00 | gp11 gp10 gp00
        if (v.qok && v.gg < p.rows) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const double a1 = comp4(sp1, e), a0 = comp4(sp0, e), b1 = comp4(g1, e), b0 = comp4(g0, e);
                val[0] += a1 * a1; val[1] += a1 * a0; val[2] += a0 * a0;
                const int o = v.q >= Hq ? 6 : 3;
                val[o] += b1 * b1; val[o + 1] += b1 * b0; val[o + 2] += b0 * b0;
            }
        }
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            const double t = warp_sum_d(val[i]);
            if (v.lane == 0) gram[(v.qw * RM + v.gg) * 12 + i] = t;
        }
    }
    // per-gene factors: thread (gene, row)
    double ug[6] = {0, 0, 0, 0, 0, 0}, ul[4] = {0, 0, 0, 0};   // gj11 gj10 gj00 s11 s10 s00 | l11 l10 l00 m
    for (int e = threadIdx.x; e < n_loc * RM; e += THREADS) {
        const RowCtl& c = rc->r[e & 3];
        const int f1 = c.fslot[sid1], f0 = sid0 >= 0 ? c.fslot[sid0] : c.fslot[sid1];
        float s1, l1, s0, l0, den;
        hill(v.ysf()[e * NFS + f1], s1, l1, den);
        hill(v.ysf()[e * NFS + f0], s0, l0, den);
        const double gj1 = v.fgj()[e * NFS + f1], gj0 = v.fgj()[e * NFS + f0];
        ug[0] += gj1 * gj1; ug[1] += gj1 * gj0; ug[2] += gj0 * gj0;
        ug[3] += (double)s1 * s1; ug[4] += (double)s1 * s0; ug[5] += (double)s0 * s0;
        ul[0] += (double)l1 * l1; ul[1] += (double)l1 * l0; ul[2] += (double)l0 * l0;
        const float km = v.fm()[e * NFS + f1] - (sid0 >= 0 ? v.fm()[e * NFS + f0] : 0.f);
        ul[3] += (double)km * (double)km;
    }
    double* tot = s.at<double>(p.so.rsum) + WARPS * RM * 8;   // [RM][8] x 2 (the tail of the per-row sum buffer)
    block_sum_rows<6>(v, ug, tot);
    double keep[6];
    if (threadIdx.x < RM)
        for (int i = 0; i < 6; ++i) keep[i] = tot[threadIdx.x * 6 + i];
    __syncthreads();
    block_sum_rows<4>(v, ul, tot);
    double res = 0;
    if (threadIdx.x < RM) {
        const int b = threadIdx.x;
        double V9[9];
        for (int i = 0; i < 9; ++i) {
            double t = 0;
            for (int w = 0; w < p.nqw; ++w) t += gram[(w * RM + b) * 12 + i];
            V9[i] = t;
        }
        const double* L = tot + b * 4;
        auto comb = [&](double u11, double u10, double u00, double v11, double v10, double v00) {
            return sid0 >= 0 ? (u11 * v11 - 2.0 * u10 * v10 + u00 * v00) : u11 * v11;
        };
        const int pm = p.pmask;   // the adjoint parameters only
        if (pm & PHX_P_WA) res += comb(keep[0], keep[1], keep[2], V9[0], V9[1], V9[2]);   // WAbar: gJ x S|Pr
        if (pm & PHX_P_WS) res += comb(keep[3], keep[4], keep[5], V9[3], V9[4], V9[5]);   // Wsbar: s x gS
        if (pm & PHX_P_WP) res += comb(L[0], L[1], L[2], V9[6], V9[7], V9[8]);             // Wpbar: l x gLP
        if (pm & PHX_P_M) res += L[3];                                                     // mbar
        if (blockIdx.x == 0) {   // (x + 0.0 == x: with both biases the sum is formed as before)
            const double bs2 = sid0 >= 0 ? (V9[3] - 2.0 * V9[4] + V9[5]) : V9[3];
            const double bp2 = sid0 >= 0 ? (V9[6] - 2.0 * V9[7] + V9[8]) : V9[6];
            if (pm & (PHX_P_BS | PHX_P_BP)) res += ((pm & PHX_P_BS) ? bs2 : 0.0) + ((pm & PHX_P_BP) ? bp2 : 0.0);
        }
        res /= (double)p.atol_f * (double)p.atol_f;
    }
    __syncthreads();
    return res;
}

// SEMI: the seminorm (p.pmask & PHX_NORM_SEMINORM), an instantiation of its own so that the default norm keeps its code
template <bool SEMI>
__global__ void __launch_bounds__(PHX_THREADS, 1) phx_rows_adj_kernel(const __grid_constant__ ResParams p) {
    Smem s(p);
    RowsView v(p, s);
    rows_prologue(p, s, v, p.ring_rows);
    Prof& pf = s.pf;
    RowsCtl* rc = v.rc();
    const int g_lo = s.g_lo, n_loc = s.n_loc;
    const int tot = n_loc * RM, BL = RM * p.gpc;
    const double Nel = (double)p.G;
    // theta block of the norm: the adjoint parameters only; with none the block is absent (th_rms == 0 never wins the
    // max over the other, non-negative blocks).  The seminorm drops it too: no theta norm pass or Gram sum runs, and the
    // theta step pass moves after the accept decision (accepted rows only, solution combination only)
    constexpr bool semi = SEMI;
    const double Pel = semi ? 0.0 : (double)phx_mask_count(p.G, p.H, p.pmask);
    auto th_rms = [&](double sum) { return Pel > 0 ? sqrtf((float)(sum / Pel)) : 0.f; };
    float* Y = v.st(0);
    float* A = v.st(1);
    float* Y1 = v.st(2);
    float* A1 = v.st(3);
    auto KY = [&](int i) { return v.st(4 + i); };
    auto KA = [&](int i) { return v.st(11 + i); };
    double* dsum = s.at<double>(p.so.dred) + 64;   // [RM * 8] block / grid totals (the first 64 doubles: theta-pass scratch)
    double* tsum = s.at<double>(p.so.dred) + 112;  // [2 * RM] theta-pass totals
    RowPP* pp = s.at<RowPP>(p.so.ppa);
    const bool dop = p.method == PHX_DOPRI5;
    // factor slots a method never writes (euler: 1..5, ...) enter the theta passes with weight 0: they must hold finite
    // values, so every table starts at zero (shared memory and tensor memory)
    for (int i = threadIdx.x; i < NFS * BL; i += THREADS) {
        v.ysf()[i] = 0.5f;
        v.fgj()[i] = 0.f;
        v.fm()[i] = 0.f;
    }
    if (v.warp < 4) {
        for (int c = 0; c < 2 * NFS * p.rows; ++c) tm_st4(v.tq + (uint32_t)(p.tm_fac + 4 * c), zero4());
        tm_wait_st();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    for (int q0 = 0; q0 < p.ntot; q0 += p.rows) {
        const int nr = min(p.rows, p.ntot - q0);
        float* const gacc = p.gsum + (size_t)(q0 / p.rows) * p.ppk;   // this group's packed cotangent sum
        if (threadIdx.x < RM) {
            RowCtl& c = rc->r[threadIdx.x];
            row_init(c, (int)threadIdx.x < nr);
            if (!dop)
                for (int i = 0; i < 7; ++i) c.fslot[i] = i < NFS ? i : -1;
        }
        if (threadIdx.x == 0) rc->spec_valid = rc->spec_pass = rc->redo = 0;
        __syncthreads();
        // Speculative final step.  When EVERY row still active is on the step that (if accepted) ends its last interval,
        // the theta pass adds the rows' final values straight into the group's sum instead of storing them per row and
        // summing afterwards (35.8 MB written + read back per sample at the headline shape).  Acceptance is only known
        // after the pass: if a row is rejected the sum is void, the accepted rows are re-run into their own buffers (their
        // factors are still on chip) and the group falls back to the explicit sum.
        auto plan_spec = [&](bool final_iv) {   // thread 0, after the RowPP block is filled
            bool any = false, all = true;
            for (int b = 0; b < RM; ++b) {
                if (!pp[b].active) continue;
                any = true;
                all = all && pp[b].last && final_iv;
            }
            const bool spec = any && all && !rc->spec_valid;
            rc->spec_pass = spec;
            bool first = true;
            for (int b = 0; b < RM; ++b) {
                pp[b].acc = gacc;
                pp[b].spec = (spec && pp[b].active) ? (first ? 1 : 2) : 0;
                if (pp[b].spec) first = false;
            }
        };
        auto set_input = [&](int e, int j, float ys, float as, int fs) {
            s.ysb()[e] = ys;
            float sv, lv, den;
            hill(ys, sv, lv, den);
            s.acts()[e] = sv;
            v.actL()[e] = lv;
            s.asb()[e] = as;
            s.gjb()[e] = as * s.relum()[j];
            if (fs >= 0) v.ysf()[e * NFS + fs] = ys;
        };
        auto no_y = [](int, int, int, float) { return 0.f; };

        for (int iv = p.T - 1; iv >= 1; --iv) {
            const bool first_iv = iv == p.T - 1;
            if (dop) {
                // dopri5 restarts every interval from the identity slot maps.  This comes before the loads: they store
                // the stage-0 input record into factor slot fslot[0], which the last interval's accepted steps may have
                // swapped to slot 5 (FSAL), where stage 0 of this interval would not read it.
                if (threadIdx.x < RM) {
                    RowCtl& c = rc->r[threadIdx.x];
                    for (int i = 0; i < 7; ++i) c.slot[i] = i;
                    c.fslot[0] = 0;
                    c.fslot[1] = -1;
                    for (int i = 2; i < 7; ++i) c.fslot[i] = i - 1;
                }
                __syncthreads();
            }
            for (int e = threadIdx.x; e < p.gpc * RM; e += THREADS) {
                const int j = e >> 2, b = e & 3;
                float y = 0.5f, av = 0.f;
                if (b < nr && j < n_loc) {
                    const size_t gi = (size_t)(q0 + b) * p.yout_stride + (size_t)iv * p.G + g_lo + j;
                    y = p.ysaved[gi];
                    av = first_iv ? p.grad_y[gi] : A[e];
                }
                Y[e] = y;
                A[e] = av;
                set_input(e, j, y, av, rc->r[b].fslot[0]);
            }
            if (threadIdx.x < RM) {
                RowCtl& c = rc->r[threadIdx.x];
                c.done = !c.valid || c.code != PHX_ST_OK;
                if (c.valid) {
                    const double ta = tget_rows(p, q0 + threadIdx.x, iv - 1), tb = tget_rows(p, q0 + threadIdx.x, iv);
                    c.tcur = c.tprev = -tb;
                    c.t_end = -ta;
                    c.n_steps_interval = 0;
                    c.dtf = p.t_is_f32 ? ((float)tb - (float)ta) : (float)(tb - ta);
                }
            }
            __syncthreads();

            if (!dop) {
                const float third = (float)(1.0 / 3.0);
                const int nst = (p.method == PHX_EULER) ? 1 : (p.method == PHX_MIDPOINT ? 2 : 4);
                // one step per interval, or the steps of each row's own grid of this interval (p.gdt): a row that has
                // taken all of its steps sits out (RowPP.active = 0) until every row has
                int nk = 1;
                if (p.gdt) {
                    nk = 0;
                    for (int b = 0; b < nr; ++b) {
                        const int sg = (q0 + b) * (p.T - 1) + iv - 1;
                        nk = max(nk, p.goff[sg + 1] - p.goff[sg]);
                    }
                }
                for (int k = 0; k < nk; ++k) {
                if (k > 0) {   // the next step starts from the state the last one left in Y / A
                    for (int e = threadIdx.x; e < p.gpc * RM; e += THREADS)
                        set_input(e, e >> 2, Y[e], A[e], rc->r[e & 3].fslot[0]);
                }
                if (threadIdx.x < RM) {
                    RowCtl& c = rc->r[threadIdx.x];
                    RowPP& a = pp[threadIdx.x];
                    int rk = 1;
                    if (p.gdt && c.valid) {
                        const int sg = (q0 + threadIdx.x) * (p.T - 1) + iv - 1;
                        rk = p.goff[sg + 1] - p.goff[sg];
                        c.dtf = k < rk ? p.gdt[p.goff[sg] + k] : 0.f;
                    }
                    c.stepping = !c.done && k < rk;
                    float* th = p.theta_ws + (size_t)(2 * threadIdx.x) * p.ppk;
                    a.src = c.theta_zero ? nullptr : th;
                    a.dst = th;
                    for (int f = 0; f < NFS; ++f) a.cs[f] = a.ce[f] = a.wo[f] = 0.f;
                    if (p.method == PHX_EULER) {
                        a.wo[0] = c.dtf;
                    } else if (p.method == PHX_MIDPOINT) {
                        a.wo[1] = c.dtf;
                    } else {   // 3/8 rule: (k1 + 3 (k2 + k3) + k4) dt / 8
                        a.wo[0] = a.wo[3] = c.dtf * 0.125f;
                        a.wo[1] = a.wo[2] = 3.f * c.dtf * 0.125f;
                    }
                    a.last = k + 1 == rk;
                    a.active = c.stepping;
                }
                __syncthreads();
                if (threadIdx.x == 0) plan_spec(iv == 1);
                const bool more = k + 1 < nk;
                for (int st = 0; st < nst; ++st) {
                    const bool last = st + 1 == nst;
                    rows_adj_eval(
                        p, s, v, st, st + 1, st > 0, !last,
                        [&](int b, int j, int li, float ky) {
                            const float dtf = rc->r[b].dtf;
                            if (p.method == PHX_MIDPOINT) return Y[li] + ky * (0.5f * dtf);
                            if (st == 0) return Y[li] + dtf * ky * third;
                            if (st == 1) return Y[li] + dtf * (ky - KY(0)[li] * third);
                            return Y[li] + dtf * (KY(0)[li] - KY(1)[li] + ky);
                        },
                        [&](int b, int j, int li, float ka) {
                            const float dtf = rc->r[b].dtf;
                            float an;
                            if (p.method == PHX_EULER) {
                                an = A[li] + dtf * ka;
                            } else if (p.method == PHX_MIDPOINT) {
                                an = (st == 0) ? A[li] + ka * (0.5f * dtf) : A[li] + dtf * ka;
                            } else {
                                if (st == 0) an = A[li] + dtf * ka * third;
                                else if (st == 1) an = A[li] + dtf * (ka - KA(0)[li] * third);
                                else if (st == 2) an = A[li] + dtf * (KA(0)[li] - KA(1)[li] + ka);
                                else an = A[li] + (KA(0)[li] + 3.f * (KA(1)[li] + KA(2)[li]) + ka) * dtf * 0.125f;
                            }
                            if (last && rc->r[b].stepping) {
                                A[li] = an;
                                if (more) {   // y at the step's end (KY of every stage is in place after pass 1)
                                    const float ky = KY(nst - 1)[li];
                                    if (p.method != PHX_RK4) Y[li] = Y[li] + dtf * ky;
                                    else Y[li] = Y[li] + (KY(0)[li] + 3.f * (KY(1)[li] + KY(2)[li]) + ky) * dtf * 0.125f;
                                }
                            }
                            return an;
                        });
                }
                __syncthreads();
                rows_theta_pass<TP_FIXED, SEMI>(p, g_lo, n_loc, s.tmem, tsum);
                pf.tick(PT_PP_STEP);
                if (threadIdx.x < RM) {
                    RowCtl& c = rc->r[threadIdx.x];
                    if (c.stepping) {
                        if (pp[threadIdx.x].spec) c.spec_done = 1;
                        else { c.theta_zero = 0; c.cur = 0; }
                        c.n_rhs += nst;
                        c.tcur = c.t_end;
                    }
                }
                if (threadIdx.x == 0 && rc->spec_pass) rc->spec_valid = 1;
                __syncthreads();
                }
            } else {
                // ------------------------------ dopri5 on the augmented state, one controller per row -----------------
                // (the slot maps were reset to the identity at the interval start: the loads above stored the stage-0
                // input record into factor slot 0)
                for (int which = 0; which < 2; ++which) {
                    const int sid = which == 0 ? 0 : 6;
                    double acc[7] = {0, 0, 0, 0, 0, 0, 0};
                    rows_adj_eval(p, s, v, sid, sid, false, false, no_y, [&](int b, int j, int li, float ka) {
                        const RowCtl& c = rc->r[b];
                        const float y = Y[li], av = A[li];
                        const float sy = p.atol_f + fabsf(y) * p.rtol_f, sa = p.atol_f + fabsf(av) * p.rtol_f;
                        float r;
                        if (which == 0) {
                            r = y / sy; acc[0] += (double)(r * r);
                            r = av / sa; acc[1] += (double)(r * r);
                            r = KY(c.slot[0])[li] / sy; acc[3] += (double)(r * r);
                            r = ka / sa; acc[4] += (double)(r * r);
                            if (!isfinite(y) || !isfinite(av)) acc[6] += 1.0;
                        } else {
                            r = (KY(c.slot[6])[li] - KY(c.slot[0])[li]) / sy; acc[0] += (double)(r * r);
                            r = (ka - KA(c.slot[0])[li]) / sa; acc[1] += (double)(r * r);
                        }
                        return 0.f;
                    });
                    // theta norms: Gram sums while a row's accumulator is still zero, a pass over memory otherwise (none
                    // under the seminorm)
                    bool any_nz = false;
                    for (int b = 0; b < RM; ++b) any_nz |= (!rc->r[b].done && !rc->r[b].theta_zero);
                    if (threadIdx.x < RM) {
                        const RowCtl& c = rc->r[threadIdx.x];
                        RowPP& a = pp[threadIdx.x];
                        a.src = p.theta_ws + (size_t)(2 * threadIdx.x + c.cur) * p.ppk;
                        a.dst = nullptr;
                        a.s0 = c.fslot[0];
                        a.s1 = c.fslot[6];
                        a.active = !c.done && !c.theta_zero;
                    }
                    __syncthreads();
                    // (a given first step needs no norm)
                    const bool thn = !semi && !(p.first_step > 0);
                    const double zn =
                        thn ? rows_theta_zero_norm(p, n_loc, s.tmem, which == 0 ? 0 : 6, which == 0 ? -1 : 0) : 0.0;
                    if (any_nz && thn) {
                        if (which == 0) rows_theta_pass<TP_D01, SEMI>(p, g_lo, n_loc, s.tmem, tsum);
                        else rows_theta_pass<TP_D2, SEMI>(p, g_lo, n_loc, s.tmem, tsum);
                    }
                    pf.tick(which == 0 ? PT_PP_D01 : PT_PP_D2);
                    block_sum_rows<7>(v, acc, dsum);
                    if (threadIdx.x < RM) {
                        const RowCtl& c = rc->r[threadIdx.x];
                        double* d = dsum + threadIdx.x * 7;
                        if (!thn) {
                            // (the seminorm has no theta block; a given first step needs none)
                        } else if (c.theta_zero) {
                            d[which == 0 ? 5 : 2] += zn;
                        } else if (which == 0) {
                            d[2] += tsum[2 * threadIdx.x];
                            d[5] += tsum[2 * threadIdx.x + 1];
                        } else {
                            d[2] += tsum[2 * threadIdx.x];
                        }
                    }
                    __syncthreads();
                    grid_sum_d(p, s, dsum, 7 * RM);
                    pf.tick(PT_NORMS);
                    if (threadIdx.x < RM) {
                        RowCtl& c = rc->r[threadIdx.x];
                        const double* d = dsum + threadIdx.x * 7;
                        if (which == 0) {
                            float d0 = fmaxf(fmaxf(sqrtf((float)(d[0] / Nel)), sqrtf((float)(d[1] / Nel))),
                                             th_rms(d[2]));
                            const bool bad_v =
                                c.valid && p.t_vjp &&
                                fold_t_vjp(p, p.t_vjp[(size_t)(q0 + threadIdx.x) * (p.T - 1) + iv - 1], d0);
                            const float d1 = fmaxf(fmaxf(sqrtf((float)(d[3] / Nel)), sqrtf((float)(d[4] / Nel))),
                                                   th_rms(d[5]));
                            c.d1 = d1;
                            c.h0 = init_h0(d0, d1);
                            c.nonfinite_prev = d[6] > 0.0 || bad_v;
                            if (p.first_step > 0) {
                                c.dt = p.first_step;
                                if (!c.done) c.n_rhs += 1;
                            }
                        } else {
                            const float d2 = fmaxf(fmaxf(sqrtf((float)(d[0] / Nel)), sqrtf((float)(d[1] / Nel))),
                                                   th_rms(d[2])) / c.h0;
                            c.dt = init_dt(c.h0, c.d1, d2);
                            if (!c.done) c.n_rhs += 2;
                        }
                    }
                    __syncthreads();
                    if (p.first_step > 0) break;   // the caller's first step (every row's): no second evaluation
                    if (which == 0) {
                        for (int e = threadIdx.x; e < tot; e += THREADS) {
                            const RowCtl& c = rc->r[e & 3];
                            set_input(e, e >> 2, Y[e] + c.h0 * KY(c.slot[0])[e], A[e] + c.h0 * KA(c.slot[0])[e], c.fslot[6]);
                        }
                        __syncthreads();
                    }
                }
                while (true) {
                    if (threadIdx.x < RM) {
                        RowCtl& c = rc->r[threadIdx.x];
                        if (!c.done && row_prestep(p, c)) {
                            // this step, if accepted, reaches t_end: same comparison as rk_common.py:153 after the step
                            c.last = !(c.t_end > c.tcur + c.dt);
                            if (c.last) row_set_interp_x(c, c.t_end, c.tcur, c.tcur + c.dt);
                        }
                    }
                    __syncthreads();
                    if (threadIdx.x == 0) {
                        int all = 1;
                        for (int b = 0; b < RM; ++b) all &= rc->r[b].done;
                        rc->all_done = all;
                    }
                    __syncthreads();
                    if (rc->all_done) break;
                    for (int e = threadIdx.x; e < tot; e += THREADS) {
                        const RowCtl& c = rc->r[e & 3];
                        const float c00 = c.cb[0][0];
                        set_input(e, e >> 2, Y[e] + KY(c.slot[0])[e] * c00, A[e] + KA(c.slot[0])[e] * c00, -1);
                    }
                    __syncthreads();
                    double acc[4] = {0, 0, 0, 0};
                    for (int st = 1; st <= 6; ++st) {
                        rows_adj_eval(
                            p, s, v, st, st + 1, st > 1, st < 6,
                            [&](int b, int j, int li, float ky) {
                                const RowCtl& c = rc->r[b];
                                const int* sl = c.slot;
                                float ay = KY(sl[0])[li] * c.cb[st][0];
                                for (int qq = 1; qq < st; ++qq) ay = fmaf(KY(sl[qq])[li], c.cb[st][qq], ay);
                                ay = fmaf(ky, c.cb[st][st], ay);
                                const float yn = Y[li] + ay;
                                if (st == 5) Y1[li] = yn;
                                return yn;
                            },
                            [&](int b, int j, int li, float ka) {
                                const RowCtl& c = rc->r[b];
                                const int* sl = c.slot;
                                if (st < 6) {
                                    float aa = KA(sl[0])[li] * c.cb[st][0];
                                    for (int qq = 1; qq < st; ++qq) aa = fmaf(KA(sl[qq])[li], c.cb[st][qq], aa);
                                    aa = fmaf(ka, c.cb[st][st], aa);
                                    const float an = A[li] + aa;
                                    if (st == 5) A1[li] = an;
                                    return an;
                                }
                                float ey = KY(sl[0])[li] * c.cerr[0];
                                float ea = KA(sl[0])[li] * c.cerr[0];
                                for (int qq = 1; qq < 6; ++qq) {
                                    ey = fmaf(KY(sl[qq])[li], c.cerr[qq], ey);
                                    ea = fmaf(KA(sl[qq])[li], c.cerr[qq], ea);
                                }
                                ey = fmaf(KY(sl[6])[li], c.cerr[6], ey);
                                ea = fmaf(ka, c.cerr[6], ea);
                                const float y1 = s.ysb()[li], a1 = s.asb()[li];
                                const float ty = p.atol_f + p.rtol_f * fmaxf(fabsf(Y[li]), fabsf(y1));
                                const float ta = p.atol_f + p.rtol_f * fmaxf(fabsf(A[li]), fabsf(a1));
                                float r;
                                r = ey / ty; acc[0] += (double)(r * r);
                                r = ea / ta; acc[1] += (double)(r * r);
                                if (!isfinite(y1) || !isfinite(a1)) acc[3] += 1.0;
                                return 0.f;
                            });
                    }
                    if (threadIdx.x < RM) {
                        const RowCtl& c = rc->r[threadIdx.x];
                        RowPP& a = pp[threadIdx.x];
                        float* t0 = p.theta_ws + (size_t)(2 * threadIdx.x) * p.ppk;
                        float* t1 = t0 + p.ppk;
                        a.src = c.theta_zero ? nullptr : (c.cur ? t1 : t0);
                        a.dst = c.theta_zero ? t0 : (c.cur ? t0 : t1);
                        a.last = c.last;
                        a.active = !c.done;
                        for (int qq = 0; qq < 7; ++qq) {
                            const int fs = c.fslot[qq];
                            if (fs < 0) continue;
                            a.cs[fs] = (qq < 6) ? c.cb[5][qq] : 0.f;
                            a.ce[fs] = c.cerr[qq];
                            a.wo[fs] = a.cs[fs];
                        }
                        if (c.last) rows_interp_weights(c, a);
                    }
                    __syncthreads();
                    if (threadIdx.x == 0 && !semi) plan_spec(iv == 1);
                    __syncthreads();
                    pf.tick(PT_COMBINE);
                    if (!semi) rows_theta_pass<TP_STEP, SEMI>(p, g_lo, n_loc, s.tmem, tsum);
                    pf.tick(PT_PP_STEP);
                    block_sum_rows<4>(v, acc, dsum);
                    if (threadIdx.x < RM && !semi) {
                        dsum[threadIdx.x * 4 + 2] += tsum[2 * threadIdx.x];
                        dsum[threadIdx.x * 4 + 3] += tsum[2 * threadIdx.x + 1];
                    }
                    __syncthreads();
                    grid_sum_d(p, s, dsum, 4 * RM);
                    pf.tick(PT_NORMS);
                    if (threadIdx.x < RM) {
                        RowCtl& c = rc->r[threadIdx.x];
                        c.accept = 0;
                        if (!c.done) {
                            const double* d = dsum + threadIdx.x * 4;
                            float ratio = fmaxf(fmaxf(sqrtf((float)(d[0] / Nel)), sqrtf((float)(d[1] / Nel))),
                                                th_rms(d[2]));
                            // torch's max() over 0-dim tensors is Python max: a NaN in a later block does not propagate
                            // the same way; treat any NaN as NaN (step rejected, dt -> NaN -> underflow assertion)
                            if (isnan(d[0]) || isnan(d[1]) || isnan(d[2])) ratio = nanf("");
                            const int accept = ratio <= 1.f;
                            row_log_step(p, c, q0 + threadIdx.x, c.tcur, c.dt, accept);
                            c.tprev = c.tcur;
                            if (accept) {
                                c.tcur = c.tcur + c.dt;
                                c.n_acc++;
                                c.nonfinite_prev = d[3] > 0.0;
                            } else {
                                c.n_rej++;
                            }
                            c.dt = next_dt(p, c.dt, ratio);
                            c.accept = accept;
                            c.n_rhs += 6;
                            c.n_steps_interval++;
                        }
                    }
                    __syncthreads();
                    if (semi) {
                        // the accepted rows' theta step, as a fixed-grid pass with the solution (or dense-output)
                        // weights wo: acceptance is known, so a speculative final step goes straight into the group sum
                        if (threadIdx.x < RM) pp[threadIdx.x].active = rc->r[threadIdx.x].accept;
                        __syncthreads();
                        if (threadIdx.x == 0) plan_spec(iv == 1);
                        __syncthreads();
                        rows_theta_pass<TP_FIXED, SEMI>(p, g_lo, n_loc, s.tmem, tsum);
                        pf.tick(PT_PP_STEP);
                        if (threadIdx.x < RM && pp[threadIdx.x].spec) rc->r[threadIdx.x].spec_done = 1;
                        if (threadIdx.x == 0 && rc->spec_pass) rc->spec_valid = 1;
                        __syncthreads();
                    } else if (rc->spec_pass) {
                        // did every speculating row accept?  otherwise materialise the accepted ones
                        if (threadIdx.x == 0) {
                            bool ok = true;
                            for (int b = 0; b < RM; ++b) ok = ok && (!pp[b].spec || rc->r[b].accept);
                            rc->spec_valid = ok;
                            rc->redo = !ok;
                            for (int b = 0; b < RM; ++b) {
                                if (ok && pp[b].spec) rc->r[b].spec_done = 1;
                                if (!ok) {
                                    pp[b].active = pp[b].spec && rc->r[b].accept;
                                    pp[b].spec = 0;
                                }
                            }
                        }
                        __syncthreads();
                        if (rc->redo) rows_theta_pass<TP_STEP, SEMI>(p, g_lo, n_loc, s.tmem, tsum);
                    }
                    for (int e = threadIdx.x; e < tot; e += THREADS) {
                        const RowCtl& c = rc->r[e & 3];
                        if (!c.accept) continue;
                        if (c.last) {
                            // last step of the interval: dense output at t_end for adj_y (adj_params: done in the pass)
                            const int* sl = c.slot;
                            const float a0 = A[e], a1 = A1[e];
                            float m = KA(sl[0])[e] * c.cmid[0];
                            for (int qq = 1; qq < 7; ++qq) m = fmaf(KA(sl[qq])[e], c.cmid[qq], m);
                            A[e] = interp_eval(a0, a1, a0 + m, KA(sl[0])[e], KA(sl[6])[e], c.dtf, c.xs);
                        } else {
                            Y[e] = Y1[e];
                            A[e] = A1[e];
                        }
                    }
                    __syncthreads();
                    if (threadIdx.x < RM) {
                        RowCtl& c = rc->r[threadIdx.x];
                        if (c.accept) {
                            if (!c.spec_done) {
                                if (c.theta_zero) { c.cur = 0; c.theta_zero = 0; } else c.cur ^= 1;
                            }
                            if (c.last) {
                                c.done = 1;
                            } else {
                                int t0 = c.slot[0]; c.slot[0] = c.slot[6]; c.slot[6] = t0;
                                t0 = c.fslot[0]; c.fslot[0] = c.fslot[6]; c.fslot[6] = t0;
                            }
                        }
                    }
                    __syncthreads();
                    pf.tick(PT_CTRL);
                }
            }
            // interval done: adj_y picks up the loss gradient at t[iv-1] (adjoint.py:152-154)
            for (int e = threadIdx.x; e < tot; e += THREADS) {
                const int j = e >> 2, b = e & 3;
                if (b < nr && rc->r[b].code == PHX_ST_OK)
                    A[e] = A[e] + p.grad_y[(size_t)(q0 + b) * p.yout_stride + (size_t)(iv - 1) * p.G + g_lo + j];
            }
            __syncthreads();
        }
        for (int e = threadIdx.x; e < tot; e += THREADS) {
            const int j = e >> 2, b = e & 3;
            if (b < nr)   // (NaN for a row stopped by a solver assertion)
                p.adj_y0[(size_t)(q0 + b) * p.adj_stride + g_lo + j] = rc->r[b].code == PHX_ST_OK ? A[e] : nanf("");
        }
        rows_theta_sum(p, g_lo, n_loc, gacc, rc->spec_valid != 0);
        pf.tick(PT_PP_COPY);
        if (threadIdx.x < nr) row_write_status(p, q0 + threadIdx.x, rc->r[threadIdx.x]);
        __syncthreads();
    }
    pf.finish();
    rows_release(p, s);
    epilogue_epoch(p, s);
}

}  // namespace
