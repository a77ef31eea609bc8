// Persistent ("resident") PHOENIX solver kernels for sm_100a: one cooperative launch integrates a whole odeint call
// (forward) or a whole adjoint sweep (backward) with the step controller on the device.
//
// Decomposition (B200-first, SURVEY.md 8a rows a3, a6-a16):
//   * the G genes are split into contiguous slices, one CTA (one SM) per slice; the CTA owns every per-gene
//     quantity of its slice -- solver state, RK stage derivatives, Hill activations, all held in SHARED MEMORY for the
//     whole solve -- and the rows W1[g][:], WA[g][:] of the packed weights, which are one contiguous block per CTA
//     and are streamed through a ring of shared-memory stages by 1-D TMA bulk copies (cp.async.bulk + mbarrier),
//     prefetched across the inter-CTA exchanges; after the first pass they come from L2 (16GH bytes << 126 MB);
//   * an RHS evaluation is: pass A over W1 (branch pre-activations, reduced over the slice's genes) -> ONE
//     grid-wide all-reduce of the K2-long branch vector -> pass B over WA (combination row-dots, decay) -> the RK
//     stage combine for the slice, all inside the same kernel: the state never makes an HBM round trip;
//   * the adjoint adds a second all-reduce (gS|gLP) and pass C over W1 (state cotangent), which is MERGED with
//     pass A of the next stage (same rows), so a VJP evaluation streams each weight matrix once; the parameter
//     cotangents stay FACTORISED per stage (rank-B outer-product factors in shared memory) and are folded into the
//     P-long accumulator once per step together with their error-norm contribution; while the accumulator is known
//     to be zero it is never read, and the last step of an interval writes the dense-output value directly (the
//     reference carries seven P-long stage tensors through every stage, adjoint.py:86-151 + rk_common.py:62-76);
//   * inter-CTA exchanges use tagged 64-bit slots ({fp32, epoch}, one relaxed store / polled relaxed loads, no
//     fences, no atomics; PhxLL in phx_common.cuh) and are summed in a fixed order: results are run-to-run
//     deterministic and identical in every CTA, which the device-side dopri5 controller relies on.
//
// Arithmetic mirrors the reference op by op where it is elementwise (compiled with -fmad=false, explicit fmaf only
// inside dot products), fp32 state, float64 time-like scalars (rk_common.py:115-131).
#include <math.h>
#include <stdio.h>
#pragma once
#include "phx_common.cuh"

namespace {

constexpr int THREADS = PHX_THREADS;
constexpr int WARPS = PHX_WARPS;

// Dormand-Prince tableau (dopri5.py:5-30), float64 constants rounded to fp32 at use like `.to(dtype=y0.dtype)`.
__constant__ double c_beta[6][6] = {
    {1.0 / 5, 0, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656, 0},
    {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84}};
__constant__ double c_err[7] = {35.0 / 384 - 1951.0 / 21600,
                                0,
                                500.0 / 1113 - 22642.0 / 50085,
                                125.0 / 192 - 451.0 / 720,
                                -2187.0 / 6784 - -12231.0 / 42400,
                                11.0 / 84 - 649.0 / 6300,
                                -1.0 / 60.0};
__constant__ double c_mid[7] = {6025192743.0 / 30085553152.0 / 2,
                                0,
                                51252292925.0 / 65400821598.0 / 2,
                                -2691868925.0 / 45128329728.0 / 2,
                                187940372067.0 / 1594534317056.0 / 2,
                                -1776094331.0 / 19743644256.0 / 2,
                                11237099.0 / 235043384.0 / 2};

struct Ctrl {
    double tcur, tprev, dt, dt_used, t_end;
    double dsum[8];
    float cb[6][6];
    float cerr[7];
    float cmid[7];
    float xs[4];  // x, x^2, x^3, x^4 for the dense output (interp.py:40-47)
    float dtf, h0, d1;
    int accept, stop, nonfinite_prev, last;
    int n_acc, n_rej, n_rhs, n_log, n_steps_interval;
    int slot[7];
    float vjp_t;  // adjoint: the time cotangent of the current interval (fold_t_vjp)
};

// Optional in-kernel phase timer (diagnostics; phx_ctx_set_profile): thread 0 of CTA 0 accumulates SM-clock deltas
// per phase into p.prof[slot].  With p.prof == nullptr every tick is one predictable branch.
enum {
    PT_SETUP = 0, PT_PHASE_A, PT_ALLRED1, PT_FINALIZE, PT_PHASE_B, PT_ALLRED2, PT_GSP, PT_PHASE_C, PT_EPILOGUE,
    PT_COMBINE, PT_PP_D01, PT_PP_D2, PT_PP_STEP, PT_PP_INTERP, PT_PP_COPY, PT_NORMS, PT_CTRL, PT_TOTAL, PT_COUNT
};
static_assert(PHX_LL_RCOPIES * 4 == 32, "replica posting assumes 8 replicas");
static_assert(sizeof(Ctrl) <= 512 && 512 + 8 * PT_COUNT <= PHX_CTRL_BYTES, "PHX_CTRL_BYTES too small");
struct Prof {
    long long* gbuf;   // global accumulators (thread 0 of CTA 0 only, else nullptr)
    long long* sbuf;   // shared-memory staging: ticks stay on chip, flushed once by finish()
    long long last, start;
    __device__ __forceinline__ void init(long long* g, long long* sm) {
        gbuf = (blockIdx.x == 0 && threadIdx.x == 0) ? g : nullptr;
        sbuf = sm;
        if (gbuf) {
            for (int i = 0; i < PT_COUNT; ++i) sbuf[i] = 0;
            last = start = clock64();
        }
    }
    __device__ __forceinline__ void tick(int slot) {
        if (gbuf) {
            long long t = clock64();
            sbuf[slot] += t - last;
            last = t;
        }
    }
    __device__ __forceinline__ void finish() {
        if (gbuf) {
            sbuf[PT_TOTAL] += clock64() - start;
            for (int i = 0; i < PT_COUNT; ++i) gbuf[i] += sbuf[i];
        }
    }
};

__device__ __forceinline__ double tget(const ResParams& p, int pi, int i) {
    return (p.T * p.nprob <= PHX_T_INLINE) ? p.t_small[pi * p.T + i] : p.t[pi * p.T + i];
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ void hill(float y, float& s, float& l, float& den) {
    float z = y - 0.5f;
    den = 1.0f + fabsf(z);
    s = z / den;
    l = log1pf(s);
}

// ---- tagged-slot ("LL") inter-CTA exchange ----------------------------------------------------------------------------
__device__ __forceinline__ void ll_put(unsigned long long* slot, float v, unsigned tag) {
    unsigned long long w = ((unsigned long long)tag << 32) | (unsigned long long)__float_as_uint(v);
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(slot), "l"(w) : "memory");
}
__device__ __forceinline__ unsigned long long ll_ld(const unsigned long long* slot) {
    unsigned long long w;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(slot) : "memory");
    return w;
}
__device__ __forceinline__ float ll_get(const unsigned long long* slot, unsigned tag) {
    unsigned long long w = ll_ld(slot);
    while ((unsigned)(w >> 32) != tag) w = ll_ld(slot);
    return __uint_as_float((unsigned)w);
}
// two adjacent slots in one 16-byte access (each 8-byte half is single-copy atomic and carries its own tag)
__device__ __forceinline__ void ll_put2(unsigned long long* slot, float v0, float v1, unsigned tag) {
    unsigned long long w0 = ((unsigned long long)tag << 32) | (unsigned long long)__float_as_uint(v0);
    unsigned long long w1 = ((unsigned long long)tag << 32) | (unsigned long long)__float_as_uint(v1);
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(slot), "l"(w0), "l"(w1) : "memory");
}
__device__ __forceinline__ void ll_ld2(const unsigned long long* slot, unsigned long long& w0, unsigned long long& w1) {
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(w0), "=l"(w1) : "l"(slot) : "memory");
}
__device__ __forceinline__ void ll_get2(const unsigned long long* slot, unsigned tag, float& v0, float& v1) {
    unsigned long long w0, w1;
    ll_ld2(slot, w0, w1);
    while ((unsigned)(w0 >> 32) != tag || (unsigned)(w1 >> 32) != tag) ll_ld2(slot, w0, w1);
    v0 = __uint_as_float((unsigned)w0);
    v1 = __uint_as_float((unsigned)w1);
}


// ---- shared-memory carve-up ---------------------------------------------------------------------------------------
// The byte offsets are computed on the host (phx_smem_layout, phx_common.cuh) and travel in the kernel parameters
// (constant bank): the views below cost no registers.  Only the three buffers that swap roles between consecutive
// stages of the adjoint keep their offsets in registers.
extern __shared__ __align__(128) unsigned char smem_raw[];

struct Xchg {
    unsigned long long ep;  // epoch counter (uniform over the grid); tags are its low 32 bits, never 0
    int ny, nd;             // one-phase / scalar exchanges done so far (double-buffer parity)
    __device__ __forceinline__ unsigned next_tag() {
        ++ep;
        if ((unsigned)ep == 0u) ++ep;
        return (unsigned)ep;
    }
};

struct Ring {
    unsigned par;   // this warp's per-slot parity of the next completion to wait for
    int pre;        // matrix (MAT_*) whose first rows are already in flight in this warp's slots, or -1
};


// Per-thread kernel context: shared-memory views + the (grid-uniform) exchange / ring / timer state.  Passed by
// reference to the __noinline__ building blocks so that the solver loops stay small enough for the instruction cache.
struct Smem {
    const ResParams& p;
    unsigned o_acts, o_actl, o_ysb, o_acts2, o_actl2, o_ysb2;
    int g_lo, n_loc;
    uint32_t tmem;   // tensor-memory base address of the parked WA slice (0: not used)
    Xchg x;
    Ring rg;
    Prof pf;
    __device__ __forceinline__ explicit Smem(const ResParams& pp)
        : p(pp), o_acts(pp.so.acts), o_actl(pp.so.actl), o_ysb(pp.so.ysb), o_acts2(pp.so.acts2),
          o_actl2(pp.so.actl2), o_ysb2(pp.so.ysb2) {
        g_lo = blockIdx.x * pp.gpc;
        n_loc = max(0, min(pp.gpc, pp.G - g_lo));
        tmem = 0u;
    }
    template <typename T>
    __device__ __forceinline__ T* at(unsigned off) const { return reinterpret_cast<T*>(smem_raw + off); }
    __device__ __forceinline__ Ctrl* ctrl() const { return at<Ctrl>(p.so.ctrl); }
    __device__ __forceinline__ double* dred() const { return at<double>(p.so.dred); }      // [WARPS][8]
    __device__ __forceinline__ double* gram() const { return at<double>(p.so.gram); }      // [2][64]   (adjoint)
    __device__ __forceinline__ float* dst16() const { return at<float>(p.so.dst16); }      // [PHX_LL_DMAX]
    __device__ __forceinline__ float* ystage() const { return at<float>(p.so.ystage); }    // [nCTA*B*K2] if use_y
    __device__ __forceinline__ float* bias() const { return at<float>(p.so.bias); }        // [K2]
    __device__ __forceinline__ float* relum() const { return at<float>(p.so.relum); }      // [gpc]
    __device__ __forceinline__ float* maskm() const { return at<float>(p.so.maskm); }      // [gpc]
    __device__ __forceinline__ float* sp() const { return at<float>(p.so.sp); }            // [B][K2]  S | Pr
    __device__ __forceinline__ float* xv() const { return at<float>(p.so.xv); }            // [2][B][K2] exchange vector
    __device__ __forceinline__ float* gsp() const { return at<float>(p.so.xv); }           // [B][K2]  gS | gLP  (= xv[0])
    __device__ __forceinline__ float* spn() const { return at<float>(p.so.xv) + p.B * p.K2; }  // next S|P (= xv[1])
    __device__ __forceinline__ float* red() const { return at<float>(p.so.red); }          // [PHX_RED_WARPS][K2]
    __device__ __forceinline__ const float4* w1g() const { return p.w.W1 + (size_t)g_lo * p.K2q; }  // my rows, global
    __device__ __forceinline__ const float4* wag() const { return p.w.WA + (size_t)g_lo * p.K2q; }
    __device__ __forceinline__ float* st() const { return at<float>(p.so.st); }            // [nslots][B][gpc]
    __device__ __forceinline__ float* jb() const { return at<float>(p.so.jb); }            // [B][gpc] ...
    __device__ __forceinline__ float* asb() const { return at<float>(p.so.asb); }
    __device__ __forceinline__ float* gjb() const { return at<float>(p.so.gjb); }
    __device__ __forceinline__ float* ub() const { return at<float>(p.so.ub); }
    __device__ __forceinline__ float* vb() const { return at<float>(p.so.vb); }
    __device__ __forceinline__ float* mt() const { return at<float>(p.so.mt); }
    __device__ __forceinline__ float* acts() const { return at<float>(o_acts); }
    __device__ __forceinline__ float* actl() const { return at<float>(o_actl); }
    __device__ __forceinline__ float* ysb() const { return at<float>(o_ysb); }
    __device__ __forceinline__ float* acts2() const { return at<float>(o_acts2); }         // next stage's input
    __device__ __forceinline__ float* actl2() const { return at<float>(o_actl2); }
    __device__ __forceinline__ float* ysb2() const { return at<float>(o_ysb2); }
    // per-stage parameter-cotangent factors, stage index innermost: [..][QB], QB = round_up(7 * BT, 4)
    __device__ __forceinline__ float* FG() const { return at<float>(p.so.FG); }            // [K2][QB]  gS|gLP
    __device__ __forceinline__ float* FSP() const { return at<float>(p.so.FSP); }          // [K2][QB]  S|Pr
    __device__ __forceinline__ float* FS() const { return at<float>(p.so.FS); }            // [gpc][QB] s
    __device__ __forceinline__ float* FL() const { return at<float>(p.so.FL); }            // [gpc][QB] l
    __device__ __forceinline__ float* FGJ() const { return at<float>(p.so.FGJ); }          // [gpc][QB] gJ
    __device__ __forceinline__ float* FM() const { return at<float>(p.so.FM); }            // [gpc][8]
    __device__ __forceinline__ float4* ring() const { return at<float4>(p.so.ring); }      // [stages][rows][K2q]
    __device__ __forceinline__ unsigned long long* bar() const { return at<unsigned long long>(p.so.bar); }
    __device__ __forceinline__ void swap_stage_buffers() {
        unsigned t;
        t = o_ysb; o_ysb = o_ysb2; o_ysb2 = t;
        t = o_acts; o_acts = o_acts2; o_acts2 = t;
        t = o_actl; o_actl = o_actl2; o_actl2 = t;
    }
};

// ---- block reductions and grid-wide exchanges -------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void block_sum_d(double (&v)[N], double* dred, double* out) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        double s = warp_sum_d(v[i]);
        if (lane == 0) dred[warp * N + i] = s;
    }
    __syncthreads();
    if (threadIdx.x < N) {
        double s = 0;
        for (int w = 0; w < WARPS; ++w) s += dred[w * N + threadIdx.x];
        out[threadIdx.x] = s;
    }
    __syncthreads();
}

// Sum over all CTAs of the nd (<= 8) doubles in vals[] (smem); the result replaces vals[] in every CTA.  Each double
// travels as two fp32 slots (hi, lo = x - hi: 48 significant bits).  Two hops: every CTA posts its partials, CTA 0
// adds them in a fixed order (one warp per value, lanes over CTAs, fixed butterfly) and posts the totals in R
// replicas, every CTA reads one replica: each hop is one L2 round trip and no slot is polled by more than nCTA / R
// readers.
__device__ __forceinline__ void grid_sum_d(const ResParams& p, Smem& s, double* vals, int nd) {
    Xchg& x = s.x;
    const int nC = gridDim.x;
    if (nC == 1) return;
    const unsigned tag = x.next_tag();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < 2 * nd) {
        double v = vals[threadIdx.x >> 1];
        float hi = (float)v;
        float w = (threadIdx.x & 1) ? (float)(v - (double)hi) : hi;
        if (!isfinite(hi)) w = hi;  // inf / nan: both halves carry it
        ll_put(p.ll.dpart + (size_t)blockIdx.x * PHX_LL_DMAX + threadIdx.x, w, tag);
    }
    if (blockIdx.x == 0) {
      for (int vi = warp; vi < nd; vi += WARPS) {   // one warp per value (nd <= PHX_LL_DMAX / 2)
        // every round (re)polls all five CTAs of the lane in one round trip; lanes past the grid re-read the last CTA
        // (unconditional loads keep the slots in registers)
        unsigned long long w0[5], w1[5];
        bool ok;
        do {
            ok = true;
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                const int c = min(lane + 32 * u, nC - 1);
                ll_ld2(p.ll.dpart + (size_t)c * PHX_LL_DMAX + 2 * vi, w0[u], w1[u]);
            }
#pragma unroll
            for (int u = 0; u < 5; ++u) ok = ok && (unsigned)(w0[u] >> 32) == tag && (unsigned)(w1[u] >> 32) == tag;
        } while (!ok);
        double t = 0;
#pragma unroll
        for (int u = 0; u < 5; ++u) {
            if (lane + 32 * u < nC) {
                float hi = __uint_as_float((unsigned)w0[u]), lo = __uint_as_float((unsigned)w1[u]);
                t += isfinite(hi) ? ((double)hi + (double)lo) : (double)hi;
            }
        }
        t = warp_sum_d(t);
        if (lane < PHX_LL_RCOPIES) {
            float hi = (float)t;
            float lo = isfinite(hi) ? (float)(t - (double)hi) : hi;
            ll_put2(p.ll.dres + (size_t)lane * PHX_LL_DMAX + 2 * vi, hi, lo, tag);
        }
      }
    }
    if (threadIdx.x < 2 * nd)
        s.dst16()[threadIdx.x] =
            ll_get(p.ll.dres + (size_t)(blockIdx.x % PHX_LL_RCOPIES) * PHX_LL_DMAX + threadIdx.x, tag);
    __syncthreads();
    if (threadIdx.x < nd) {
        float hi = s.dst16()[2 * threadIdx.x], lo = s.dst16()[2 * threadIdx.x + 1];
        vals[threadIdx.x] = isfinite(hi) ? ((double)hi + (double)lo) : (double)hi;
    }
    __syncthreads();
}

// Sum over all CTAs of the n-float vector vec[] (smem, n a multiple of 4); the result replaces vec[] in every CTA.
// Small grids: one phase (every CTA reads every partial).  Large grids: reduce-scatter by column quads (one warp per
// quad, lanes over CTAs, fixed butterfly), the reduced quads posted in R replicas, then all-gather from one replica.
__device__ __forceinline__ void grid_allreduce_f(const ResParams& p, Smem& s, float* vec, int n) {
    Xchg& x = s.x;
    const int nC = gridDim.x;
    if (nC == 1) return;
    const unsigned tag = x.next_tag();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (p.so.ystage != PHX_NONE) {
        unsigned long long* base = p.ll.ypart + (size_t)(x.ny & 1) * PHX_LL_YMAX;
        x.ny++;
        for (int i = 2 * threadIdx.x; i < n; i += 2 * THREADS) ll_put2(base + (size_t)blockIdx.x * n + i, vec[i], vec[i + 1], tag);
        const int tot = nC * n;
        for (int e0 = 2 * threadIdx.x; e0 < tot; e0 += 8 * THREADS) {
            unsigned long long w[4][2];
            bool ok;
            do {   // all four pairs are (re)polled in the same round trip (past the end: the last pair again)
                ok = true;
#pragma unroll
                for (int u = 0; u < 4; ++u) ll_ld2(base + min(e0 + u * 2 * THREADS, tot - 2), w[u][0], w[u][1]);
#pragma unroll
                for (int u = 0; u < 4; ++u) ok = ok && (unsigned)(w[u][0] >> 32) == tag && (unsigned)(w[u][1] >> 32) == tag;
            } while (!ok);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * 2 * THREADS;
                if (e < tot) {
                    s.ystage()[e] = __uint_as_float((unsigned)w[u][0]);
                    s.ystage()[e + 1] = __uint_as_float((unsigned)w[u][1]);
                }
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += THREADS) {
            float t = 0.f;
            for (int c = 0; c < nC; ++c) t += s.ystage()[c * n + i];
            vec[i] = t;
        }
        __syncthreads();
        return;
    }
    unsigned long long* mine = p.ll.xpart + (size_t)blockIdx.x * PHX_LL_NMAX;
    for (int i = 2 * threadIdx.x; i < n; i += 2 * THREADS) ll_put2(mine + i, vec[i], vec[i + 1], tag);
    const int nq = n >> 2;
    for (int q = blockIdx.x + nC * warp; q < nq; q += nC * WARPS) {
        // every round (re)polls all five CTAs of the lane in one round trip; lanes past the grid re-read the last CTA
        unsigned long long w[5][4];
        bool ok;
        do {
            ok = true;
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                const unsigned long long* src = p.ll.xpart + (size_t)min(lane + 32 * u, nC - 1) * PHX_LL_NMAX + 4 * q;
                ll_ld2(src, w[u][0], w[u][1]);
                ll_ld2(src + 2, w[u][2], w[u][3]);
            }
#pragma unroll
            for (int u = 0; u < 5; ++u)
                ok = ok && (unsigned)(w[u][0] >> 32) == tag && (unsigned)(w[u][1] >> 32) == tag &&
                     (unsigned)(w[u][2] >> 32) == tag && (unsigned)(w[u][3] >> 32) == tag;
        } while (!ok);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int u = 0; u < 5; ++u) {
            if (lane + 32 * u < nC) {
                a0 += __uint_as_float((unsigned)w[u][0]);
                a1 += __uint_as_float((unsigned)w[u][1]);
                a2 += __uint_as_float((unsigned)w[u][2]);
                a3 += __uint_as_float((unsigned)w[u][3]);
            }
        }
        a0 = warp_sum(a0);
        a1 = warp_sum(a1);
        a2 = warp_sum(a2);
        a3 = warp_sum(a3);
        // lanes 0..15 post: replica (l >> 1), half (l & 1) of the quad, 16 bytes each
        if (lane < 2 * PHX_LL_RCOPIES)
            ll_put2(p.ll.xres + (size_t)(lane >> 1) * PHX_LL_NMAX + 4 * q + 2 * (lane & 1), (lane & 1) ? a2 : a0,
                    (lane & 1) ? a3 : a1, tag);
    }
    const unsigned long long* res = p.ll.xres + (size_t)(blockIdx.x % PHX_LL_RCOPIES) * PHX_LL_NMAX;
    for (int i0 = 2 * threadIdx.x; i0 < n; i0 += 8 * THREADS) {
        // up to four pairs per thread, all (re)polled in the same round trip (past the end: the last pair again)
        unsigned long long w[4][2];
        bool ok;
        do {
            ok = true;
#pragma unroll
            for (int u = 0; u < 4; ++u) ll_ld2(res + min(i0 + u * 2 * THREADS, n - 2), w[u][0], w[u][1]);
#pragma unroll
            for (int u = 0; u < 4; ++u) ok = ok && (unsigned)(w[u][0] >> 32) == tag && (unsigned)(w[u][1] >> 32) == tag;
        } while (!ok);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * 2 * THREADS;
            if (i < n) {
                vec[i] = __uint_as_float((unsigned)w[u][0]);
                vec[i + 1] = __uint_as_float((unsigned)w[u][1]);
            }
        }
    }
    __syncthreads();
}

// ---- weight access: slices resident in shared memory, or a ring of stages filled by 1-D TMA bulk copies ---------------
// A CTA's rows of W1 / WA are one contiguous block of global memory.  If the plan found room, a slice is copied into
// shared memory ONCE (prologue) and every pass over it is a shared-memory pass; otherwise its passes stream the slice
// from L2 through the ring (cp.async.bulk + mbarrier), the first chunks of the next streamed pass prefetched across
// the inter-CTA exchange that precedes it.
__device__ __forceinline__ unsigned smem_u32(const void* ptr) { return (unsigned)__cvta_generic_to_shared(ptr); }

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

__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

enum { MAT_W1 = 0, MAT_WA = 1, MAT_NONE = -1 };

__device__ __forceinline__ bool mat_resident(const ResParams& p, int which) {
    return (which == MAT_W1 ? p.so.w1r : p.so.war) != PHX_NONE || (which == MAT_WA && p.so.watm != PHX_NONE);
}
__device__ __forceinline__ const float4* mat_global(const Smem& s, int which) { return which == MAT_W1 ? s.w1g() : s.wag(); }

// ---- tensor memory as a weight store ---------------------------------------------------------------------------------
// TMEM (256 KB per SM: 128 lanes x 512 columns x 32 bit) normally holds tcgen05.mma accumulators; the B = 1 solves do
// GEMV-shaped work that never touches the tensor cores, so the whole TMEM is free and serves as a second on-chip home
// for weights next to shared memory: the CTA's WA slice is written there once (tcgen05.st) and every pass reads its
// rows back with tcgen05.ld (LDTM) straight into the registers of the lanes that own the columns -- no L2 traffic, no
// shared-memory bandwidth.  Warp w may only touch lanes 32 (w % 4) .. + 31; the four warps of a quarter take 128
// columns each; row i of the warp occupies columns 4 NV i .. of every lane (the lane's float4 columns l + 32 v).
template <int NV>
__device__ __forceinline__ void tmem_ld_row(uint32_t taddr, float4 (&w)[NV]) {
    uint32_t u[4 * NV];
    if constexpr (NV == 1) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3])
                     : "r"(taddr));
    } else if constexpr (NV == 2) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
                     : "r"(taddr));
    } else {
        static_assert(NV == 4, "NV must be 1, 2 or 4");
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
            : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
              "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
            : "r"(taddr));
    }
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int v = 0; v < NV; ++v)
        w[v] = make_float4(__uint_as_float(u[4 * v]), __uint_as_float(u[4 * v + 1]), __uint_as_float(u[4 * v + 2]),
                           __uint_as_float(u[4 * v + 3]));
}
template <int NV>
__device__ __forceinline__ void tmem_st_row(uint32_t taddr, const float4 (&w)[NV]) {
    uint32_t u[4 * NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        u[4 * v] = __float_as_uint(w[v].x);
        u[4 * v + 1] = __float_as_uint(w[v].y);
        u[4 * v + 2] = __float_as_uint(w[v].z);
        u[4 * v + 3] = __float_as_uint(w[v].w);
    }
    if constexpr (NV == 1) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(u[0]), "r"(u[1]),
                     "r"(u[2]), "r"(u[3])
                     : "memory");
    } else if constexpr (NV == 2) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(u[0]),
                     "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7])
                     : "memory");
    } else {
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(
                taddr),
            "r"(u[0]), "r"(u[1]), "r"(u[2]), "r"(u[3]), "r"(u[4]), "r"(u[5]), "r"(u[6]), "r"(u[7]), "r"(u[8]), "r"(u[9]),
            "r"(u[10]), "r"(u[11]), "r"(u[12]), "r"(u[13]), "r"(u[14]), "r"(u[15])
            : "memory");
    }
}
// TMEM address of row i of this warp
template <int NV>
__device__ __forceinline__ uint32_t tmem_row_addr(uint32_t base, int i) {
    const int warp = threadIdx.x >> 5;
    return base + ((uint32_t)(32 * (warp & 3)) << 16) + (uint32_t)((warp >> 2) * 128 + i * 4 * NV);
}

// allocate all 512 columns (one CTA per SM) and park this CTA's WA rows; every warp fills its own rows
template <int NV>
__device__ __forceinline__ uint32_t tmem_setup(const ResParams& p, const Smem& s) {
    if (p.so.watm == PHX_NONE) return 0u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* slot = s.at<uint32_t>(p.so.watm);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t base = *slot;
    const int nw = (s.n_loc > warp) ? (s.n_loc - warp + WARPS - 1) / WARPS : 0;
    const float4* mat = s.wag();
    for (int i = 0; i < nw; ++i) {
        const float4* row = mat + (size_t)(warp + WARPS * i) * p.K2q;
        float4 w[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            int q = lane + 32 * v;
            w[v] = (q < p.K2q) ? __ldg(row + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        tmem_st_row<NV>(tmem_row_addr<NV>(base, i), w);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    return base;
}
__device__ __forceinline__ void tmem_release(const ResParams& p, uint32_t base) {
    if (p.so.watm == PHX_NONE) return;
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if ((threadIdx.x >> 5) == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(512u) : "memory");
}

// where a pass finds a row: shared memory (resident slice or ring slot) or tensor memory
struct RowSrc {
    const float4* sm;
    uint32_t tm;
};
template <int NV>
__device__ __forceinline__ void load_row_src(const RowSrc& src, int K2q, float4 (&w)[NV]) {
    if (src.sm) {
        const int lane = threadIdx.x & 31;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            int q = lane + 32 * v;
            w[v] = (q < K2q) ? src.sm[q] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    } else {
        tmem_ld_row<NV>(src.tm, w);
    }
}

// barriers + the one-time copy of the resident slices (all threads wait for it before the first pass)
__device__ __forceinline__ void ring_init(const ResParams& p, const Smem& s) {
    if (threadIdx.x == 0) {
        for (int i = 0; i < p.ring_stages * WARPS; ++i)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(s.bar() + i)));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(s.at<unsigned long long>(p.so.resbar))));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const unsigned bytes = (unsigned)s.n_loc * p.K2q * 16u;
        const unsigned nres = (p.so.w1r != PHX_NONE ? 1u : 0u) + (p.so.war != PHX_NONE ? 1u : 0u);
        if (nres && bytes) {
            const unsigned bar = smem_u32(s.at<unsigned long long>(p.so.resbar));
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * nres) : "memory");
            if (p.so.w1r != PHX_NONE) bulk_g2s(smem_u32(smem_raw + p.so.w1r), s.w1g(), bytes, bar);
            if (p.so.war != PHX_NONE) bulk_g2s(smem_u32(smem_raw + p.so.war), s.wag(), bytes, bar);
        }
    }
    __syncthreads();
}
__device__ __forceinline__ void resident_wait(const ResParams& p, const Smem& s) {
    if ((p.so.w1r != PHX_NONE || p.so.war != PHX_NONE) && s.n_loc > 0)
        mbar_wait(smem_u32(s.at<unsigned long long>(p.so.resbar)), 0u);
}

// Streaming is PER WARP: warp w owns rows w, w + 16, ... of the CTA's slice and a private ring of S row-sized slots
// with one mbarrier each; its lane 0 issues the bulk copies, so a pass needs no block-wide synchronisation and the
// warps drift freely against each other.
__device__ __forceinline__ int warp_rows(const Smem& s) {
    const int warp = threadIdx.x >> 5;
    return (s.n_loc > warp) ? (s.n_loc - warp + WARPS - 1) / WARPS : 0;
}
// lane 0 only: row i of this warp (row index warp + 16 i of the slice) -> slot i % S
__device__ __forceinline__ void ring_issue(const ResParams& p, const Smem& s, const float4* mat, int i) {
    const int warp = threadIdx.x >> 5;
    const int slot = warp * p.ring_stages + i % p.ring_stages;
    const unsigned bytes = (unsigned)p.K2q * 16u;
    const unsigned bar = smem_u32(s.bar() + slot);
    const unsigned dst = smem_u32(s.ring() + (size_t)slot * p.K2q);
    const float4* src = mat + (size_t)(warp + WARPS * i) * p.K2q;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
    bulk_g2s(dst, src, bytes, bar);
}

// wait for a prefetch nobody will consume (end of the kernel, or a change of plan): no bulk copy may be in flight
// when the CTA exits or when the slots are re-targeted
__device__ __forceinline__ void ring_drain(const ResParams& p, Smem& s) {
    Ring& r = s.rg;
    if (r.pre < 0) return;
    const int warp = threadIdx.x >> 5;
    const int nw = warp_rows(s);
    for (int i = 0; i < min(nw, p.ring_stages); ++i) {
        mbar_wait(smem_u32(s.bar() + warp * p.ring_stages + i), (r.par >> i) & 1u);
        r.par ^= 1u << i;
    }
    r.pre = -1;
}

// Start the first rows of the next pass over `which` if that matrix streams (no-op when it is resident).  The ring
// slots double as the cross-warp reduction buffer, so call this only (a) after a block barrier that follows the last
// generic-proxy use of the slots and (b) when no reduction happens before the prefetched rows are consumed.
__device__ __forceinline__ void ring_prefetch(const ResParams& p, Smem& s, int which) {
    Ring& r = s.rg;
    if (which == MAT_NONE || p.ring_stages == 0 || r.pre >= 0 || mat_resident(p, which)) return;
    if ((threadIdx.x & 31) == 0) {
        const int nw = warp_rows(s);
        const float4* mat = mat_global(s, which);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        for (int i = 0; i < min(nw, p.ring_stages); ++i) ring_issue(p, s, mat, i);
    }
    r.pre = which;
}

// One pass over this CTA's rows of W1 / WA: fn(j, row) is called by one warp (all lanes) per row j with the row in
// shared memory; fn must have consumed the row (into registers and through at least one use) when it returns.
// Ends with a block barrier.
template <typename RowFn>
__device__ __forceinline__ void mat_pass(const ResParams& p, Smem& s, int which, RowFn fn) {
    Ring& r = s.rg;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned roff = (which == MAT_W1) ? p.so.w1r : p.so.war;
    if (roff != PHX_NONE) {
        const float4* base = s.at<float4>(roff);
        for (int rr = warp; rr < s.n_loc; rr += WARPS) fn(rr, base + (size_t)rr * p.K2q);
        __syncthreads();
        return;
    }
    const float4* mat = mat_global(s, which);
    const int S = p.ring_stages;
    const int nw = warp_rows(s);
    if (r.pre != which) {
        ring_drain(p, s);
        ring_prefetch(p, s, which);
    }
    r.pre = -1;
    for (int i = 0; i < nw; ++i) {
        const int sl = i % S;
        mbar_wait(smem_u32(s.bar() + warp * S + sl), (r.par >> sl) & 1u);
        r.par ^= 1u << sl;
        fn(warp + WARPS * i, s.ring() + (size_t)(warp * S + sl) * p.K2q);
        __syncwarp();
        if (lane == 0 && i + S < nw) ring_issue(p, s, mat, i + S);
    }
    __syncthreads();
}

// Grouped variant: a warp's rows are taken RG at a time.  row_fn(r, j, row) consumes row j (slot r of the group) --
// typically per-lane partial dot products kept in registers -- and group_fn(g0, ng) then finishes the ng rows
// j = warp + 16 (g0 + r) together: one interleaved butterfly for all their dot products, the per-element algebra on
// one lane per element, and whatever needs the results.  The latency chain of a pass is paid once per group instead
// of once per row.
template <int NV, int RG, typename RowFn, typename GroupFn>
__device__ __forceinline__ void mat_pass_grouped(const ResParams& p, Smem& s, int which, RowFn row_fn, GroupFn group_fn) {
    Ring& r = s.rg;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned roff = (which == MAT_W1) ? p.so.w1r : p.so.war;
    const int nw = warp_rows(s);
    const bool in_tmem = which == MAT_WA && p.so.watm != PHX_NONE;
    if (roff != PHX_NONE || in_tmem) {
        const float4* base = in_tmem ? nullptr : s.at<float4>(roff);
        for (int g0 = 0; g0 < nw; g0 += RG) {
            const int ng = min(RG, nw - g0);
#pragma unroll
            for (int q = 0; q < RG; ++q) {
                if (q < ng) {
                    RowSrc src;
                    src.sm = in_tmem ? nullptr : base + (size_t)(warp + WARPS * (g0 + q)) * p.K2q;
                    src.tm = in_tmem ? tmem_row_addr<NV>(s.tmem, g0 + q) : 0u;
                    row_fn(q, warp + WARPS * (g0 + q), src);
                }
            }
            group_fn(g0, ng);
        }
        __syncthreads();
        return;
    }
    const float4* mat = mat_global(s, which);
    const int S = p.ring_stages;
    if (r.pre != which) {
        ring_drain(p, s);
        ring_prefetch(p, s, which);
    }
    r.pre = -1;
    for (int g0 = 0; g0 < nw; g0 += RG) {
        const int ng = min(RG, nw - g0);
#pragma unroll
        for (int q = 0; q < RG; ++q) {
            if (q < ng) {
                const int i = g0 + q, sl = i % S;
                mbar_wait(smem_u32(s.bar() + warp * S + sl), (r.par >> sl) & 1u);
                r.par ^= 1u << sl;
                RowSrc src;
                src.sm = s.ring() + (size_t)(warp * S + sl) * p.K2q;
                src.tm = 0u;
                row_fn(q, warp + WARPS * i, src);
                __syncwarp();
                if (lane == 0 && i + S < nw) ring_issue(p, s, mat, i + S);
            }
        }
        group_fn(g0, ng);
    }
    __syncthreads();
}

// ---- the weight passes --------------------------------------------------------------------------------------------------
// Mapping common to all passes: a warp owns one row at a time; lane l owns the float4 columns q = l + 32 v (v < NV) of
// the K2-long row.  Column accumulators live in registers for the whole pass and are combined across warps in a fixed
// order through s.red().
template <int NV, int BT>
__device__ __forceinline__ void acc_zero(float4 (&acc)[BT][NV]) {
#pragma unroll
    for (int b = 0; b < BT; ++b)
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[b][v] = make_float4(0.f, 0.f, 0.f, 0.f);
}

__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

// out[(b0+b)][k] = sum over the 16 warps of acc[b] (fixed order: warps w and w+8 first, then 0..7)
template <int NV, int BT>
__device__ __forceinline__ void acc_reduce(const ResParams& p, const Smem& s, float4 (&acc)[BT][NV], float* out, int b0, int nb) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int K2q = p.K2q;
    float4* red4 = reinterpret_cast<float4*>(s.red());
    static_assert(WARPS == 2 * PHX_RED_WARPS, "two-round fold");
#pragma unroll
    for (int b = 0; b < BT; ++b) {
        if (b < nb) {
            if (warp >= PHX_RED_WARPS) {
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    int q = lane + 32 * v;
                    if (q < K2q) red4[(warp - PHX_RED_WARPS) * K2q + q] = acc[b][v];
                }
            }
            __syncthreads();
            if (warp < PHX_RED_WARPS) {
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    int q = lane + 32 * v;
                    if (q < K2q) red4[warp * K2q + q] = add4(acc[b][v], red4[warp * K2q + q]);
                }
            }
            __syncthreads();
            for (int k = threadIdx.x; k < p.K2; k += THREADS) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < PHX_RED_WARPS; ++w) t += s.red()[w * p.K2 + k];
                out[(b0 + b) * p.K2 + k] = t;
            }
            __syncthreads();
        }
    }
}

template <int NV>
__device__ __forceinline__ void load_row(const float4* row, int K2q, float4 (&w)[NV]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        int q = lane + 32 * v;
        w[v] = (q < K2q) ? row[q] : make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// acc[b][:] += c_b * w  with c_b = cs[b] on the sums half (q < Hq) and cl[b] on the prods half
template <int NV, int BT>
__device__ __forceinline__ void axpy_row(const float4 (&w)[NV], float4 (&acc)[BT][NV], const float* cs, const float* cl,
                                         int stride, int j, int nb, int Hq) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int b = 0; b < BT; ++b) {
        if (b < nb) {
            float sv = cs[b * stride + j], lv = cl[b * stride + j];
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                int q = lane + 32 * v;
                float c = (q >= Hq) ? lv : sv;
                acc[b][v].x = fmaf(w[v].x, c, acc[b][v].x);
                acc[b][v].y = fmaf(w[v].y, c, acc[b][v].y);
                acc[b][v].z = fmaf(w[v].z, c, acc[b][v].z);
                acc[b][v].w = fmaf(w[v].w, c, acc[b][v].w);
            }
        }
    }
}

// Pass A: out[b][k] (this CTA's partial) = sum_{g in slice} act[b][g] * W1[g][k], act = s for k < Hp, l for k >= Hp.
template <int NV, int BT>
__device__ __forceinline__ void passA(const ResParams& p, Smem& s, const float* acts, const float* actl, float* out,
                                      int next) {
    const int Hq = p.Hp >> 2;
    for (int b0 = 0; b0 < p.B; b0 += BT) {
        const int nb = min(BT, p.B - b0);
        float4 acc[BT][NV];
        acc_zero<NV, BT>(acc);
        mat_pass(p, s, MAT_W1, [&](int j, const float4* row) {
            float4 w[NV];
            load_row<NV>(row, p.K2q, w);
            axpy_row<NV, BT>(w, acc, acts + b0 * p.gpc, actl + b0 * p.gpc, p.gpc, j, nb, Hq);
        });
        acc_reduce<NV, BT>(p, s, acc, out, b0, nb);
    }
    ring_prefetch(p, s, next);
}

// rows of the batch handled per fused pass (register budget: accumulators are PB x NV float4 each)
template <int NV, int BT> struct PassRows {
    static constexpr int FWD = (BT < 8 / NV) ? BT : (8 / NV > 1 ? 8 / NV : 1);
    static constexpr int ADJ = (BT < 4 / NV) ? BT : (4 / NV > 1 ? 4 / NV : 1);
};

__device__ __forceinline__ float dot4(const float4& w, const float4& x) {
    float t = w.x * x.x;
    t = fmaf(w.y, x.y, t);
    t = fmaf(w.z, x.z, t);
    t = fmaf(w.w, x.w, t);
    return t;
}

// per-lane partial of sum_k w[k] * x[k] (x in shared memory)
template <int NV>
__device__ __forceinline__ float row_dot_partial(const float4 (&w)[NV], const float4* x4, int K2q) {
    const int lane = threadIdx.x & 31;
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        int q = lane + 32 * v;
        if (q < K2q) {
            if (v & 1) t1 += dot4(w[v], x4[q]); else t0 += dot4(w[v], x4[q]);
        }
    }
    return t0 + t1;
}

// the lane's own float4 columns of PB K2-long vectors (x[b][:], shared memory) into registers: the passes dot every
// row with the same vectors, so they are loaded once per pass instead of once per row
template <int NV, int PB>
__device__ __forceinline__ void hoist_vec(const float4* x4, int K2q, int nb, float4 (&x)[PB][NV]) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int b = 0; b < PB; ++b)
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            int q = lane + 32 * v;
            x[b][v] = (b < nb && q < K2q) ? x4[b * K2q + q] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
}
template <int NV>
__device__ __forceinline__ float row_dot_reg(const float4 (&w)[NV], const float4 (&x)[NV]) {
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        if (v & 1) t1 += dot4(w[v], x[v]); else t0 += dot4(w[v], x[v]);
    }
    return t0 + t1;
}

// all lanes end up with the warp-wide sums of the N per-lane values (N independent butterflies, interleaved)
template <int N>
__device__ __forceinline__ void warp_sum_n(float (&d)[N]) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int i = 0; i < N; ++i) d[i] += __shfl_xor_sync(0xffffffffu, d[i], o);
}
template <int N>
__device__ __forceinline__ float pick_lane(const float (&d)[N]) {
    const int lane = threadIdx.x & 31;
    float v = 0.f;
#pragma unroll
    for (int i = 0; i < N; ++i) v = (lane == i) ? d[i] : v;
    return v;
}

// acc[b][:] += c[b] * w  (one coefficient per row of the batch)
template <int NV, int PB>
__device__ __forceinline__ void axpy1(const float4 (&w)[NV], float4 (&acc)[PB][NV], const float (&c)[PB], int nb) {
#pragma unroll
    for (int b = 0; b < PB; ++b) {
        if (b < nb) {
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                acc[b][v].x = fmaf(w[v].x, c[b], acc[b][v].x);
                acc[b][v].y = fmaf(w[v].y, c[b], acc[b][v].y);
                acc[b][v].z = fmaf(w[v].z, c[b], acc[b][v].z);
                acc[b][v].w = fmaf(w[v].w, c[b], acc[b][v].w);
            }
        }
    }
}
// acc[b][:] += (cs[b] on the sums half, cl[b] on the prods half) * w
template <int NV, int PB>
__device__ __forceinline__ void axpy2(const float4 (&w)[NV], float4 (&acc)[PB][NV], const float (&cs)[PB],
                                      const float (&cl)[PB], int nb, int Hq) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int b = 0; b < PB; ++b) {
        if (b < nb) {
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                int q = lane + 32 * v;
                float c = (q >= Hq) ? cl[b] : cs[b];
                acc[b][v].x = fmaf(w[v].x, c, acc[b][v].x);
                acc[b][v].y = fmaf(w[v].y, c, acc[b][v].y);
                acc[b][v].z = fmaf(w[v].z, c, acc[b][v].z);
                acc[b][v].w = fmaf(w[v].w, c, acc[b][v].w);
            }
        }
    }
}

// Fused forward pass over WA: for every local gene row j and batch row b
//     J = WA[g][:] . sp[b][:]              f = fsign * relu(m)[g] * (J - y_stage)          (odenet.py:88-90)
//     y_next = post(b, j, li, f, true)     (the caller's RK stage algebra, run by ONE lane per element)
// and, with do_next, the Hill activations of y_next become the next stage input (ysb / acts / actl) and -- when the W1
// slice is resident -- are contracted with W1[g][:] on the spot, so that pass A of the NEXT evaluation costs no extra
// pass: its partial branch vector lands in s.sp().  With a streamed W1 the contraction is a separate pass A.
template <int NV, int BT, typename Post>
__device__ __forceinline__ void fwd_passBA(const ResParams& p, Smem& s, bool do_next, Post post) {
    constexpr int PB = PassRows<NV, BT>::FWD;
    constexpr int RG = 8 / PB;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int K2q = p.K2q, Hq = p.Hp >> 2;
    const bool fuse = do_next && p.so.w1r != PHX_NONE;
    const float4* sp4 = reinterpret_cast<const float4*>(s.sp());
    const float4* w1res = s.at<float4>(p.so.w1r);
    float4 acc[PB][NV];
    for (int b0 = 0; b0 < p.B; b0 += PB) {
        const int nb = min(PB, p.B - b0);
        acc_zero<NV, PB>(acc);
        float d[RG * PB] = {};
        float4 x[PB][NV];
        hoist_vec<NV, PB>(sp4 + (size_t)b0 * K2q, K2q, nb, x);
        mat_pass_grouped<NV, RG>(
            p, s, MAT_WA,
            [&](int r, int j, const RowSrc& row) {
                float4 w[NV];
                load_row_src<NV>(row, K2q, w);
#pragma unroll
                for (int b = 0; b < PB; ++b) d[r * PB + b] = row_dot_reg<NV>(w, x[b]);
            },
            [&](int g0, int ng) {
                warp_sum_n<RG * PB>(d);
                const float mine = pick_lane<RG * PB>(d);
                float sv = 0.f, lv = 0.f;
                {
                    const int r = lane / PB, b = lane - r * PB;
                    if (r < ng && b < nb) {
                        const int j = warp + WARPS * (g0 + r);
                        const int li = (b0 + b) * p.gpc + j;
                        const float f = p.fsign * (s.relum()[j] * (mine - s.ysb()[li]));
                        const float yn = post(b0 + b, j, li, f, true);
                        if (do_next) {
                            float den;
                            hill(yn, sv, lv, den);
                            s.ysb()[li] = yn;
                            s.acts()[li] = sv;
                            s.actl()[li] = lv;
                        }
                    }
                }
                if (fuse) {
#pragma unroll
                    for (int r = 0; r < RG; ++r) {
                        if (r < ng) {
                            float cs[PB], cl[PB];
#pragma unroll
                            for (int b = 0; b < PB; ++b) {
                                cs[b] = __shfl_sync(0xffffffffu, sv, r * PB + b);
                                cl[b] = __shfl_sync(0xffffffffu, lv, r * PB + b);
                            }
                            float4 w[NV];
                            load_row<NV>(w1res + (size_t)(warp + WARPS * (g0 + r)) * K2q, K2q, w);
                            axpy2<NV, PB>(w, acc, cs, cl, nb, Hq);
                        }
                    }
                }
            });
        if (fuse) acc_reduce<NV, PB>(p, s, acc, s.sp(), b0, nb);   // sp is dead once every row-dot of the pass is done
    }
    // what streams next (the ring slots double as the reduction buffer: only prefetch what is consumed before the
    // next reduction): fused -> the next evaluation's WA pass; not fused -> pass A over W1; last stage -> the next
    // step's stand-alone pass A over W1
    if (do_next && !fuse) passA<NV, BT>(p, s, s.acts(), s.actl(), s.sp(), MAT_WA);
    else ring_prefetch(p, s, fuse ? MAT_WA : MAT_W1);
}

// Fused adjoint pass 1 over WA at the current stage input (ysb / acts / actl, cotangent asb, gj = a relu(m) in gjb):
//     J = WA[g][:] . sp[b][:]        ky = -relu(m) (J - y)       gSP partial += gj[b][g] * WA[g][:]  -> s.gsp()
//     theta factors of this stage (FS, FL, FGJ, FM) into column `slot`
//     with has_next: y_next = ynext(b, j, li, ky) -> ysb2 / acts2 / actl2 and (resident W1) its pass A -> s.spn()
template <int NV, int BT, typename YNext>
__device__ __forceinline__ void adj_pass1(const ResParams& p, Smem& s, int slot, bool has_next, YNext ynext) {
    constexpr int PB = PassRows<NV, BT>::ADJ;
    constexpr int RG = 8 / PB;
    constexpr int QB = (7 * BT + 3) & ~3;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int K2q = p.K2q, Hq = p.Hp >> 2;
    const bool fuse = has_next && p.so.w1r != PHX_NONE;
    const float4* sp4 = reinterpret_cast<const float4*>(s.sp());
    const float4* w1res = s.at<float4>(p.so.w1r);
    float* KYs = s.st() + (4 + slot) * p.B * p.gpc;
    float4 accg[PB][NV], acca[PB][NV];
    for (int b0 = 0; b0 < p.B; b0 += PB) {
        const int nb = min(PB, p.B - b0);
        acc_zero<NV, PB>(accg);
        acc_zero<NV, PB>(acca);
        float d[RG * PB] = {};
        float4 x[PB][NV];
        hoist_vec<NV, PB>(sp4 + (size_t)b0 * K2q, K2q, nb, x);
        mat_pass_grouped<NV, RG>(
            p, s, MAT_WA,
            [&](int r, int j, const RowSrc& row) {
                float4 w[NV];
                load_row_src<NV>(row, K2q, w);
                float gj[PB];
#pragma unroll
                for (int b = 0; b < PB; ++b) {
                    d[r * PB + b] = row_dot_reg<NV>(w, x[b]);
                    gj[b] = (b < nb) ? s.gjb()[(b0 + b) * p.gpc + j] : 0.f;
                }
                axpy1<NV, PB>(w, accg, gj, nb);
            },
            [&](int g0, int ng) {
                warp_sum_n<RG * PB>(d);
                const float mine = pick_lane<RG * PB>(d);
                float sv = 0.f, lv = 0.f, mt = 0.f;
                const int r = lane / PB, b = lane - r * PB;
                const int j = warp + WARPS * (g0 + r);
                const bool active = r < ng && b < nb;
                if (active) {
                    const int li = (b0 + b) * p.gpc + j;
                    const float jm = mine - s.ysb()[li];
                    const float ky = -(s.relum()[j] * jm);
                    mt = s.asb()[li] * jm;
                    KYs[li] = ky;
                    s.FS()[j * QB + slot * BT + b0 + b] = s.acts()[li];
                    s.FL()[j * QB + slot * BT + b0 + b] = s.actl()[li];
                    s.FGJ()[j * QB + slot * BT + b0 + b] = s.gjb()[li];
                    if (has_next) {
                        const float yn = ynext(b0 + b, j, li, ky);
                        float den;
                        hill(yn, sv, lv, den);
                        s.ysb2()[li] = yn;
                        s.acts2()[li] = sv;
                        s.actl2()[li] = lv;
                    }
                }
                // multiplier cotangent of the row: sum over the batch rows (adjacent lanes), masked by m > 0
#pragma unroll
                for (int o = PB / 2; o > 0; o >>= 1) mt += __shfl_xor_sync(0xffffffffu, mt, o);
                if (r < ng && b == 0) {
                    const float prev = (b0 == 0) ? 0.f : s.FM()[j * 8 + slot];
                    s.FM()[j * 8 + slot] = prev + mt * s.maskm()[j];
                }
                if (fuse) {
#pragma unroll
                    for (int q = 0; q < RG; ++q) {
                        if (q < ng) {
                            float cs[PB], cl[PB];
#pragma unroll
                            for (int bb = 0; bb < PB; ++bb) {
                                cs[bb] = __shfl_sync(0xffffffffu, sv, q * PB + bb);
                                cl[bb] = __shfl_sync(0xffffffffu, lv, q * PB + bb);
                            }
                            float4 w[NV];
                            load_row<NV>(w1res + (size_t)(warp + WARPS * (g0 + q)) * K2q, K2q, w);
                            axpy2<NV, PB>(w, acca, cs, cl, nb, Hq);
                        }
                    }
                }
            });
        acc_reduce<NV, PB>(p, s, accg, s.gsp(), b0, nb);
        if (fuse) acc_reduce<NV, PB>(p, s, acca, s.spn(), b0, nb);
    }
    // next streamed pass: pass A (not fused) or pass 2 over W1; with W1 resident the next evaluation's WA pass (pass 2
    // does no cross-warp reduction, so the ring slots stay untouched until then)
    if (has_next && !fuse) passA<NV, BT>(p, s, s.acts2(), s.actl2(), s.spn(), MAT_W1);
    else ring_prefetch(p, s, (has_next && mat_resident(p, MAT_W1)) ? MAT_WA : MAT_W1);
}

// Fused adjoint pass 2 over W1 (after the exchange; s.gsp() = gS | gLP):
//     u = W1[g][:Hp] . gS     v = W1[g][Hp:] . gLP      ka = (u + v / (1 + s)) / (1 + |y - .5|)^2 - gj   -> KA(slot)
//     a_next = anext(b, j, li, ka, true); with has_next it becomes the next stage's cotangent input (asb, gjb)
template <int NV, int BT, typename ANext>
__device__ __forceinline__ void adj_pass2(const ResParams& p, Smem& s, int slot, bool has_next, ANext anext) {
    constexpr int PB = PassRows<NV, BT>::ADJ;
    constexpr int RG = 8 / PB;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int K2q = p.K2q, Hq = p.Hp >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(s.gsp());
    float* KAs = s.st() + (11 + slot) * p.B * p.gpc;
    for (int b0 = 0; b0 < p.B; b0 += PB) {
        const int nb = min(PB, p.B - b0);
        float du[RG * PB] = {}, dv[RG * PB] = {};
        float4 x[PB][NV];
        hoist_vec<NV, PB>(g4 + (size_t)b0 * K2q, K2q, nb, x);
        mat_pass_grouped<NV, RG>(
            p, s, MAT_W1,
            [&](int r, int j, const RowSrc& row) {
                float4 w[NV];
                load_row_src<NV>(row, K2q, w);
#pragma unroll
                for (int b = 0; b < PB; ++b) {
                    float tu = 0.f, tv = 0.f;
#pragma unroll
                    for (int v = 0; v < NV; ++v) {
                        const float t = dot4(w[v], x[b][v]);   // zero beyond the row / the batch
                        if (lane + 32 * v >= Hq) tv += t; else tu += t;
                    }
                    du[r * PB + b] = tu;
                    dv[r * PB + b] = tv;
                }
            },
            [&](int g0, int ng) {
                warp_sum_n<RG * PB>(du);
                warp_sum_n<RG * PB>(dv);
                const float u = pick_lane<RG * PB>(du), v = pick_lane<RG * PB>(dv);
                const int r = lane / PB, b = lane - r * PB;
                if (r < ng && b < nb) {
                    const int j = warp + WARPS * (g0 + r);
                    const int li = (b0 + b) * p.gpc + j;
                    const float z = s.ysb()[li] - 0.5f;
                    const float den = 1.0f + fabsf(z);
                    const float yb = (u + v / (1.0f + s.acts()[li])) / (den * den);
                    const float ka = yb - s.gjb()[li];
                    KAs[li] = ka;
                    const float an = anext(b0 + b, j, li, ka, true);
                    if (has_next) {
                        s.asb()[li] = an;
                        s.gjb()[li] = an * s.relum()[j];
                    }
                }
            });
    }
    ring_prefetch(p, s, has_next ? MAT_WA : MAT_W1);
}

template <typename F>
__device__ __forceinline__ void for_local(const ResParams& p, int g_lo, int n_loc, F f) {
    const int tot = p.B * n_loc;
    for (int e = threadIdx.x; e < tot; e += THREADS) {
        int b = e / n_loc, j = e - b * n_loc;
        f(b, j, g_lo + j, (size_t)b * p.G + g_lo + j, b * p.gpc + j);
    }
}

// branch vector after the all-reduce: add bias, exponentiate the prods half (odenet.py:86-87); padded columns -> 0
__device__ __forceinline__ void finalize_sp(const ResParams& p, const Smem& s, const float* src, float* dst) {
    for (int i = threadIdx.x; i < p.B * p.K2; i += THREADS) {
        int k = i % p.K2;
        float v = src[i] + s.bias()[k];
        if (k >= p.Hp) v = (k - p.Hp < p.H) ? expf(v) : 0.f;
        dst[i] = v;
    }
    __syncthreads();
}

// controller pieces (thread 0 only) --------------------------------------------------------------------------------
__device__ void set_step_coeffs(Ctrl* c) {
    float dtf = (float)c->dt;
    c->dtf = dtf;
    for (int i = 0; i < 6; ++i)
        for (int j = 0; j <= i; ++j) c->cb[i][j] = (float)c_beta[i][j] * dtf;
    for (int j = 0; j < 7; ++j) {
        c->cerr[j] = dtf * (float)c_err[j];
        c->cmid[j] = dtf * (float)c_mid[j];
    }
}

// misc.py:94-103 with order 5 and the request's safety, ifactor, dfactor (defaults 0.9, 10, 0.2)
__device__ double next_dt(const ResParams& p, double dt, float ratio) {
    if (ratio == 0.f) return dt * p.ifactor;
    double dfactor = (ratio < 1.f) ? 1.0 : p.dfactor;
    double r = (double)ratio;
    if (isnan(r)) return nan("");
    double f = p.safety / pow(r, 0.2);
    f = fmax(f, dfactor);
    f = fmin(p.ifactor, f);
    return dt * f;
}

// the caller gives the first step of a dopri5 solve (phx_solve_desc.first_step; never with a step grid, which is
// fixed-grid only).  Read at each use rather than held in a variable: the default instantiations then keep their
// register allocation
template <bool GRID>
__device__ __forceinline__ bool given_step(const ResParams& p) { return !GRID && p.first_step > 0; }

// whether the adjoint has time cotangents (phx_solve_desc.t_vjp; never in the step-grid instantiations, which are
// fixed-grid only).  Read at each use, like given_step
template <bool GRID>
__device__ __forceinline__ bool has_t_vjp(const ResParams& p) { return !GRID && p.t_vjp != nullptr; }
// the time cotangent v of an adjoint interval (Ctrl.vjp_t) as the one-element block of the mixed norm in d0 of Hairer's
// estimate; returns whether v is non-finite (the reference asserts a finite augmented state)
__device__ __forceinline__ bool fold_t_vjp(const ResParams& p, float v, float& d0) {
    const float r = v / (p.atol_f + fabsf(v) * p.rtol_f);
    d0 = fmaxf(d0, sqrtf(r * r));
    return !isfinite(v);
}

// misc.py:47-86 tail: h0 from d0, d1
__device__ float init_h0(float d0, float d1) {
    if (d0 < 1e-5f || d1 < 1e-5f) return 1e-6f;
    return 0.01f * d0 / d1;
}
__device__ double init_dt(float h0, float d1, float d2) {
    float h1;
    if (d1 <= 1e-15f && d2 <= 1e-15f)
        h1 = fmaxf(1e-6f, h0 * 1e-3f);
    else
        h1 = powf(0.01f / fmaxf(d1, d2), 0.2f);
    return (double)fminf(100.f * h0, h1);
}

__device__ void log_step(const ResParams& p, Ctrl* c, double t0, double dt, int accepted) {
    if (blockIdx.x == 0 && p.steplog && c->n_log < p.steplog_cap) {
        p.steplog[3 * c->n_log + 0] = t0;
        p.steplog[3 * c->n_log + 1] = dt;
        p.steplog[3 * c->n_log + 2] = (double)accepted;
    }
    c->n_log++;
}

__device__ void set_interp_x(Ctrl* c, double t, double t0, double t1) {
    double x = (t - t0) / (t1 - t0);
    double xp = x;
    c->xs[0] = (float)xp;
    xp = xp * x;
    c->xs[1] = (float)xp;
    xp = xp * x;
    c->xs[2] = (float)xp;
    xp = xp * x;
    c->xs[3] = (float)xp;
}

// quartic dense output (interp.py:1-47) from the step's end values and derivatives
__device__ __forceinline__ float interp_eval(float y0, float y1, float ymid, float f0, float f1, float dt,
                                             const float* xs) {
    float a = 2.f * dt * (f1 - f0) - 8.f * (y1 + y0) + 16.f * ymid;
    float b = dt * (5.f * f0 - 3.f * f1) + 18.f * y0 + 14.f * y1 - 32.f * ymid;
    float c = dt * (f1 - 4.f * f0) - 11.f * y0 - 5.f * y1 + 16.f * ymid;
    float d = dt * f0;
    float total = y0 + xs[0] * d;
    total = total + xs[1] * c;
    total = total + xs[2] * b;
    total = total + xs[3] * a;
    return total;
}

__device__ void write_status(const ResParams& p, int pi, const Ctrl* c, int code) {
    if (blockIdx.x == 0 && threadIdx.x == 0 && p.status) {
        phx_status* st = p.status + pi;
        st->n_accepted = c->n_acc;
        st->n_rejected = c->n_rej;
        st->n_rhs = c->n_rhs;
        st->n_logged = min(c->n_log, p.steplog_cap);
        st->reserved = 0;
        st->t_fail = c->tcur;
        st->dt_fail = c->dt;
        __threadfence_system();
        st->code = code;
    }
}

// common prologue: shared-memory views, epoch, constant per-gene / per-column vectors
__device__ __forceinline__ void prologue(const ResParams& p, Smem& s) {
    Xchg& x = s.x;
    Ring& ring = s.rg;
    const int g_lo = s.g_lo, n_loc = s.n_loc;
    s.pf.init(p.prof, reinterpret_cast<long long*>(smem_raw + p.so.ctrl + 512));
    x.ep = __ldcg(p.ll.epoch);
    x.ny = x.nd = 0;
    ring.par = 0;
    ring.pre = -1;
    for (int k = threadIdx.x; k < p.K2; k += THREADS) s.bias()[k] = p.w.bias[k];
    for (int j = threadIdx.x; j < n_loc; j += THREADS) {
        s.relum()[j] = p.w.relum[g_lo + j];
        s.maskm()[j] = p.w.maskm[g_lo + j];
    }
    ring_init(p, s);
    ring_prefetch(p, s, MAT_W1);
    resident_wait(p, s);
}

__device__ __forceinline__ void epilogue_epoch(const ResParams& p, const Smem& s) {
    const Xchg& x = s.x;
    // every CTA has read the launch's starting epoch before CTA 0 can get here (it took part in >= 1 exchange)
    if (blockIdx.x == 0 && threadIdx.x == 0) *p.ll.epoch = x.ep;
}

// Stand-alone pass A at the stage input (acts / actl) + its exchange: leaves the finalised branch vector in s.sp().
template <int NV, int BT>
__device__ __forceinline__ void eval_A(const ResParams& __restrict__ p, Smem& __restrict__ s) {
    Prof& pf = s.pf;
    pf.tick(PT_COMBINE);
    passA<NV, BT>(p, s, s.acts(), s.actl(), s.sp(), MAT_WA);
    pf.tick(PT_PHASE_A);
    grid_allreduce_f(p, s, s.sp(), p.B * p.K2);
    pf.tick(PT_ALLRED1);
    finalize_sp(p, s, s.sp(), s.sp());
    pf.tick(PT_FINALIZE);
}

// The rest of a forward evaluation: fused pass B (+ the caller's stage algebra + pass A of the next stage input) and,
// with do_next, the exchange that completes the next stage's branch vector.
template <int NV, int BT, typename Post>
__device__ __forceinline__ void eval_B(const ResParams& __restrict__ p, Smem& __restrict__ s, bool do_next, Post post) {
    Prof& pf = s.pf;
    fwd_passBA<NV, BT>(p, s, do_next, post);
    pf.tick(PT_PHASE_B);
    if (do_next) {
        grid_allreduce_f(p, s, s.sp(), p.B * p.K2);
        pf.tick(PT_ALLRED1);
        finalize_sp(p, s, s.sp(), s.sp());
        pf.tick(PT_FINALIZE);
    }
}

// =====================================================================================================================
// Forward solve
// =====================================================================================================================
// GRID: the fixed grid is the caller's step grid (p.gdt != nullptr), an instantiation of its own so that the default
// (one step per output interval) and dopri5 keep their code
template <int NV, int BT, bool GRID>
__global__ void __launch_bounds__(PHX_THREADS, 1) phx_fwd_kernel(const __grid_constant__ ResParams p) {
    Smem s(p);
    const int g_lo = s.g_lo, n_loc = s.n_loc;
    prologue(p, s);
    s.tmem = tmem_setup<NV>(p, s);
    Prof& pf = s.pf;
    Ctrl* c = s.ctrl();
    const size_t BG = (size_t)p.B * p.G;
    const int BL = p.B * p.gpc;
    const double Nel = (double)p.B * (double)p.G;
    float* Y = s.st();
    float* Y1 = s.st() + BL;
    auto K = [&](int i) { return s.st() + (2 + i) * BL; };

    // independent problems, one after the other: the weights stay on chip (shared / tensor memory) across them
    for (int pi = 0; pi < p.nprob; ++pi) {
    const float* y0p = p.y0 + (size_t)pi * p.y0_stride;
    float* youtp = p.yout + (size_t)pi * p.yout_stride;
    if (threadIdx.x == 0) {
        c->n_acc = c->n_rej = c->n_rhs = c->n_log = 0;
        c->stop = 0;
        c->tcur = tget(p, pi, 0);
        c->dt = 0;
        for (int i = 0; i < 7; ++i) c->slot[i] = i;
    }
    auto set_stage_input = [&](int li, float ys) {
        s.ysb()[li] = ys;
        float sv, lv, den;
        hill(ys, sv, lv, den);
        s.acts()[li] = sv;
        s.actl()[li] = lv;
    };
    for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
        float y = y0p[gi];
        Y[li] = y;
        youtp[gi] = y;
        set_stage_input(li, y);
    });
    __syncthreads();

    if (p.method != PHX_DOPRI5) {
        // ---- fixed grid (solvers.py:48-50, 77-103): one step per output interval, or the steps of the caller's grid
        // (p.gdt), whose output times are written from the step that reaches them: y1 on an exact hit, else y + s (y1 - y)
        const float third = (float)(1.0 / 3.0);
        const int nk = GRID ? p.goff[pi + 1] - p.goff[pi] : p.T - 1;
        int jn = 1;   // first output time not written yet (grid)
        eval_A<NV, BT>(p, s);
        for (int i = 0; i < nk; ++i) {
            const float dtf = GRID ? p.gdt[p.goff[pi] + i]
                                    : (p.t_is_f32 ? ((float)tget(p, pi, i + 1) - (float)tget(p, pi, i)) : (float)(tget(p, pi, i + 1) - tget(p, pi, i)));
            float* yo = youtp + (size_t)(i + 1) * BG;
            int je = jn;   // grid: outputs [jn, je) are written by this step
            if (GRID)
                while (je < p.T && p.gout[pi * (p.T - 1) + je - 1] == i) ++je;
            const bool more = i + 1 < nk;   // another step follows: its first pass A is fused into the last stage
            // one call site for every stage of every fixed-grid method (the stage algebra switches at run time)
            const int nst = (p.method == PHX_EULER) ? 1 : (p.method == PHX_MIDPOINT ? 2 : 4);
            const float half = 0.5f * dtf;
            for (int st = 0; st < nst; ++st) {
                const bool last = st + 1 == nst;
                eval_B<NV, BT>(p, s, !last || more, [&](int b, int j, int li, float f, bool lead) {
                    float yn;
                    if (p.method == PHX_EULER) {
                        yn = Y[li] + dtf * f;
                    } else if (p.method == PHX_MIDPOINT) {
                        yn = (st == 0) ? Y[li] + f * half : Y[li] + dtf * f;
                    } else {  // 3/8-rule RK4 (rk_common.py:96-103)
                        if (st == 0) yn = Y[li] + dtf * f * third;
                        else if (st == 1) yn = Y[li] + dtf * (f - K(0)[li] * third);
                        else if (st == 2) yn = Y[li] + dtf * (K(0)[li] - K(1)[li] + f);
                        else yn = Y[li] + (K(0)[li] + 3.f * (K(1)[li] + K(2)[li]) + f) * dtf * 0.125f;
                        if (lead && !last) K(st)[li] = f;
                    }
                    if (last && lead) {
                        if (GRID) {
                            // (op by op, solvers.py:97-103; the build does not contract to fma)
                            for (int jj = jn; jj < je; ++jj) {
                                const float sl = p.gsl[pi * (p.T - 1) + jj - 1];
                                youtp[(size_t)jj * BG + (size_t)b * p.G + g_lo + j] = sl < 0.f ? yn : Y[li] + sl * (yn - Y[li]);
                            }
                        } else {
                            yo[(size_t)b * p.G + g_lo + j] = yn;
                        }
                        Y[li] = yn;
                    }
                    return yn;
                });
            }
            jn = je;
        }
        if (threadIdx.x == 0) {
            int per = (p.method == PHX_EULER) ? 1 : (p.method == PHX_MIDPOINT ? 2 : 4);
            c->n_rhs = per * nk;
            c->tcur = tget(p, pi, p.T - 1);
        }
        __syncthreads();
        ring_drain(p, s);
        pf.tick(PT_CTRL);
        write_status(p, pi, c, PHX_ST_OK);
        __syncthreads();
        continue;
    }

    // ---- dopri5 (rk_common.py:111-228) ----
    // f0 and the initial step (misc.py:47-86): two evaluations through one call site, or f0 alone when the caller gives
    // the first step
    for (int which = 0; which < 2; ++which) {
        double acc[3] = {0, 0, 0};
        eval_A<NV, BT>(p, s);
        eval_B<NV, BT>(p, s, false, [&](int b, int j, int li, float f, bool lead) {
            if (lead) {
                float y = Y[li];
                float scale = p.atol_f + fabsf(y) * p.rtol_f;
                if (which == 0) {
                    K(0)[li] = f;
                    float r0 = y / scale, r1 = f / scale;
                    acc[0] += (double)(r0 * r0);
                    acc[1] += (double)(r1 * r1);
                    if (!isfinite(y)) acc[2] += 1.0;
                } else {
                    float r = (f - K(0)[li]) / scale;
                    acc[0] += (double)(r * r);
                }
            }
            return 0.f;
        });
        block_sum_d<3>(acc, s.dred(), c->dsum);
        grid_sum_d(p, s, c->dsum, which == 0 ? 3 : 1);
        pf.tick(PT_NORMS);
        if (which == 0) {
            if (threadIdx.x == 0) {
                float d0 = sqrtf((float)(c->dsum[0] / Nel));
                float d1 = sqrtf((float)(c->dsum[1] / Nel));
                c->d1 = d1;
                c->h0 = init_h0(d0, d1);
                c->nonfinite_prev = c->dsum[2] > 0.0;
                if (given_step<GRID>(p)) {
                    c->dt = p.first_step;
                    c->tprev = c->tcur;
                    c->n_rhs = 1;
                    c->n_steps_interval = 0;
                }
            }
            __syncthreads();
            if (given_step<GRID>(p)) break;   // the caller's first step: no second evaluation
            const float h0 = c->h0;
            for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                set_stage_input(li, Y[li] + h0 * K(0)[li]);
            });
            __syncthreads();
        } else {
            if (threadIdx.x == 0) {
                float d2 = sqrtf((float)(c->dsum[0] / Nel)) / c->h0;
                c->dt = init_dt(c->h0, c->d1, d2);
                c->tprev = c->tcur;
                c->n_rhs = 2;
                c->n_steps_interval = 0;
            }
            __syncthreads();
        }
    }

    int next_out = 1;
    int code = PHX_ST_OK;
    while (next_out < p.T) {
        // ---- assertions of rk_common.py:154,175-176 + coefficient table for this dt ----
        if (threadIdx.x == 0) {
            int st = 0;
            if ((long long)c->n_steps_interval >= p.max_steps) st = PHX_ST_MAX_STEPS;
            else if (!(c->tcur + c->dt > c->tcur)) st = PHX_ST_DT_UNDERFLOW;
            else if (c->nonfinite_prev) st = PHX_ST_NONFINITE;
            c->stop = st;
            if (!st) set_step_coeffs(c);
        }
        __syncthreads();
        if (c->stop) {
            code = c->stop;
            break;
        }
        const int* sl = c->slot;   // FSAL slot permutation, read from shared memory (a dynamically indexed local array
                                   // would live in local memory)
        {
            const float c00 = c->cb[0][0];
            const float* K0 = K(sl[0]);
            for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                set_stage_input(li, Y[li] + K0[li] * c00);
            });
            __syncthreads();
        }
        eval_A<NV, BT>(p, s);
        double acc[2] = {0, 0};
        for (int st = 1; st <= 6; ++st) {
            eval_B<NV, BT>(p, s, st < 6, [&](int b, int j, int li, float f, bool lead) {
                if (lead) K(sl[st])[li] = f;
                if (st < 6) {
                    float a = K(sl[0])[li] * c->cb[st][0];
                    for (int q = 1; q < st; ++q) a = fmaf(K(sl[q])[li], c->cb[st][q], a);
                    a = fmaf(f, c->cb[st][st], a);
                    float yn = Y[li] + a;
                    if (st == 5 && lead) Y1[li] = yn;
                    return yn;
                }
                if (lead) {
                    float ys = s.ysb()[li];
                    float e = K(sl[0])[li] * c->cerr[0];
                    for (int q = 1; q < 6; ++q) e = fmaf(K(sl[q])[li], c->cerr[q], e);
                    e = fmaf(f, c->cerr[6], e);
                    float tol = p.atol_f + p.rtol_f * fmaxf(fabsf(Y[li]), fabsf(ys));
                    float r = e / tol;
                    acc[0] += (double)(r * r);
                    if (!isfinite(ys)) acc[1] += 1.0;
                }
                return 0.f;
            });
        }
        pf.tick(PT_COMBINE);
        block_sum_d<2>(acc, s.dred(), c->dsum);
        grid_sum_d(p, s, c->dsum, 2);
        pf.tick(PT_NORMS);
        if (threadIdx.x == 0) {
            float ratio = sqrtf((float)(c->dsum[0] / Nel));
            int accept = ratio <= 1.f;
            log_step(p, c, c->tcur, c->dt, accept);
            c->dt_used = c->dt;
            c->tprev = c->tcur;
            if (accept) {
                c->tcur = c->tcur + c->dt;
                c->n_acc++;
                c->nonfinite_prev = c->dsum[1] > 0.0;
            } else {
                c->n_rej++;
            }
            c->dt = next_dt(p, c->dt, ratio);
            c->accept = accept;
            c->n_rhs += 6;
            c->n_steps_interval++;
        }
        __syncthreads();
        if (c->accept) {
            // emit every pending output inside (tprev, tcur] from the quartic interpolant (rk_common.py:157)
            while (next_out < p.T && tget(p, pi, next_out) <= c->tcur) {
                if (threadIdx.x == 0) set_interp_x(c, tget(p, pi, next_out), c->tprev, c->tcur);
                __syncthreads();
                float* yo = youtp + (size_t)next_out * BG;
                const float dtf = c->dtf;
                for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                    float y0 = Y[li], y1 = Y1[li];
                    float m = K(sl[0])[li] * c->cmid[0];
                    for (int q = 1; q < 7; ++q) m = fmaf(K(sl[q])[li], c->cmid[q], m);
                    float ymid = y0 + m;
                    yo[gi] = interp_eval(y0, y1, ymid, K(sl[0])[li], K(sl[6])[li], dtf, c->xs);
                });
                __syncthreads();
                ++next_out;
                if (threadIdx.x == 0) c->n_steps_interval = 0;
            }
            for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) { Y[li] = Y1[li]; });
            if (threadIdx.x == 0) {
                int t0 = c->slot[0];
                c->slot[0] = c->slot[6];
                c->slot[6] = t0;
            }
            __syncthreads();
        }
        pf.tick(PT_CTRL);
    }
    __syncthreads();
    ring_drain(p, s);
    pf.tick(PT_CTRL);
    write_status(p, pi, c, code);
    __syncthreads();
    }   // problems
    pf.finish();
    tmem_release(p, s.tmem);
    epilogue_epoch(p, s);
}

// =====================================================================================================================
// Adjoint sweep
// =====================================================================================================================
// Parameter-cotangent ("theta") passes.  The stage derivative of a theta element in physical slot q is the rank-B
// outer product of that stage's factors (SURVEY.md a15):
//   m[g]      : FM[g][q]
//   Wp[h][g]  : sum_b gLP[q][b][h] * l[q][b][g]        bp[h] : sum_b gLP[q][b][h]
//   Ws[h][g]  : sum_b gS [q][b][h] * s[q][b][g]        bs[h] : sum_b gS [q][b][h]
//   Wa[g][k]  : sum_b gJ [q][b][g] * SP[q][b][k]
// PP_SOL: PP_STEP without the error estimate and its norm sums -- the seminorm's pass, run after the accept decision
enum { PP_D01 = 0, PP_D2 = 1, PP_STEP = 2, PP_FIXED = 3, PP_COPY = 4, PP_SOL = 5 };

struct PPArgs {
    const float* src;   // theta at step start; nullptr while theta is known to be identically zero
    float* dst;         // where the pass writes (may alias src: every element is read before it is written)
    int s0, s1;         // D01: s0; D2: s0, s1
    int method;         // PP_FIXED: PHX_EULER / MIDPOINT / RK4 (slots 0..3)
    int last;           // PP_STEP: this step, if accepted, ends the interval -> write the dense output at t_end
    float coef_sol[7];  // indexed by PHYSICAL slot
    float coef_err[7];
    float coef_mid[7];
    int slot_first, slot_last;
    float dtf;
    float xs[4];
};

template <int MODE>
__device__ __forceinline__ void theta_elem(const float atol_f, const float rtol_f, const PPArgs& a, size_t idx,
                                           const float (&k)[7], double& acc0, double& acc1) {
    if (MODE == PP_COPY) {
        a.dst[idx] = a.src[idx];
        return;
    }
    const float th0 = a.src ? a.src[idx] : 0.f;
    if (MODE == PP_D01) {
        float scale = atol_f + fabsf(th0) * rtol_f;
        float r0 = th0 / scale, r1 = k[0] / scale;
        acc0 += (double)(r0 * r0);
        acc1 += (double)(r1 * r1);
    } else if (MODE == PP_D2) {
        float scale = atol_f + fabsf(th0) * rtol_f;
        float r = (k[1] - k[0]) / scale;
        acc0 += (double)(r * r);
    } else if (MODE == PP_STEP) {
        float inc = k[0] * a.coef_sol[0], e = k[0] * a.coef_err[0];
#pragma unroll
        for (int q = 1; q < 7; ++q) {
            inc = fmaf(k[q], a.coef_sol[q], inc);
            e = fmaf(k[q], a.coef_err[q], e);
        }
        float th1 = th0 + inc;
        float tol = atol_f + rtol_f * fmaxf(fabsf(th0), fabsf(th1));
        float r = e / tol;
        acc0 += (double)(r * r);
        if (!isfinite(th1)) acc1 += 1.0;
        if (a.last) {
            float md = k[0] * a.coef_mid[0];
            float kf = 0.f, kl = 0.f;
#pragma unroll
            for (int q = 0; q < 7; ++q) {
                if (q > 0) md = fmaf(k[q], a.coef_mid[q], md);
                kf = (q == a.slot_first) ? k[q] : kf;
                kl = (q == a.slot_last) ? k[q] : kl;
            }
            a.dst[idx] = interp_eval(th0, th1, th0 + md, kf, kl, a.dtf, a.xs);
        } else {
            a.dst[idx] = th1;
        }
    } else if (MODE == PP_FIXED) {
        float r;
        if (a.method == PHX_EULER) r = th0 + a.dtf * k[0];
        else if (a.method == PHX_MIDPOINT) r = th0 + a.dtf * k[1];
        else r = th0 + (k[0] + 3.f * (k[1] + k[2]) + k[3]) * a.dtf * 0.125f;
        a.dst[idx] = r;
    }
}

// PP_STEP for one theta element with the seven stage derivatives produced on the fly by kq(q) (q = physical slot):
// no k[] array exists, so nothing can be demoted to local memory (a select chain over an array is turned into a
// dynamically indexed load by the optimiser).  Same operation order as the reference's k.matmul(dt * c).
// ERR == false (PP_SOL): the written value only -- no error combination, no norm sums.
template <bool ERR = true, typename KQ>
__device__ __forceinline__ float theta_step_val(const float atol_f, const float rtol_f, const PPArgs& a, const float th0, KQ kq,
                                                double& acc0, double& acc1) {
    float inc = 0.f, e = 0.f, md = 0.f, kf = 0.f, kl = 0.f;
#pragma unroll
    for (int q = 0; q < 7; ++q) {
        const float t = kq(q);
        if (q == 0) {
            inc = t * a.coef_sol[0];
            if (ERR) e = t * a.coef_err[0];
            md = t * a.coef_mid[0];
        } else {
            inc = fmaf(t, a.coef_sol[q], inc);
            if (ERR) e = fmaf(t, a.coef_err[q], e);
            md = fmaf(t, a.coef_mid[q], md);
        }
        kf = (q == a.slot_first) ? t : kf;
        kl = (q == a.slot_last) ? t : kl;
    }
    const float th1 = th0 + inc;
    if (ERR) {
        const float tol = atol_f + rtol_f * fmaxf(fabsf(th0), fabsf(th1));
        const float r = e / tol;
        acc0 += (double)(r * r);
        if (!isfinite(th1)) acc1 += 1.0;
    }
    return a.last ? interp_eval(th0, th1, th0 + md, kf, kl, a.dtf, a.xs) : th1;
}
template <bool ERR = true, typename KQ>
__device__ __forceinline__ void theta_step(const float atol_f, const float rtol_f, const PPArgs& a, size_t idx, KQ kq,
                                           double& acc0, double& acc1) {
    const float th0 = a.src ? a.src[idx] : 0.f;
    a.dst[idx] = theta_step_val<ERR>(atol_f, rtol_f, a, th0, kq, acc0, acc1);
}

// which factor slots a mode needs, as k[0..NK): D01 {s0}, D2 {s0, s1}, STEP / SOL all seven physical slots, FIXED 0..3
template <int MODE>
struct PPSlots {
    static constexpr int NK = (MODE == PP_D01) ? 1
                            : (MODE == PP_D2 ? 2 : ((MODE == PP_STEP || MODE == PP_SOL) ? 7 : (MODE == PP_FIXED ? 4 : 0)));
};
template <int MODE>
__device__ __forceinline__ int pp_slot(const PPArgs& a, int i) {
    if (MODE == PP_D01) return a.s0;
    if (MODE == PP_D2) return i == 0 ? a.s0 : a.s1;
    return i;
}

// One R x C outer-product block of theta: element (r, c) at gbase + r * ld + c, factors U[r][QB] (smem, broadcast
// loads) and V[vcol(c)][QB] (held in registers by the thread that owns column c).
template <int MODE, int BT, typename VCol>
__device__ __forceinline__ void pp_block(const float atol_f, const float rtol_f, const PPArgs& a, int R, int C,
                                         const float* U, const float* V, VCol vcol, size_t gbase, size_t ld,
                                         double& acc0, double& acc1) {
    constexpr int NK = PPSlots<MODE>::NK;
    constexpr int NKA = NK > 0 ? NK : 1;
    constexpr int QB = (7 * BT + 3) & ~3;
    if (C <= 0 || R <= 0) return;
    for (int c0 = 0; c0 < C; c0 += THREADS) {
        const int Cw = min(C - c0, THREADS);
        const int RG = THREADS / Cw;
        const int ry = threadIdx.x / Cw, cx = threadIdx.x - ry * Cw;
        if (ry >= RG) continue;
        float v[NKA][BT];
        int uo[NKA];
        const float* vp = V + (size_t)vcol(c0 + cx) * QB;
#pragma unroll
        for (int i = 0; i < NKA; ++i) {
            uo[i] = pp_slot<MODE>(a, i) * BT;
#pragma unroll
            for (int b = 0; b < BT; ++b) v[i][b] = vp[uo[i] + b];
        }
        if constexpr (MODE == PP_STEP || MODE == PP_SOL) {
            // two rows per iteration: the per-element chain (7-term combinations, a division, the quartic) is long
            // and the rows are independent, so interleaving them doubles the instruction-level parallelism
            for (int r = ry; r < R; r += 2 * RG) {
                const int r2 = r + RG;
                const bool two = r2 < R;
                const float* upA = U + (size_t)r * QB;
                const float* upB = U + (size_t)(two ? r2 : r) * QB;
                float uA[QB], uB[QB];
#pragma unroll
                for (int i = 0; i < QB / 4; ++i) {
                    float4 t = reinterpret_cast<const float4*>(upA)[i];
                    uA[4 * i] = t.x; uA[4 * i + 1] = t.y; uA[4 * i + 2] = t.z; uA[4 * i + 3] = t.w;
                    t = reinterpret_cast<const float4*>(upB)[i];
                    uB[4 * i] = t.x; uB[4 * i + 1] = t.y; uB[4 * i + 2] = t.z; uB[4 * i + 3] = t.w;
                }
                const size_t iA = gbase + (size_t)r * ld + c0 + cx, iB = gbase + (size_t)(two ? r2 : r) * ld + c0 + cx;
                const float thA = a.src ? a.src[iA] : 0.f, thB = a.src ? a.src[iB] : 0.f;
                double b0 = 0, b1 = 0;
                const float oA = theta_step_val<MODE == PP_STEP>(atol_f, rtol_f, a, thA,
                                                [&](int q) {
                                                    float t = 0.f;
#pragma unroll
                                                    for (int b = 0; b < BT; ++b) t = fmaf(uA[q * BT + b], v[q < NKA ? q : 0][b], t);
                                                    return t;
                                                },
                                                acc0, acc1);
                const float oB = theta_step_val<MODE == PP_STEP>(atol_f, rtol_f, a, thB,
                                                [&](int q) {
                                                    float t = 0.f;
#pragma unroll
                                                    for (int b = 0; b < BT; ++b) t = fmaf(uB[q * BT + b], v[q < NKA ? q : 0][b], t);
                                                    return t;
                                                },
                                                b0, b1);
                a.dst[iA] = oA;
                if (two) {
                    a.dst[iB] = oB;
                    acc0 += b0;
                    acc1 += b1;
                }
            }
            continue;
        }
        for (int r = ry; r < R; r += RG) {
            const float* up = U + (size_t)r * QB;
            float k[7];
#pragma unroll
            for (int i = 0; i < 7; ++i) {
                float t = 0.f;
                if (i < NK) {
#pragma unroll
                    for (int b = 0; b < BT; ++b) t = fmaf(up[uo[i < NKA ? i : 0] + b], v[i < NKA ? i : 0][b], t);
                }
                k[i] = t;
            }
            theta_elem<MODE>(atol_f, rtol_f, a, gbase + (size_t)r * ld + c0 + cx, k, acc0, acc1);
        }
    }
}

// One pass over this CTA's share of the P-long parameter-cotangent vector.
struct PPSums {
    double a0, a1;
};
// (returns its two partial sums BY VALUE and builds its own shared-memory view: nothing of the caller's per-thread
// state may have its address taken, or it would live in local memory for the whole kernel)
static_assert(sizeof(PPArgs) <= 256, "PPArgs must fit its shared-memory slot");
template <int MODE, int BT>
__device__ __noinline__ PPSums ppass(const ResParams& __restrict__ p, int g_lo, int n_loc) {
    const Smem s(p);
    // the arguments travel through shared memory (written by thread 0, block barrier before the call); private copy:
    // the stores to theta may not force reloads of the coefficients
    const PPArgs a = *s.at<PPArgs>(p.so.ppa);
    double acc0 = 0, acc1 = 0;
    constexpr int NK = PPSlots<MODE>::NK;
    constexpr int QB = (7 * BT + 3) & ~3;
    const PhxGradOff off = phx_grad_offsets(p.G, p.H);
    const int Hp = p.Hp, H = p.H, G = p.G;
    const float atol_f = p.atol_f, rtol_f = p.rtol_f;
    // only the blocks of the adjoint parameters are read or written (p.pmask); the others are zeroed once at the end
    const int pm = p.pmask;
    if (MODE == PP_COPY) {
        float k[7] = {0, 0, 0, 0, 0, 0, 0};
        if (pm & PHX_P_M)
            for (int j = threadIdx.x; j < n_loc; j += THREADS) theta_elem<MODE>(atol_f, rtol_f, a, off.m + g_lo + j, k, acc0, acc1);
        for (int h = 0; h < H; ++h)
            for (int j = threadIdx.x; j < n_loc; j += THREADS) {
                if (pm & PHX_P_WP) theta_elem<MODE>(atol_f, rtol_f, a, off.Wp + (size_t)h * G + g_lo + j, k, acc0, acc1);
                if (pm & PHX_P_WS) theta_elem<MODE>(atol_f, rtol_f, a, off.Ws + (size_t)h * G + g_lo + j, k, acc0, acc1);
            }
        if (pm & PHX_P_WA)
            for (size_t e = threadIdx.x; e < (size_t)n_loc * 2 * H; e += THREADS)
                theta_elem<MODE>(atol_f, rtol_f, a, off.Wa + (size_t)g_lo * 2 * H + e, k, acc0, acc1);
        if (blockIdx.x == 0)
            for (int h = threadIdx.x; h < H; h += THREADS) {
                if (pm & PHX_P_BP) theta_elem<MODE>(atol_f, rtol_f, a, off.bp + h, k, acc0, acc1);
                if (pm & PHX_P_BS) theta_elem<MODE>(atol_f, rtol_f, a, off.bs + h, k, acc0, acc1);
            }
        return PPSums{acc0, acc1};
    }
    // m
    if (pm & PHX_P_M)
    for (int j = threadIdx.x; j < n_loc; j += THREADS) {
        if constexpr (MODE == PP_STEP || MODE == PP_SOL) {
            theta_step<MODE == PP_STEP>(atol_f, rtol_f, a, off.m + g_lo + j, [&](int q) { return s.FM()[j * 8 + q]; },
                                        acc0, acc1);
        } else {
            float k[7];
#pragma unroll
            for (int i = 0; i < 7; ++i) k[i] = (i < NK) ? s.FM()[j * 8 + pp_slot<MODE>(a, i)] : 0.f;
            theta_elem<MODE>(atol_f, rtol_f, a, off.m + g_lo + j, k, acc0, acc1);
        }
    }
    auto ident = [](int c) { return c; };
    // Wp, Ws : rows h (factors FG), this CTA's gene columns (factors FL / FS)
    if (pm & PHX_P_WP)
        pp_block<MODE, BT>(atol_f, rtol_f, a, H, n_loc, s.FG() + (size_t)Hp * QB, s.FL(), ident, off.Wp + g_lo, (size_t)G, acc0, acc1);
    if (pm & PHX_P_WS)
        pp_block<MODE, BT>(atol_f, rtol_f, a, H, n_loc, s.FG(), s.FS(), ident, off.Ws + g_lo, (size_t)G, acc0, acc1);
    // Wa : this CTA's gene rows (factors FGJ), 2H columns (factors FSP, skipping the padded columns)
    if (pm & PHX_P_WA)
        pp_block<MODE, BT>(atol_f, rtol_f, a, n_loc, 2 * H, s.FGJ(), s.FSP(), [&](int kk) { return kk < H ? kk : Hp + kk - H; },
                           off.Wa + (size_t)g_lo * 2 * H, (size_t)2 * H, acc0, acc1);
    // biases : CTA 0
    if (blockIdx.x == 0) {
        for (int h = threadIdx.x; h < 2 * H; h += THREADS) {
            const bool prod = h >= H;
            if (!(pm & (prod ? PHX_P_BP : PHX_P_BS))) continue;
            const float* up = s.FG() + (size_t)(prod ? Hp + h - H : h) * QB;
            if constexpr (MODE == PP_STEP || MODE == PP_SOL) {
                theta_step<MODE == PP_STEP>(atol_f, rtol_f, a, (prod ? off.bp + (h - H) : off.bs + h),
                           [&](int q) {
                               float t = 0.f;
                               for (int b = 0; b < BT; ++b) t += up[q * BT + b];
                               return t;
                           },
                           acc0, acc1);
                continue;
            }
            float k[7];
#pragma unroll
            for (int i = 0; i < 7; ++i) {
                float t = 0.f;
                if (i < NK) {
                    int o = pp_slot<MODE>(a, i) * BT;
                    for (int b = 0; b < BT; ++b) t += up[o + b];
                }
                k[i] = t;
            }
            theta_elem<MODE>(atol_f, rtol_f, a, (prod ? off.bp + (h - H) : off.bs + h), k, acc0, acc1);
        }
    }
    return PPSums{acc0, acc1};
}

// sum over (r, c) of (sum_m sgn_m U[r][idx_m] V[c][idx_m])^2 through the two M x M Gram matrices (theta == 0 norms:
// no pass over memory).  All threads return the same value.
__device__ __noinline__ double gram_sq(const Smem& s, const float* U, int R, const float* V, int C, int QB, const int* idx,
                          const float* sgn, int M) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int MM = M * M;
    __syncthreads();
    for (int pr = warp; pr < 2 * MM; pr += WARPS) {
        const int which = pr / MM, m = (pr % MM) / M, m2 = pr % M;
        const float* X = which ? V : U;
        const int n = which ? C : R;
        double t = 0;
        for (int r = lane; r < n; r += 32) t += (double)X[(size_t)r * QB + idx[m]] * (double)X[(size_t)r * QB + idx[m2]];
        t = warp_sum_d(t);
        if (lane == 0) s.gram()[pr] = t;
    }
    __syncthreads();
    double tot = 0;
    for (int m = 0; m < M; ++m)
        for (int m2 = 0; m2 < M; ++m2)
            tot += (double)(sgn[m] * sgn[m2]) * s.gram()[m * M + m2] * s.gram()[MM + m * M + m2];
    return tot;
}

// this thread's share of the sum over this CTA's theta elements of (k / atol)^2 with k = k[s1] - k[s0]
// (s0 < 0: k = k[s1]); valid while theta == 0 (scale = atol, misc.py:63).
template <int BT>
__device__ __noinline__ double theta_zero_norm(const ResParams& p, int n_loc, int s1, int s0) {
    const Smem s(p);
    constexpr int QB = (7 * BT + 3) & ~3;
    int idx[8];
    float sgn[8];
    int M = 0;
    for (int b = 0; b < BT; ++b) { idx[M] = s1 * BT + b; sgn[M] = 1.f; ++M; }
    if (s0 >= 0)
        for (int b = 0; b < BT; ++b) { idx[M] = s0 * BT + b; sgn[M] = -1.f; ++M; }
    const int Hp = p.Hp, pm = p.pmask;
    double tot = 0;
    // Wp, Ws (padded branch columns hold zeros), Wa -- the adjoint parameters only (every thread takes the same branches)
    if (pm & PHX_P_WP) tot += gram_sq(s, s.FG() + (size_t)Hp * QB, Hp, s.FL(), n_loc, QB, idx, sgn, M);
    if (pm & PHX_P_WS) tot += gram_sq(s, s.FG(), Hp, s.FS(), n_loc, QB, idx, sgn, M);
    if (pm & PHX_P_WA) tot += gram_sq(s, s.FGJ(), n_loc, s.FSP(), p.K2, QB, idx, sgn, M);
    // m (per gene) and, on CTA 0, the biases: direct
    double loc = 0;
    if (pm & PHX_P_M)
    for (int j = threadIdx.x; j < n_loc; j += THREADS) {
        float k = s.FM()[j * 8 + s1] - (s0 >= 0 ? s.FM()[j * 8 + s0] : 0.f);
        loc += (double)k * (double)k;
    }
    if (blockIdx.x == 0) {
        for (int h = threadIdx.x; h < p.K2; h += THREADS) {
            if (!(pm & (h < Hp ? PHX_P_BS : PHX_P_BP))) continue;
            float k1 = 0.f, k0 = 0.f;
            for (int b = 0; b < BT; ++b) {
                k1 += s.FG()[(size_t)h * QB + s1 * BT + b];
                if (s0 >= 0) k0 += s.FG()[(size_t)h * QB + s0 * BT + b];
            }
            float k = k1 - k0;
            loc += (double)k * (double)k;
        }
    }
    double mine = loc + (threadIdx.x == 0 ? tot : 0.0);
    return mine / ((double)p.atol_f * (double)p.atol_f);
}

// One RHS + VJP evaluation at the current stage input (ysb / acts / actl, cotangent asb / gjb); stage derivatives land
// in KY(slot) / KA(slot), the theta factors in column `slot` of the factor tables.
//   sp_ready: the branch vector of this input is already in s.sp() (it was all-reduced together with the previous
//             evaluation's gS|gP); otherwise a stand-alone pass A + exchange runs first.
//   has_next: ynext(b, j, li, ky) returns the NEXT stage's y input per element; its pass A is fused into pass 1 and its
//             branch vector shares this evaluation's single all-reduce.  anext(b, j, li, ka, lead) returns the next
//             stage's cotangent input (and is where the caller does its per-element stage algebra).
template <int NV, int BT, typename YNext, typename ANext>
__device__ __forceinline__ void adj_eval(const ResParams& __restrict__ p, Smem& __restrict__ s, int slot, bool sp_ready,
                                         bool has_next, YNext ynext, ANext anext) {
    constexpr int QB = (7 * BT + 3) & ~3;
    Prof& pf = s.pf;
    const int n = p.B * p.K2;
    if (!sp_ready) eval_A<NV, BT>(p, s);
    pf.tick(PT_COMBINE);
    adj_pass1<NV, BT>(p, s, slot, has_next, ynext);
    pf.tick(PT_PHASE_B);
    grid_allreduce_f(p, s, s.xv(), has_next ? 2 * n : n);
    pf.tick(PT_ALLRED2);
    // gLP = gPr * Pr (exp backward); record the stage's K2-long theta factors; the next stage's branch vector replaces
    // this one (bias, exp) -- every index is handled by one thread, reads before writes
    for (int i = threadIdx.x; i < n; i += THREADS) {
        const int b = i / p.K2, k = i - b * p.K2;
        const float spv = s.sp()[i];
        float gv = s.gsp()[i];
        if (k >= p.Hp) gv = gv * spv;
        s.gsp()[i] = gv;
        s.FSP()[k * QB + slot * BT + b] = spv;
        s.FG()[k * QB + slot * BT + b] = gv;
        if (has_next) {
            float v = s.spn()[i] + s.bias()[k];
            if (k >= p.Hp) v = (k - p.Hp < p.H) ? expf(v) : 0.f;
            s.sp()[i] = v;
        }
    }
    __syncthreads();
    pf.tick(PT_FINALIZE);
    adj_pass2<NV, BT>(p, s, slot, has_next, anext);
    if (has_next) s.swap_stage_buffers();
    pf.tick(PT_PHASE_C);
}

// SEMI: the seminorm (p.pmask & PHX_NORM_SEMINORM), an instantiation of its own so that the default norm keeps its code
// GRID: as in phx_fwd_kernel (fixed grids use no norm: the grid instantiations are the default-norm ones)
template <int NV, int BT, bool SEMI, bool GRID>
__global__ void __launch_bounds__(PHX_THREADS, 1) phx_adj_kernel(const __grid_constant__ ResParams p) {
    constexpr int QB = (7 * BT + 3) & ~3;
    Smem s(p);
    const int g_lo = s.g_lo, n_loc = s.n_loc;
    prologue(p, s);
    s.tmem = tmem_setup<NV>(p, s);
    Prof& pf = s.pf;
    Ctrl* c = s.ctrl();
    const size_t BG = (size_t)p.B * p.G;
    const int BL = p.B * p.gpc;
    const double Nel = (double)p.B * (double)p.G;
    const PhxGradOff goff = phx_grad_offsets(p.G, p.H);
    // theta block of the norm: the adjoint parameters only; with none the block is absent (th_rms == 0 never wins the
    // max over the other, non-negative blocks).  The seminorm drops it too: no theta norm pass runs, and the theta step
    // pass moves after the accept decision (accepted attempts only, solution combination only, in place)
    const double Pel = SEMI ? 0.0 : (double)phx_mask_count(p.G, p.H, p.pmask);
    auto th_rms = [&](double sum) { return Pel > 0 ? sqrtf((float)(sum / Pel)) : 0.f; };
    float* Y = s.st();
    float* A = s.st() + BL;
    float* Y1 = s.st() + 2 * BL;
    float* A1 = s.st() + 3 * BL;
    auto KY = [&](int i) { return s.st() + (4 + i) * BL; };
    auto KA = [&](int i) { return s.st() + (11 + i) * BL; };
    // independent problems, one after the other: the weights stay on chip (shared / tensor memory) across them
    for (int pi = 0; pi < p.nprob; ++pi) {
    const float* ysavedp = p.ysaved + (size_t)pi * p.yout_stride;
    const float* gradyp = p.grad_y + (size_t)pi * p.yout_stride;
    float* adjy0p = p.adj_y0 + (size_t)pi * p.adj_stride;
    float* theta0p = p.theta0 + (size_t)pi * p.theta_stride;
    int cur = 0;             // which theta buffer holds the current value (meaningful once !theta_zero)
    bool theta_zero = true;  // the accumulator has not been written yet: it is identically zero and never read

    if (threadIdx.x == 0) {
        c->n_acc = c->n_rej = c->n_rhs = c->n_log = 0;
        c->stop = 0;
        c->tcur = 0;
        c->dt = 0;
    }
    // zero the factor tables once (padded entries are read by the float4 loads of the theta passes)
    for (int i = threadIdx.x; i < p.K2 * QB; i += THREADS) { s.FG()[i] = 0.f; s.FSP()[i] = 0.f; }
    for (int i = threadIdx.x; i < p.gpc * QB; i += THREADS) { s.FS()[i] = 0.f; s.FL()[i] = 0.f; s.FGJ()[i] = 0.f; }
    for (int i = threadIdx.x; i < p.gpc * 8; i += THREADS) s.FM()[i] = 0.f;
    __syncthreads();

    // stage input (y, a) -> smem activations and gJ = a * relu(m)
    auto set_y_input = [&](float* ysb, float* acts, float* actl, int li, float ys) {
        ysb[li] = ys;
        float sv, lv, den;
        hill(ys, sv, lv, den);
        acts[li] = sv;
        actl[li] = lv;
    };
    auto set_a_input = [&](int li, int j, float as) {
        s.asb()[li] = as;
        s.gjb()[li] = as * s.relum()[j];
    };

    auto no_y = [](int, int, int, float) { return 0.f; };
    auto no_a = [](int, int, int, float, bool) { return 0.f; };

    int code = PHX_ST_OK;
    for (int iv = p.T - 1; iv >= 1 && code == PHX_ST_OK; --iv) {
        const float* ysv = ysavedp + (size_t)iv * BG;
        const float* gy = gradyp + (size_t)iv * BG;
        const bool first_iv = (iv == p.T - 1);
        for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
            float y = ysv[gi];
            float av = first_iv ? gy[gi] : A[li];
            Y[li] = y;
            A[li] = av;
            set_y_input(s.ysb(), s.acts(), s.actl(), li, y);
            set_a_input(li, j, av);
        });
        __syncthreads();
        const double t_start = -tget(p, pi, iv), t_end = -tget(p, pi, iv - 1);

        if (p.method != PHX_DOPRI5) {
            // one step per interval, or the steps of the interval's own grid (p.gdt): y and adj_y advance together, and
            // every step runs its own theta pass
            const int seg = pi * (p.T - 1) + iv - 1;
            const int nk = GRID ? p.goff[seg + 1] - p.goff[seg] : 1;
            for (int k = 0; k < nk; ++k) {
            const float dtf = GRID ? p.gdt[p.goff[seg] + k]
                                    : (p.t_is_f32 ? ((float)tget(p, pi, iv) - (float)tget(p, pi, iv - 1)) : (float)(tget(p, pi, iv) - tget(p, pi, iv - 1)));
            const bool more = k + 1 < nk;
            const float third = (float)(1.0 / 3.0);
            if (k > 0) {   // the next step starts from the state the last one left in Y / A
                for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                    set_y_input(s.ysb(), s.acts(), s.actl(), li, Y[li]);
                    set_a_input(li, j, A[li]);
                });
                __syncthreads();
            }
            if (threadIdx.x == 0) {
                PPArgs& pa = *s.at<PPArgs>(p.so.ppa);
                pa.src = theta_zero ? nullptr : theta0p;
                pa.dst = theta0p;
                pa.dtf = dtf;
                pa.method = p.method;
            }
            // one call site for every stage of every fixed-grid method (stage algebra switches at run time)
            const int nst = (p.method == PHX_EULER) ? 1 : (p.method == PHX_MIDPOINT ? 2 : 4);
            const float half = 0.5f * dtf;
            for (int st = 0; st < nst; ++st) {
                const bool last = st + 1 == nst;
                adj_eval<NV, BT>(
                    p, s, st, st > 0, !last,
                    [&](int b, int j, int li, float ky) {
                        if (p.method == PHX_MIDPOINT) return Y[li] + ky * half;
                        if (st == 0) return Y[li] + dtf * ky * third;
                        if (st == 1) return Y[li] + dtf * (ky - KY(0)[li] * third);
                        return Y[li] + dtf * (KY(0)[li] - KY(1)[li] + ky);
                    },
                    [&](int b, int j, int li, float ka, bool lead) {
                        float an;
                        if (p.method == PHX_EULER) {
                            an = A[li] + dtf * ka;
                        } else if (p.method == PHX_MIDPOINT) {
                            an = (st == 0) ? A[li] + ka * half : A[li] + dtf * ka;
                        } else {
                            if (st == 0) an = A[li] + dtf * ka * third;
                            else if (st == 1) an = A[li] + dtf * (ka - KA(0)[li] * third);
                            else if (st == 2) an = A[li] + dtf * (KA(0)[li] - KA(1)[li] + ka);
                            else an = A[li] + (KA(0)[li] + 3.f * (KA(1)[li] + KA(2)[li]) + ka) * dtf * 0.125f;
                        }
                        if (last && lead) {
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
            pf.tick(PT_COMBINE);
            ppass<PP_FIXED, BT>(p, g_lo, n_loc);
            pf.tick(PT_PP_STEP);
            theta_zero = false;
            if (threadIdx.x == 0) {
                int per = (p.method == PHX_EULER) ? 1 : (p.method == PHX_MIDPOINT ? 2 : 4);
                c->n_rhs += per;
                c->tcur = t_end;
            }
            __syncthreads();
            }
        } else {
            // ------------------------------ dopri5 on the augmented state ------------------------------
            if (threadIdx.x == 0) {
                c->tcur = t_start;
                c->tprev = t_start;
                c->t_end = t_end;
                c->n_steps_interval = 0;
                for (int i = 0; i < 7; ++i) c->slot[i] = i;
                if (has_t_vjp<GRID>(p)) c->vjp_t = p.t_vjp[(size_t)pi * (p.T - 1) + iv - 1];
            }
            __syncthreads();
            // f0 and Hairer's initial step under the mixed norm max(RMS_y, RMS_a, RMS_theta): two evaluations through
            // one call site, or f0 alone when the caller gives the first step
            for (int which = 0; which < 2; ++which) {
                double acc[7] = {0, 0, 0, 0, 0, 0, 0};
                adj_eval<NV, BT>(p, s, which, false, false, no_y, [&](int b, int j, int li, float ka, bool lead) {
                    if (lead) {
                        float y = Y[li], av = A[li];
                        float sy = p.atol_f + fabsf(y) * p.rtol_f, sa = p.atol_f + fabsf(av) * p.rtol_f;
                        float r;
                        if (which == 0) {
                            r = y / sy; acc[0] += (double)(r * r);
                            r = av / sa; acc[1] += (double)(r * r);
                            r = KY(0)[li] / sy; acc[3] += (double)(r * r);
                            r = ka / sa; acc[4] += (double)(r * r);
                            if (!isfinite(y) || !isfinite(av)) acc[6] += 1.0;
                        } else {
                            r = (KY(1)[li] - KY(0)[li]) / sy; acc[0] += (double)(r * r);
                            r = (ka - KA(0)[li]) / sa; acc[1] += (double)(r * r);
                        }
                    }
                    return 0.f;
                });
                if (threadIdx.x == 0) {
                    PPArgs& pa = *s.at<PPArgs>(p.so.ppa);
                    pa.src = theta_zero ? nullptr : (cur ? p.theta1 : theta0p);
                    pa.dst = nullptr;
                    pa.s0 = 0;
                    pa.s1 = 1;
                }
                __syncthreads();
                pf.tick(PT_COMBINE);
                if (which == 0) {
                    if (!SEMI && !given_step<GRID>(p)) {   // (the seminorm has no theta block; a given first step
                                                          // needs no norm)
                        if (theta_zero) {
                            acc[5] += theta_zero_norm<BT>(p, n_loc, 0, -1);
                        } else {
                            PPSums ps = ppass<PP_D01, BT>(p, g_lo, n_loc);
                            acc[2] += ps.a0;
                            acc[5] += ps.a1;
                        }
                    }
                    pf.tick(PT_PP_D01);
                    block_sum_d<7>(acc, s.dred(), c->dsum);
                    grid_sum_d(p, s, c->dsum, 7);
                    pf.tick(PT_NORMS);
                    if (threadIdx.x == 0) {
                        float d0 = fmaxf(fmaxf(sqrtf((float)(c->dsum[0] / Nel)), sqrtf((float)(c->dsum[1] / Nel))),
                                         th_rms(c->dsum[2]));
                        float d1 = fmaxf(fmaxf(sqrtf((float)(c->dsum[3] / Nel)), sqrtf((float)(c->dsum[4] / Nel))),
                                         th_rms(c->dsum[5]));
                        c->d1 = d1;
                        c->nonfinite_prev = c->dsum[6] > 0.0;
                        if (has_t_vjp<GRID>(p) && fold_t_vjp(p, c->vjp_t, d0)) c->nonfinite_prev = 1;
                        c->h0 = init_h0(d0, d1);
                        if (given_step<GRID>(p)) {
                            c->dt = p.first_step;
                            c->n_rhs += 1;
                        }
                    }
                    __syncthreads();
                    if (given_step<GRID>(p)) break;   // the caller's first step: no second evaluation
                    const float h0 = c->h0;
                    for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                        set_y_input(s.ysb(), s.acts(), s.actl(), li, Y[li] + h0 * KY(0)[li]);
                        set_a_input(li, j, A[li] + h0 * KA(0)[li]);
                    });
                    __syncthreads();
                } else {
                    if (!SEMI) {
                        if (theta_zero) acc[2] += theta_zero_norm<BT>(p, n_loc, 1, 0);
                        else acc[2] += ppass<PP_D2, BT>(p, g_lo, n_loc).a0;
                    }
                    pf.tick(PT_PP_D2);
                    block_sum_d<7>(acc, s.dred(), c->dsum);
                    grid_sum_d(p, s, c->dsum, 3);
                    pf.tick(PT_NORMS);
                    if (threadIdx.x == 0) {
                        float d2 = fmaxf(fmaxf(sqrtf((float)(c->dsum[0] / Nel)), sqrtf((float)(c->dsum[1] / Nel))),
                                         th_rms(c->dsum[2])) / c->h0;
                        c->dt = init_dt(c->h0, c->d1, d2);
                        c->n_rhs += 2;
                    }
                    __syncthreads();
                }
            }
            bool done = false;
            while (!done) {
                if (threadIdx.x == 0) {
                    int st = 0;
                    if ((long long)c->n_steps_interval >= p.max_steps) st = PHX_ST_MAX_STEPS;
                    else if (!(c->tcur + c->dt > c->tcur)) st = PHX_ST_DT_UNDERFLOW;
                    else if (c->nonfinite_prev) st = PHX_ST_NONFINITE;
                    c->stop = st;
                    if (!st) {
                        set_step_coeffs(c);
                        // this step, if accepted, reaches t_end: same comparison as rk_common.py:153 after the step
                        c->last = !(c->t_end > c->tcur + c->dt);
                        if (c->last) set_interp_x(c, c->t_end, c->tcur, c->tcur + c->dt);
                    }
                }
                __syncthreads();
                if (c->stop) {
                    code = c->stop;
                    break;
                }
                const int* sl = c->slot;   // FSAL slot permutation, read from shared memory
                {
                    const float c00 = c->cb[0][0];
                    for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                        set_y_input(s.ysb(), s.acts(), s.actl(), li, Y[li] + KY(sl[0])[li] * c00);
                        set_a_input(li, j, A[li] + KA(sl[0])[li] * c00);
                    });
                    __syncthreads();
                }
                double acc[4] = {0, 0, 0, 0};
                for (int st = 1; st <= 6; ++st) {
                    adj_eval<NV, BT>(
                        p, s, sl[st], st > 1, st < 6,
                        // next stage's y input from ky of stages 0..st (the newest one still in a register)
                        [&](int b, int j, int li, float ky) {
                            float ay = KY(sl[0])[li] * c->cb[st][0];
                            for (int q = 1; q < st; ++q) ay = fmaf(KY(sl[q])[li], c->cb[st][q], ay);
                            ay = fmaf(ky, c->cb[st][st], ay);
                            float yn = Y[li] + ay;
                            if (st == 5) Y1[li] = yn;
                            return yn;
                        },
                        [&](int b, int j, int li, float ka, bool lead) {
                            if (st < 6) {
                                float aa = KA(sl[0])[li] * c->cb[st][0];
                                for (int q = 1; q < st; ++q) aa = fmaf(KA(sl[q])[li], c->cb[st][q], aa);
                                aa = fmaf(ka, c->cb[st][st], aa);
                                float an = A[li] + aa;
                                if (st == 5 && lead) A1[li] = an;
                                return an;
                            }
                            if (lead) {
                                float ey = KY(sl[0])[li] * c->cerr[0];
                                float ea = KA(sl[0])[li] * c->cerr[0];
                                for (int q = 1; q < 6; ++q) {
                                    ey = fmaf(KY(sl[q])[li], c->cerr[q], ey);
                                    ea = fmaf(KA(sl[q])[li], c->cerr[q], ea);
                                }
                                ey = fmaf(KY(sl[6])[li], c->cerr[6], ey);
                                ea = fmaf(ka, c->cerr[6], ea);
                                float y1 = s.ysb()[li], a1 = s.asb()[li];
                                float ty = p.atol_f + p.rtol_f * fmaxf(fabsf(Y[li]), fabsf(y1));
                                float ta = p.atol_f + p.rtol_f * fmaxf(fabsf(A[li]), fabsf(a1));
                                float r;
                                r = ey / ty; acc[0] += (double)(r * r);
                                r = ea / ta; acc[1] += (double)(r * r);
                                if (!isfinite(y1) || !isfinite(a1)) acc[3] += 1.0;
                            }
                            return 0.f;
                        });
                }
                if (threadIdx.x == 0) {
                    PPArgs& pa = *s.at<PPArgs>(p.so.ppa);
                    pa.src = theta_zero ? nullptr : (cur ? p.theta1 : theta0p);
                    // (seminorm: cur stays 0, the pass writes in place)
                    pa.dst = (theta_zero || SEMI) ? theta0p : (cur ? theta0p : p.theta1);
                    pa.dtf = c->dtf;
                    pa.last = c->last;
                    for (int q = 0; q < 7; ++q) {
                        pa.coef_sol[sl[q]] = (q < 6) ? c->cb[5][q] : 0.f;
                        pa.coef_err[sl[q]] = c->cerr[q];
                        pa.coef_mid[sl[q]] = c->cmid[q];
                    }
                    pa.slot_first = sl[0];
                    pa.slot_last = sl[6];
                    for (int q = 0; q < 4; ++q) pa.xs[q] = c->xs[q];
                }
                __syncthreads();
                pf.tick(PT_COMBINE);
                if (!SEMI) {
                    PPSums ps = ppass<PP_STEP, BT>(p, g_lo, n_loc);
                    acc[2] += ps.a0;
                    acc[3] += ps.a1;
                }
                pf.tick(PT_PP_STEP);
                block_sum_d<4>(acc, s.dred(), c->dsum);
                grid_sum_d(p, s, c->dsum, 4);
                pf.tick(PT_NORMS);
                if (threadIdx.x == 0) {
                    float ratio = fmaxf(fmaxf(sqrtf((float)(c->dsum[0] / Nel)), sqrtf((float)(c->dsum[1] / Nel))),
                                        th_rms(c->dsum[2]));
                    // torch's max() over 0-dim tensors is Python max: a NaN in a later block does not propagate the
                    // same way; treat any NaN as NaN (step rejected, dt -> NaN -> underflow assertion)
                    if (isnan(c->dsum[0]) || isnan(c->dsum[1]) || isnan(c->dsum[2])) ratio = nanf("");
                    int accept = ratio <= 1.f;
                    log_step(p, c, c->tcur, c->dt, accept);
                    c->tprev = c->tcur;
                    if (accept) {
                        c->tcur = c->tcur + c->dt;
                        c->n_acc++;
                        c->nonfinite_prev = c->dsum[3] > 0.0;
                    } else {
                        c->n_rej++;
                    }
                    c->dt = next_dt(p, c->dt, ratio);
                    c->accept = accept;
                    c->n_rhs += 6;
                    c->n_steps_interval++;
                }
                __syncthreads();
                if (c->accept) {
                    if (SEMI) {
                        // the seminorm's theta step: accepted attempts only, in place (cur stays 0)
                        ppass<PP_SOL, BT>(p, g_lo, n_loc);
                        pf.tick(PT_PP_STEP);
                        theta_zero = false;
                    } else if (theta_zero) {
                        cur = 0;
                        theta_zero = false;
                    } else {
                        cur ^= 1;
                    }
                    if (c->last) {
                        // last step of the interval: dense output at t_end for adj_y (adj_params: done in the pass)
                        const float dtf = c->dtf;
                        for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                            float a0 = A[li], a1 = A1[li];
                            float m = KA(sl[0])[li] * c->cmid[0];
                            for (int q = 1; q < 7; ++q) m = fmaf(KA(sl[q])[li], c->cmid[q], m);
                            A[li] = interp_eval(a0, a1, a0 + m, KA(sl[0])[li], KA(sl[6])[li], dtf, c->xs);
                        });
                        done = true;
                    } else {
                        for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) {
                            Y[li] = Y1[li];
                            A[li] = A1[li];
                        });
                        if (threadIdx.x == 0) {
                            int t0 = c->slot[0];
                            c->slot[0] = c->slot[6];
                            c->slot[6] = t0;
                        }
                    }
                    __syncthreads();
                }
                pf.tick(PT_CTRL);
            }
        }
        // interval done: adj_y picks up the loss gradient at t[iv-1] (adjoint.py:152-154)
        if (code == PHX_ST_OK) {
            const float* gprev = gradyp + (size_t)(iv - 1) * BG;
            for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) { A[li] = A[li] + gprev[gi]; });
            __syncthreads();
        }
    }
    for_local(p, g_lo, n_loc, [&](int b, int j, int g, size_t gi, int li) { adjy0p[gi] = A[li]; });
    pf.tick(PT_COMBINE);
    if (theta_zero) {
        // nothing was ever written (a solver assertion fired before the first accepted step): report zeros
        const size_t tot = goff.total;
        for (size_t i = (size_t)blockIdx.x * THREADS + threadIdx.x; i < tot; i += (size_t)gridDim.x * THREADS)
            theta0p[i] = 0.f;
    } else if (cur != 0) {
        // the last accepted step landed in the scratch twin
        if (threadIdx.x == 0) {
            PPArgs& pa = *s.at<PPArgs>(p.so.ppa);
            pa.src = p.theta1;
            pa.dst = theta0p;
        }
        __syncthreads();
        ppass<PP_COPY, BT>(p, g_lo, n_loc);
    }
    if (!theta_zero && (SEMI ? p.pmask & PHX_P_ALL : p.pmask) != PHX_P_ALL) {
        // the blocks of parameters outside the adjoint set were never touched: report zeros
        const int pm = p.pmask;
        const size_t HG = (size_t)p.H * p.G;
        const size_t lo[6] = {goff.m, goff.Wp, goff.bp, goff.Ws, goff.bs, goff.Wa};
        const size_t n[6] = {(size_t)p.G, HG, (size_t)p.H, HG, (size_t)p.H, 2 * HG};
        for (int q = 0; q < 6; ++q) {
            if (pm & (1 << q)) continue;
            for (size_t i = (size_t)blockIdx.x * THREADS + threadIdx.x; i < n[q]; i += (size_t)gridDim.x * THREADS)
                theta0p[lo[q] + i] = 0.f;
        }
    }
    pf.tick(PT_PP_COPY);
    __syncthreads();
    ring_drain(p, s);
    pf.tick(PT_CTRL);
    write_status(p, pi, c, code);
    __syncthreads();
    }   // problems
    pf.finish();
    tmem_release(p, s.tmem);
    epilogue_epoch(p, s);
}

}  // namespace
