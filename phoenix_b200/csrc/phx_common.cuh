// Shared definitions of the phoenix_b200 CUDA library (sm_100a).
//
// Data layout in HBM (all fp32):
//   packed weights  (built once per optimiser step by phx_pack_weights, constant during a solve)
//     W1[G][K2]   row g = [ Ws[0:H, g] | 0-pad to Hp | Wp[0:H, g] | 0-pad to Hp ]   (gene-major transposes of the
//                 two branch matrices, so the weights of one gene are one contiguous K2*4-byte row)
//     WA[G][K2]   row g = [ Wa[g, 0:H] | 0-pad | Wa[g, H:2H] | 0-pad ]
//     bias[K2]    [ bs | 0 | bp | 0 ]
//     relum[G]    relu(gene_multipliers)            maskm[G]  (gene_multipliers > 0)
//   Hp = round_up(H, 4), K2 = 2*Hp, so every row is a whole number of float4 and each float4 lies in one half.
//   solver state [slot][B][G]: every (row b, gene g) element is owned by exactly one thread of the CTA that owns
//   gene g, so state never needs cross-CTA synchronisation; only the K2-long branch vectors do.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <vector>
#include "../../include/phoenix_b200.h"

#define PHX_THREADS 512
#define PHX_WARPS 16
#define PHX_MAX_B_FWD 8
#define PHX_MAX_B_ADJ 4
#define PHX_SMEM_LIMIT (227 * 1024)

static inline __host__ __device__ int phx_round_up(int x, int m) { return (x + m - 1) / m * m; }
static inline __host__ __device__ int phx_Hp(int H) { return phx_round_up(H, 4); }
static inline __host__ __device__ int phx_K2(int H) { return 2 * phx_Hp(H); }
#include "phx_tc.cuh"

struct PhxPacked {
    const float4* W1;
    const float4* WA;
    const float* bias;
    const float* relum;
    const float* maskm;
    // tensor-core operand images (phx_tc.cuh), the tail of the packed buffer; valid only once tc_pack has run on it
    const float* w1img;
    const float* waimg;
    const float* watimg;
    const float* w1kimg;
    int tc;   // 0: fp32 CUDA-core contractions; 3: 3xTF32 tcgen05; 1: single-pass TF32 tcgen05 (set by the entry points)
};

// base part (W1, WA, bias, relum, maskm) rounded up to 128 bytes so that the tensor-core images that follow are aligned
static inline __host__ __device__ size_t phx_packed_base_floats(int G, int H) {
    size_t K2 = (size_t)phx_K2(H);
    size_t n = 2 * (size_t)G * K2 + K2 + 2 * (size_t)phx_round_up(G, 4);
    return (n + 31) & ~(size_t)31;
}
static inline __host__ __device__ size_t phx_packed_floats(int G, int H) {
    return phx_packed_base_floats(G, H) + 2 * (phx_tc_w1img_floats(G, H) + phx_tc_waimg_floats(G, H));
}

static inline __host__ __device__ PhxPacked phx_packed_view(const float* base, int G, int H) {
    size_t K2 = (size_t)phx_K2(H);
    PhxPacked v;
    v.W1 = reinterpret_cast<const float4*>(base);
    v.WA = reinterpret_cast<const float4*>(base + (size_t)G * K2);
    v.bias = base + 2 * (size_t)G * K2;
    v.relum = v.bias + K2;
    v.maskm = v.relum + phx_round_up(G, 4);
    v.w1img = base + phx_packed_base_floats(G, H);
    v.waimg = v.w1img + phx_tc_w1img_floats(G, H);
    v.watimg = v.waimg + phx_tc_waimg_floats(G, H);
    v.w1kimg = v.watimg + phx_tc_w1img_floats(G, H);
    v.tc = 0;
    return v;
}

// flat-gradient offsets, reference parameter order (SURVEY.md appendix A)
struct PhxGradOff {
    size_t m, Wp, bp, Ws, bs, Wa, total;
};
static inline __host__ __device__ PhxGradOff phx_grad_offsets(int G, int H) {
    PhxGradOff o;
    o.m = 0;
    o.Wp = (size_t)G;
    o.bp = o.Wp + (size_t)H * G;
    o.Ws = o.bp + (size_t)H;
    o.bs = o.Ws + (size_t)H * G;
    o.Wa = o.bs + (size_t)H;
    o.total = o.Wa + (size_t)G * 2 * H;
    return o;
}

// Adjoint parameter mask: bit i = the i-th parameter in reference order (m, Wp, bp, Ws, bs, Wa).  The adjoint solvers
// integrate, put in the error norm and return only the cotangents of the parameters in the mask; the others come back
// as zeros.
enum { PHX_P_M = 1, PHX_P_WP = 2, PHX_P_BP = 4, PHX_P_WS = 8, PHX_P_BS = 16, PHX_P_WA = 32, PHX_P_ALL = 63 };
// number of cotangent elements in the mask
static inline __host__ __device__ size_t phx_mask_count(int G, int H, int mask) {
    const size_t HG = (size_t)H * G;
    return ((mask & PHX_P_M) ? (size_t)G : 0) + ((mask & PHX_P_WP) ? HG : 0) + ((mask & PHX_P_BP) ? (size_t)H : 0) +
           ((mask & PHX_P_WS) ? HG : 0) + ((mask & PHX_P_BS) ? (size_t)H : 0) + ((mask & PHX_P_WA) ? 2 * HG : 0);
}
// offsets of the masked-in blocks when only they are stored, back to back in reference order (masked-out blocks get the
// offset of the next kept one and are never addressed); phx_compact_grad_offsets(G, H, PHX_P_ALL) == phx_grad_offsets
static inline __host__ __device__ PhxGradOff phx_compact_grad_offsets(int G, int H, int mask) {
    PhxGradOff o;
    const size_t HG = (size_t)H * G;
    size_t at = 0;
    o.m = at;  at += (mask & PHX_P_M) ? (size_t)G : 0;
    o.Wp = at; at += (mask & PHX_P_WP) ? HG : 0;
    o.bp = at; at += (mask & PHX_P_BP) ? (size_t)H : 0;
    o.Ws = at; at += (mask & PHX_P_WS) ? HG : 0;
    o.bs = at; at += (mask & PHX_P_BS) ? (size_t)H : 0;
    o.Wa = at; at += (mask & PHX_P_WA) ? 2 * HG : 0;
    o.total = at;
    return o;
}

// Parameter cotangents in the PACKED layout = the layout of the packed weights themselves: W1bar[G][K2] (row g =
// [Wsbar[:, g] | Wpbar[:, g]]), WAbar[G][K2], biasbar[K2] ([bs | bp]), mbar[G]; every row 16-byte aligned, the rows of one
// CTA's gene slice contiguous.  phx_unpack_grads converts to the reference's flat order.
struct PhxPackedGradOff {
    size_t W1, WA, bias, m, total;
};
static inline __host__ __device__ PhxPackedGradOff phx_packed_grad_offsets(int G, int H) {
    const size_t K2 = (size_t)phx_K2(H);
    PhxPackedGradOff o;
    o.W1 = 0;
    o.WA = (size_t)G * K2;
    o.bias = 2 * (size_t)G * K2;
    o.m = o.bias + K2;
    o.total = (o.m + (size_t)G + 3) & ~(size_t)3;
    return o;
}

// ---- inter-CTA exchange area ("LL" = low-latency tagged slots), at the START of every resident-solver workspace -----
// Each slot is one naturally aligned 64-bit word {fp32 payload, 32-bit epoch tag} written with a single relaxed
// gpu-scope store and polled with relaxed gpu-scope loads until the tag matches: the payload arrives with its flag, so
// an exchange costs one L2 round trip and needs no fences or atomics.  Tags are a per-workspace monotonically
// increasing epoch (word 0 of the area carries it from launch to launch), so the area has to be zero exactly once,
// when the workspace is allocated (phx_solve_workspace_init).
#define PHX_LL_MAXC 160                      /* CTAs (>= SM count of any sm_100 part)                    */
#define PHX_LL_NMAX 4096                     /* longest all-reduced vector: max rows (8) x max K2 (512)  */
#define PHX_LL_YMAX 16384                    /* one-phase exchange: nCTA * n <= YMAX                     */
#define PHX_LL_DMAX 64                       /* scalar (norm) exchange: floats per CTA (hi/lo pairs of <= 32 sums) */
#define PHX_LL_RCOPIES 8                     /* replicas of every reduced result: CTA c polls copy c % R, so the
                                                readers of one exchange spread over R x as many L2 slices */
struct PhxLL {
    unsigned long long* epoch;   // [1] (+7 pad)
    unsigned long long* xpart;   // [MAXC][NMAX]   two-phase all-reduce: per-CTA partials
    unsigned long long* xres;    // [R][NMAX]      two-phase all-reduce: reduced vector, R replicas
    unsigned long long* ypart;   // [2][YMAX]      one-phase all-reduce (small grids), double-buffered
    unsigned long long* dpart;   // [MAXC][DMAX]   scalar sums (error norms): per-CTA partials
    unsigned long long* dres;    // [R][DMAX]      scalar sums: totals, R replicas
};
static inline __host__ __device__ size_t phx_ll_words() {
    return 8 + (size_t)PHX_LL_MAXC * PHX_LL_NMAX + (size_t)PHX_LL_RCOPIES * PHX_LL_NMAX + 2 * (size_t)PHX_LL_YMAX +
           (size_t)PHX_LL_MAXC * PHX_LL_DMAX + (size_t)PHX_LL_RCOPIES * PHX_LL_DMAX;
}
static inline __host__ __device__ PhxLL phx_ll_view(void* base) {
    PhxLL v;
    unsigned long long* p = reinterpret_cast<unsigned long long*>(base);
    v.epoch = p; p += 8;
    v.xpart = p; p += (size_t)PHX_LL_MAXC * PHX_LL_NMAX;
    v.xres = p; p += (size_t)PHX_LL_RCOPIES * PHX_LL_NMAX;
    v.ypart = p; p += 2 * (size_t)PHX_LL_YMAX;
    v.dpart = p; p += (size_t)PHX_LL_MAXC * PHX_LL_DMAX;
    v.dres = p;
    return v;
}

// Byte offsets of the resident kernels' shared-memory views (PHX_NONE: not present), computed by phx_smem_layout.
#define PHX_NONE 0xffffffffu
#define PHX_RED_WARPS 8   /* slots of the cross-warp column-sum buffer (16 warps fold into 8, then 8 -> 1) */
struct SmemOff {
    unsigned w1r, war;   // this CTA's gpc rows of W1 / WA when they stay resident in shared memory for the whole solve
    unsigned watm;       // != PHX_NONE: the WA slice is parked in TENSOR MEMORY (value = smem word that receives the
                         // tcgen05.alloc base address); each warp keeps its own rows in its own TMEM lanes / columns
    unsigned ring, bar, resbar, ctrl, dred, gram, dst16, ystage, bias, relum, maskm, sp, xv, red, st;
    unsigned acts, actl, ysb, jb, acts2, actl2, ysb2, asb, gjb, ub, vb, mt;
    unsigned FG, FSP, FS, FL, FGJ, FM, ppa;
    // rows kernels (phx_rows.cuh): J partials per quad-warp, stage inputs kept for the theta passes, next-stage
    // activation staging, per-row controller block, per-row block sums
    unsigned jred, ysf, actS, actL, rctl, rsum;
};
#define PHX_CTRL_BYTES 1024  /* >= sizeof(Ctrl) in phx_resident.cuh (static_assert there) */
#define PHX_ROWS_MAX 4        /* independent problems in lock-step per pass of the rows kernels */
#define PHX_RCTL_BYTES 2048   /* >= sizeof(RowsCtl) in phx_rows.cuh (static_assert there) */

static inline int phx_QB(int B) { return (7 * (B > 1 ? 4 : 1) + 3) & ~3; }
static inline bool phx_use_y(int nCTA, int B, int K2, int adjoint) {
    return (size_t)nCTA * B * K2 * (adjoint ? 2 : 1) <= 4096;
}

// wa_res: 0 = WA streams through the ring, 1 = resident in shared memory, 2 = resident in tensor memory
static inline size_t phx_smem_layout(int nCTA, int B, int K2, int gpc, int adjoint, int w1_res, int wa_res,
                                     int ring_rows, int ring_stages, SmemOff* o) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t at = off;
        off += (bytes + 15) & ~size_t(15);
        return (unsigned)at;
    };
    SmemOff t;
    const unsigned none = PHX_NONE;
    const int QB = phx_QB(B);
    const size_t bl = sizeof(float) * B * gpc;
    const size_t slice = sizeof(float) * (size_t)gpc * K2;
    // bulk-copy targets first (128-byte aligned: every size below is a multiple of 32 bytes)
    t.w1r = w1_res ? take(slice) : none;
    t.war = wa_res == 1 ? take(slice) : none;
    t.watm = wa_res == 2 ? take(16) : none;
    // per-warp ring: PHX_WARPS x ring_stages row-sized slots, one mbarrier each
    t.ring = ring_stages ? take(sizeof(float) * (size_t)ring_stages * PHX_WARPS * K2) : none;
    t.bar = take(sizeof(unsigned long long) * (ring_stages ? ring_stages * PHX_WARPS : 1));
    t.resbar = take(sizeof(unsigned long long));
    t.ctrl = take(PHX_CTRL_BYTES);
    t.dred = take(sizeof(double) * PHX_WARPS * 8);
    t.gram = adjoint ? take(sizeof(double) * 128) : none;
    t.dst16 = take(sizeof(float) * PHX_LL_DMAX);
    t.ystage = phx_use_y(nCTA, B, K2, adjoint) ? take(sizeof(float) * (size_t)nCTA * B * K2 * (adjoint ? 2 : 1)) : none;
    t.bias = take(sizeof(float) * K2);
    t.relum = take(sizeof(float) * gpc);
    t.maskm = take(sizeof(float) * gpc);
    t.sp = take(sizeof(float) * B * K2);
    t.xv = adjoint ? take(sizeof(float) * 2 * B * K2) : none;   // [gS|gLP partial][next stage's S|P partial]
    // cross-warp column-sum buffer: aliases the ring when there is one (no bulk copy is ever in flight during a
    // reduction: see the prefetch rules in phx_resident.cuh)
    t.red = ring_stages ? t.ring : take(sizeof(float) * PHX_RED_WARPS * K2);
    t.st = take((adjoint ? 18 : 9) * bl);
    t.acts = take(bl); t.actl = take(bl); t.ysb = take(bl); t.jb = take(bl);
    t.acts2 = t.actl2 = t.ysb2 = t.asb = t.gjb = t.ub = t.vb = t.mt = none;
    t.FG = t.FSP = t.FS = t.FL = t.FGJ = t.FM = t.ppa = none;
    if (adjoint) {
        t.acts2 = take(bl); t.actl2 = take(bl); t.ysb2 = take(bl); t.asb = take(bl); t.gjb = take(bl);
        t.ub = take(bl); t.vb = take(bl); t.mt = take(bl);
        t.FG = take(sizeof(float) * K2 * QB);
        t.FSP = take(sizeof(float) * K2 * QB);
        t.FS = take(sizeof(float) * gpc * QB);
        t.FL = take(sizeof(float) * gpc * QB);
        t.FGJ = take(sizeof(float) * gpc * QB);
        t.FM = take(sizeof(float) * gpc * 8);
        t.ppa = take(256);   // PPArgs of the theta passes (phx_resident.cuh)
    }
    if (o) *o = t;
    return off;
}

// Parameters of the persistent ("resident") solver kernels.
struct ResParams {
    int G, H, Hp, K2, K2q, B, T, method, gpc, t_is_f32, adjoint;
    int ring_rows, ring_stages;   // weight-streaming ring: rows per chunk, chunks in flight
    SmemOff so;
    float rtol_f, atol_f;
    float fsign;           // +1, or -1 when the caller's t was decreasing (f -> -f(-t, y), misc.py:159-162)
    long long max_steps;
    // dopri5 step control (phx_solve_desc): first_step > 0 replaces Hairer's initial-step estimate (of every output
    // interval in the adjoint); the controller constants of next_dt, defaults filled in by the host
    double first_step, safety, ifactor, dfactor;
    PhxPacked w;
    const double* t;       // [T] device copy of the output times (only used when T > PHX_T_INLINE)
    double t_small[64];    // the output times themselves when nprob * T <= PHX_T_INLINE (no host->device copy per call)
    // forward
    const float* y0;       // [B][G]
    float* yout;           // [T][B][G]
    // adjoint
    const float* ysaved;   // [T][B][G]
    const float* grad_y;   // [T][B][G]
    float* adj_y0;         // [B][G]
    float* theta0;         // [P] caller's flat grads (result lands here)
    float* theta1;         // [P] scratch twin
    // several independent problems per launch (phx_solve with N > 1): problem i reads / writes base + i * stride (floats),
    // its output times are t_small[i*T .. i*T+T) and its status record is status[i]; nprob == 1 for the plain calls
    int nprob;
    long long y0_stride, yout_stride, adj_stride, theta_stride;
    // workspace
    PhxLL ll;
    phx_status* status;
    double* steplog;
    int steplog_cap;
    long long* prof;       // optional [PHX_PROF_SLOTS] phase-timer accumulators (phx_ctx_set_profile), else nullptr
    // rows kernels (phx_rows.cuh): `ntot` independent one-row problems, `rows` of them in lock-step per pass, each with its
    // own step controller; thread mapping constants; parameter cotangents in the PACKED layout (phx_packed_grad_*)
    int rows, ntot, nqw, ngg, gpg, tm_wa, tm_fac;
    float* theta_ws;       // [rows][2][ppk] per-row packed cotangent double buffers (workspace)
    float* gsum;           // [ppk] packed cotangents summed over all problems of the launch
    int gsum_acc;          // != 0: add to gsum instead of overwriting it
    long long ppk;
    int pmask;             // adjoint: parameters whose cotangents are integrated (PHX_P_*)
    // fixed-grid solves on the caller's step grid (phx_solve_desc.grid_*, options=dict(step_size=...)); gdt == nullptr:
    // one step per output interval.  Segment q (forward: problem q; adjoint: interval iv of problem pi, q = pi*(T-1)+iv-1)
    // takes the steps gdt[goff[q] .. goff[q+1]).  Forward output j >= 1 of problem pi is written in step
    // gout[pi*(T-1)+j-1] of its problem, as y + gsl[...] * (y1 - y), or as y1 itself when gsl[...] < 0
    const float* gdt;
    const int* goff;
    const int* gout;
    const float* gsl;
    // adjoint: the time cotangent v of every output interval (phx_solve_desc.t_vjp, [N][T-1], interval [t[i-1], t[i]] of
    // problem pi at pi*(T-1) + i-1), or nullptr for v = 0.  dopri5 folds it into d0 of the interval's initial step
    const float* t_vjp;
};
#define PHX_PROF_SLOTS 32
#define PHX_T_INLINE 64

struct ResLaunchPlan {
    int nCTA, gpc, NV, ring_rows, ring_stages, w1_res, wa_res;
    size_t smem_bytes;
    SmemOff so;
};


// ---- rows kernels (phx_rows.cuh): shared-memory layout and launch plan --------------------------------------------------
#define PHX_ROWS_NFS 6   /* factor slots per row: dopri5 stages {0,2,3,4,5,6} (stage 1 has zero weight in the solution,
                            error and mid-point combinations, dopri5.py:15-30); rk4: its 4 stages */
struct RowsPlan {
    int nCTA, gpc, nqw, ngg, gpg, wa_res, rows, w1_stride_q, tm_wa, tm_fac;
    size_t smem_bytes;
    SmemOff so;
};
// wa_res: 1 = WA slice in shared memory, 2 = in tensor memory.  Per-(gene,row) arrays are [gpc][PHX_ROWS_MAX].
static inline size_t phx_rows_smem_layout(int nCTA, int K2, int gpc, int adjoint, int wa_res, int nqw, int w1_stride_q,
                                          SmemOff* o) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t at = off;
        off += (bytes + 15) & ~size_t(15);
        return (unsigned)at;
    };
    SmemOff t;
    const unsigned none = PHX_NONE;
    const int RMx = PHX_ROWS_MAX, ngg = PHX_WARPS / nqw;
    const size_t bl = sizeof(float) * RMx * gpc;
    t.w1r = take(sizeof(float) * 4 * (size_t)gpc * w1_stride_q);
    t.war = wa_res == 1 ? take(sizeof(float) * (size_t)gpc * K2) : none;
    t.watm = take(16);                       // tcgen05.alloc result (tensor memory is always allocated: factor tables)
    t.ring = none;
    t.bar = take(sizeof(unsigned long long));
    t.resbar = take(sizeof(unsigned long long));
    t.ctrl = take(PHX_CTRL_BYTES);           // phase-timer staging lives in its tail, as in the resident kernels
    t.rctl = take(PHX_RCTL_BYTES);
    t.dred = take(sizeof(double) * PHX_WARPS * 8);
    t.rsum = take(sizeof(double) * (PHX_WARPS + 1) * RMx * 8);
    t.gram = adjoint ? take(sizeof(double) * 4 * RMx * 12) : none;
    t.dst16 = take(sizeof(float) * PHX_LL_DMAX);
    const int nvec = RMx * K2 * (adjoint ? 2 : 1);
    t.ystage = ((size_t)nCTA * nvec <= 4096) ? take(sizeof(float) * (size_t)nCTA * nvec) : none;
    t.bias = take(sizeof(float) * K2);
    t.relum = take(sizeof(float) * gpc);
    t.maskm = take(sizeof(float) * gpc);
    t.sp = take(sizeof(float) * RMx * K2);
    t.xv = adjoint ? take(sizeof(float) * 2 * RMx * K2) : none;
    // cross-group fold buffer [ngg/2][RM][K2] followed by the J partials [nqw][gpc][RM]: together they are the scratch
    // of the theta passes (per-gene activation tables rebuilt from the stored stage inputs).  The adjoint's state-cotangent
    // pass keeps its v partials [nqw][gpc][RM] in the fold buffer (the u partials sit in the J partials): it must hold
    // them too, or a CTA with more than (ngg/2) K2 / nqw genes overwrites its own u partials.
    const size_t fold = (size_t)(ngg / 2) * K2, vpart = adjoint ? (size_t)nqw * gpc : 0;
    t.red = take(sizeof(float) * RMx * (fold > vpart ? fold : vpart));
    t.jred = take(sizeof(float) * nqw * RMx * gpc);
    if (adjoint) {
        const size_t have = off - t.red, need = 2 * sizeof(float) * PHX_ROWS_NFS * RMx * gpc;
        if (have < need) take(need - have);
    }
    t.st = take((adjoint ? 18 : 9) * bl);
    t.ysb = take(bl); t.acts = take(bl); t.actL = take(bl);
    t.actl = t.jb = none;
    t.acts2 = t.actl2 = t.ysb2 = t.asb = t.gjb = t.ub = t.vb = t.mt = none;
    t.FG = t.FSP = t.FS = t.FL = t.FGJ = t.FM = t.ppa = t.ysf = t.actS = none;
    if (adjoint) {
        t.ysb2 = take(bl); t.acts2 = take(bl); t.asb = take(bl); t.gjb = take(bl);
        t.ysf = take(PHX_ROWS_NFS * bl);
        t.FGJ = take(PHX_ROWS_NFS * bl);
        t.FM = take(PHX_ROWS_NFS * bl);
        t.ppa = take(1024);
    }
    if (o) *o = t;
    return off;
}
int phx_rows_plan(int num_sms, int G, int H, int adjoint, RowsPlan* plan);
size_t phx_rows_workspace_floats(int G, int H, int N, int T, int rows, int adjoint, size_t* off_t, size_t* off_theta);
int phx_rows_launch(const ResParams& p, const RowsPlan& plan, cudaStream_t stream);

// host helpers implemented in phx_resident.cu
int phx_resident_plan(int num_sms, int G, int H, int B, int adjoint, ResLaunchPlan* plan);
size_t phx_resident_workspace_floats(int G, int H, int B, int T, int adjoint, size_t* off_t, size_t* off_theta1);
int phx_resident_launch(const ResParams& p, const ResLaunchPlan& plan, cudaStream_t stream);

// A fixed-grid solve's step grid as phx_solve takes it (include/phoenix_b200.h): nseg segments (forward: the
// N problems; adjoint: the N * (T-1) intervals, problem-major), steps[q] >= 1 steps each, their dt back to back; forward
// only: out_step / out_slope [N][T-1], the step of each output time j >= 1 and its slope (< 0: exact hit, take y1).
struct PhxGridHost {
    const float* dt;
    const int32_t* steps;
    const int32_t* out_step;
    const float* out_slope;
};
// Validates the grid (phx_set_error + PHX_ERR_INVALID otherwise); with `room` (device, >= phx_grid_workspace_bytes) set,
// copies it there on `stream` and points p->gdt / goff / gout / gsl at it.  `off` (may be null) receives the segment
// offsets into dt (nseg + 1 entries).
int phx_grid_stage(const PhxGridHost& g, int N, int T, int method, int forward, void* room, cudaStream_t stream,
                   ResParams* p, std::vector<int>* off);
// the streaming engine's solves (phx_stream.cu), called by phx_solve once it has checked the request's combination of
// fields, its param_mask and its y0 / y_out or adjoint pointers
int phx_stream_forward(phx_ctx* ctx, const phx_solve_desc& d, cudaStream_t stream);
int phx_stream_adjoint(phx_ctx* ctx, const phx_solve_desc& d, cudaStream_t stream);

// ---- RK stage algebra fused into the RHS (streaming solvers, forward solves on the tensor-core path) ------------------
// With k = the stage derivative a forward RHS launch produces, the epilogue of the joint contraction also writes
//   PHX_POST_CHAIN : out = x0 + (c[0] k[0] + ... + c[nk-1] k[nk-1] + cr k)   one fmaf chain in this order (the adaptive
//                    solver's next stage input / y1, rk_common.py:66)
//   PHX_POST_FX_*  : one of the fixed-grid formulas exactly as fixed_grid.py / rk_common.py:96-103 write them, with k in
//                    the place of the newest derivative and k[0..] the older ones
// next to (store_f) or instead of k itself.  out may be the buffer the launch reads its state from: every element is read
// and written by the same thread.  phx_fixed_formula is THE definition both the fused epilogue and the stand-alone
// elementwise kernels of phx_stream.cu evaluate (no FMA contraction: the library is built with -fmad=false).
enum { PHX_POST_NONE = 0, PHX_POST_CHAIN = 1, PHX_POST_FX = 2 };   // mode = PHX_POST_FX + one of the PHX_FX_* below
enum { PHX_FX_EULER_END = 0, PHX_FX_MID_IN = 1, PHX_FX_RK4_IN2 = 2, PHX_FX_RK4_IN3 = 3, PHX_FX_RK4_IN4 = 4,
       PHX_FX_RK4_END = 5 };
struct PhxRhsPost {
    int mode;      // PHX_POST_*
    int nk;        // older derivatives read from k[0..nk-1]
    int store_f;   // 0: the launch's own f is not written (the last stage of a fixed-grid step)
    float dt;      // PHX_POST_FX_*: the step (half the step for PHX_FX_MID_IN)
    const float* x0;
    const float* k[6];
    float c[6];    // PHX_POST_CHAIN: coefficients of k[0..nk-1]
    float cr;      // PHX_POST_CHAIN: coefficient of the launch's own derivative
    float* out;
};
static __host__ __device__ __forceinline__ float phx_fixed_formula(int mode, float x, float a1, float a2, float a3, float a4,
                                                            float dt) {
    const float third = (float)(1.0 / 3.0);
    switch (mode) {
        case PHX_FX_EULER_END: return x + dt * a1;
        case PHX_FX_MID_IN: return x + a1 * dt;  // dt carries half_dt here
        case PHX_FX_RK4_IN2: return x + dt * a1 * third;
        case PHX_FX_RK4_IN3: return x + dt * (a2 - a1 * third);
        case PHX_FX_RK4_IN4: return x + dt * (a1 - a2 + a3);
        default: return x + (a1 + 3.f * (a2 + a3) + a4) * dt * 0.125f;
    }
}

// host helpers implemented in phx_rhs.cu.  `post` (optional) needs phx_rhs_post_supported(w, H, B).
int phx_rhs_forward_launch(int G, int H, int B, const PhxPacked& w, const float* y, float* f, int decay, float fscale,
                           float* ws, cudaStream_t stream, const PhxRhsPost* post = nullptr);
bool phx_rhs_post_supported(const PhxPacked& w, int H, int B);
int phx_rhs_vjp_launch(int G, int H, int B, const PhxPacked& w, const float* y, const float* g, int decay,
                       float* ybar, float* grads_flat, int accumulate, float* f_out, float fscale, float* ws,
                       cudaStream_t stream, int pmask = PHX_P_ALL, const PhxGradOff* goff = nullptr);
size_t phx_rhs_workspace_floats(int G, int H, int B);
int phx_prior_loss_launch(int G, int H, int B, const PhxPacked& w, const float* x, const float* prior_grad, float scale,
                          float* gcot, float* loss, float* ws, cudaStream_t stream);
int phx_prior_setup_launch(int G, int B, const float* x, const int* colptr, const int* rowidx, const float* val,
                           float* out, cudaStream_t stream);

// tensor-core path (phx_tc.cu).  phx_tc_prepare (phx_api.cu) decides per call whether the contractions of a B-row call
// run on tcgen05 (ctx precision, shape), (re)builds the operand images in the tail of `packed` if phx_pack_weights has
// run since they were last built, and returns the view with .tc set.
struct phx_ctx;
int phx_tc_prepare(phx_ctx* ctx, int G, int H, int B, const float* packed, PhxPacked* view, cudaStream_t stream);
int phx_tc_pack_launch(int G, int H, const PhxPacked& w, cudaStream_t stream);
int phx_tc_rhs_forward_launch(int G, int H, int B, const PhxPacked& w, const float* y, float* f, int decay,
                              float fscale, float* SP, float* tcws, cudaStream_t stream, const PhxRhsPost* post = nullptr);
// after phx_tc_rhs_forward_launch on the same scratch: GS = (g relu(m)) WA (prods half scaled by Pr) and, if ybar != 0,
// ybar = (GS_s Ws + (GS_p Wp)/(1+s)) / (1+|y-.5|)^2 - g relu(m); if J != 0 also the un-decayed joint J = [S|P] WA^T
int phx_tc_vjp_state_launch(int G, int H, int B, const PhxPacked& w, const float* y, const float* g, int decay,
                            float* ybar, const float* SP, float* GS, float* J, float* tcws, cudaStream_t stream);
int phx_tc_joint_launch(int G, int H, int B, const PhxPacked& w, const float* y, float* f, int decay, float fscale,
                        float* tcws, cudaStream_t stream);
int phx_tc_prior_loss_launch(int G, int H, int B, const PhxPacked& w, const float* x, const float* prior_grad, float scale,
                             float* gcot, float* loss, float* SP, double* part, float* tcws, cudaStream_t stream);
int phx_tc_vjp_params_launch(int G, int H, int B, const PhxPacked& w, const float* y, const float* g, int decay,
                             float* grads_flat, int accumulate, float* tcws, cudaStream_t stream,
                             int pmask = PHX_P_ALL, const PhxGradOff* goff = nullptr);

void phx_set_error(const char* fmt, ...);
int phx_ctx_device(const phx_ctx* ctx);
int phx_ctx_sum_hook(const phx_ctx* ctx, phx_sum_hook* hook, void** user);   // returns the world size (1: no hook)
// Every entry point that enqueues work makes the context's device current for the duration of the call (the caller may be
// sitting on another GPU) and restores the previous one.
struct PhxDevGuard {
    int prev = -1;
    bool sw = false;
    explicit PhxDevGuard(const phx_ctx* ctx) {
        if (!ctx) return;
        const int d = phx_ctx_device(ctx);
        if (cudaGetDevice(&prev) == cudaSuccess && prev != d) sw = cudaSetDevice(d) == cudaSuccess;
    }
    ~PhxDevGuard() {
        if (sw) cudaSetDevice(prev);
    }
    PhxDevGuard(const PhxDevGuard&) = delete;
    PhxDevGuard& operator=(const PhxDevGuard&) = delete;
};
