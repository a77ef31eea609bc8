// Streaming engine: the same solvers as the resident kernels for ANY number of rows B (gene-influence scan B=60,
// synthetic sweep B=4096, batched adjoint), driven from the host.  The state is too large to live on chip, so each RK
// stage is: one fused elementwise combine over the state -> the batched RHS / RHS-VJP contractions of phx_rhs.cu.
// Fixed-grid methods stay fully asynchronous; dopri5 reads ONE small record (the error sums) back per step attempt
// for the controller, negligible next to the B*G*H contractions of a step at these sizes.
// Forward solves on the tensor-core path can go one step further (`fuse`, PHX_STREAM_FUSE=1): the stage algebra that
// FOLLOWS a stage derivative -- the next stage input, y1, the end value of a fixed-grid step -- evaluated in the epilogue
// of the joint contraction that produces the derivative (PhxRhsPost, phx_common.cuh): a fixed-grid step is then RHS
// launches only (its last derivative is never written), a dopri5 attempt keeps one stand-alone combine (the first stage
// input, which needs the step size the controller has just chosen) and the error pass.  Same formulas, same operation
// order: bit-identical to the stand-alone kernels -- and measured SLOWER than them at every shape, so it is off by
// default (numbers and the reason in phx_stream_solve_forward).
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <stdint.h>
#include <vector>
#include "phx_common.cuh"

namespace {

constexpr int EB = 256;        // elementwise block
constexpr int MAXBLK = 1184;   // 8 x 148

const double H_BETA[6][6] = {
    {1.0 / 5, 0, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656, 0},
    {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84}};
const double H_CERR[7] = {35.0 / 384 - 1951.0 / 21600, 0, 500.0 / 1113 - 22642.0 / 50085, 125.0 / 192 - 451.0 / 720,
                          -2187.0 / 6784 - -12231.0 / 42400, 11.0 / 84 - 649.0 / 6300, -1.0 / 60.0};
const double H_CMID[7] = {6025192743.0 / 30085553152.0 / 2, 0, 51252292925.0 / 65400821598.0 / 2,
                          -2691868925.0 / 45128329728.0 / 2, 187940372067.0 / 1594534317056.0 / 2,
                          -1776094331.0 / 19743644256.0 / 2, 11237099.0 / 235043384.0 / 2};

struct KSet {
    int nk;
    const float* k[7];
    float c[7];
};

__device__ __forceinline__ float ksum(const KSet& a, size_t i) {
    float v = a.k[0][i] * a.c[0];
    for (int j = 1; j < a.nk; ++j) v = fmaf(a.k[j][i], a.c[j], v);
    return v;
}
// the same for four consecutive elements (i a multiple of 4, 16-byte aligned arrays): one 128-bit load per array
__device__ __forceinline__ float4 ksum4(const KSet& a, size_t i) {
    float4 k = *reinterpret_cast<const float4*>(a.k[0] + i);
    float4 v = make_float4(k.x * a.c[0], k.y * a.c[0], k.z * a.c[0], k.w * a.c[0]);
    for (int j = 1; j < a.nk; ++j) {
        k = *reinterpret_cast<const float4*>(a.k[j] + i);
        v.x = fmaf(k.x, a.c[j], v.x);
        v.y = fmaf(k.y, a.c[j], v.y);
        v.z = fmaf(k.z, a.c[j], v.z);
        v.w = fmaf(k.w, a.c[j], v.w);
    }
    return v;
}
__device__ __forceinline__ float4 ld4(const float* p, size_t i) { return *reinterpret_cast<const float4*>(p + i); }

// out = x0 + sum_j c_j k_j           (rk_common.py:66).  V = 4: n is a multiple of 4 and every array is 16-byte aligned
template <int V>
__global__ void combine_kernel(float* out, const float* x0, KSet a, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x * V;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * V; i < n; i += stride) {
        if (V == 4) {
            const float4 x = ld4(x0, i), k = ksum4(a, i);
            *reinterpret_cast<float4*>(out + i) = make_float4(x.x + k.x, x.y + k.y, x.z + k.z, x.w + k.w);
        } else {
            out[i] = x0[i] + ksum(a, i);
        }
    }
}

// fixed-grid formulas, exactly as written in fixed_grid.py / rk_common.py:96-103 (phx_fixed_formula, phx_common.cuh: the
// fused epilogue evaluates the very same function)
enum { FX_EULER_END = PHX_FX_EULER_END, FX_MID_IN = PHX_FX_MID_IN, FX_RK4_IN2 = PHX_FX_RK4_IN2, FX_RK4_IN3 = PHX_FX_RK4_IN3,
       FX_RK4_IN4 = PHX_FX_RK4_IN4, FX_RK4_END = PHX_FX_RK4_END };
__device__ __forceinline__ float fixed_one(int mode, float x, float a1, float a2, float a3, float a4, float dt) {
    return phx_fixed_formula(mode, x, a1, a2, a3, a4, dt);
}
template <int V>
__global__ void fixed_kernel(int mode, float* out, const float* x0, const float* k1, const float* k2, const float* k3,
                             const float* k4, float dt, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x * V;
    const bool u2 = mode >= FX_RK4_IN3, u3 = mode >= FX_RK4_IN4, u4 = mode == FX_RK4_END;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * V; i < n; i += stride) {
        if (V == 4) {
            const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 x = ld4(x0, i), a1 = ld4(k1, i), a2 = u2 ? ld4(k2, i) : z, a3 = u3 ? ld4(k3, i) : z,
                         a4 = u4 ? ld4(k4, i) : z;
            *reinterpret_cast<float4*>(out + i) =
                make_float4(fixed_one(mode, x.x, a1.x, a2.x, a3.x, a4.x, dt), fixed_one(mode, x.y, a1.y, a2.y, a3.y, a4.y, dt),
                            fixed_one(mode, x.z, a1.z, a2.z, a3.z, a4.z, dt), fixed_one(mode, x.w, a1.w, a2.w, a3.w, a4.w, dt));
        } else {
            out[i] = fixed_one(mode, x0[i], k1[i], u2 ? k2[i] : 0.f, u3 ? k3[i] : 0.f, u4 ? k4[i] : 0.f, dt);
        }
    }
}

template <int NV>
__device__ void block_partials(double (&v)[NV], double* partial) {
    __shared__ double sh[EB / 32][NV];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        double s = v[q];
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) sh[warp][q] = s;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double s = 0;
        for (int w = 0; w < EB / 32; ++w) s += sh[w][threadIdx.x];
        partial[(size_t)blockIdx.x * NV + threadIdx.x] = s;
    }
}

// sums for Hairer's initial step (misc.py:63-66): [0]=sum (x0/scale)^2, [1]=sum (k0/scale)^2, [2]=#non-finite
__global__ void init01_kernel(const float* x0, const float* k0, float rtol, float atol, size_t n, double* partial) {
    double v[3] = {0, 0, 0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float x = x0[i];
        float scale = atol + fabsf(x) * rtol;
        float r0 = x / scale, r1 = k0[i] / scale;
        v[0] += (double)(r0 * r0);
        v[1] += (double)(r1 * r1);
        if (!isfinite(x)) v[2] += 1.0;
    }
    block_partials<3>(v, partial);
}
// [0] = sum ((k1-k0)/scale)^2   (misc.py:76)
__global__ void initd2_kernel(const float* x0, const float* k0, const float* k1, float rtol, float atol, size_t n,
                              double* partial) {
    double v[3] = {0, 0, 0};
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float scale = atol + fabsf(x0[i]) * rtol;
        float r = (k1[i] - k0[i]) / scale;
        v[0] += (double)(r * r);
    }
    block_partials<3>(v, partial);
}
// [0] = sum (err/tol)^2, [1] = #non-finite in x1   (misc.py:89-91)
template <int V>
__global__ void err_kernel(const float* x0, const float* x1, KSet a, float rtol, float atol, size_t n,
                           double* partial) {
    double v[3] = {0, 0, 0};
    const size_t stride = (size_t)gridDim.x * blockDim.x * V;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * V; i < n; i += stride) {
        float e[4], xa[4], xb[4];
        if (V == 4) {
            const float4 e4 = ksum4(a, i), a4 = ld4(x0, i), b4 = ld4(x1, i);
            e[0] = e4.x; e[1] = e4.y; e[2] = e4.z; e[3] = e4.w;
            xa[0] = a4.x; xa[1] = a4.y; xa[2] = a4.z; xa[3] = a4.w;
            xb[0] = b4.x; xb[1] = b4.y; xb[2] = b4.z; xb[3] = b4.w;
        } else {
            e[0] = ksum(a, i); xa[0] = x0[i]; xb[0] = x1[i];
        }
        float s = 0.f;   // squares of (at most) four neighbours in fp32, then into the double running sum
        bool bad = false;
#pragma unroll
        for (int q = 0; q < V; ++q) {
            const float tol = atol + rtol * fmaxf(fabsf(xa[q]), fabsf(xb[q]));
            const float r = e[q] / tol;
            s += r * r;
            bad = bad || !isfinite(xb[q]);
            if (V == 4 && !isfinite(xb[q])) v[1] += 1.0;
        }
        v[0] += (double)s;
        if (V == 1 && bad) v[1] += 1.0;
    }
    block_partials<3>(v, partial);
}
// out[seg*3 + q] = sum over blocks, fixed order: lane l adds blocks l, l+32, ... then a fixed butterfly (one warp)
__global__ void final_reduce_kernel(const double* partial, int nblocks, double* out) {
    const int lane = threadIdx.x;
    double s[3] = {0, 0, 0};
    for (int b = lane; b < nblocks; b += 32)
        for (int q = 0; q < 3; ++q) s[q] += partial[(size_t)b * 3 + q];
    for (int q = 0; q < 3; ++q) {
        for (int o = 16; o > 0; o >>= 1) s[q] += __shfl_xor_sync(0xffffffffu, s[q], o);
        if (lane == 0) out[q] = s[q];
    }
}
// quartic dense output at x (interp.py:1-47)
__device__ __forceinline__ float interp_one(float y0, float y1, float f0, float f1, float ks, float dt, float xs0,
                                            float xs1, float xs2, float xs3) {
    float ymid = y0 + ks;
    float a = 2.f * dt * (f1 - f0) - 8.f * (y1 + y0) + 16.f * ymid;
    float b = dt * (5.f * f0 - 3.f * f1) + 18.f * y0 + 14.f * y1 - 32.f * ymid;
    float c = dt * (f1 - 4.f * f0) - 11.f * y0 - 5.f * y1 + 16.f * ymid;
    float d = dt * f0;
    float total = y0 + xs0 * d;
    total = total + xs1 * c;
    total = total + xs2 * b;
    total = total + xs3 * a;
    return total;
}
template <int V>
__global__ void interp_kernel(float* out, const float* x0, const float* x1, KSet mid, const float* kf, const float* kl,
                              float dt, float xs0, float xs1, float xs2, float xs3, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x * V;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * V; i < n; i += stride) {
        if (V == 4) {
            const float4 a = ld4(x0, i), b = ld4(x1, i), f0 = ld4(kf, i), f1 = ld4(kl, i), m = ksum4(mid, i);
            *reinterpret_cast<float4*>(out + i) =
                make_float4(interp_one(a.x, b.x, f0.x, f1.x, m.x, dt, xs0, xs1, xs2, xs3),
                            interp_one(a.y, b.y, f0.y, f1.y, m.y, dt, xs0, xs1, xs2, xs3),
                            interp_one(a.z, b.z, f0.z, f1.z, m.z, dt, xs0, xs1, xs2, xs3),
                            interp_one(a.w, b.w, f0.w, f1.w, m.w, dt, xs0, xs1, xs2, xs3));
        } else {
            out[i] = interp_one(x0[i], x1[i], kf[i], kl[i], ksum(mid, i), dt, xs0, xs1, xs2, xs3);
        }
    }
}
__global__ void add_kernel(float* x, const float* y, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        x[i] = x[i] + y[i];
}
// an output time inside a fixed-grid step (solvers.py:97-103): y0 + slope * (y1 - y0), op by op
__global__ void lerp_kernel(float* out, const float* y0, const float* y1, float slope, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = y0[i] + slope * (y1[i] - y0[i]);
}

inline bool al16(const void* p) { return p == nullptr || ((uintptr_t)p & 15) == 0; }
inline bool kset_al16(const KSet& a) {
    for (int j = 0; j < a.nk; ++j)
        if (!al16(a.k[j])) return false;
    return true;
}

int nblk(size_t n) {
    size_t b = (n + EB - 1) / EB;
    return (int)(b < (size_t)MAXBLK ? (b ? b : 1) : MAXBLK);
}

struct Seg {
    size_t n;
    float* x0;
    float* x1;
    float* xs;   // stage input (null for the parameter segment: the dynamics do not depend on it)
    float* k[7];
    double count;
    bool in_norm = true;   // false: the seminorm's parameter segment -- no norm sums, no error kernel
};

// misc.py:94-103 with order 5 (next_dt of the resident kernels)
double next_dt_host(double dt, float ratio, double safety, double ifactor, double dfactor_ge1) {
    if (ratio == 0.f) return dt * ifactor;
    double dfactor = (ratio < 1.f) ? 1.0 : dfactor_ge1;
    double r = (double)ratio;
    if (isnan(r)) return nan("");
    double f = safety / pow(r, 0.2);
    f = fmax(f, dfactor);
    f = fmin(ifactor, f);
    return dt * f;
}

struct Stream {
    phx_ctx* ctx;
    int G, H, B, T, method, t_is_f32, adjoint;
    float rtol_f, atol_f, fsign;
    long long max_steps;
    PhxPacked w;
    cudaStream_t st;
    std::vector<Seg> segs;
    float* rhs_ws;
    double* partial;   // [MAXBLK][3]
    double* sums_dev;  // [nseg][3]
    double* sums_host; // pinned
    phx_status status;
    double* steplog;
    int steplog_cap;
    std::vector<double> log;
    phx_sum_hook sum_hook = nullptr;   // exact-global-norm mode (forward solves only)
    void* sum_user = nullptr;
    int sum_world = 1;
    bool fuse = false;                 // stage algebra in the RHS epilogue (forward solves on the tensor-core path)
    // dopri5 step control (phx_solve_desc): first_step > 0 replaces Hairer's estimate; the controller constants
    double first_step = 0, safety = 0.9, ifactor = 10.0, dfactor = 0.2;
    // adjoint: the time cotangent v of the interval being solved (phx_solve_desc.t_vjp), in pinned host memory that is
    // filled on the stream before the first synchronisation of the solve; nullptr: v = 0
    const float* vjp_t = nullptr;
    int pmask = PHX_P_ALL;            // adjoint: parameters whose cotangents make up the theta segment
    PhxGradOff goff{};                 // adjoint: their offsets in the theta segment (back to back, reference order)

    // stage derivative `slot` of every segment at the current stage inputs (at_x0: at the step's start values themselves,
    // read in place -- no copy into the stage-input buffers)
    enum { AT_XS = 0, AT_X0 = 1, AT_X1 = 2 };
    int eval(int slot, int at = AT_XS, const PhxRhsPost* post = nullptr) {
        auto in = [&](Seg& s) -> const float* { return at == AT_X0 ? s.x0 : (at == AT_X1 ? s.x1 : s.xs); };
        if (!adjoint)
            return phx_rhs_forward_launch(G, H, B, w, in(segs[0]), segs[0].k[slot], 1, fsign, rhs_ws, st, post);
        // reverse time: ky = -f, ka = VJP_y(cotangent a), ktheta = VJP_theta(cotangent a)
        // (no theta segment when no parameter is integrated)
        return phx_rhs_vjp_launch(G, H, B, w, in(segs[0]), in(segs[1]), 1, segs[1].k[slot],
                                  segs.size() > 2 ? segs[2].k[slot] : nullptr, 0, segs[0].k[slot], -1.f, rhs_ws, st,
                                  pmask, &goff);
    }
    // reduce a 3-value kernel result for segment si into sums_dev[si]
    // reduce the per-block partials of the LAST 3-value kernel launched for segment si (`blocks` = its grid size)
    void finish_sums(int si, int blocks = -1) {
        final_reduce_kernel<<<1, 32, 0, st>>>(partial, blocks < 0 ? nblk(segs[si].n) : blocks, sums_dev + 3 * si);
    }
    void combine(float* out, const float* x0, const KSet& a, size_t n) {
        if (n % 4 == 0 && al16(out) && al16(x0) && kset_al16(a)) combine_kernel<4><<<nblk(n / 4), EB, 0, st>>>(out, x0, a, n);
        else combine_kernel<1><<<nblk(n), EB, 0, st>>>(out, x0, a, n);
    }
    void fixed(int mode, float* out, const float* x0, const float* k1, const float* k2, const float* k3, const float* k4,
               float dt, size_t n) {
        if (n % 4 == 0 && al16(out) && al16(x0) && al16(k1) && al16(k2) && al16(k3) && al16(k4))
            fixed_kernel<4><<<nblk(n / 4), EB, 0, st>>>(mode, out, x0, k1, k2, k3, k4, dt, n);
        else
            fixed_kernel<1><<<nblk(n), EB, 0, st>>>(mode, out, x0, k1, k2, k3, k4, dt, n);
    }
    int fetch_sums() {
        if (sum_hook) sum_hook(sums_dev, 3 * (int)segs.size(), (void*)st, sum_user);   // sum over the ranks, in place
        cudaError_t e = cudaMemcpyAsync(sums_host, sums_dev, sizeof(double) * 3 * segs.size(), cudaMemcpyDeviceToHost,
                                        st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            phx_set_error("stream engine sync: %s", cudaGetErrorString(e));
            return PHX_ERR_CUDA;
        }
        return PHX_OK;
    }
    float block_norm(int q) {  // max over segments of sqrt(mean) in fp32 (misc.py:10-24)
        float m = 0.f;
        bool any_nan = false;
        for (size_t si = 0; si < segs.size(); ++si) {
            if (!segs[si].in_norm) continue;
            double s = sums_host[3 * si + q];
            if (isnan(s)) any_nan = true;
            m = fmaxf(m, sqrtf((float)(s / (segs[si].count * (double)sum_world))));
        }
        return any_nan ? nanf("") : m;
    }
    void set_inputs(const KSet* per_seg) {
        for (size_t si = 0; si < segs.size(); ++si) {
            Seg& s = segs[si];
            if (s.xs) combine(s.xs, s.x0, per_seg[si], s.n);
        }
    }
    KSet kset(int si, const int* slots, const float* coef, int nk) {
        KSet a;
        a.nk = nk;
        for (int j = 0; j < nk; ++j) {
            a.k[j] = segs[si].k[slots[j]];
            a.c[j] = coef[j];
        }
        for (int j = nk; j < 7; ++j) {
            a.k[j] = nullptr;
            a.c[j] = 0.f;
        }
        return a;
    }
    // ---- one fixed-grid step of size dtf on all segments.  The new values replace x0 in place -- or, with `dst0`
    // (forward solves: the caller's output slice of this interval), segment 0's go straight there and x0 is re-pointed
    // at them: no copy of the state into the output, and the start values of a solve are read where the caller put them ----
    // fixed-grid stage record: the derivative of this launch is the newest of `nk + 1`, the older ones sit in k[0..nk-1]
    PhxRhsPost fx_post(int fx, int nk, float dt, float* out, bool store) {
        PhxRhsPost po;
        memset(&po, 0, sizeof(po));
        Seg& s = segs[0];
        po.mode = PHX_POST_FX + fx; po.nk = nk; po.store_f = store ? 1 : 0; po.dt = dt; po.x0 = s.x0; po.out = out;
        for (int j = 0; j < nk; ++j) po.k[j] = s.k[j];
        return po;
    }
    int fixed_step_fused(float dtf, float* dst0) {
        int rc;
        Seg& s = segs[0];
        float* end = dst0 ? dst0 : s.x1;   // never x0 itself: other threads still read x0 while this one writes
        PhxRhsPost po;
        if (method == PHX_EULER) {
            po = fx_post(FX_EULER_END, 0, dtf, end, false);
            if ((rc = eval(0, AT_X0, &po)) != PHX_OK) return rc;
            status.n_rhs += 1;
        } else if (method == PHX_MIDPOINT) {
            po = fx_post(FX_MID_IN, 0, 0.5f * dtf, s.xs, false);   // k1 is only ever used here
            if ((rc = eval(0, AT_X0, &po)) != PHX_OK) return rc;
            po = fx_post(FX_EULER_END, 0, dtf, end, false);   // x + dt * k2: k2 is this launch's own derivative
            if ((rc = eval(1, AT_XS, &po)) != PHX_OK) return rc;
            status.n_rhs += 2;
        } else {
            po = fx_post(FX_RK4_IN2, 0, dtf, s.xs, true);
            if ((rc = eval(0, AT_X0, &po)) != PHX_OK) return rc;
            po = fx_post(FX_RK4_IN3, 1, dtf, s.xs, true);
            if ((rc = eval(1, AT_XS, &po)) != PHX_OK) return rc;
            po = fx_post(FX_RK4_IN4, 2, dtf, s.xs, true);
            if ((rc = eval(2, AT_XS, &po)) != PHX_OK) return rc;
            po = fx_post(FX_RK4_END, 3, dtf, end, false);
            if ((rc = eval(3, AT_XS, &po)) != PHX_OK) return rc;
            status.n_rhs += 4;
        }
        if (dst0) s.x0 = dst0;
        else std::swap(s.x0, s.x1);
        return PHX_OK;
    }
    int fixed_step(float dtf, float* dst0 = nullptr) {
        int rc;
        if (fuse) return fixed_step_fused(dtf, dst0);
        if ((rc = eval(0, AT_X0)) != PHX_OK) return rc;
        auto endp = [&](Seg& s) { return (dst0 && &s == &segs[0]) ? dst0 : s.x0; };
        auto fx = [&](int mode, Seg& s, float* out, float dt) {
            fixed(mode, out, s.x0, s.k[0], s.k[1], s.k[2], s.k[3], dt, s.n);
        };
        if (method == PHX_EULER) {
            for (auto& s : segs) fx(FX_EULER_END, s, endp(s), dtf);
            status.n_rhs += 1;
        } else if (method == PHX_MIDPOINT) {
            for (auto& s : segs)
                if (s.xs) fx(FX_MID_IN, s, s.xs, 0.5f * dtf);
            if ((rc = eval(1)) != PHX_OK) return rc;
            for (auto& s : segs)
                fixed(FX_EULER_END, endp(s), s.x0, s.k[1], nullptr, nullptr, nullptr, dtf, s.n);
            status.n_rhs += 2;
        } else {
            for (auto& s : segs)
                if (s.xs) fx(FX_RK4_IN2, s, s.xs, dtf);
            if ((rc = eval(1)) != PHX_OK) return rc;
            for (auto& s : segs)
                if (s.xs) fx(FX_RK4_IN3, s, s.xs, dtf);
            if ((rc = eval(2)) != PHX_OK) return rc;
            for (auto& s : segs)
                if (s.xs) fx(FX_RK4_IN4, s, s.xs, dtf);
            if ((rc = eval(3)) != PHX_OK) return rc;
            for (auto& s : segs) fx(FX_RK4_END, s, endp(s), dtf);
            status.n_rhs += 4;
        }
        if (dst0) segs[0].x0 = dst0;
        return PHX_OK;
    }

    // ---- dopri5 from t_start until every time in outs[] (increasing, > t_start) has been emitted ----
    // emit(j, xs[4], slots, dtf) writes the dense output for outs[j].
    template <typename Emit>
    int dopri5(double t_start, const double* outs, int nout, Emit emit) {
        int rc;
        const size_t ns = segs.size();
        int sl[7] = {0, 1, 2, 3, 4, 5, 6};
        if ((rc = eval(0, AT_X0)) != PHX_OK) return rc;
        for (size_t si = 0; si < ns; ++si) {
            Seg& s = segs[si];
            if (!s.in_norm) continue;
            init01_kernel<<<nblk(s.n), EB, 0, st>>>(s.x0, s.k[0], rtol_f, atol_f, s.n, partial);
            finish_sums((int)si);
        }
        if ((rc = fetch_sums()) != PHX_OK) return rc;
        bool nonfinite = false;
        for (size_t si = 0; si < ns; ++si) nonfinite = nonfinite || (segs[si].in_norm && sums_host[3 * si + 2] > 0.0);
        // v as the one-element block of the mixed norm (read after the fetch: its copy was enqueued before it)
        float d0v = 0.f;
        if (vjp_t) {
            const float v = *vjp_t, r = v / (atol_f + fabsf(v) * rtol_f);
            d0v = sqrtf(r * r);
            nonfinite = nonfinite || !isfinite(v);
        }
        double dt = first_step;
        if (first_step > 0) {
            // the caller's first step: the fetch above was for the non-finite count only
            status.n_rhs += 1;
        } else {
            float d0 = block_norm(0), d1 = block_norm(1);
            if (vjp_t) d0 = fmaxf(d0, d0v);
            float h0 = (d0 < 1e-5f || d1 < 1e-5f) ? 1e-6f : 0.01f * d0 / d1;
            {
                std::vector<KSet> ks(ns);
                int s0[1] = {0};
                float c0[1] = {h0};
                for (size_t si = 0; si < ns; ++si) ks[si] = kset((int)si, s0, c0, 1);
                set_inputs(ks.data());
            }
            if ((rc = eval(1)) != PHX_OK) return rc;
            for (size_t si = 0; si < ns; ++si) {
                Seg& s = segs[si];
                if (!s.in_norm) continue;
                initd2_kernel<<<nblk(s.n), EB, 0, st>>>(s.x0, s.k[0], s.k[1], rtol_f, atol_f, s.n, partial);
                finish_sums((int)si);
            }
            if ((rc = fetch_sums()) != PHX_OK) return rc;
            float d2 = block_norm(0) / h0;
            float h1 = (d1 <= 1e-15f && d2 <= 1e-15f) ? fmaxf(1e-6f, h0 * 1e-3f) : powf(0.01f / fmaxf(d1, d2), 0.2f);
            dt = (double)fminf(100.f * h0, h1);
            status.n_rhs += 2;
        }
        double tcur = t_start, tprev = t_start;
        int next_out = 0;
        long long nsteps = 0;
        while (next_out < nout) {
            if (nsteps >= max_steps) return fail(PHX_ST_MAX_STEPS, tcur, dt);
            if (!(tcur + dt > tcur)) return fail(PHX_ST_DT_UNDERFLOW, tcur, dt);
            if (nonfinite) return fail(PHX_ST_NONFINITE, tcur, dt);
            const float dtf = (float)dt;
            float cb[6][6], cerr[7], cmid[7];
            for (int i = 0; i < 6; ++i)
                for (int j = 0; j <= i; ++j) cb[i][j] = (float)H_BETA[i][j] * dtf;
            for (int j = 0; j < 7; ++j) {
                cerr[j] = dtf * (float)H_CERR[j];
                cmid[j] = dtf * (float)H_CMID[j];
            }
            for (int stg = 1; stg <= 6; ++stg) {
                // stage input from beta[stg-1]; the last one is y1 and is written to x1 as well
                if (!fuse || stg == 1) {
                    for (size_t si = 0; si < ns; ++si) {
                        Seg& s = segs[si];
                        KSet a = kset((int)si, sl, cb[stg - 1], stg);
                        if (stg == 6) combine(s.x1, s.x0, a, s.n);   // y1: the last stage is evaluated there, in place
                        else if (s.xs) combine(s.xs, s.x0, a, s.n);
                    }
                }
                if (fuse && stg < 6) {
                    // this launch's derivative k_stg closes the chain of the NEXT stage input (y1 after stage 5)
                    Seg& s = segs[0];
                    PhxRhsPost po;
                    memset(&po, 0, sizeof(po));
                    po.mode = PHX_POST_CHAIN; po.nk = stg; po.store_f = 1; po.x0 = s.x0;
                    po.out = stg == 5 ? s.x1 : s.xs;
                    for (int j = 0; j < stg; ++j) po.k[j] = s.k[sl[j]];
                    for (int j = 0; j < stg; ++j) po.c[j] = cb[stg][j];
                    po.cr = cb[stg][stg];
                    if ((rc = eval(sl[stg], AT_XS, &po)) != PHX_OK) return rc;
                    continue;
                }
                if ((rc = eval(sl[stg], stg == 6 ? AT_X1 : AT_XS)) != PHX_OK) return rc;
            }
            for (size_t si = 0; si < ns; ++si) {
                Seg& s = segs[si];
                if (!s.in_norm) continue;
                KSet a = kset((int)si, sl, cerr, 7);
                if (s.n % 4 == 0 && al16(s.x0) && al16(s.x1) && kset_al16(a)) {
                    err_kernel<4><<<nblk(s.n / 4), EB, 0, st>>>(s.x0, s.x1, a, rtol_f, atol_f, s.n, partial);
                    finish_sums((int)si, nblk(s.n / 4));
                } else {
                    err_kernel<1><<<nblk(s.n), EB, 0, st>>>(s.x0, s.x1, a, rtol_f, atol_f, s.n, partial);
                    finish_sums((int)si);
                }
            }
            if ((rc = fetch_sums()) != PHX_OK) return rc;
            float ratio = block_norm(0);
            bool accept = ratio <= 1.f;
            if ((int)log.size() / 3 < steplog_cap) {
                log.push_back(tcur);
                log.push_back(dt);
                log.push_back(accept ? 1.0 : 0.0);
            }
            status.n_rhs += 6;
            tprev = tcur;
            ++nsteps;
            double dt_used = dt;
            dt = next_dt_host(dt, ratio, safety, ifactor, dfactor);
            if (!accept) {
                status.n_rejected++;
                continue;
            }
            status.n_accepted++;
            tcur = tcur + dt_used;
            nonfinite = false;
            for (size_t si = 0; si < ns; ++si) nonfinite = nonfinite || (segs[si].in_norm && sums_host[3 * si + 1] > 0.0);
            while (next_out < nout && outs[next_out] <= tcur) {
                double x = (outs[next_out] - tprev) / (tcur - tprev);
                float xs[4];
                double xp = x;
                xs[0] = (float)xp; xp *= x; xs[1] = (float)xp; xp *= x; xs[2] = (float)xp; xp *= x; xs[3] = (float)xp;
                emit(next_out, xs, sl, dtf, cmid);
                ++next_out;
                nsteps = 0;
            }
            for (auto& s : segs) std::swap(s.x0, s.x1);
            std::swap(sl[0], sl[6]);
        }
        return PHX_OK;
    }
    void interp_seg(int si, float* out, const float* xs, const int* sl, float dtf, const float* cmid) {
        Seg& s = segs[si];
        KSet mid = kset(si, sl, cmid, 7);
        if (s.n % 4 == 0 && al16(out) && al16(s.x0) && al16(s.x1) && kset_al16(mid))
            interp_kernel<4><<<nblk(s.n / 4), EB, 0, st>>>(out, s.x0, s.x1, mid, s.k[sl[0]], s.k[sl[6]], dtf, xs[0], xs[1],
                                                           xs[2], xs[3], s.n);
        else
            interp_kernel<1><<<nblk(s.n), EB, 0, st>>>(out, s.x0, s.x1, mid, s.k[sl[0]], s.k[sl[6]], dtf, xs[0], xs[1],
                                                       xs[2], xs[3], s.n);
    }
    int fail(int code, double t, double dt) {
        status.code = code;
        status.t_fail = t;
        status.dt_fail = dt;
        return PHX_OK;  // a solver assertion is reported through the status record, like the resident kernels
    }
};

size_t stream_ws_floats(int G, int H, int B, int T, int adjoint, size_t* o_rhs, size_t* o_partial, size_t* o_sums,
                        size_t* o_seg) {
    size_t off = 0;
    auto take = [&](size_t nfloats) {
        size_t o = off;
        off += (nfloats + 3) & ~size_t(3);
        return o;
    };
    size_t partial = take(2 * (size_t)MAXBLK * 3);
    size_t sums = take(2 * 3 * 3 + 2);
    size_t rhs = take(phx_rhs_workspace_floats(G, H, B));
    size_t BG = (size_t)B * G;
    size_t seg = take(adjoint ? 2 * 10 * BG + 8 * phx_grad_offsets(G, H).total + 64 : 10 * BG + 16);
    if (o_rhs) *o_rhs = rhs;
    if (o_partial) *o_partial = partial;
    if (o_sums) *o_sums = sums;
    if (o_seg) *o_seg = seg;
    return off;
}

void write_back(Stream& S, phx_status* status_out) {
    S.status.n_logged = (int)(S.log.size() / 3);
    cudaPointerAttributes at;
    bool dev_status = false, dev_log = false;
    if (status_out && cudaPointerGetAttributes(&at, status_out) == cudaSuccess) dev_status = at.type == cudaMemoryTypeDevice;
    if (S.steplog && cudaPointerGetAttributes(&at, S.steplog) == cudaSuccess) dev_log = at.type == cudaMemoryTypeDevice;
    cudaGetLastError();
    cudaStreamSynchronize(S.st);
    if (S.steplog && !S.log.empty()) {
        if (dev_log) cudaMemcpy(S.steplog, S.log.data(), S.log.size() * sizeof(double), cudaMemcpyHostToDevice);
        else memcpy(S.steplog, S.log.data(), S.log.size() * sizeof(double));
    }
    if (status_out) {
        if (dev_status) cudaMemcpy(status_out, &S.status, sizeof(phx_status), cudaMemcpyHostToDevice);
        else *status_out = S.status;
    }
}

int setup(Stream& S, phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T, int t_is_f32,
          int method, double rtol, double atol, int64_t max_steps, int adjoint, void* workspace, size_t ws_bytes,
          double* steplog, int steplog_cap, cudaStream_t st, float** seg_base) {
    if (!ctx || G < 1 || H < 1 || B < 1 || !packed || !t_host || !workspace || T < 2) {
        phx_set_error("stream solve: invalid argument");
        return PHX_ERR_INVALID;
    }
    for (int i = 1; i < T; ++i)
        if (!(t_host[i] > t_host[i - 1])) {
            phx_set_error("t must be strictly increasing at the C boundary");
            return PHX_ERR_INVALID;
        }
    if (method < PHX_EULER || method > PHX_DOPRI5) {
        phx_set_error("unknown method id %d", method);
        return PHX_ERR_INVALID;
    }
    size_t o_rhs, o_partial, o_sums, o_seg;
    size_t need = stream_ws_floats(G, H, B, T, adjoint, &o_rhs, &o_partial, &o_sums, &o_seg) * sizeof(float);
    if (ws_bytes < need) {
        phx_set_error("stream workspace too small: %zu < %zu", ws_bytes, need);
        return PHX_ERR_WORKSPACE;
    }
    float* ws = (float*)workspace;
    S.ctx = ctx; S.G = G; S.H = H; S.B = B; S.T = T; S.method = method; S.t_is_f32 = t_is_f32; S.adjoint = adjoint;
    if (!adjoint) S.sum_world = phx_ctx_sum_hook(ctx, &S.sum_hook, &S.sum_user);
    S.rtol_f = (float)rtol; S.atol_f = (float)atol; S.fsign = 1.f; S.max_steps = (long long)max_steps;
    int rc_tc = phx_tc_prepare(ctx, G, H, B, packed, &S.w, st);
    if (rc_tc != PHX_OK) return rc_tc;
    S.st = st;
    S.rhs_ws = ws + o_rhs;
    S.partial = (double*)(ws + o_partial);
    S.sums_dev = (double*)(ws + o_sums);
    S.steplog = steplog;
    S.steplog_cap = steplog ? steplog_cap : 0;
    memset(&S.status, 0, sizeof(S.status));
    static thread_local double* pinned = nullptr;
    if (!pinned && cudaMallocHost((void**)&pinned, sizeof(double) * 16) != cudaSuccess) {
        phx_set_error("cudaMallocHost failed");
        return PHX_ERR_CUDA;
    }
    S.sums_host = pinned;
    *seg_base = ws + o_seg;
    return PHX_OK;
}

// the request's dopri5 step control (0: the default)
void set_step_control(Stream& S, const phx_solve_desc& d) {
    S.first_step = d.first_step;
    if (d.safety > 0) S.safety = d.safety;
    if (d.ifactor > 0) S.ifactor = d.ifactor;
    if (d.dfactor > 0) S.dfactor = d.dfactor;
}

float fixed_dt(const double* t, int i, int t_is_f32) {
    return t_is_f32 ? ((float)t[i + 1] - (float)t[i]) : (float)(t[i + 1] - t[i]);
}

}  // namespace

extern "C" {

size_t phx_stream_workspace_bytes(const phx_ctx* ctx, int G, int H, int B, int T, int adjoint) {
    if (!ctx || G < 1 || H < 1 || B < 1 || T < 2) return 0;
    return stream_ws_floats(G, H, B, T, adjoint, nullptr, nullptr, nullptr, nullptr) * sizeof(float);
}

}  // extern "C"

int phx_stream_forward(phx_ctx* ctx, const phx_solve_desc& d, cudaStream_t st) {
    const int G = d.G, H = d.H, B = d.B, T = d.T, method = d.method;
    const double* t_host = d.t_host;
    float* y_out = d.y_out;
    Stream S;
    float* base;
    const PhxGridHost g{d.grid_dt, d.grid_steps, d.grid_out_step, d.grid_out_slope};
    const PhxGridHost* grid = d.grid_dt ? &g : nullptr;
    if (grid && phx_grid_stage(*grid, 1, T, method, 1, nullptr, st, nullptr, nullptr) != PHX_OK) return PHX_ERR_INVALID;
    int rc = setup(S, ctx, G, H, B, d.packed, t_host, T, d.t_is_f32, method, d.rtol, d.atol, d.max_num_steps, 0,
                   d.workspace, d.workspace_bytes, d.steplog, d.steplog_cap, st, &base);
    if (rc != PHX_OK) return rc;
    S.fsign = d.reversed ? -1.f : 1.f;
    set_step_control(S, d);
    {
        // OFF unless PHX_STREAM_FUSE=1: measured slower at every shape (tools/stream_fuse_ab.py,
        // profiles/r04d_stream_fuse_ab.txt -- 60 rows x 11 165 genes rk4 0.40 ms fused / 0.34 ms not; 4 096 x 20 000:
        // 4.68 / 3.59 ms; the scan 242 / 261 genes/s).  The eight epilogue warps of a joint CTA hold at most ~48 loads
        // per thread in flight (168 registers at 320 threads), wait for them chunk by chunk, and the MMAs of the next tile
        // wait for the epilogue; the 1 184-block elementwise kernels stream the same arrays at HBM speed and cost one
        // launch.  Kept because it is bit-identical (tests/test_gpu_stream_fused.py) and documents the experiment.
        const char* e = getenv("PHX_STREAM_FUSE");
        const bool want = e && e[0] == '1';
        S.fuse = want && phx_rhs_post_supported(S.w, H, B);
    }
    const size_t BG = (size_t)B * G;
    Seg y;
    y.n = BG; y.count = (double)BG;
    y.x0 = base; y.x1 = base + BG; y.xs = base + 2 * BG;
    for (int i = 0; i < 7; ++i) y.k[i] = base + (3 + i) * BG;
    S.segs.push_back(y);
    cudaMemcpyAsync(y_out, d.y0, BG * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (method != PHX_DOPRI5 && grid) {
        // the caller's grid: a step that ends on an output time writes that output slice, the others a scratch slot
        // (x0 / x1, never the step's own input); output times inside the step are interpolated between the two
        S.segs[0].x0 = y_out;
        float* cur = y_out;
        int jn = 1;
        for (int k = 0; k < grid->steps[0] && rc == PHX_OK; ++k) {
            int je = jn;
            while (je < T && grid->out_step[je - 1] == k) ++je;
            const bool hit = je > jn && grid->out_slope[je - 2] < 0.f;   // an exact hit is the step's last output
            float* dst = hit ? y_out + (size_t)(je - 1) * BG : (cur == base ? base + BG : base);
            rc = S.fixed_step(grid->dt[k], dst);
            for (int j = jn; j < je && rc == PHX_OK; ++j)
                if (!(grid->out_slope[j - 1] < 0.f))
                    lerp_kernel<<<nblk(BG), EB, 0, st>>>(y_out + (size_t)j * BG, cur, dst, grid->out_slope[j - 1], BG);
            cur = dst;
            jn = je;
        }
    } else if (method != PHX_DOPRI5) {
        // fixed grid: the state of interval i is read from the output slice i and written to slice i + 1
        S.segs[0].x0 = y_out;
        for (int i = 0; i + 1 < T && rc == PHX_OK; ++i) rc = S.fixed_step(fixed_dt(t_host, i, d.t_is_f32), y_out + (size_t)(i + 1) * BG);
    } else {
        cudaMemcpyAsync(y.x0, d.y0, BG * sizeof(float), cudaMemcpyDeviceToDevice, st);
        rc = S.dopri5(t_host[0], t_host + 1, T - 1,
                      [&](int j, const float* xs, const int* sl, float dtf, const float* cmid) {
                          S.interp_seg(0, y_out + (size_t)(j + 1) * BG, xs, sl, dtf, cmid);
                      });
    }
    if (rc != PHX_OK) return rc;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("stream forward: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    write_back(S, d.status);
    return PHX_OK;
}

int phx_stream_adjoint(phx_ctx* ctx, const phx_solve_desc& d, cudaStream_t st) {
    const int G = d.G, H = d.H, B = d.B, T = d.T, method = d.method, param_mask = d.param_mask;
    const double* t_host = d.t_host;
    const float *y_saved = d.y_saved, *grad_y = d.grad_y, *grid_dt = d.grid_dt;
    float* grads_flat = d.grads;
    Stream S;
    float* base;
    std::vector<int> goff;   // the grid's interval offsets into grid_dt
    const PhxGridHost grid{grid_dt, d.grid_steps, nullptr, nullptr};
    if (grid_dt && phx_grid_stage(grid, 1, T, method, 0, nullptr, st, nullptr, &goff) != PHX_OK) return PHX_ERR_INVALID;
    int rc = setup(S, ctx, G, H, B, d.packed, t_host, T, d.t_is_f32, method, d.rtol, d.atol, d.max_num_steps, 1,
                   d.workspace, d.workspace_bytes, d.steplog, d.steplog_cap, st, &base);
    if (rc != PHX_OK) return rc;
    set_step_control(S, d);
    const size_t BG = (size_t)B * G, P = phx_grad_offsets(G, H).total;
    // the theta segment holds the adjoint parameters' cotangents only, back to back in reference order (all six: the
    // flat layout itself), at the start of grads_flat; it is absent when there are none
    // (PHX_NORM_SEMINORM: the segment is integrated but kept out of every norm)
    const int pm = param_mask & PHX_P_ALL;
    const size_t PS = phx_mask_count(G, H, pm);
    S.pmask = pm;
    S.goff = phx_compact_grad_offsets(G, H, pm);
    Seg y, a, th;
    y.n = a.n = BG; y.count = a.count = (double)BG;
    y.x0 = base; y.x1 = base + BG; y.xs = base + 2 * BG;
    for (int i = 0; i < 7; ++i) y.k[i] = base + (3 + i) * BG;
    float* ab = base + 10 * BG;
    a.x0 = ab; a.x1 = ab + BG; a.xs = ab + 2 * BG;
    for (int i = 0; i < 7; ++i) a.k[i] = ab + (3 + i) * BG;
    float* tb = ab + 10 * BG;
    tb += (4 - ((size_t)(tb - (float*)d.workspace) & 3)) & 3;
    th.n = PS; th.count = (double)PS;
    th.in_norm = !(param_mask & PHX_NORM_SEMINORM);
    th.x0 = grads_flat; th.x1 = tb; th.xs = nullptr;
    for (int i = 0; i < 7; ++i) th.k[i] = tb + (size_t)(1 + i) * PS;
    S.segs.push_back(y);
    S.segs.push_back(a);
    if (PS > 0) S.segs.push_back(th);
    cudaMemsetAsync(grads_flat, 0, P * sizeof(float), st);
    cudaMemcpyAsync(S.segs[1].x0, grad_y + (size_t)(T - 1) * BG, BG * sizeof(float), cudaMemcpyDeviceToDevice, st);
    // the time cotangents of the T-1 intervals, fetched once: dopri5 reads interval iv's after its first synchronisation
    float* tv = nullptr;
    if (d.t_vjp && method == PHX_DOPRI5) {
        static thread_local float* pinned_tv = nullptr;
        static thread_local int pinned_cap = 0;
        if (pinned_cap < T - 1) {
            if (pinned_tv) cudaFreeHost(pinned_tv);
            pinned_cap = 0;
            if (cudaMallocHost((void**)&pinned_tv, sizeof(float) * (T - 1)) != cudaSuccess) {
                pinned_tv = nullptr;
                phx_set_error("cudaMallocHost failed");
                return PHX_ERR_CUDA;
            }
            pinned_cap = T - 1;
        }
        tv = pinned_tv;
        cudaError_t e = cudaMemcpyAsync(tv, d.t_vjp, sizeof(float) * (T - 1), cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) {
            phx_set_error("cudaMemcpyAsync(t_vjp): %s", cudaGetErrorString(e));
            return PHX_ERR_CUDA;
        }
    }
    for (int iv = T - 1; iv >= 1 && rc == PHX_OK && S.status.code == PHX_ST_OK; --iv) {
        S.vjp_t = tv ? tv + iv - 1 : nullptr;
        cudaMemcpyAsync(S.segs[0].x0, y_saved + (size_t)iv * BG, BG * sizeof(float), cudaMemcpyDeviceToDevice, st);
        if (method != PHX_DOPRI5 && grid_dt) {
            for (int k = goff[iv - 1]; k < goff[iv] && rc == PHX_OK; ++k) rc = S.fixed_step(grid_dt[k]);
        } else if (method != PHX_DOPRI5) {
            rc = S.fixed_step(fixed_dt(t_host, iv - 1, d.t_is_f32));
        } else {
            double t_end = -t_host[iv - 1];
            rc = S.dopri5(-t_host[iv], &t_end, 1,
                          [&](int, const float* xs, const int* sl, float dtf, const float* cmid) {
                              // dense output at t_end for adj_y and adj_params, written into x1 so that the swap
                              // after the step leaves it in x0; y is replaced by the saved state anyway
                              // (in place: every element is read before it is overwritten)
                              S.interp_seg(1, S.segs[1].x1, xs, sl, dtf, cmid);
                              if (PS > 0) S.interp_seg(2, S.segs[2].x1, xs, sl, dtf, cmid);
                          });
        }
        if (rc != PHX_OK) break;
        Seg& as = S.segs[1];
        add_kernel<<<nblk(BG), EB, 0, st>>>(as.x0, grad_y + (size_t)(iv - 1) * BG, BG);
    }
    if (rc != PHX_OK) return rc;
    cudaMemcpyAsync(d.adj_y0, S.segs[1].x0, BG * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (pm == PHX_P_ALL) {
        if (S.segs[2].x0 != grads_flat)
            cudaMemcpyAsync(grads_flat, S.segs[2].x0, P * sizeof(float), cudaMemcpyDeviceToDevice, st);
    } else {
        // back to the flat layout: the kept blocks from the segment (moved out of grads_flat first), zeros elsewhere
        const float* src = nullptr;
        if (PS > 0) {
            src = S.segs[2].x0;
            if (src == grads_flat) {
                cudaMemcpyAsync(S.segs[2].x1, grads_flat, PS * sizeof(float), cudaMemcpyDeviceToDevice, st);
                src = S.segs[2].x1;
            }
        }
        cudaMemsetAsync(grads_flat, 0, P * sizeof(float), st);
        const PhxGradOff fo = phx_grad_offsets(G, H), co = S.goff;
        const size_t HG = (size_t)H * G;
        const size_t flo[6] = {fo.m, fo.Wp, fo.bp, fo.Ws, fo.bs, fo.Wa}, clo[6] = {co.m, co.Wp, co.bp, co.Ws, co.bs, co.Wa};
        const size_t n[6] = {(size_t)G, HG, (size_t)H, HG, (size_t)H, 2 * HG};
        for (int q = 0; q < 6; ++q)
            if (pm & (1 << q))
                cudaMemcpyAsync(grads_flat + flo[q], src + clo[q], n[q] * sizeof(float), cudaMemcpyDeviceToDevice, st);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("stream adjoint: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    write_back(S, d.status);
    return PHX_OK;
}
