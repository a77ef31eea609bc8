// Stand-alone batched RHS and RHS-VJP for any number of rows B (ODENet.forward / prior_only_forward called directly,
// e.g. the 10 000-row prior batch of train_insilico.py:134, and their ordinary-autograd backward).
//
// fp32 CUDA-core path: every contraction is one launch of a functor-driven tiled SGEMM (64x64x16 tiles, 4x4 register
// micro-tiles) whose operand loaders fuse the Hill activations / decay factors and whose epilogues fuse bias, exp, the
// decay term and the cotangent algebra, so no activation tensor is ever materialised in HBM:
//   SP  [B][K2] = act(y) W1            (+bias, exp on the prods half)                    odenet.py:86-88
//   f   [B][G]  = relu(m) (SP WA^T - y)                                                 odenet.py:89-90
//   GS  [B][K2] = (g relu(m)) WA       (prods half scaled by Pr)                         exp / Linear backward
//   ybar[B][G]  = (GS_s Ws + (GS_p Wp)/(1+s)) / (1+|y-.5|)^2 - g relu(m)                 soft-sign / log1p backward
//   Wa_bar = gJ^T SP,  Ws_bar = GS_s^T s,  Wp_bar = GS_p^T l,  biases / multipliers: column sums
// The tcgen05 (3xTF32) variant of the same decomposition replaces sgemm_kernel for large B in a later round.
#include <math.h>
#include "phx_common.cuh"

namespace {

constexpr int BM = 64, BN = 64, BK = 16, GT = 256;

template <typename LA, typename LB, typename EPI>
__global__ void __launch_bounds__(GT) sgemm_kernel(int M, int N, int K, LA la, LB lb, EPI epi) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < K; k0 += BK) {
        for (int i = tid; i < BM * BK; i += GT) {
            int m, kk;
            if (LA::k_contig) { kk = i % BK; m = i / BK; } else { m = i % BM; kk = i / BM; }
            As[kk][m] = (m0 + m < M && k0 + kk < K) ? la(m0 + m, k0 + kk) : 0.f;
        }
        for (int i = tid; i < BN * BK; i += GT) {
            int n, kk;
            if (LB::n_contig) { n = i % BN; kk = i / BN; } else { kk = i % BK; n = i / BK; }
            Bs[kk][n] = (n0 + n < N && k0 + kk < K) ? lb(k0 + kk, n0 + n) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
            for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
            if (m < M && n < N) epi(m, n, acc[i][j]);
        }
}

template <typename LA, typename LB, typename EPI>
void sgemm(int M, int N, int K, LA la, LB lb, EPI epi, cudaStream_t st) {
    if (M <= 0 || N <= 0) return;
    dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM);
    sgemm_kernel<<<grid, GT, 0, st>>>(M, N, K, la, lb, epi);
}

__device__ __forceinline__ void hill(float y, float& s, float& l, float& den) {
    float z = y - 0.5f;
    den = 1.0f + fabsf(z);
    s = z / den;
    l = log1pf(s);
}

// ---- operand loaders -----------------------------------------------------------------------------------------------
// A(b, g) = s(y[b][g]) or l(y[b][g])
struct LoadAct {
    static constexpr bool k_contig = true;
    const float* y; int G; int use_l;
    __device__ float operator()(int b, int g) const {
        float s, l, den;
        hill(y[(size_t)b * G + g], s, l, den);
        return use_l ? l : s;
    }
};
// B(g, n) = W[g][col0 + n]   (row-major packed weight, n contiguous)
struct LoadWrow {
    static constexpr bool n_contig = true;
    const float* W; int ld; int col0;
    __device__ float operator()(int g, int n) const { return __ldg(W + (size_t)g * ld + col0 + n); }
};
// A(b, k) = X[b][col0 + k]
struct LoadRowMajorA {
    static constexpr bool k_contig = true;
    const float* X; int ld; int col0;
    __device__ float operator()(int b, int k) const { return X[(size_t)b * ld + col0 + k]; }
};
// B(k, g) = W[g][col0 + k]  (transposed use of a packed weight: k contiguous)
struct LoadWcol {
    static constexpr bool n_contig = false;
    const float* W; int ld; int col0;
    __device__ float operator()(int k, int g) const { return __ldg(W + (size_t)g * ld + col0 + k); }
};
// A(b, g) = g_cot[b][g] * (decay ? relum[g] : 1)
struct LoadGJ {
    static constexpr bool k_contig = true;
    const float* g; const float* relum; int G; int decay;
    __device__ float operator()(int b, int gg) const {
        float v = g[(size_t)b * G + gg];
        return decay ? v * relum[gg] : v;
    }
};
// A(m, b) = X[b][col0 + m]  (X^T, m contiguous)
struct LoadTransA {
    static constexpr bool k_contig = false;
    const float* X; int ld; int col0;
    __device__ float operator()(int m, int b) const { return X[(size_t)b * ld + col0 + m]; }
};
struct LoadGJT {  // A(g, b) = gJ[b][g]
    static constexpr bool k_contig = false;
    const float* g; const float* relum; int G; int decay;
    __device__ float operator()(int gg, int b) const {
        float v = g[(size_t)b * G + gg];
        return decay ? v * relum[gg] : v;
    }
};
struct LoadActB {  // B(b, g) = s or l of y[b][g]
    static constexpr bool n_contig = true;
    const float* y; int G; int use_l;
    __device__ float operator()(int b, int g) const {
        float s, l, den;
        hill(y[(size_t)b * G + g], s, l, den);
        return use_l ? l : s;
    }
};
struct LoadRowMajorB {  // B(b, n) = X[b][col0+n]
    static constexpr bool n_contig = true;
    const float* X; int ld; int col0;
    __device__ float operator()(int b, int n) const { return X[(size_t)b * ld + col0 + n]; }
};

// ---- epilogues --------------------------------------------------------------------------------------------------------
struct EpiSP {  // SP[b][col0+n] = acc + bias ; exp on prods half ; pads -> 0
    float* SP; const float* bias; int K2, Hp, H, col0;
    __device__ void operator()(int b, int n, float acc) const {
        int k = col0 + n;
        float v = acc + bias[k];
        if (k >= Hp) v = (k - Hp < H) ? expf(v) : 0.f;
        SP[(size_t)b * K2 + k] = v;
    }
};
struct EpiF {  // f = fscale * (decay ? relum*(J - y) : J)
    float* f; const float* y; const float* relum; int G; int decay; float fscale;
    __device__ void operator()(int b, int g, float acc) const {
        size_t i = (size_t)b * G + g;
        f[i] = fscale * (decay ? relum[g] * (acc - y[i]) : acc);
    }
};
struct EpiGS {  // GS[b][k] = acc (sums half) or acc * Pr (prods half)
    float* GS; const float* SP; int K2, Hp;
    __device__ void operator()(int b, int k, float acc) const {
        size_t i = (size_t)b * K2 + k;
        GS[i] = (k >= Hp) ? acc * SP[i] : acc;
    }
};
struct EpiStore {  // plain store into [M][ld]
    float* C; int ld;
    __device__ void operator()(int m, int n, float acc) const { C[(size_t)m * ld + n] = acc; }
};
struct EpiYbar {  // ybar = (u + v/(1+s))/den^2 - gJ   (u held in ybar from the first pass, acc = v)
    float* ybar; const float* y; const float* g; const float* relum; int G; int decay;
    __device__ void operator()(int b, int gg, float acc) const {
        size_t i = (size_t)b * G + gg;
        float s, l, den;
        hill(y[i], s, l, den);
        float r = (ybar[i] + acc / (1.0f + s)) / (den * den);
        if (decay) r = r - g[i] * relum[gg];
        ybar[i] = r;
    }
};
struct EpiGrad {  // grads[off + m*ld + n] (+)= acc
    float* dst; int ld; int accumulate;
    __device__ void operator()(int m, int n, float acc) const {
        size_t i = (size_t)m * ld + n;
        dst[i] = accumulate ? dst[i] + acc : acc;
    }
};
struct EpiGradWa {  // m = gene, n = packed column -> Wa_bar[g][2H] (skip pads)
    float* dst; int H, Hp; int accumulate;
    __device__ void operator()(int gg, int k, float acc) const {
        int col;
        if (k < Hp) { if (k >= H) return; col = k; } else { if (k - Hp >= H) return; col = H + k - Hp; }
        size_t i = (size_t)gg * 2 * H + col;
        dst[i] = accumulate ? dst[i] + acc : acc;
    }
};

// column sums over the B rows (biases, multipliers).  Block = 32 columns x 32 row lanes: a warp reads 128 contiguous
// bytes of one row, every row lane walks rows ty, ty+32, ... and the 32 lane totals are added in fixed order, so the
// result is deterministic.
constexpr int CS = 32;
__device__ __forceinline__ float colsum_fold(float t, float (*sh)[CS + 1]) {
    const int tx = threadIdx.x, ty = threadIdx.y;
    sh[ty][tx] = t;
    __syncthreads();
    float r = 0.f;
    if (ty == 0)
        for (int i = 0; i < CS; ++i) r += sh[i][tx];
    return r;
}
__global__ void colsum_bias_kernel(const float* GS, int B, int K2, int Hp, int H, float* bs_bar, float* bp_bar,
                                   int accumulate) {
    __shared__ float sh[CS][CS + 1];
    const int k = blockIdx.x * CS + threadIdx.x;
    const bool ok = k < 2 * H;
    const int col = ok ? ((k < H) ? k : (Hp + k - H)) : 0;
    float t = 0.f;
    if (ok)
        for (int b = threadIdx.y; b < B; b += CS) t += GS[(size_t)b * K2 + col];
    t = colsum_fold(t, sh);
    float* const base = (k < H) ? bs_bar : bp_bar;   // nullptr: that bias is not wanted
    if (ok && threadIdx.y == 0 && base) {
        float* dst = base + ((k < H) ? k : k - H);
        *dst = accumulate ? *dst + t : t;
    }
}
// f_out = fscale * relum * (J - y) from the un-decayed J
__global__ void decay_kernel(const float* J, const float* y, const float* relum, int G, size_t n, float fscale,
                             float* f_out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        f_out[i] = fscale * (relum[i % G] * (J[i] - y[i]));
}
// m_bar[g] = mask[g] * sum_b g[b][g] * (J - y)[b][g].  from_f != 0: `f_nodecay` is the finished RHS value
// f = fscale * relu(m) * (J - y) instead of J, and (J - y) is recovered per gene after the column sum
// (mask[g] != 0  <=>  relu(m)[g] > 0).
__global__ void colsum_mult_kernel(const float* g, const float* f_nodecay, const float* y, const float* maskm, int B,
                                   int G, float* m_bar, int accumulate, int decay, int from_f, const float* relum,
                                   float fscale) {
    __shared__ float sh[CS][CS + 1];
    const int gg = blockIdx.x * CS + threadIdx.x;
    const bool ok = gg < G;
    float t = 0.f;
    if (ok && decay)
        for (int b = threadIdx.y; b < B; b += CS) {
            size_t i = (size_t)b * G + gg;
            t += from_f ? g[i] * f_nodecay[i] : g[i] * (f_nodecay[i] - y[i]);
        }
    t = colsum_fold(t, sh);
    if (ok && threadIdx.y == 0) {
        if (!decay || maskm[gg] == 0.f) t = 0.f;
        else if (from_f) t = t / (fscale * relum[gg]);
        m_bar[gg] = accumulate ? m_bar[gg] + t : t;
    }
}

}  // namespace

static size_t rhs_base_floats(int G, int H, int B) {
    size_t K2 = (size_t)phx_K2(H);
    // SP, GS, J (+ 16, rounded to an even count), then 2 * 8 * 160 floats = the per-warp double partial sums of the fused
    // prior loss
    return ((2 * (size_t)B * K2 + (size_t)B * G + 16 + 1) & ~(size_t)1) + 2 * 8 * 160;
}
size_t phx_rhs_workspace_floats(int G, int H, int B) {
    size_t K2 = (size_t)phx_K2(H);
    // SP, GS : [B][K2] each ; J : [B][G] ; scratch of the tensor-core path (K-split partials, [S|P] operand image)
    return rhs_base_floats(G, H, B) + (phx_tc_shape_ok(H, B) ? phx_tc_scratch_floats(G, H, B) : 0);
}

static void rhs_sp(int G, int H, int B, const PhxPacked& w, const float* y, float* SP, cudaStream_t st) {
    const int Hp = phx_Hp(H), K2 = 2 * Hp;
    const float* W1 = reinterpret_cast<const float*>(w.W1);
    for (int half = 0; half < 2; ++half) {
        LoadAct la{y, G, half};
        LoadWrow lb{W1, K2, half * Hp};
        EpiSP ep{SP, w.bias, K2, Hp, H, half * Hp};
        sgemm(B, Hp, G, la, lb, ep, st);
    }
}

bool phx_rhs_post_supported(const PhxPacked& w, int H, int B) { return w.tc && phx_tc_shape_ok(H, B); }

int phx_rhs_forward_launch(int G, int H, int B, const PhxPacked& w, const float* y, float* f, int decay, float fscale,
                           float* ws, cudaStream_t st, const PhxRhsPost* post) {
    const int K2 = phx_K2(H);
    float* SP = ws;
    if (w.tc && phx_tc_shape_ok(H, B))   // tcgen05 path: both contractions on the tensor cores
        return phx_tc_rhs_forward_launch(G, H, B, w, y, f, decay, fscale, SP, ws + rhs_base_floats(G, H, B), st, post);
    if (post && post->mode != PHX_POST_NONE) {
        phx_set_error("rhs_forward: the fused stage algebra needs the tensor-core path (phx_rhs_post_supported)");
        return PHX_ERR_INVALID;
    }
    rhs_sp(G, H, B, w, y, SP, st);
    LoadRowMajorA la{SP, K2, 0};
    LoadWcol lb{reinterpret_cast<const float*>(w.WA), K2, 0};
    EpiF ep{f, y, w.relum, G, decay, fscale};
    sgemm(B, G, K2, la, lb, ep, st);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("rhs_forward launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

int phx_rhs_vjp_launch(int G, int H, int B, const PhxPacked& w, const float* y, const float* g, int decay,
                       float* ybar, float* grads, int accumulate_flags, float* f_out, float fscale, float* ws,
                       cudaStream_t st, int pmask, const PhxGradOff* goff) {
    const int Hp = phx_Hp(H), K2 = 2 * Hp;
    const int accumulate = accumulate_flags & 1;
    float* SP = ws;
    float* GS = ws + (size_t)B * K2;
    float* J = GS + (size_t)B * K2;
    const float* W1 = reinterpret_cast<const float*>(w.W1);
    const float* WA = reinterpret_cast<const float*>(w.WA);
    const bool tc = w.tc && phx_tc_shape_ok(H, B);
    const bool needJ = (f_out != nullptr) || (grads && decay && (pmask & PHX_P_M));
    bool direct_f = false;
    if (tc) {
        // tensor cores: [S|P], gSP, the state cotangent and the un-decayed joint (phx_tc.cu); the K = B parameter
        // contractions below stay on the fp32 path
        float* tcws = ws + rhs_base_floats(G, H, B);
        int rc = PHX_OK;
        if (!(accumulate_flags & 2))   // bit 1: the workspace still holds [S|P] (+ images) of this (weights, y)
            rc = phx_tc_rhs_forward_launch(G, H, B, w, y, nullptr, 0, 1.f, SP, tcws, st);
        if (rc != PHX_OK) return rc;
        // with the decay term and an RHS output requested (the streaming adjoint) the joint kernel writes f itself and
        // the multiplier cotangent is recovered from it: no un-decayed J, no separate decay pass
        direct_f = f_out != nullptr && decay;
        rc = phx_tc_vjp_state_launch(G, H, B, w, y, g, decay, ybar, SP, GS, (needJ && !direct_f) ? J : nullptr, tcws, st);
        if (rc != PHX_OK) return rc;
        if (direct_f) {
            rc = phx_tc_joint_launch(G, H, B, w, y, f_out, 1, fscale, tcws, st);
            if (rc != PHX_OK) return rc;
        }
    } else {
        rhs_sp(G, H, B, w, y, SP, st);
        // GS = gJ WA, prods half scaled by Pr
        {
            LoadGJ la{g, w.relum, G, decay};
            LoadWrow lb{WA, K2, 0};
            EpiGS ep{GS, SP, K2, Hp};
            sgemm(B, K2, G, la, lb, ep, st);
        }
        if (ybar) {
            {   // u = GS_s Ws
                LoadRowMajorA la{GS, K2, 0};
                LoadWcol lb{W1, K2, 0};
                EpiStore ep{ybar, G};
                sgemm(B, G, Hp, la, lb, ep, st);
            }
            {   // v = GS_p Wp, combine
                LoadRowMajorA la{GS, K2, Hp};
                LoadWcol lb{W1, K2, Hp};
                EpiYbar ep{ybar, y, g, w.relum, G, decay};
                sgemm(B, G, Hp, la, lb, ep, st);
            }
        }
        if (needJ) {   // un-decayed joint, for the multiplier cotangent and/or the RHS value itself
            LoadRowMajorA la{SP, K2, 0};
            LoadWcol lb{WA, K2, 0};
            EpiF ep{J, y, w.relum, G, 0, 1.f};
            sgemm(B, G, K2, la, lb, ep, st);
        }
    }
    if (f_out && !direct_f) {
        size_t n = (size_t)B * G;
        int blocks = (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
        if (decay) decay_kernel<<<blocks, 256, 0, st>>>(J, y, w.relum, G, n, fscale, f_out);
        else cudaMemcpyAsync(f_out, J, n * sizeof(float), cudaMemcpyDeviceToDevice, st);
    }
    // parameter cotangents: only the blocks in pmask, at the offsets `goff` (default: the flat reference layout)
    if (grads && pmask) {
        const PhxGradOff off = goff ? *goff : phx_grad_offsets(G, H);
        if (tc) {
            int rc = phx_tc_vjp_params_launch(G, H, B, w, y, g, decay, grads, accumulate,
                                              ws + rhs_base_floats(G, H, B), st, pmask, &off);
            if (rc != PHX_OK) return rc;
        } else {
            if (pmask & PHX_P_WA) {   // Wa_bar[g][k] = sum_b gJ[b][g] SP[b][k]
                LoadGJT la{g, w.relum, G, decay};
                LoadRowMajorB lb{SP, K2, 0};
                EpiGradWa ep{grads + off.Wa, H, Hp, accumulate};
                sgemm(G, K2, B, la, lb, ep, st);
            }
            if (pmask & PHX_P_WS) {   // Ws_bar[h][g] = sum_b GS[b][h] s[b][g]
                LoadTransA la{GS, K2, 0};
                LoadActB lb{y, G, 0};
                EpiGrad ep{grads + off.Ws, G, accumulate};
                sgemm(H, G, B, la, lb, ep, st);
            }
            if (pmask & PHX_P_WP) {   // Wp_bar[h][g] = sum_b GS[b][Hp+h] l[b][g]
                LoadTransA la{GS, K2, Hp};
                LoadActB lb{y, G, 1};
                EpiGrad ep{grads + off.Wp, G, accumulate};
                sgemm(H, G, B, la, lb, ep, st);
            }
        }
        if (pmask & (PHX_P_BS | PHX_P_BP))
            colsum_bias_kernel<<<(2 * H + CS - 1) / CS, dim3(CS, CS), 0, st>>>(
                GS, B, K2, Hp, H, (pmask & PHX_P_BS) ? grads + off.bs : nullptr,
                (pmask & PHX_P_BP) ? grads + off.bp : nullptr, accumulate);
        if (pmask & PHX_P_M)
            colsum_mult_kernel<<<(G + CS - 1) / CS, dim3(CS, CS), 0, st>>>(g, direct_f ? f_out : J, y, w.maskm, B, G,
                                                                           grads + off.m, accumulate, decay, direct_f,
                                                                           w.relum, fscale);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("rhs_vjp launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}


// ---- prior-constrained loss (train_insilico.py:134-135, 208-209) ---------------------------------------------------------
namespace {
// fallback for batches below the tensor-core threshold / fp32 precision: J is materialised, then one elementwise pass
__global__ void prior_loss_elem_kernel(const float* __restrict__ J, const float* __restrict__ pg, size_t n, float scale,
                                       float* __restrict__ gcot, double* __restrict__ part) {
    double sq = 0.0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float d = J[i] - pg[i];
        sq += (double)(d * d);
        gcot[i] = scale * d;
    }
    __shared__ double red[256];
    red[threadIdx.x] = sq;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) part[blockIdx.x] = red[0];
}
__global__ void prior_loss_sum_kernel(const double* __restrict__ part, int n, double inv_n, float* __restrict__ loss) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < n; ++i) t += part[i];
        *loss = (float)(t * inv_n);
    }
}
// prior_grad = batch_for_prior @ prior_mat (train_insilico.py:209) with the 0.5-3 % dense prior in CSC form: one CTA per
// R batch rows (staged in shared memory, interleaved [gene][R]), one thread per output gene walking that gene's column of
// the prior -- every (row index, value) pair fetched from L2 serves R rows.  Each output is one fmaf chain over its
// column in storage order, whatever R is.
template <int R>
__global__ void prior_setup_kernel(int G, int B, const float* __restrict__ x, const int* __restrict__ colptr,
                                   const int* __restrict__ rowidx, const float* __restrict__ val, float* __restrict__ out) {
    extern __shared__ float xrow[];
    const size_t b0 = (size_t)blockIdx.x * R;
    for (int i = threadIdx.x; i < G; i += blockDim.x) {
#pragma unroll
        for (int r = 0; r < R; ++r) xrow[(size_t)i * R + r] = (b0 + r < (size_t)B) ? x[(b0 + r) * G + i] : 0.f;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < G; j += blockDim.x) {
        float t[R];
#pragma unroll
        for (int r = 0; r < R; ++r) t[r] = 0.f;
        for (int e = colptr[j]; e < colptr[j + 1]; ++e) {
            const float v = val[e];
            const float* xr = xrow + (size_t)rowidx[e] * R;
#pragma unroll
            for (int r = 0; r < R; ++r) t[r] = fmaf(xr[r], v, t[r]);
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (b0 + r < (size_t)B) out[(b0 + r) * G + j] = t[r];
    }
}
template <int R>
cudaError_t prior_setup_run(int G, int B, const float* x, const int* colptr, const int* rowidx, const float* val,
                            float* out, cudaStream_t st) {
    const size_t smem = (size_t)G * R * sizeof(float);
    cudaFuncSetAttribute(prior_setup_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    prior_setup_kernel<R><<<(B + R - 1) / R, 512, smem, st>>>(G, B, x, colptr, rowidx, val, out);
    return cudaGetLastError();
}
}  // namespace

int phx_prior_loss_launch(int G, int H, int B, const PhxPacked& w, const float* x, const float* prior_grad, float scale,
                          float* gcot, float* loss, float* ws, cudaStream_t st) {
    const int K2 = phx_K2(H);
    float* SP = ws;
    float* J = ws + 2 * (size_t)B * K2;
    double* part = reinterpret_cast<double*>(ws + rhs_base_floats(G, H, B) - 2 * 8 * 160);
    if (w.tc && phx_tc_shape_ok(H, B))
        return phx_tc_prior_loss_launch(G, H, B, w, x, prior_grad, scale, gcot, loss, SP, part,
                                        ws + rhs_base_floats(G, H, B), st);
    int rc = phx_rhs_forward_launch(G, H, B, w, x, J, 0, 1.f, ws, st);
    if (rc != PHX_OK) return rc;
    const size_t n = (size_t)B * G;
    const int blocks = (int)((n + 255) / 256 < 1024 ? (n + 255) / 256 : 1024);
    prior_loss_elem_kernel<<<blocks, 256, 0, st>>>(J, prior_grad, n, scale, gcot, part);
    prior_loss_sum_kernel<<<1, 32, 0, st>>>(part, blocks, 1.0 / (double)n, loss);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("prior_loss launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

int phx_prior_setup_launch(int G, int B, const float* x, const int* colptr, const int* rowidx, const float* val,
                           float* out, cudaStream_t st) {
    const size_t row = (size_t)G * sizeof(float), budget = 200 * 1024;
    if (row > budget) {
        phx_set_error("prior_setup supports up to 51200 genes (got %d)", G);
        return PHX_ERR_UNSUPPORTED;
    }
    // as many batch rows per CTA as fit beside each other in shared memory (4 at 11 165 genes, 2 at 20 000)
    cudaError_t e;
    if (4 * row <= budget) e = prior_setup_run<4>(G, B, x, colptr, rowidx, val, out, st);
    else if (2 * row <= budget) e = prior_setup_run<2>(G, B, x, colptr, rowidx, val, out, st);
    else e = prior_setup_run<1>(G, B, x, colptr, rowidx, val, out, st);
    if (e != cudaSuccess) {
        phx_set_error("prior_setup launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}
