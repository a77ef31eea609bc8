// extern "C" entry points of libphoenix_b200.so (declared in include/phoenix_b200.h).
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <unordered_map>
#include <vector>
#include "phx_common.cuh"

static thread_local char g_err[512] = "";

void phx_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

struct phx_ctx {
    int device;
    int num_sms;
    int coop;
    long long* prof;
    int precision;                                   // PHX_PREC_*
    std::mutex mu;
    std::unordered_map<const float*, int> tc_valid;  // packed buffer -> its tensor-core images are current
    phx_sum_hook sum_hook;                           // exact-global-norm mode of sharded batched dopri5 solves
    void* sum_user;
    int sum_world;
};

namespace {

__global__ void pack_kernel(int G, int H, int Hp, int K2, const float* __restrict__ m, const float* __restrict__ Wp,
                            const float* __restrict__ bp, const float* __restrict__ Ws, const float* __restrict__ bs,
                            const float* __restrict__ Wa, float* __restrict__ W1, float* __restrict__ WA,
                            float* __restrict__ bias, float* __restrict__ relum, float* __restrict__ maskm) {
    const size_t n = (size_t)G * K2;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        int g = (int)(i / K2), k = (int)(i % K2);
        int half = k >= Hp, h = half ? k - Hp : k;
        float w1 = 0.f, wa = 0.f;
        if (h < H) {
            w1 = half ? Wp[(size_t)h * G + g] : Ws[(size_t)h * G + g];
            wa = Wa[(size_t)g * 2 * H + (half ? H + h : h)];
        }
        W1[i] = w1;
        WA[i] = wa;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)K2; i += stride) {
        int k = (int)i, half = k >= Hp, h = half ? k - Hp : k;
        bias[k] = (h < H) ? (half ? bp[h] : bs[h]) : 0.f;
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)G; i += stride) {
        float v = m[i];
        relum[i] = v > 0.f ? v : 0.f;
        maskm[i] = v > 0.f ? 1.f : 0.f;
    }
}


// packed-layout cotangents (phx_packed_grad_offsets) -> the reference's flat order (phx_grad_offsets).  The two branch
// matrices are transposed ([G][K2] gene-major -> [H][G]) through a 32 x 33 shared-memory tile so that both the reads
// (along k) and the writes (along g) are coalesced.
// Blocks outside `mask` (PHX_P_*) are not read: they are written as zeros, or left as they are when accumulating.
__global__ void unpack_w1_kernel(int G, int H, int Hp, int K2, const float* __restrict__ w1bar, int nparts, size_t pstride,
                                 float* __restrict__ Ws, float* __restrict__ Wp, int accumulate, int mask) {
    __shared__ float tile[32][33];
    const int g0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int g = g0 + r, k = k0 + threadIdx.x;
        float t = 0.f;
        if (g < G && k < K2 && (mask & (k >= Hp ? PHX_P_WP : PHX_P_WS)))
            for (int q = 0; q < nparts; ++q) t += w1bar[q * pstride + (size_t)g * K2 + k];   // fixed order over the parts
        tile[r][threadIdx.x] = t;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int k = k0 + r, g = g0 + threadIdx.x;
        if (g >= G || k >= K2) continue;
        const int half = k >= Hp, h = half ? k - Hp : k;
        if (h >= H) continue;
        float* dst = (half ? Wp : Ws) + (size_t)h * G + g;
        const float v = tile[threadIdx.x][r];
        if (!(mask & (half ? PHX_P_WP : PHX_P_WS))) {
            if (!accumulate) *dst = 0.f;
            continue;
        }
        *dst = accumulate ? *dst + v : v;
    }
}
// cotangent of the data loss of training_step (train_insilico.py:132, torch.mean((predictions - targets)**2)):
// grad[r][g] = scale * (pred[r][g] - target[r][g]), rows of pred / grad `stride` floats apart (the t1 slices of [N][T][G])
__global__ void mse_grad_kernel(int rows, int G, const float* __restrict__ pred, size_t pred_stride,
                                const float* __restrict__ target, float scale, float* __restrict__ grad,
                                size_t grad_stride) {
    const size_t n = (size_t)rows * G, step = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        const size_t r = i / G, g = i - r * G;
        grad[r * grad_stride + g] = scale * (pred[r * pred_stride + g] - target[i]);
    }
}
__global__ void unpack_rest_kernel(int G, int H, int Hp, int K2, const float* __restrict__ wabar,
                                   const float* __restrict__ biasbar, const float* __restrict__ mbar, int nparts,
                                   size_t pstride, float* __restrict__ Wa, float* __restrict__ bs,
                                   float* __restrict__ bp, float* __restrict__ m, int accumulate, int mask) {
    auto psum = [&](const float* base, size_t i) {
        float t = 0.f;
        for (int q = 0; q < nparts; ++q) t += base[q * pstride + i];
        return t;
    };
    // a block outside `mask` is not read: zeros, or left as it is when accumulating
    auto put = [&](float* dst, int bit, const float* base, size_t i) {
        if (mask & bit) {
            const float v = psum(base, i);
            *dst = accumulate ? *dst + v : v;
        } else if (!accumulate) {
            *dst = 0.f;
        }
    };
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t n = (size_t)G * 2 * H;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const size_t g = i / (2 * H);
        const int kk = (int)(i - g * 2 * H);
        put(Wa + i, PHX_P_WA, wabar, g * K2 + (kk < H ? kk : Hp + kk - H));
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)H; i += stride) {
        put(bs + i, PHX_P_BS, biasbar, i);
        put(bp + i, PHX_P_BP, biasbar, Hp + i);
    }
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)G; i += stride) put(m + i, PHX_P_M, mbar, i);
}

bool check_mask(int mask) {
    if (mask < 0 || mask > PHX_P_ALL) {
        phx_set_error("param_mask must be a 6-bit mask (0 .. 0x3F), got %d", mask);
        return false;
    }
    return true;
}

// the adjoint solves also take PHX_NORM_SEMINORM
bool check_adjoint_mask(int mask) {
    if (mask < 0 || mask > (PHX_P_ALL | PHX_NORM_SEMINORM)) {
        phx_set_error("param_mask must be a 6-bit mask, optionally with PHX_NORM_SEMINORM (0 .. 0x7F), got %d", mask);
        return false;
    }
    return true;
}

bool check_dims(int G, int H, int B) {
    if (G < 1 || H < 1 || B < 1) {
        phx_set_error("invalid dims G=%d H=%d B=%d", G, H, B);
        return false;
    }
    return true;
}

// ---- fixed-grid step grids (the *_grid entry points) -----------------------------------------------------------------
// the grid goes to the workspace right after the solver's own part, 16-byte aligned
size_t grid_room(size_t need) { return (need + 15) & ~(size_t)15; }

// total steps of a grid (for the workspace check; a negative count is refused by phx_grid_stage afterwards)
long long grid_steps(const PhxGridHost& g, int N, int T, int adjoint) {
    const long long nseg = adjoint ? (long long)N * (T - 1) : N;
    long long tot = 0;
    if (g.steps)
        for (long long q = 0; q < nseg; ++q) tot += g.steps[q] > 0 ? g.steps[q] : 0;
    return tot;
}

}  // namespace

int phx_grid_stage(const PhxGridHost& g, int N, int T, int method, int forward, void* room, cudaStream_t stream,
                   ResParams* p, std::vector<int>* off) {
    if (method == PHX_DOPRI5 || method < PHX_EULER || method > PHX_DOPRI5) {
        phx_set_error("a step grid is for the fixed-grid methods (euler, midpoint, rk4), got method id %d", method);
        return PHX_ERR_INVALID;
    }
    if (!g.dt || !g.steps || (forward && (!g.out_step || !g.out_slope))) {
        phx_set_error("null grid array");
        return PHX_ERR_INVALID;
    }
    const int nseg = forward ? N : N * (T - 1), nout = forward ? N * (T - 1) : 0;
    std::vector<int> o(nseg + 1, 0);
    for (int q = 0; q < nseg; ++q) {
        if (g.steps[q] < 1 || (long long)o[q] + g.steps[q] > (1LL << 30)) {
            phx_set_error("grid segment %d: step count %d out of range", q, g.steps[q]);
            return PHX_ERR_INVALID;
        }
        o[q + 1] = o[q] + g.steps[q];
    }
    for (int k = 0; k < o[nseg]; ++k)
        if (!(g.dt[k] >= 0.f) || isinf(g.dt[k])) {
            phx_set_error("grid step %d: dt %g is not a finite non-negative number", k, (double)g.dt[k]);
            return PHX_ERR_INVALID;
        }
    for (int q = 0; q < N && forward; ++q)
        for (int j = 0; j + 1 < T; ++j) {
            const int k = g.out_step[q * (T - 1) + j];
            if (k < 0 || k >= g.steps[q] || (j > 0 && k < g.out_step[q * (T - 1) + j - 1])) {
                phx_set_error("problem %d, output %d: step %d is out of range or the output map decreases", q, j + 1, k);
                return PHX_ERR_INVALID;
            }
            if (isnan(g.out_slope[q * (T - 1) + j])) {
                phx_set_error("problem %d, output %d: the slope is NaN", q, j + 1);
                return PHX_ERR_INVALID;
            }
        }
    if (off) *off = o;
    if (!room) return PHX_OK;
    // one copy: dt | goff | gout | gsl, each part padded to 16 bytes
    auto pad = [](size_t n) { return (n + 3) & ~(size_t)3; };
    const size_t n_dt = pad(o[nseg]), n_off = pad(nseg + 1), n_out = pad(nout);
    std::vector<uint32_t> buf(n_dt + n_off + 2 * n_out, 0);
    memcpy(buf.data(), g.dt, sizeof(float) * o[nseg]);
    memcpy(buf.data() + n_dt, o.data(), sizeof(int) * (nseg + 1));
    if (nout) {
        memcpy(buf.data() + n_dt + n_off, g.out_step, sizeof(int) * nout);
        memcpy(buf.data() + n_dt + n_off + n_out, g.out_slope, sizeof(float) * nout);
    }
    cudaError_t e = cudaMemcpyAsync(room, buf.data(), sizeof(uint32_t) * buf.size(), cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) {
        phx_set_error("cudaMemcpyAsync(grid): %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    const uint32_t* d = (const uint32_t*)room;
    p->gdt = (const float*)d;
    p->goff = (const int*)(d + n_dt);
    p->gout = nout ? (const int*)(d + n_dt + n_off) : nullptr;
    p->gsl = nout ? (const float*)(d + n_dt + n_off + n_out) : nullptr;
    return PHX_OK;
}

int phx_tc_prepare(phx_ctx* ctx, int G, int H, int B, const float* packed, PhxPacked* view, cudaStream_t stream) {
    *view = phx_packed_view(packed, G, H);
    if (!ctx || ctx->precision == PHX_PREC_FP32 || !phx_tc_shape_ok(H, B)) return PHX_OK;
    if ((uintptr_t)packed & 127) {
        phx_set_error("packed weights must be 128-byte aligned for the tensor-core path");
        return PHX_ERR_INVALID;
    }
    bool stale;
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        auto it = ctx->tc_valid.find(packed);
        stale = (it == ctx->tc_valid.end()) || it->second == 0;
        ctx->tc_valid[packed] = 1;
    }
    if (stale) {
        int rc = phx_tc_pack_launch(G, H, *view, stream);
        if (rc != PHX_OK) return rc;
    }
    view->tc = ctx->precision == PHX_PREC_TF32 ? 1 : 3;
    return PHX_OK;
}

extern "C" {

const char* phx_last_error(void) { return g_err; }

int phx_ctx_create(int device, phx_ctx** out) {
    if (!out) return PHX_ERR_INVALID;
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) {
        phx_set_error("cudaGetDeviceProperties(%d): %s", device, cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    if (prop.major < 10) {
        phx_set_error("phoenix_b200 needs an sm_100a (B200) device; device %d is sm_%d%d", device, prop.major,
                      prop.minor);
        return PHX_ERR_UNSUPPORTED;
    }
    phx_ctx* c = new phx_ctx;
    c->device = device;
    c->num_sms = prop.multiProcessorCount;
    c->coop = prop.cooperativeLaunch;
    c->prof = nullptr;
    c->precision = PHX_PREC_3XTF32;
    c->sum_hook = nullptr;
    c->sum_user = nullptr;
    c->sum_world = 1;
    if (const char* e = getenv("PHX_PRECISION")) c->precision = atoi(e);
    if (!c->coop) {
        delete c;
        phx_set_error("device %d does not support cooperative launch", device);
        return PHX_ERR_UNSUPPORTED;
    }
    *out = c;
    return PHX_OK;
}

void phx_ctx_destroy(phx_ctx* ctx) { delete ctx; }

int phx_ctx_num_sms(const phx_ctx* ctx) { return ctx ? ctx->num_sms : 0; }
}  // extern "C"
int phx_ctx_device(const phx_ctx* ctx) { return ctx ? ctx->device : 0; }
int phx_ctx_sum_hook(const phx_ctx* ctx, phx_sum_hook* hook, void** user) {
    if (!ctx || !ctx->sum_hook) return 1;
    *hook = ctx->sum_hook;
    *user = ctx->sum_user;
    return ctx->sum_world;
}
extern "C" {

int phx_ctx_set_profile(phx_ctx* ctx, void* slots) {
    if (!ctx) return PHX_ERR_INVALID;
    ctx->prof = (long long*)slots;
    return PHX_OK;
}
int phx_profile_slots(void) { return PHX_PROF_SLOTS; }

int phx_resident_max_rows(int adjoint) { return adjoint ? PHX_MAX_B_ADJ : PHX_MAX_B_FWD; }

int phx_plan_describe(int num_sms, int G, int H, int B, int adjoint, int32_t out[8]) {
    ResLaunchPlan plan;
    if (!out || !check_dims(G, H, B)) return PHX_ERR_INVALID;
    int rc = phx_resident_plan(num_sms, G, H, B, adjoint, &plan);
    if (rc != PHX_OK) return rc;
    out[0] = plan.nCTA; out[1] = plan.gpc; out[2] = plan.NV; out[3] = plan.w1_res; out[4] = plan.wa_res;
    out[5] = plan.ring_rows; out[6] = plan.ring_stages; out[7] = (int32_t)plan.smem_bytes;
    return PHX_OK;
}

int phx_ctx_set_precision(phx_ctx* ctx, int precision) {
    if (!ctx || (precision != PHX_PREC_FP32 && precision != PHX_PREC_3XTF32 && precision != PHX_PREC_TF32)) {
        phx_set_error("set_precision: unknown mode %d", precision);
        return PHX_ERR_INVALID;
    }
    ctx->precision = precision;
    return PHX_OK;
}
int phx_ctx_get_precision(const phx_ctx* ctx) { return ctx ? ctx->precision : PHX_ERR_INVALID; }
int phx_ctx_set_global_norm(phx_ctx* ctx, phx_sum_hook hook, void* user, int world_size) {
    if (!ctx || world_size < 1) return PHX_ERR_INVALID;
    ctx->sum_hook = hook;
    ctx->sum_user = user;
    ctx->sum_world = hook ? world_size : 1;
    return PHX_OK;
}
int phx_tc_min_rows(void) { return phx_tc_min_rows_rt(); }

int phx_tc_plan_describe(int K, int M, int32_t out[6]) {
    if (!out || K < 1 || M < 1) return PHX_ERR_INVALID;
    const PhxTcBranchPlan pl = phx_tc_branch_plan(K, M);
    out[0] = pl.mtiles; out[1] = pl.ks_p; out[2] = pl.per_p; out[3] = pl.ks_s; out[4] = pl.per_s; out[5] = pl.slots;
    return PHX_OK;
}

size_t phx_packed_bytes(int G, int H) { return phx_packed_floats(G, H) * sizeof(float); }

int phx_pack_weights(phx_ctx* ctx, int G, int H, const float* m, const float* Wp, const float* bp, const float* Ws,
                     const float* bs, const float* Wa, float* packed, void* stream) {
    PhxDevGuard dev_guard(ctx);
    if (!ctx || !check_dims(G, H, 1) || !m || !Wp || !bp || !Ws || !bs || !Wa || !packed) return PHX_ERR_INVALID;
    const int Hp = phx_Hp(H), K2 = 2 * Hp;
    PhxPacked v = phx_packed_view(packed, G, H);
    pack_kernel<<<ctx->num_sms * 4, 256, 0, (cudaStream_t)stream>>>(
        G, H, Hp, K2, m, Wp, bp, Ws, bs, Wa, (float*)v.W1, (float*)v.WA, (float*)v.bias, (float*)v.relum,
        (float*)v.maskm);
    {
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->tc_valid[packed] = 0;   // the tensor-core operand images are rebuilt lazily by the first large-B call
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("pack_weights launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

size_t phx_rhs_workspace_bytes(int G, int H, int B) { return phx_rhs_workspace_floats(G, H, B) * sizeof(float); }

int phx_rhs_forward(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y, float* f, int decay,
                    void* workspace, size_t workspace_bytes, void* stream) {
    PhxDevGuard dev_guard(ctx);
    if (!ctx || !check_dims(G, H, B) || !packed || !y || !f || !workspace) return PHX_ERR_INVALID;
    if (workspace_bytes < phx_rhs_workspace_bytes(G, H, B)) {
        phx_set_error("rhs workspace too small: %zu < %zu", workspace_bytes, phx_rhs_workspace_bytes(G, H, B));
        return PHX_ERR_WORKSPACE;
    }
    PhxPacked w;
    int rc = phx_tc_prepare(ctx, G, H, B, packed, &w, (cudaStream_t)stream);
    if (rc != PHX_OK) return rc;
    return phx_rhs_forward_launch(G, H, B, w, y, f, decay, 1.f, (float*)workspace, (cudaStream_t)stream);
}

int phx_rhs_vjp(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y, const float* g, int decay,
                float* ybar, float* grads_flat, int accumulate, void* workspace, size_t workspace_bytes,
                void* stream) {
    PhxDevGuard dev_guard(ctx);
    if (!ctx || !check_dims(G, H, B) || !packed || !y || !g || !workspace) return PHX_ERR_INVALID;
    if (workspace_bytes < phx_rhs_workspace_bytes(G, H, B)) {
        phx_set_error("rhs workspace too small: %zu < %zu", workspace_bytes, phx_rhs_workspace_bytes(G, H, B));
        return PHX_ERR_WORKSPACE;
    }
    PhxPacked w;
    int rc = phx_tc_prepare(ctx, G, H, B, packed, &w, (cudaStream_t)stream);
    if (rc != PHX_OK) return rc;
    return phx_rhs_vjp_launch(G, H, B, w, y, g, decay, ybar, grads_flat, accumulate, nullptr, 1.f, (float*)workspace,
                              (cudaStream_t)stream);
}

int phx_prior_loss(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* x, const float* prior_grad,
                   float scale, float* gcot, float* loss, void* workspace, size_t workspace_bytes, void* stream) {
    PhxDevGuard dev_guard(ctx);
    if (!ctx || !check_dims(G, H, B) || !packed || !x || !prior_grad || !gcot || !loss || !workspace) return PHX_ERR_INVALID;
    if (workspace_bytes < phx_rhs_workspace_bytes(G, H, B)) {
        phx_set_error("rhs workspace too small: %zu < %zu", workspace_bytes, phx_rhs_workspace_bytes(G, H, B));
        return PHX_ERR_WORKSPACE;
    }
    PhxPacked w;
    int rc = phx_tc_prepare(ctx, G, H, B, packed, &w, (cudaStream_t)stream);
    if (rc != PHX_OK) return rc;
    return phx_prior_loss_launch(G, H, B, w, x, prior_grad, scale, gcot, loss, (float*)workspace, (cudaStream_t)stream);
}

int phx_prior_setup(phx_ctx* ctx, int G, int B, const float* x, const int32_t* colptr, const int32_t* rowidx,
                    const float* val, float* out, void* stream) {
    PhxDevGuard dev_guard(ctx);
    if (!ctx || G < 1 || B < 1 || !x || !colptr || !rowidx || !val || !out) return PHX_ERR_INVALID;
    return phx_prior_setup_launch(G, B, x, colptr, rowidx, val, out, (cudaStream_t)stream);
}

size_t phx_solve_workspace_bytes(const phx_ctx* ctx, int G, int H, int B, int T, int adjoint) {
    if (!ctx) return 0;
    ResLaunchPlan plan;
    if (phx_resident_plan(ctx->num_sms, G, H, B, adjoint, &plan) != PHX_OK) return 0;
    return phx_resident_workspace_floats(G, H, B, T, adjoint, nullptr, nullptr) * sizeof(float);
}

size_t phx_solve_workspace_init_bytes(void) { return phx_ll_words() * sizeof(unsigned long long); }

int phx_solve_workspace_init(void* workspace, size_t workspace_bytes, void* stream) {
    const size_t need = phx_solve_workspace_init_bytes();
    if (!workspace || workspace_bytes < need) {
        phx_set_error("workspace_init: workspace smaller than the %zu-byte exchange area", need);
        return PHX_ERR_WORKSPACE;
    }
    cudaError_t e = cudaMemsetAsync(workspace, 0, need, (cudaStream_t)stream);
    if (e != cudaSuccess) {
        phx_set_error("cudaMemsetAsync(workspace): %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

static int solve_common(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                        int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps, int adjoint,
                        void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                        int steplog_cap, cudaStream_t stream, ResParams* p, ResLaunchPlan* plan, int nprob = 1,
                        const PhxGridHost* grid = nullptr) {
    if (!ctx || !check_dims(G, H, B) || !packed || !t_host || !workspace) {
        if (g_err[0] == 0) phx_set_error("null argument");
        return PHX_ERR_INVALID;
    }
    if (T < 2) {
        phx_set_error("t must hold at least two time points (got %d)", T);
        return PHX_ERR_INVALID;
    }
    if (nprob < 1 || (nprob > 1 && nprob * T > PHX_T_INLINE)) {
        phx_set_error("a multi-problem launch takes 1 <= N and N * T <= %d output times (got N=%d, T=%d)", PHX_T_INLINE,
                      nprob, T);
        return PHX_ERR_INVALID;
    }
    for (int q = 0; q < nprob; ++q)
        for (int i = 1; i < T; ++i) {
            if (!(t_host[q * T + i] > t_host[q * T + i - 1])) {
                phx_set_error("t must be strictly increasing at the C boundary (the Python shim negates decreasing t)");
                return PHX_ERR_INVALID;
            }
        }
    if (method < PHX_EULER || method > PHX_DOPRI5) {
        phx_set_error("unknown method id %d", method);
        return PHX_ERR_INVALID;
    }
    if (((uintptr_t)workspace & 15) || ((uintptr_t)packed & 15)) {
        phx_set_error("workspace and packed weights must be 16-byte aligned");
        return PHX_ERR_INVALID;
    }
    int rc = phx_resident_plan(ctx->num_sms, G, H, B, adjoint, plan);
    if (rc != PHX_OK) return rc;
    size_t o_t, o_th;
    size_t need = phx_resident_workspace_floats(G, H, B, T, adjoint, &o_t, &o_th) * sizeof(float);
    const size_t need_grid = grid ? grid_room(need) + phx_grid_workspace_bytes(nprob, T, grid_steps(*grid, nprob, T, adjoint)) : need;
    if (workspace_bytes < need_grid) {
        phx_set_error("solve workspace too small: %zu < %zu", workspace_bytes, need_grid);
        return PHX_ERR_WORKSPACE;
    }
    float* ws = (float*)workspace;
    memset(p, 0, sizeof(*p));
    p->G = G; p->H = H; p->Hp = phx_Hp(H); p->K2 = 2 * p->Hp; p->K2q = p->K2 / 4; p->B = B; p->T = T;
    p->method = method; p->gpc = plan->gpc; p->t_is_f32 = t_is_f32; p->adjoint = adjoint;
    p->ring_rows = plan->ring_rows; p->ring_stages = plan->ring_stages;
    p->so = plan->so;
    p->rtol_f = (float)rtol; p->atol_f = (float)atol; p->fsign = 1.f;
    p->max_steps = (long long)max_num_steps;
    p->w = phx_packed_view(packed, G, H);
    p->ll = phx_ll_view(workspace);
    p->t = (const double*)(ws + o_t);
    p->theta1 = adjoint ? ws + o_th : nullptr;
    p->status = status; p->steplog = steplog; p->steplog_cap = steplog ? steplog_cap : 0;
    p->prof = ctx->prof;
    p->nprob = nprob;
    if (grid && (rc = phx_grid_stage(*grid, nprob, T, method, !adjoint, (char*)workspace + grid_room(need), stream, p,
                                     nullptr)) != PHX_OK)
        return rc;
    if (T * nprob <= PHX_T_INLINE) {
        for (int i = 0; i < T * nprob; ++i) p->t_small[i] = t_host[i];  // travels with the kernel parameters
        return PHX_OK;
    }
    cudaError_t e = cudaMemcpyAsync((void*)p->t, t_host, sizeof(double) * T, cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) {
        phx_set_error("cudaMemcpyAsync(t): %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

int phx_solve_forward(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y0,
                      const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol, double atol,
                      int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                      phx_status* status, double* steplog, int steplog_cap, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!y0 || !y_out) {
        phx_set_error("null y0 / y_out");
        return PHX_ERR_INVALID;
    }
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 0, workspace,
                          workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan);
    if (rc != PHX_OK) return rc;
    p.y0 = y0;
    p.yout = y_out;
    p.fsign = reversed ? -1.f : 1.f;
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}

int phx_solve_adjoint(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                      int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                      const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat, void* workspace,
                      size_t workspace_bytes, phx_status* status, double* steplog, int steplog_cap, void* stream) {
    return phx_solve_adjoint_masked(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, y_saved,
                                    grad_y, adj_y0, grads_flat, workspace, workspace_bytes, status, steplog, steplog_cap,
                                    PHX_P_ALL, stream);
}

int phx_solve_adjoint_masked(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                             int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                             const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat, void* workspace,
                             size_t workspace_bytes, phx_status* status, double* steplog, int steplog_cap,
                             int param_mask, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!check_adjoint_mask(param_mask)) return PHX_ERR_INVALID;
    if (!y_saved || !grad_y || !adj_y0 || !grads_flat) {
        phx_set_error("null y_saved / grad_y / adj_y0 / grads_flat");
        return PHX_ERR_INVALID;
    }
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 1, workspace,
                          workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan);
    if (rc != PHX_OK) return rc;
    p.ysaved = y_saved;
    p.grad_y = grad_y;
    p.adj_y0 = adj_y0;
    p.theta0 = grads_flat;  // written once by the kernel (never read while still zero): no memset needed
    p.pmask = param_mask;
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}

/* ---- several independent problems per launch (SURVEY.md section 8 f1) -------------------------------------------- */
int phx_solve_forward_many(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const float* y0,
                           const double* t_host, int T, int t_is_f32, int method, double rtol, double atol,
                           int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                           phx_status* status, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!y0 || !y_out) {
        phx_set_error("null y0 / y_out");
        return PHX_ERR_INVALID;
    }
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 0, workspace,
                          workspace_bytes, status, nullptr, 0, (cudaStream_t)stream, &p, &plan, N);
    if (rc != PHX_OK) return rc;
    p.y0 = y0;
    p.yout = y_out;
    p.y0_stride = (long long)B * G;
    p.yout_stride = (long long)T * B * G;
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}

int phx_solve_adjoint_many(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const double* t_host, int T,
                           int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                           const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                           void* workspace, size_t workspace_bytes, phx_status* status, void* stream) {
    return phx_solve_adjoint_many_masked(ctx, G, H, B, N, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps,
                                         y_saved, grad_y, adj_y0, grads_flat, workspace, workspace_bytes, status, PHX_P_ALL,
                                         stream);
}

int phx_solve_adjoint_many_masked(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const double* t_host,
                                  int T, int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                                  const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                                  void* workspace, size_t workspace_bytes, phx_status* status, int param_mask,
                                  void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!check_adjoint_mask(param_mask)) return PHX_ERR_INVALID;
    if (!y_saved || !grad_y || !adj_y0 || !grads_flat) {
        phx_set_error("null y_saved / grad_y / adj_y0 / grads_flat");
        return PHX_ERR_INVALID;
    }
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 1, workspace,
                          workspace_bytes, status, nullptr, 0, (cudaStream_t)stream, &p, &plan, N);
    if (rc != PHX_OK) return rc;
    p.ysaved = y_saved;
    p.grad_y = grad_y;
    p.adj_y0 = adj_y0;
    p.theta0 = grads_flat;
    p.yout_stride = (long long)T * B * G;
    p.adj_stride = (long long)B * G;
    p.theta_stride = (long long)phx_grad_offsets(G, H).total;
    p.pmask = param_mask;
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}


/* ---- rows kernels: N independent one-row problems in lock-step (phx_rows.cuh) ------------------------------------------- */
static int rows_common(phx_ctx* ctx, int G, int H, int N, const float* packed, const double* t_host, int T, int t_is_f32,
                       int method, double rtol, double atol, int64_t max_num_steps, int adjoint, void* workspace,
                       size_t workspace_bytes, phx_status* status, double* steplog, int steplog_cap, cudaStream_t stream,
                       ResParams* p, RowsPlan* plan, size_t* off_theta, const PhxGridHost* grid = nullptr) {
    if (!ctx || !check_dims(G, H, 1) || !packed || !t_host || !workspace || N < 1) {
        if (g_err[0] == 0) phx_set_error("null argument");
        return PHX_ERR_INVALID;
    }
    if (T < 2) {
        phx_set_error("t must hold at least two time points (got %d)", T);
        return PHX_ERR_INVALID;
    }
    for (int q = 0; q < N; ++q)
        for (int i = 1; i < T; ++i)
            if (!(t_host[q * T + i] > t_host[q * T + i - 1])) {
                phx_set_error("t must be strictly increasing at the C boundary (the Python shim negates decreasing t)");
                return PHX_ERR_INVALID;
            }
    if (method < PHX_EULER || method > PHX_DOPRI5) {
        phx_set_error("unknown method id %d", method);
        return PHX_ERR_INVALID;
    }
    if (((uintptr_t)workspace & 127) || ((uintptr_t)packed & 15)) {
        phx_set_error("workspace must be 128-byte and packed weights 16-byte aligned");
        return PHX_ERR_INVALID;
    }
    int rc = phx_rows_plan(ctx->num_sms, G, H, adjoint, plan);
    if (rc != PHX_OK) return rc;
    size_t o_t;
    const size_t need = phx_rows_workspace_floats(G, H, N, T, plan->rows, adjoint, &o_t, off_theta) * sizeof(float);
    const size_t need_grid = grid ? grid_room(need) + phx_grid_workspace_bytes(N, T, grid_steps(*grid, N, T, adjoint)) : need;
    if (workspace_bytes < need_grid) {
        phx_set_error("rows workspace too small: %zu < %zu", workspace_bytes, need_grid);
        return PHX_ERR_WORKSPACE;
    }
    float* ws = (float*)workspace;
    memset(p, 0, sizeof(*p));
    p->G = G; p->H = H; p->Hp = phx_Hp(H); p->K2 = 2 * p->Hp; p->K2q = p->K2 / 4; p->B = 1; p->T = T;
    p->method = method; p->gpc = plan->gpc; p->t_is_f32 = t_is_f32; p->adjoint = adjoint;
    p->ring_rows = plan->w1_stride_q;   // rows kernels: W1 row stride in shared memory (float4 units)
    p->ring_stages = 0;
    p->so = plan->so;
    p->rtol_f = (float)rtol; p->atol_f = (float)atol; p->fsign = 1.f;
    p->max_steps = (long long)max_num_steps;
    p->w = phx_packed_view(packed, G, H);
    p->ll = phx_ll_view(workspace);
    p->t = (const double*)(ws + o_t);
    p->status = status; p->steplog = steplog; p->steplog_cap = steplog ? steplog_cap : 0;
    p->prof = ctx->prof;
    p->nprob = 1;
    p->rows = plan->rows; p->ntot = N; p->nqw = plan->nqw; p->ngg = plan->ngg; p->gpg = plan->gpg;
    p->tm_wa = plan->tm_wa; p->tm_fac = plan->tm_fac;
    p->y0_stride = G; p->yout_stride = (long long)T * G; p->adj_stride = G;
    p->ppk = (long long)phx_packed_grad_offsets(G, H).total;
    if (grid && (rc = phx_grid_stage(*grid, N, T, method, !adjoint, (char*)workspace + grid_room(need), stream, p,
                                     nullptr)) != PHX_OK)
        return rc;
    if ((size_t)T * N <= PHX_T_INLINE) {
        for (int i = 0; i < T * N; ++i) p->t_small[i] = t_host[i];
        return PHX_OK;
    }
    cudaError_t e = cudaMemcpyAsync((void*)p->t, t_host, sizeof(double) * T * N, cudaMemcpyHostToDevice, stream);
    if (e != cudaSuccess) {
        phx_set_error("cudaMemcpyAsync(t): %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

int phx_rows_supported(const phx_ctx* ctx, int G, int H, int adjoint) {
    if (!ctx) return 0;
    RowsPlan plan;
    return phx_rows_plan(ctx->num_sms, G, H, adjoint, &plan) == PHX_OK ? plan.rows : 0;
}

int phx_rows_plan_describe(int num_sms, int G, int H, int adjoint, int32_t out[10]) {
    RowsPlan plan;
    if (!out || !check_dims(G, H, 1)) return PHX_ERR_INVALID;
    int rc = phx_rows_plan(num_sms, G, H, adjoint, &plan);
    if (rc != PHX_OK) return rc;
    out[0] = plan.nCTA; out[1] = plan.gpc; out[2] = plan.nqw; out[3] = plan.ngg; out[4] = plan.gpg;
    out[5] = plan.wa_res; out[6] = plan.rows; out[7] = plan.w1_stride_q;
    out[8] = plan.tm_wa + (adjoint ? 2 * PHX_ROWS_NFS * 4 * plan.rows : 0);
    out[9] = (int32_t)plan.smem_bytes;
    return PHX_OK;
}

size_t phx_rows_workspace_bytes(const phx_ctx* ctx, int G, int H, int N, int T, int adjoint) {
    if (!ctx || N < 1 || T < 2) return 0;
    RowsPlan plan;
    if (phx_rows_plan(ctx->num_sms, G, H, adjoint, &plan) != PHX_OK) return 0;
    return phx_rows_workspace_floats(G, H, N, T, plan.rows, adjoint, nullptr, nullptr) * sizeof(float);
}

int phx_solve_forward_rows(phx_ctx* ctx, int G, int H, int N, const float* packed, const float* y0, const double* t_host,
                           int T, int t_is_f32, int reversed, int method, double rtol, double atol, int64_t max_num_steps,
                           float* y_out, void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                           int steplog_cap, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!y0 || !y_out) {
        phx_set_error("null y0 / y_out");
        return PHX_ERR_INVALID;
    }
    ResParams p;
    RowsPlan plan;
    int rc = rows_common(ctx, G, H, N, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 0, workspace,
                         workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan, nullptr);
    if (rc != PHX_OK) return rc;
    p.y0 = y0;
    p.yout = y_out;
    p.fsign = reversed ? -1.f : 1.f;
    return phx_rows_launch(p, plan, (cudaStream_t)stream);
}

int phx_rows_grad_parts(const phx_ctx* ctx, int G, int H, int N) {
    if (!ctx || N < 1) return 0;
    RowsPlan plan;
    if (phx_rows_plan(ctx->num_sms, G, H, 1, &plan) != PHX_OK) return 0;
    return (N + plan.rows - 1) / plan.rows;
}

int phx_unpack_grads(phx_ctx* ctx, int G, int H, const float* packed_grads, int nparts, float* grads_flat,
                     int accumulate, void* stream) {
    return phx_unpack_grads_masked(ctx, G, H, packed_grads, nparts, grads_flat, accumulate, PHX_P_ALL, stream);
}

int phx_unpack_grads_masked(phx_ctx* ctx, int G, int H, const float* packed_grads, int nparts, float* grads_flat,
                            int accumulate, int param_mask, void* stream) {
    PhxDevGuard dev_guard(ctx);
    if (!ctx || !check_dims(G, H, 1) || !packed_grads || !grads_flat || nparts < 1 || !check_mask(param_mask))
        return PHX_ERR_INVALID;
    const int Hp = phx_Hp(H), K2 = 2 * Hp;
    const PhxPackedGradOff po = phx_packed_grad_offsets(G, H);
    const PhxGradOff fo = phx_grad_offsets(G, H);
    dim3 grid((G + 31) / 32, (K2 + 31) / 32), block(32, 8);
    unpack_w1_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(G, H, Hp, K2, packed_grads + po.W1, nparts, po.total,
                                                               grads_flat + fo.Ws, grads_flat + fo.Wp, accumulate,
                                                               param_mask);
    unpack_rest_kernel<<<ctx->num_sms * 4, 256, 0, (cudaStream_t)stream>>>(
        G, H, Hp, K2, packed_grads + po.WA, packed_grads + po.bias, packed_grads + po.m, nparts, po.total,
        grads_flat + fo.Wa, grads_flat + fo.bs, grads_flat + fo.bp, grads_flat + fo.m, accumulate, param_mask);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("unpack_grads launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

size_t phx_packed_grad_bytes(int G, int H) { return phx_packed_grad_offsets(G, H).total * sizeof(float); }

int phx_mse_grad(phx_ctx* ctx, int rows, int G, const float* pred, size_t pred_stride, const float* target, float scale,
                 float* grad, size_t grad_stride, void* stream) {
    if (!ctx || rows < 1 || G < 1 || !pred || !target || !grad) {
        phx_set_error("mse_grad: invalid argument");
        return PHX_ERR_INVALID;
    }
    PhxDevGuard dev_guard(ctx);
    const size_t n = (size_t)rows * G;
    int blocks = (int)((n + 255) / 256);
    if (blocks > ctx->num_sms * 8) blocks = ctx->num_sms * 8;
    mse_grad_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(rows, G, pred, pred_stride, target, scale, grad, grad_stride);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        phx_set_error("mse_grad launch: %s", cudaGetErrorString(e));
        return PHX_ERR_CUDA;
    }
    return PHX_OK;
}

int phx_solve_adjoint_rows(phx_ctx* ctx, int G, int H, int N, const float* packed, const double* t_host, int T,
                           int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                           const float* y_saved, const float* grad_y, float* adj_y0, float* grads_packed_parts,
                           void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                           int steplog_cap, void* stream) {
    return phx_solve_adjoint_rows_masked(ctx, G, H, N, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps,
                                         y_saved, grad_y, adj_y0, grads_packed_parts, workspace, workspace_bytes, status,
                                         steplog, steplog_cap, PHX_P_ALL, stream);
}

int phx_solve_adjoint_rows_masked(phx_ctx* ctx, int G, int H, int N, const float* packed, const double* t_host, int T,
                                  int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                                  const float* y_saved, const float* grad_y, float* adj_y0, float* grads_packed_parts,
                                  void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                                  int steplog_cap, int param_mask, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!check_adjoint_mask(param_mask)) return PHX_ERR_INVALID;
    if (!y_saved || !grad_y || !adj_y0 || !grads_packed_parts) {
        phx_set_error("null y_saved / grad_y / adj_y0 / grads_packed_parts");
        return PHX_ERR_INVALID;
    }
    if ((uintptr_t)grads_packed_parts & 15) {
        phx_set_error("grads_packed_parts must be 16-byte aligned");
        return PHX_ERR_INVALID;
    }
    ResParams p;
    RowsPlan plan;
    size_t o_th = 0;
    int rc = rows_common(ctx, G, H, N, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 1, workspace,
                         workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan, &o_th);
    if (rc != PHX_OK) return rc;
    p.ysaved = y_saved;
    p.grad_y = grad_y;
    p.adj_y0 = adj_y0;
    p.theta_ws = (float*)workspace + o_th;
    p.gsum = grads_packed_parts;
    p.gsum_acc = 0;
    p.pmask = param_mask;
    return phx_rows_launch(p, plan, (cudaStream_t)stream);
}


/* ---- fixed-grid solves on the caller's step grid (options=dict(step_size=...), solvers.py:48-50, 77-103) ---------------- */
size_t phx_grid_workspace_bytes(int N, int T, int64_t total_steps) {
    if (N < 1 || T < 2 || total_steps < 0) return 0;
    const size_t nseg = (size_t)N * (T - 1);
    return 4 * (((size_t)total_steps + 3) / 4 * 4 + (nseg + 4) / 4 * 4 + 2 * ((nseg + 3) / 4 * 4)) + 16;
}

int phx_solve_forward_grid(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y0, const double* t_host,
                           int T, int t_is_f32, int reversed, int method, double rtol, double atol, int64_t max_num_steps,
                           float* y_out, void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                           int steplog_cap, const float* grid_dt, const int32_t* grid_steps_, const int32_t* grid_out_step,
                           const float* grid_out_slope, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!y0 || !y_out) {
        phx_set_error("null y0 / y_out");
        return PHX_ERR_INVALID;
    }
    const PhxGridHost grid{grid_dt, grid_steps_, grid_out_step, grid_out_slope};
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 0, workspace,
                          workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan, 1, &grid);
    if (rc != PHX_OK) return rc;
    p.y0 = y0;
    p.yout = y_out;
    p.fsign = reversed ? -1.f : 1.f;
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}

int phx_solve_adjoint_grid(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                           int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                           const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat, void* workspace,
                           size_t workspace_bytes, phx_status* status, double* steplog, int steplog_cap, int param_mask,
                           const float* grid_dt, const int32_t* grid_steps_, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!check_adjoint_mask(param_mask)) return PHX_ERR_INVALID;
    if (!y_saved || !grad_y || !adj_y0 || !grads_flat) {
        phx_set_error("null y_saved / grad_y / adj_y0 / grads_flat");
        return PHX_ERR_INVALID;
    }
    const PhxGridHost grid{grid_dt, grid_steps_, nullptr, nullptr};
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 1, workspace,
                          workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan, 1, &grid);
    if (rc != PHX_OK) return rc;
    p.ysaved = y_saved;
    p.grad_y = grad_y;
    p.adj_y0 = adj_y0;
    p.theta0 = grads_flat;
    p.pmask = param_mask & PHX_P_ALL;   // (a fixed grid uses no norm)
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}

int phx_solve_forward_many_grid(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const float* y0,
                                const double* t_host, int T, int t_is_f32, int method, double rtol, double atol,
                                int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                                phx_status* status, const float* grid_dt, const int32_t* grid_steps_,
                                const int32_t* grid_out_step, const float* grid_out_slope, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!y0 || !y_out) {
        phx_set_error("null y0 / y_out");
        return PHX_ERR_INVALID;
    }
    const PhxGridHost grid{grid_dt, grid_steps_, grid_out_step, grid_out_slope};
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 0, workspace,
                          workspace_bytes, status, nullptr, 0, (cudaStream_t)stream, &p, &plan, N, &grid);
    if (rc != PHX_OK) return rc;
    p.y0 = y0;
    p.yout = y_out;
    p.y0_stride = (long long)B * G;
    p.yout_stride = (long long)T * B * G;
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}

int phx_solve_adjoint_many_grid(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const double* t_host, int T,
                                int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                                const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                                void* workspace, size_t workspace_bytes, phx_status* status, int param_mask,
                                const float* grid_dt, const int32_t* grid_steps_, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!check_adjoint_mask(param_mask)) return PHX_ERR_INVALID;
    if (!y_saved || !grad_y || !adj_y0 || !grads_flat) {
        phx_set_error("null y_saved / grad_y / adj_y0 / grads_flat");
        return PHX_ERR_INVALID;
    }
    const PhxGridHost grid{grid_dt, grid_steps_, nullptr, nullptr};
    ResParams p;
    ResLaunchPlan plan;
    int rc = solve_common(ctx, G, H, B, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 1, workspace,
                          workspace_bytes, status, nullptr, 0, (cudaStream_t)stream, &p, &plan, N, &grid);
    if (rc != PHX_OK) return rc;
    p.ysaved = y_saved;
    p.grad_y = grad_y;
    p.adj_y0 = adj_y0;
    p.theta0 = grads_flat;
    p.yout_stride = (long long)T * B * G;
    p.adj_stride = (long long)B * G;
    p.theta_stride = (long long)phx_grad_offsets(G, H).total;
    p.pmask = param_mask & PHX_P_ALL;   // (a fixed grid uses no norm)
    return phx_resident_launch(p, plan, (cudaStream_t)stream);
}

int phx_solve_forward_rows_grid(phx_ctx* ctx, int G, int H, int N, const float* packed, const float* y0,
                                const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol,
                                double atol, int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                                phx_status* status, double* steplog, int steplog_cap, const float* grid_dt,
                                const int32_t* grid_steps_, const int32_t* grid_out_step, const float* grid_out_slope,
                                void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!y0 || !y_out) {
        phx_set_error("null y0 / y_out");
        return PHX_ERR_INVALID;
    }
    const PhxGridHost grid{grid_dt, grid_steps_, grid_out_step, grid_out_slope};
    ResParams p;
    RowsPlan plan;
    int rc = rows_common(ctx, G, H, N, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 0, workspace,
                         workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan, nullptr, &grid);
    if (rc != PHX_OK) return rc;
    p.y0 = y0;
    p.yout = y_out;
    p.fsign = reversed ? -1.f : 1.f;
    return phx_rows_launch(p, plan, (cudaStream_t)stream);
}

int phx_solve_adjoint_rows_grid(phx_ctx* ctx, int G, int H, int N, const float* packed, const double* t_host, int T,
                                int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                                const float* y_saved, const float* grad_y, float* adj_y0, float* grads_packed_parts,
                                void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                                int steplog_cap, int param_mask, const float* grid_dt, const int32_t* grid_steps_,
                                void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!check_adjoint_mask(param_mask)) return PHX_ERR_INVALID;
    if (!y_saved || !grad_y || !adj_y0 || !grads_packed_parts) {
        phx_set_error("null y_saved / grad_y / adj_y0 / grads_packed_parts");
        return PHX_ERR_INVALID;
    }
    if ((uintptr_t)grads_packed_parts & 15) {
        phx_set_error("grads_packed_parts must be 16-byte aligned");
        return PHX_ERR_INVALID;
    }
    const PhxGridHost grid{grid_dt, grid_steps_, nullptr, nullptr};
    ResParams p;
    RowsPlan plan;
    size_t o_th = 0;
    int rc = rows_common(ctx, G, H, N, packed, t_host, T, t_is_f32, method, rtol, atol, max_num_steps, 1, workspace,
                         workspace_bytes, status, steplog, steplog_cap, (cudaStream_t)stream, &p, &plan, &o_th, &grid);
    if (rc != PHX_OK) return rc;
    p.ysaved = y_saved;
    p.grad_y = grad_y;
    p.adj_y0 = adj_y0;
    p.theta_ws = (float*)workspace + o_th;
    p.gsum = grads_packed_parts;
    p.gsum_acc = 0;
    p.pmask = param_mask;
    return phx_rows_launch(p, plan, (cudaStream_t)stream);
}

}  // extern "C"
