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

// ---- fixed-grid step grids (phx_solve_desc.grid_*) ------------------------------------------------------------------
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

}  // extern "C"

/* ---- phx_solve: one request per solve, for every engine (include/phoenix_b200.h) ------------------------------------- */
namespace {

// the combinations of fields some engine takes
bool check_request(const phx_solve_desc& d) {
    if (d.engine < PHX_ENGINE_RESIDENT || d.engine > PHX_ENGINE_STREAM) {
        phx_set_error("unknown engine id %d", d.engine);
        return false;
    }
    const char* why = nullptr;
    if (d.adjoint && d.reversed) why = "an adjoint solve takes no `reversed`";
    else if (!d.adjoint && d.param_mask) why = "param_mask is for adjoint solves";
    else if (d.adjoint && (d.grid_out_step || d.grid_out_slope)) why = "grid_out_step / grid_out_slope are for forward solves";
    else if (!d.grid_dt && (d.grid_steps || d.grid_out_step || d.grid_out_slope)) why = "a step grid needs grid_dt";
    else if (d.engine == PHX_ENGINE_STREAM && d.N != 1) why = "the streaming engine solves one problem per call (N = 1)";
    else if (d.engine == PHX_ENGINE_ROWS && d.B != 1) why = "the rows engine solves one-row problems (B = 1)";
    else if (d.engine == PHX_ENGINE_RESIDENT && d.N > 1 && (d.reversed || d.steplog))
        why = "a resident solve of several problems takes no `reversed` and no step log";
    if (why) phx_set_error("%s (engine %d, adjoint %d, N=%d, B=%d)", why, d.engine, d.adjoint, d.N, d.B);
    return !why;
}

// the dopri5 step-control fields: 0 (the default) or a positive finite number, and only with dopri5
bool check_step_control(const phx_solve_desc& d) {
    const char* names[4] = {"first_step", "safety", "ifactor", "dfactor"};
    const double v[4] = {d.first_step, d.safety, d.ifactor, d.dfactor};
    for (int i = 0; i < 4; ++i) {
        if (!(v[i] >= 0.0 && v[i] < INFINITY)) {
            phx_set_error("%s must be 0 (the default) or a positive finite number (got %g)", names[i], v[i]);
            return false;
        }
        if (v[i] != 0.0 && d.method != PHX_DOPRI5) {
            phx_set_error("%s is a dopri5 option (method %d)", names[i], d.method);
            return false;
        }
    }
    return true;
}

// the resident and rows engines: the whole solve in one persistent launch
int solve_on_chip(phx_ctx* ctx, const phx_solve_desc& d, cudaStream_t stream) {
    const bool rows = d.engine == PHX_ENGINE_ROWS;
    const int G = d.G, H = d.H, B = d.B, N = d.N, T = d.T, adjoint = d.adjoint ? 1 : 0;
    if (!ctx || !check_dims(G, H, B) || !d.packed || !d.t_host || !d.workspace || (rows && N < 1)) {
        if (g_err[0] == 0) phx_set_error("null argument");
        return PHX_ERR_INVALID;
    }
    if (T < 2) {
        phx_set_error("t must hold at least two time points (got %d)", T);
        return PHX_ERR_INVALID;
    }
    if (!rows && (N < 1 || (N > 1 && N * T > PHX_T_INLINE))) {
        phx_set_error("a multi-problem launch takes 1 <= N and N * T <= %d output times (got N=%d, T=%d)", PHX_T_INLINE, N,
                      T);
        return PHX_ERR_INVALID;
    }
    for (int q = 0; q < N; ++q)
        for (int i = 1; i < T; ++i)
            if (!(d.t_host[q * T + i] > d.t_host[q * T + i - 1])) {
                phx_set_error("t must be strictly increasing at the C boundary (the Python shim negates decreasing t)");
                return PHX_ERR_INVALID;
            }
    if (d.method < PHX_EULER || d.method > PHX_DOPRI5) {
        phx_set_error("unknown method id %d", d.method);
        return PHX_ERR_INVALID;
    }
    if (((uintptr_t)d.workspace & (rows ? 127 : 15)) || ((uintptr_t)d.packed & 15)) {
        phx_set_error(rows ? "workspace must be 128-byte and packed weights 16-byte aligned"
                           : "workspace and packed weights must be 16-byte aligned");
        return PHX_ERR_INVALID;
    }
    ResLaunchPlan rplan;
    RowsPlan wplan;
    int rc = rows ? phx_rows_plan(ctx->num_sms, G, H, adjoint, &wplan)
                  : phx_resident_plan(ctx->num_sms, G, H, B, adjoint, &rplan);
    if (rc != PHX_OK) return rc;
    size_t o_t, o_th;   // o_th: the rows kernels' per-row cotangent buffers, or the resident adjoint's scratch twin
    const size_t need = (rows ? phx_rows_workspace_floats(G, H, N, T, wplan.rows, adjoint, &o_t, &o_th)
                              : phx_resident_workspace_floats(G, H, B, T, adjoint, &o_t, &o_th)) * sizeof(float);
    const PhxGridHost grid{d.grid_dt, d.grid_steps, d.grid_out_step, d.grid_out_slope};
    const bool gridded = d.grid_dt != nullptr;
    const size_t need_grid = gridded ? grid_room(need) + phx_grid_workspace_bytes(N, T, grid_steps(grid, N, T, adjoint))
                                     : need;
    if (d.workspace_bytes < need_grid) {
        phx_set_error("%s workspace too small: %zu < %zu", rows ? "rows" : "solve", d.workspace_bytes, need_grid);
        return PHX_ERR_WORKSPACE;
    }
    float* ws = (float*)d.workspace;
    ResParams p;
    memset(&p, 0, sizeof(p));
    p.G = G; p.H = H; p.Hp = phx_Hp(H); p.K2 = 2 * p.Hp; p.K2q = p.K2 / 4; p.B = B; p.T = T;
    p.method = d.method; p.t_is_f32 = d.t_is_f32; p.adjoint = adjoint;
    p.gpc = rows ? wplan.gpc : rplan.gpc;
    p.ring_rows = rows ? wplan.w1_stride_q : rplan.ring_rows;   // rows kernels: W1 row stride in shared memory (float4)
    p.ring_stages = rows ? 0 : rplan.ring_stages;
    p.so = rows ? wplan.so : rplan.so;
    p.rtol_f = (float)d.rtol; p.atol_f = (float)d.atol; p.fsign = d.reversed ? -1.f : 1.f;
    p.max_steps = (long long)d.max_num_steps;
    p.first_step = d.first_step;
    p.safety = d.safety > 0 ? d.safety : 0.9;
    p.ifactor = d.ifactor > 0 ? d.ifactor : 10.0;
    p.dfactor = d.dfactor > 0 ? d.dfactor : 0.2;
    p.w = phx_packed_view(d.packed, G, H);
    p.ll = phx_ll_view(d.workspace);
    p.t = (const double*)(ws + o_t);
    p.status = d.status; p.steplog = d.steplog; p.steplog_cap = d.steplog ? d.steplog_cap : 0;
    p.prof = ctx->prof;
    // problem i reads and writes base + i * stride; the rows engine runs its N problems as the rows of one problem
    p.nprob = rows ? 1 : N;
    p.y0_stride = (long long)B * G; p.yout_stride = (long long)T * B * G; p.adj_stride = (long long)B * G;
    if (rows) {
        p.rows = wplan.rows; p.ntot = N; p.nqw = wplan.nqw; p.ngg = wplan.ngg; p.gpg = wplan.gpg;
        p.tm_wa = wplan.tm_wa; p.tm_fac = wplan.tm_fac;
        p.ppk = (long long)phx_packed_grad_offsets(G, H).total;
    }
    if (!adjoint) {
        p.y0 = d.y0;
        p.yout = d.y_out;
    } else {
        p.ysaved = d.y_saved;
        p.grad_y = d.grad_y;
        p.adj_y0 = d.adj_y0;
        if (rows) {
            p.theta_ws = ws + o_th;
            p.gsum = d.grads;
            p.gsum_acc = 0;
            p.pmask = d.param_mask;
        } else {
            p.theta0 = d.grads;  // written once by the kernel (never read while still zero): no memset needed
            p.theta1 = ws + o_th;
            p.theta_stride = (long long)phx_grad_offsets(G, H).total;
            // A resident grid solve drops PHX_NORM_SEMINORM (a fixed grid uses no norm) where the rows engine passes it
            // on; both have always done so, and making them agree could change which kernel runs and its bits.
            p.pmask = gridded ? d.param_mask & PHX_P_ALL : d.param_mask;
        }
    }
    if (gridded && (rc = phx_grid_stage(grid, N, T, d.method, !adjoint, (char*)d.workspace + grid_room(need), stream, &p,
                                        nullptr)) != PHX_OK)
        return rc;
    if ((size_t)T * N <= PHX_T_INLINE) {
        for (int i = 0; i < T * N; ++i) p.t_small[i] = d.t_host[i];  // travels with the kernel parameters
    } else {
        cudaError_t e = cudaMemcpyAsync((void*)p.t, d.t_host, sizeof(double) * T * N, cudaMemcpyHostToDevice, stream);
        if (e != cudaSuccess) {
            phx_set_error("cudaMemcpyAsync(t): %s", cudaGetErrorString(e));
            return PHX_ERR_CUDA;
        }
    }
    return rows ? phx_rows_launch(p, wplan, stream) : phx_resident_launch(p, rplan, stream);
}

// the request of one of the entry points that predate phx_solve: a forward solve, or an adjoint one of all six parameters
phx_solve_desc forward_desc(int engine, int G, int H, int B, int N, const float* packed, const float* y0,
                            const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol, double atol,
                            int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                            phx_status* status, double* steplog, int steplog_cap) {
    phx_solve_desc d;
    memset(&d, 0, sizeof(d));
    d.engine = engine; d.G = G; d.H = H; d.B = B; d.N = N; d.T = T;
    d.packed = packed; d.t_host = t_host; d.t_is_f32 = t_is_f32; d.reversed = reversed; d.method = method;
    d.rtol = rtol; d.atol = atol; d.max_num_steps = max_num_steps;
    d.y0 = y0; d.y_out = y_out;
    d.workspace = workspace; d.workspace_bytes = workspace_bytes; d.status = status;
    d.steplog = steplog; d.steplog_cap = steplog_cap;
    return d;
}

phx_solve_desc adjoint_desc(int engine, int G, int H, int B, int N, const float* packed, const double* t_host, int T,
                            int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                            const float* y_saved, const float* grad_y, float* adj_y0, float* grads, void* workspace,
                            size_t workspace_bytes, phx_status* status, double* steplog, int steplog_cap) {
    phx_solve_desc d = forward_desc(engine, G, H, B, N, packed, nullptr, t_host, T, t_is_f32, 0, method, rtol, atol,
                                    max_num_steps, nullptr, workspace, workspace_bytes, status, steplog, steplog_cap);
    d.adjoint = 1;
    d.y_saved = y_saved; d.grad_y = grad_y; d.adj_y0 = adj_y0; d.grads = grads;
    d.param_mask = PHX_P_ALL;
    return d;
}

}  // namespace

extern "C" {

int phx_solve(phx_ctx* ctx, const phx_solve_desc* desc, void* stream) {
    PhxDevGuard dev_guard(ctx);
    g_err[0] = 0;
    if (!desc) {
        phx_set_error("null solve request");
        return PHX_ERR_INVALID;
    }
    const phx_solve_desc& d = *desc;
    if (!check_request(d) || !check_step_control(d)) return PHX_ERR_INVALID;
    const bool rows = d.engine == PHX_ENGINE_ROWS;
    if (d.adjoint) {
        if (!check_adjoint_mask(d.param_mask)) return PHX_ERR_INVALID;
        if (!d.y_saved || !d.grad_y || !d.adj_y0 || !d.grads) {
            phx_set_error(rows ? "null y_saved / grad_y / adj_y0 / grads_packed_parts"
                               : "null y_saved / grad_y / adj_y0 / grads_flat");
            return PHX_ERR_INVALID;
        }
        if (rows && ((uintptr_t)d.grads & 15)) {
            phx_set_error("grads_packed_parts must be 16-byte aligned");
            return PHX_ERR_INVALID;
        }
    } else if (!d.y0 || !d.y_out) {
        phx_set_error("null y0 / y_out");
        return PHX_ERR_INVALID;
    }
    if (d.engine == PHX_ENGINE_STREAM)
        return d.adjoint ? phx_stream_adjoint(ctx, d, (cudaStream_t)stream) : phx_stream_forward(ctx, d, (cudaStream_t)stream);
    return solve_on_chip(ctx, d, (cudaStream_t)stream);
}

int phx_solve_forward(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y0,
                      const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol, double atol,
                      int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                      phx_status* status, double* steplog, int steplog_cap, void* stream) {
    const phx_solve_desc d = forward_desc(PHX_ENGINE_RESIDENT, G, H, B, 1, packed, y0, t_host, T, t_is_f32, reversed, method,
                                          rtol, atol, max_num_steps, y_out, workspace, workspace_bytes, status, steplog,
                                          steplog_cap);
    return phx_solve(ctx, &d, stream);
}

int phx_solve_adjoint(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                      int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                      const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat, void* workspace,
                      size_t workspace_bytes, phx_status* status, double* steplog, int steplog_cap, void* stream) {
    const phx_solve_desc d = adjoint_desc(PHX_ENGINE_RESIDENT, G, H, B, 1, packed, t_host, T, t_is_f32, method, rtol, atol,
                                          max_num_steps, y_saved, grad_y, adj_y0, grads_flat, workspace, workspace_bytes,
                                          status, steplog, steplog_cap);
    return phx_solve(ctx, &d, stream);
}

/* ---- several independent problems per launch (SURVEY.md section 8 f1) -------------------------------------------- */
int phx_solve_forward_many(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const float* y0,
                           const double* t_host, int T, int t_is_f32, int method, double rtol, double atol,
                           int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                           phx_status* status, void* stream) {
    const phx_solve_desc d = forward_desc(PHX_ENGINE_RESIDENT, G, H, B, N, packed, y0, t_host, T, t_is_f32, 0, method, rtol,
                                          atol, max_num_steps, y_out, workspace, workspace_bytes, status, nullptr, 0);
    return phx_solve(ctx, &d, stream);
}

int phx_solve_adjoint_many(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const double* t_host, int T,
                           int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                           const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                           void* workspace, size_t workspace_bytes, phx_status* status, void* stream) {
    const phx_solve_desc d = adjoint_desc(PHX_ENGINE_RESIDENT, G, H, B, N, packed, t_host, T, t_is_f32, method, rtol, atol,
                                          max_num_steps, y_saved, grad_y, adj_y0, grads_flat, workspace, workspace_bytes,
                                          status, nullptr, 0);
    return phx_solve(ctx, &d, stream);
}

/* ---- the streaming engine (phx_stream.cu) ------------------------------------------------------------------------- */
int phx_stream_solve_forward(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y0,
                             const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol,
                             double atol, int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                             phx_status* status, double* steplog, int steplog_cap, void* stream) {
    const phx_solve_desc d = forward_desc(PHX_ENGINE_STREAM, G, H, B, 1, packed, y0, t_host, T, t_is_f32, reversed, method,
                                          rtol, atol, max_num_steps, y_out, workspace, workspace_bytes, status, steplog,
                                          steplog_cap);
    return phx_solve(ctx, &d, stream);
}

int phx_stream_solve_adjoint(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                             int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                             const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                             void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                             int steplog_cap, void* stream) {
    const phx_solve_desc d = adjoint_desc(PHX_ENGINE_STREAM, G, H, B, 1, packed, t_host, T, t_is_f32, method, rtol, atol,
                                          max_num_steps, y_saved, grad_y, adj_y0, grads_flat, workspace, workspace_bytes,
                                          status, steplog, steplog_cap);
    return phx_solve(ctx, &d, stream);
}

/* ---- rows kernels: N independent one-row problems in lock-step (phx_rows.cuh) ------------------------------------------- */
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
    const phx_solve_desc d = forward_desc(PHX_ENGINE_ROWS, G, H, 1, N, packed, y0, t_host, T, t_is_f32, reversed, method,
                                          rtol, atol, max_num_steps, y_out, workspace, workspace_bytes, status, steplog,
                                          steplog_cap);
    return phx_solve(ctx, &d, stream);
}

int phx_solve_adjoint_rows(phx_ctx* ctx, int G, int H, int N, const float* packed, const double* t_host, int T,
                           int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                           const float* y_saved, const float* grad_y, float* adj_y0, float* grads_packed_parts,
                           void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                           int steplog_cap, void* stream) {
    const phx_solve_desc d = adjoint_desc(PHX_ENGINE_ROWS, G, H, 1, N, packed, t_host, T, t_is_f32, method, rtol, atol,
                                          max_num_steps, y_saved, grad_y, adj_y0, grads_packed_parts, workspace,
                                          workspace_bytes, status, steplog, steplog_cap);
    return phx_solve(ctx, &d, stream);
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


/* ---- fixed-grid solves on the caller's step grid (options=dict(step_size=...), solvers.py:48-50, 77-103) ---------------- */
size_t phx_grid_workspace_bytes(int N, int T, int64_t total_steps) {
    if (N < 1 || T < 2 || total_steps < 0) return 0;
    const size_t nseg = (size_t)N * (T - 1);
    return 4 * (((size_t)total_steps + 3) / 4 * 4 + (nseg + 4) / 4 * 4 + 2 * ((nseg + 3) / 4 * 4)) + 16;
}

}  // extern "C"
