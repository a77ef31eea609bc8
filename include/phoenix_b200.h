/*
 * phoenix_b200 — C ABI of the B200-native PHOENIX NeuralODE hot path (libphoenix_b200.so).
 *
 * The reference (QuackenbushLab/phoenix) has no process / FFI boundary on this path: it is Python calling Python
 * (SURVEY.md section 8b).  The entry points below are what a binding for that path would bind; each one names the
 * reference interface it replaces.  Citations are relative to the reference root, `ode_net/code/...`.
 *
 * Conventions
 *   - every data pointer is a DEVICE pointer to contiguous fp32 unless the name ends in `_host`;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); nothing is allocated or freed
 *     behind the caller's back except inside phx_ctx_create / phx_ctx_destroy;
 *   - the library only borrows the caller's buffers for the duration of the enqueued work;
 *   - return value: PHX_OK or a negative phx_err; phx_last_error() returns a thread-local message;
 *   - solver-side conditions the reference reports with Python `assert` (dt underflow, non-finite state,
 *     max_num_steps; torchdiffeq/_impl/rk_common.py:154,175-176) are written to a phx_status record that the
 *     caller reads after synchronising the stream.
 *   - parameter order is the reference's `ODENet.parameters()` order: gene_multipliers[1,G], Wp[H,G], bp[H],
 *     Ws[H,G], bs[H], Wa[G,2H]  (odenet.py:49-61); "flat grads" is their concatenation, P = 4GH + 2H + G floats.
 */
#ifndef PHOENIX_B200_H
#define PHOENIX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct phx_ctx phx_ctx;

typedef enum phx_err {
    PHX_OK = 0,
    PHX_ERR_INVALID = -1,      /* bad argument (shape, null pointer, unsupported size)            */
    PHX_ERR_CUDA = -2,         /* a CUDA runtime call failed                                      */
    PHX_ERR_UNSUPPORTED = -3,  /* valid request this build has no kernel for                      */
    PHX_ERR_WORKSPACE = -4     /* workspace too small                                             */
} phx_err;

/* torchdiffeq method strings (torchdiffeq/_impl/odeint.py:9-22) this path implements */
typedef enum phx_method {
    PHX_EULER = 0,     /* 'euler'    fixed_grid.py:6-14                                           */
    PHX_MIDPOINT = 1,  /* 'midpoint' fixed_grid.py:17-27                                          */
    PHX_RK4 = 2,       /* 'rk4' = 3/8 rule, fixed_grid.py:30-38 + rk_common.py:96-103             */
    PHX_DOPRI5 = 3     /* 'dopri5'   dopri5.py:5-36 + rk_common.py:111-228                        */
} phx_method;

/* solver status codes written to phx_status.code */
enum {
    PHX_ST_OK = 0,
    PHX_ST_DT_UNDERFLOW = 1,  /* assert t0 + dt > t0          rk_common.py:175                    */
    PHX_ST_NONFINITE = 2,     /* assert isfinite(y0).all()    rk_common.py:176                    */
    PHX_ST_MAX_STEPS = 3,     /* assert n_steps < max_num_steps rk_common.py:154                  */
    PHX_ST_RUNNING = 99       /* kernel has not finished (status record not yet written)          */
};

typedef struct phx_status {
    int32_t code;        /* PHX_ST_*                                                              */
    int32_t n_accepted;  /* accepted adaptive steps                                               */
    int32_t n_rejected;  /* rejected adaptive steps                                               */
    int32_t n_rhs;       /* RHS (forward) or RHS-VJP (adjoint) evaluations                        */
    int32_t n_logged;    /* entries written to the step log                                       */
    int32_t reserved;
    double t_fail;       /* time at which a non-OK code was raised                                */
    double dt_fail;      /* dt at that moment                                                     */
} phx_status;

/* ---- context --------------------------------------------------------------------------------------------- */
int phx_ctx_create(int device, phx_ctx** out);
void phx_ctx_destroy(phx_ctx* ctx);
const char* phx_last_error(void);
/* number of SMs the persistent kernels will use on this device, and the largest B the resident solver accepts */
int phx_ctx_num_sms(const phx_ctx* ctx);
int phx_resident_max_rows(int adjoint);
/* Diagnostics (no reference counterpart): while `slots` (a device array of phx_profile_slots() int64, zeroed by the
 * caller) is set, CTA 0 of every resident solve adds the SM-clock cycles it spends in each phase of the kernel
 * (phase ids: PT_* in csrc/phx_resident.cuh).  NULL switches the timer off. */
/* Host-only: how a resident solve of this shape would be laid out on a device with num_sms SMs (needs no GPU).
 * out = {CTAs, genes per CTA, float4 columns per lane, W1 slice resident in shared memory?, WA slice resident?,
 * ring rows per chunk, ring stages, dynamic shared memory bytes}.  PHX_ERR_UNSUPPORTED if the shape does not fit. */
int phx_plan_describe(int num_sms, int G, int H, int B, int adjoint, int32_t out[8]);
int phx_ctx_set_profile(phx_ctx* ctx, void* slots);
int phx_profile_slots(void);

/* ---- precision of the batched contractions ------------------------------------------------------------------ */
/* Calls with B >= phx_tc_min_rows() rows (the 10 000-row prior batch train_insilico.py:134,209; the batched sweeps)
 * are dense contractions and run on the tcgen05 tensor cores.  PHX_PREC_3XTF32 (default) keeps fp32 parity with the
 * reference's ATen fp32 matmuls by splitting every operand into two TF32 terms (three MMAs per product);
 * PHX_PREC_TF32 is the single-pass TF32 mode (relative error ~1e-3, reported separately); PHX_PREC_FP32 forces the
 * fp32 CUDA-core contractions.  Calls with fewer rows are GEMV-bound and never use the tensor cores. */
enum { PHX_PREC_FP32 = 0, PHX_PREC_TF32 = 1, PHX_PREC_3XTF32 = 3 };
int phx_ctx_set_precision(phx_ctx* ctx, int precision);
int phx_ctx_get_precision(const phx_ctx* ctx);
int phx_tc_min_rows(void);
/* Host-only: how a branch-type tensor-core contraction with K k-elements (genes, or batch rows for the parameter
 * cotangents) and M rows is split over CTAs.  out = {128-row tiles, K-splits of the prods half, k-blocks per split,
 * K-splits of the sums half, k-blocks per split, partial-sum slots}; a k-block is 16 k-elements. */
int phx_tc_plan_describe(int K, int M, int32_t out[6]);
/* Diagnostics (no reference counterpart).  phx_tc_set_pair(1): run the branch-type tensor-core contractions as CTA pairs
 * (tcgen05 cta_group::2) -- bit-identical results, measured slower on B200, off by default (tests compare the two).
 * phx_tc_prof_dump: print and reset the device counters collected when the process runs with PHX_TC_PROF=1. */
void phx_tc_set_pair(int on);
void phx_tc_prof_dump(void);

/* ---- weights --------------------------------------------------------------------------------------------- */
/* Bytes of the packed (kernel-layout) copy of the six parameters for an ODENet(ndim=G, neurons=H). */
size_t phx_packed_bytes(int G, int H);
/* Re-lay the six reference parameter tensors (odenet.py:49-61) into the kernel layout:
 * W1[G][K2] = [Ws^T | Wp^T], WA[G][K2] = Wa (halves padded to a multiple of 4), bias[K2], relu(m)[G], (m>0)[G].
 * The tail of the buffer holds the tensor-core operand images; they are rebuilt on `stream` by the first large-B call
 * that follows a phx_pack_weights of the same buffer, so all calls sharing a packed buffer must share a stream. */
int phx_pack_weights(phx_ctx* ctx, int G, int H, const float* gene_multipliers, const float* Wp, const float* bp,
                     const float* Ws, const float* bs, const float* Wa, float* packed, void* stream);

/* ---- RHS: ODENet.forward / ODENet.prior_only_forward (odenet.py:85-98) ----------------------------------- */
/* f[B][G] = relu(m) * (joint(y) - y)   (decay != 0)    or    joint(y)   (decay == 0) */
int phx_rhs_forward(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y, float* f, int decay,
                    void* workspace, size_t workspace_bytes, void* stream);
/* VJP of the call above for cotangent g[B][G] (what torch.autograd computes through odenet.py:85-98):
 * ybar[B][G] (may be NULL) and the flat parameter cotangents grads_flat[P] (may be NULL); accumulate bit 0 adds into
 * grads_flat instead of overwriting it.  accumulate bit 1 (PHX_VJP_REUSE_FORWARD = 2) is a promise by the caller that
 * `workspace` has not been touched since a phx_rhs_forward call with the same packed weights, the same y and the same
 * B ran on it: the branch contraction [S|P] it left there is reused instead of recomputed (what autograd's saved
 * activations give the reference).  Ignored on the fp32 path. */
#define PHX_VJP_REUSE_FORWARD 2
int phx_rhs_vjp(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y, const float* g, int decay,
                float* ybar, float* grads_flat, int accumulate, void* workspace, size_t workspace_bytes,
                void* stream);
size_t phx_rhs_workspace_bytes(int G, int H, int B);

/* ---- prior-constrained loss term of training_step (train_insilico.py:134-137, 208-209) -------------------------------- */
/* loss[0] = mean((prior_only_forward(x) - prior_grad)^2) over the B rows (device scalar) and
 * gcot[B][G] = scale * (prior_only_forward(x) - prior_grad) -- with scale = 2 / (B * G) the cotangent of that mean --
 * in one fused pass (B >= phx_tc_min_rows(): the joint contraction's epilogue compares with prior_grad, the joint itself
 * never goes to memory).  `workspace` is an RHS workspace (phx_rhs_workspace_bytes); it is left holding [S|P] of x, so the
 * backward is  phx_rhs_vjp(ctx, G, H, B, packed, x, gcot, 0, NULL, grads_flat, PHX_VJP_REUSE_FORWARD, workspace, ...). */
int phx_prior_loss(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* x, const float* prior_grad,
                   float scale, float* gcot, float* loss, void* workspace, size_t workspace_bytes, void* stream);
/* Cached Hill activations of a CONSTANT input.  batch_for_prior is drawn once before the epoch loop
 * (train_insilico.py:208) and is the same matrix at every optimiser step; phx_hill_planes evaluates
 * s = SoftsignMod(x) and l = LogShiftedSoftSignMod(x) (odenet.py:21-35) for n = rows * G elements once, and while
 * phx_hill_cache_set(ctx, x, n, s, l) is in force every tensor-core contraction whose activation operand is that x
 * (phx_prior_loss, phx_rhs_forward, the Ws_bar | Wp_bar part of phx_rhs_vjp) reads the planes instead of
 * re-evaluating the activations (same values bit for bit).  The caller scopes the entry around its launches and
 * clears it with s = l = NULL; the planes must stay valid until the enqueued work has run. */
int phx_hill_planes(phx_ctx* ctx, size_t n, const float* x, float* s_plane, float* l_plane, void* stream);
int phx_hill_cache_set(phx_ctx* ctx, const float* x, size_t n, const float* s_plane, const float* l_plane);
/* prior_grad[B][G] = x[B][G] @ prior_mat[G][G] (train_insilico.py:209) for a sparse prior in CSC form (column j of
 * prior_mat = rows rowidx[colptr[j] .. colptr[j+1]) with values val[...]; all device pointers). */
int phx_prior_setup(phx_ctx* ctx, int G, int B, const float* x, const int32_t* colptr, const int32_t* rowidx,
                    const float* val, float* out, void* stream);

/* ---- odeint (torchdiffeq/_impl/odeint.py:25-69) ---------------------------------------------------------- */
size_t phx_solve_workspace_bytes(const phx_ctx* ctx, int G, int H, int B, int T, int adjoint);
/* The first phx_solve_workspace_init_bytes() bytes of a resident-solver workspace hold the inter-CTA exchange area
 * (tagged slots carrying a per-workspace epoch from launch to launch).  Call phx_solve_workspace_init ONCE after
 * allocating a workspace (it zeroes that area on `stream`); afterwards the same workspace serves any sequence of
 * phx_solve_forward / phx_solve_adjoint calls of any shape, as long as calls sharing it are ordered on one stream. */
size_t phx_solve_workspace_init_bytes(void);
int phx_solve_workspace_init(void* workspace, size_t workspace_bytes, void* stream);
/* y_out[T][B][G] = solution at the T increasing times t_host (float64; t_is_f32 != 0 says the caller's tensor was
 * float32, which changes how fixed-grid dt is rounded, solvers.py:84-86).  reversed != 0: the caller's t was
 * decreasing and has been negated, so the kernel integrates -f (misc.py:159-162,210-212).  Reference defaults: rtol 1e-7,
 * atol 1e-9, max_num_steps 2^31-1, norm = RMS over the whole [B][G] state (misc.py:198-201).
 * steplog (may be NULL): steplog_cap rows of (t0, dt, accepted) float64, one per attempted adaptive step. */
int phx_solve_forward(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y0,
                      const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol,
                      double atol, int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                      phx_status* status, double* steplog, int steplog_cap, void* stream);

/* ---- OdeintAdjointMethod.backward (torchdiffeq/_impl/adjoint.py:32-162) ---------------------------------- */
/* Integrates the augmented system (y, adj_y, adj_params) backwards over every output interval with the forward
 * method / tolerances and the mixed max-of-RMS norm (adjoint.py:72-78,198-200).  y_saved and grad_y are
 * [T][B][G]; outputs adj_y0[B][G] and grads_flat[P] (overwritten). */
int phx_solve_adjoint(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                      int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                      const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                      void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                      int steplog_cap, void* stream);
/* ---- adjoint parameters (adjoint.py:185-193: the members of adjoint_params that require grad) -------------------------
 * An adjoint phx_solve (below) takes param_mask, a 6-bit set of parameters in reference order: bit i = the i-th of
 * (gene_multipliers, Wp, bp, Ws, bs, Wa), PHX_PARAMS_ALL = all six (what the other adjoint entry points pass).  Only the
 * cotangents of the parameters in the mask are integrated, and only they make up the parameter block of the error norm
 * (count = their total size; with an empty mask the block is absent).  The blocks of grads_flat outside the mask are
 * written as zeros (phx_unpack_grads_masked with accumulate != 0 leaves them as they are).  A mask outside 0 .. 0x3F
 * returns PHX_ERR_INVALID.
 * PHX_NORM_SEMINORM may be OR-ed into the param_mask of an adjoint phx_solve (not phx_unpack_grads_masked): dopri5 then
 * measures the error with the seminorm of Kidger, Chen & Lyons (2021), the mixed norm without the parameter block, in
 * Hairer's initial step and in every error ratio, while the low six bits still choose the integrated cotangents.
 * Fixed grids use no norm and are unaffected.  With it the accepted range is 0 .. 0x7F. */
#define PHX_PARAMS_ALL 0x3F
#define PHX_NORM_SEMINORM 0x40

/* ---- N independent problems per launch (the per-sample loop of training_step, train_insilico.py:128-130) -------- */
/* Problem i: initial state y0 + i*B*G, its own T increasing times t_host[i*T .. i*T+T), outputs y_out + i*T*B*G, its own
 * step controller and its own status[i] (an array of N records).  The solves run one after the other inside ONE
 * persistent launch, so the weights are staged on chip once for all of them; results are bit-identical to N calls of
 * phx_solve_forward / phx_solve_adjoint.  Limits: the rows fit the resident kernels and N * T <= 64.
 * Adjoint: y_saved / grad_y are [N][T][B][G], adj_y0 [N][B][G], grads_flat [N][P] (one cotangent vector per problem). */
int phx_solve_forward_many(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const float* y0,
                           const double* t_host, int T, int t_is_f32, int method, double rtol, double atol,
                           int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                           phx_status* status, void* stream);
int phx_solve_adjoint_many(phx_ctx* ctx, int G, int H, int B, int N, const float* packed, const double* t_host, int T,
                           int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                           const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                           void* workspace, size_t workspace_bytes, phx_status* status, void* stream);

/* ---- the same two solves for ANY number of rows B (streaming engine) ---------------------------------------- */
/* phx_solve_forward / phx_solve_adjoint keep the whole solve in one persistent cooperative launch and need the rows
 * to fit on chip (B <= phx_resident_max_rows()).  These variants stream the [B][G] state through HBM and run the
 * branch contractions as batched GEMM-shaped launches; they cover the batched callers of the reference
 * (find_gene_influences.py:64-73 with B=60, the 4096-row synthetic sweep).  Identical arguments and semantics; with
 * method = PHX_DOPRI5 the call synchronises `stream` once per attempted step (host-side step controller). */
size_t phx_stream_workspace_bytes(const phx_ctx* ctx, int G, int H, int B, int T, int adjoint);
/* Exact-global-norm mode for a batched dopri5 FORWARD solve whose rows are sharded over several GPUs (SURVEY 8e): the
 * reference's error norm is the RMS over ALL rows of the batch (torchdiffeq/_impl/misc.py:10-11), so every rank must take
 * the same accept / reject decisions.  With a hook installed, phx_stream_solve_forward calls it once per norm evaluation
 * with the DEVICE array of this rank's n partial sums (float64), enqueued on `stream`; the hook must sum the array over
 * the ranks in place (an NCCL all-reduce of n doubles) and every rank then counts world_size x its own elements.  All
 * ranks must hold the same number of rows.  The adjoint keeps per-shard controllers (its norm involves the parameter
 * cotangents of the WHOLE batch).  hook = NULL switches the mode off. */
typedef void (*phx_sum_hook)(double* sums_device, int n, void* stream, void* user);
int phx_ctx_set_global_norm(phx_ctx* ctx, phx_sum_hook hook, void* user, int world_size);
int phx_stream_solve_forward(phx_ctx* ctx, int G, int H, int B, const float* packed, const float* y0,
                             const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol,
                             double atol, int64_t max_num_steps, float* y_out, void* workspace,
                             size_t workspace_bytes, phx_status* status, double* steplog, int steplog_cap,
                             void* stream);
int phx_stream_solve_adjoint(phx_ctx* ctx, int G, int H, int B, const float* packed, const double* t_host, int T,
                             int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                             const float* y_saved, const float* grad_y, float* adj_y0, float* grads_flat,
                             void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                             int steplog_cap, void* stream);

/* ---- the sample loop of training_step as rows of ONE launch (train_insilico.py:128-130) ------------------------------- */
/* N independent ONE-ROW problems (y0 [N][G], each with its own T increasing times t_host[i*T .. i*T+T), its own dopri5 step
 * controller and its own status[i]) advance in lock-step, phx_rows_supported() of them at a time as the rows of one
 * pass: the RHS is autonomous, so every weight-slice pass and every inter-CTA exchange serves all rows.  A problem's results
 * are bit-identical whether it runs alone or beside others.  phx_rows_supported returns the rows per pass (0: the model's
 * weight slices do not fit on chip -- use phx_solve_forward / phx_solve_adjoint).
 * steplog (may be NULL): [N][steplog_cap][3] float64 rows of (t0, dt, accepted), one block per problem. */
int phx_rows_supported(const phx_ctx* ctx, int G, int H, int adjoint);
/* Host-only: out = {CTAs, genes per CTA, quad-warps, gene groups, genes per group, WA slice in shared (1) / tensor (2)
 * memory, rows per pass, W1 row stride (float4), tensor-memory columns used, dynamic shared memory bytes}. */
int phx_rows_plan_describe(int num_sms, int G, int H, int adjoint, int32_t out[10]);
size_t phx_rows_workspace_bytes(const phx_ctx* ctx, int G, int H, int N, int T, int adjoint);
/* y_out [N][T][G].  The workspace starts with the exchange area of phx_solve_workspace_init (same rules). */
int phx_solve_forward_rows(phx_ctx* ctx, int G, int H, int N, const float* packed, const float* y0,
                           const double* t_host, int T, int t_is_f32, int reversed, int method, double rtol, double atol,
                           int64_t max_num_steps, float* y_out, void* workspace, size_t workspace_bytes,
                           phx_status* status, double* steplog, int steplog_cap, void* stream);
/* OdeintAdjointMethod.backward (adjoint.py:32-162) of the N problems: y_saved / grad_y [N][T][G], adj_y0 [N][G], and the
 * parameter cotangents in the PACKED layout -- W1bar[G][K2] | WAbar[G][K2] | biasbar[K2] | mbar[G], the layout of
 * phx_pack_weights, phx_packed_grad_bytes() bytes, 16-byte aligned -- as phx_rows_grad_parts() PARTIAL SUMS (one per pass
 * of phx_rows_supported() problems): grads_packed_parts [parts][phx_packed_grad_bytes / 4].  phx_unpack_grads adds the
 * parts in a fixed order and converts to the reference's flat order (gene_multipliers, Wp, bp, Ws, bs, Wa): what autograd
 * accumulates into .grad over the samples; accumulate != 0 adds to grads_flat instead of overwriting it. */
int phx_solve_adjoint_rows(phx_ctx* ctx, int G, int H, int N, const float* packed, const double* t_host, int T,
                           int t_is_f32, int method, double rtol, double atol, int64_t max_num_steps,
                           const float* y_saved, const float* grad_y, float* adj_y0, float* grads_packed_parts,
                           void* workspace, size_t workspace_bytes, phx_status* status, double* steplog,
                           int steplog_cap, void* stream);
size_t phx_packed_grad_bytes(int G, int H);
int phx_rows_grad_parts(const phx_ctx* ctx, int G, int H, int N);

/* ---- every solve through one request (phx_solve) --------------------------------------------------------------------
 * phx_solve runs one solve described by a phx_solve_desc; each entry point above is a phx_solve call with the options it
 * does not take at their defaults.  `engine` picks the solver (PHX_ENGINE_RESIDENT: phx_solve_forward / _adjoint, and
 * phx_solve_*_many when N > 1; PHX_ENGINE_ROWS: phx_solve_*_rows, B = 1; PHX_ENGINE_STREAM: phx_stream_solve_*, N = 1),
 * `adjoint` the direction.  The fields mean what the arguments of the same names mean there, and the workspace is sized
 * by the engine's own size function.  Forward solves read y0 and write y_out; adjoint solves read y_saved and grad_y and
 * write adj_y0 and `grads` (flat [N][P] on the resident and streaming engines, the packed partial sums of
 * phx_solve_adjoint_rows on the rows engine), with `param_mask` as described above (PHX_PARAMS_ALL for all six).
 * The combinations no engine takes return PHX_ERR_INVALID: an unknown engine; `reversed` or `grid_out_*` on an adjoint
 * solve; a nonzero param_mask on a forward solve; grid arrays without grid_dt; N != 1 on the streaming engine; B != 1 on
 * the rows engine; `reversed` or a step log on the resident engine with N > 1.
 *
 * Fixed-grid solves on a step grid (odeint options=dict(step_size=h), torchdiffeq solvers.py:48-50, 77-103): with grid_dt
 * set (NULL: one step per output interval) the method must be euler, midpoint or rk4, and PHX_NORM_SEMINORM is accepted
 * and has no effect.  The caller builds the grid (the Python layer does it with the reference's own tensor ops) and no
 * kernel computes one; its arrays are HOST arrays:
 *   grid_steps[q] >= 1 steps per segment and their float32 dt back to back in grid_dt (in segment order).  A forward
 *     segment is a problem (N of them); an adjoint segment is an output interval of a problem, [N][T-1] with the interval
 *     [t[i], t[i+1]] at index i, its steps in the order the backward takes them (from t[i+1]).
 *   forward only, [N][T-1]: grid_out_step[j-1] = the step (counted from 0 within the problem, non-decreasing in j) whose
 *     end is the first grid point >= t[j], and grid_out_slope[j-1] = (t[j] - t0) / (t1 - t0) of that step, rounded to
 *     float32; output j is then y0 + slope * (y1 - y0), or y1 itself when the slope is negative (t[j] == t1).
 * Between the steps the state is not restarted at the output times.  status.n_rhs = stages x steps.  The grid is copied
 * into the workspace (not on the streaming engine), which must then hold phx_grid_workspace_bytes(N, T, total steps)
 * more bytes than the engine's own size function asks for.  An invalid grid (a step count < 1, a dt that is negative or
 * not finite, an output step out of range or decreasing, a NaN slope) returns PHX_ERR_INVALID.
 *
 * dopri5 step control (odeint options first_step, safety, ifactor, dfactor; rk_common.py:111-228, misc.py:94-103):
 * 0 in a field means its default -- Hairer's initial-step estimate (misc.py:47-86), 0.9, 10 and 0.2 -- so a
 * zero-initialised request and every entry point above keep the reference's default controller.
 *   first_step > 0: the first attempted dt of the solve, and of every output interval of an adjoint solve (each is its
 *     own odeint call in the reference's backward), in the increasing time the solve runs in.  f0 is still evaluated
 *     (it counts in status.n_rhs and gives the non-finite check of the initial state); Hairer's second evaluation and
 *     its norms (in the adjoint also those of the parameter cotangents) are skipped.  A first step beyond the next
 *     output time is legal: steps are never clipped to output times.
 *   safety, ifactor, dfactor: with the error ratio r, the next dt is dt * ifactor when r == 0, else
 *     dt * min(ifactor, max(safety / r^(1/5), r < 1 ? 1 : dfactor)).
 * A negative, NaN or infinite value in any of the four, or a nonzero one with a method other than dopri5, returns
 * PHX_ERR_INVALID. */
enum { PHX_ENGINE_RESIDENT = 0, PHX_ENGINE_ROWS = 1, PHX_ENGINE_STREAM = 2 };
typedef struct phx_solve_desc {
    const float* packed;
    const double* t_host;            /* [N][T] */
    const float* y0;                 /* forward */
    float* y_out;
    const float* y_saved;            /* adjoint */
    const float* grad_y;
    float* adj_y0;
    float* grads;
    const float* grid_dt;            /* step grid (host arrays); NULL grid_dt: one step per output interval */
    const int32_t* grid_steps;
    const int32_t* grid_out_step;    /* forward grids only */
    const float* grid_out_slope;
    void* workspace;
    size_t workspace_bytes;
    phx_status* status;              /* [N] */
    double* steplog;                 /* may be NULL */
    double rtol, atol;
    int64_t max_num_steps;
    double first_step, safety, ifactor, dfactor;   /* dopri5 step control; 0: the default */
    int32_t engine, adjoint, G, H, B, N, T, t_is_f32, reversed, method, param_mask, steplog_cap;
} phx_solve_desc;
int phx_solve(phx_ctx* ctx, const phx_solve_desc* desc, void* stream);
size_t phx_grid_workspace_bytes(int N, int T, int64_t total_steps);
int phx_unpack_grads(phx_ctx* ctx, int G, int H, const float* packed_grads, int nparts, float* grads_flat,
                     int accumulate, void* stream);
int phx_unpack_grads_masked(phx_ctx* ctx, int G, int H, const float* packed_grads, int nparts, float* grads_flat,
                            int accumulate, int param_mask, void* stream);
/* Cotangent of the data loss of training_step, loss = torch.mean((predictions - targets)**2) (train_insilico.py:132):
 * grad[r][g] = scale * (pred[r][g] - target[r][g]) for `rows` samples of G genes, scale = 2 / (rows * G); pred and grad
 * rows are pred_stride / grad_stride floats apart (the t1 slices of the [N][T][G] solver output and of grad_y), target is
 * dense [rows][G].  What autograd computes for that line; lets a C-ABI caller go from phx_solve_forward_rows to
 * phx_solve_adjoint_rows without leaving the library. */
int phx_mse_grad(phx_ctx* ctx, int rows, int G, const float* pred, size_t pred_stride, const float* target, float scale,
                 float* grad, size_t grad_stride, void* stream);

/* ---- multi-GPU: the one exchange of the path (SURVEY 8e) ------------------------------------------------------------------
 * The reference has no distributed code; with the samples of train_insilico.py:128-130 sharded over the GPUs of one box
 * the parameter gradients must be summed once per optimiser step.  phx_peer_allreduce does that sum IN PLACE over peer
 * memory (NVLink 5 / NVSwitch), one kernel per rank, no NCCL call: bufs[r] / flags[r] are the device pointers of rank r's
 * gradient buffer (n floats, 16-byte aligned) and flag pad (2 * world uint32, zeroed once) as mapped into THIS process
 * (e.g. torch symmetric memory); `epoch` grows by one per call and is the same on every rank; every rank's buffer ends up
 * holding scale * (sum over ranks), bit-identical everywhere, summed in rank order.  world in {2, 4, 8}.  The call is
 * asynchronous on `stream`; all ranks must make it (it spins on the peers' flags). */
int phx_peer_allreduce(phx_ctx* ctx, void* const* bufs, void* const* flags, int rank, int world, size_t n,
                       unsigned epoch, float scale, void* stream);
/* The same with the sums formed inside the NVSwitch (NVLS: multimem.ld_reduce / multimem.st): multicast_buf is the
 * multicast address of the W gradient buffers (cuMulticast* / torch symmetric memory `multicast_ptr`). */
int phx_peer_allreduce_nvls(phx_ctx* ctx, void* multicast_buf, void* const* flags, int rank, int world, size_t n,
                            unsigned epoch, float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PHOENIX_B200_H */
