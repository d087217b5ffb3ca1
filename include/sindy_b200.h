/*
 * sindy_b200.h — C ABI of libsindy_b200.so: the B200 (sm_100a) implementation of the SINDy-family
 * hot path of Rose-STL-Lab/symmetry-ode-discovery.
 *
 * The reference is pure Python/PyTorch and has no FFI of its own; every entry point below
 * replaces the tensor arithmetic of one reference function (cited as file:line relative to the
 * reference root). The host side that binds these symbols is
 * `symmetry-ode-discovery_b200/sindy_b200/native.py` (ctypes); `INTEGRATION.md` shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *  - every data pointer is a DEVICE pointer on the current CUDA device, row-major, contiguous;
 *  - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream); every call is
 *    asynchronous on that stream and never synchronises the device;
 *  - the caller owns all buffers, including workspaces (`sb_workspace_bytes`); nothing is retained
 *    after the call returns except per-device constant tables;
 *  - return value: 0 = ok, negative = `sb_status`; `sb_last_error()` gives a thread-local message;
 *  - re-entrant from several host threads. The specialised kernels read the coefficient matrix from per-device
 *    constant-bank slots: the stateless entry points (sb_train_step, sb_closure[_peer], sb_forward, sb_backward) share
 *    scratch slot 0 — each call packs its coefficients on its own stream right before its kernel, and a call arriving
 *    on a different stream than the previous one waits (event) for it, so concurrent streams are serialised at that
 *    point rather than racing (inside a CUDA-graph capture the wait cannot be inserted: captured calls that use
 *    different coefficients must then be ordered by the graph); sb_fit_step / sb_load_w keep their coefficients in
 *    the RESIDENT slot 1, which no stateless entry point writes — forward / closure / STLSQ calls may run between two
 *    iterations of a fit; two fits alternating on one device must re-load the slot when they take turns (sb_load_w, or
 *    a call without SB_FIT_W_RESIDENT);
 *  - no C++ exception crosses the ABI; there is NO CPU fallback: without a CUDA device every
 *    compute entry point returns SB_ERR_CUDA.
 *
 * Library column order (reference `sindy.py:7-30,68-77`): 1; x_0..x_{d-1}; then for n = 2..poly_order
 * the degree-n monomials over non-decreasing index tuples in lexicographic order, each formed
 * left to right ((x_i*x_j)*x_k...); then sin(x_i) (if include_sine); then exp(x_i) (if include_exp).
 * The reference stops at degree 3 (`sindy.py:37`); degrees 4 and 5 continue the same enumeration.
 */
#ifndef SINDY_B200_H
#define SINDY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB_MAX_DIM 8
#define SB_MAX_POLY 5
#define SB_MAX_TERMS 256
#define SB_MAX_PEERS 8

typedef enum {
  SB_OK = 0,
  SB_ERR_INVALID = -1,     /* bad argument (NULL pointer, negative size, misaligned buffer ...) */
  SB_ERR_UNSUPPORTED = -2, /* library outside the supported range (dim, poly_order, K) */
  SB_ERR_CUDA = -3,        /* CUDA runtime error (message in sb_last_error) */
  SB_ERR_WORKSPACE = -4    /* workspace too small */
} sb_status;

/* Function library Θ: mirrors SINDyRegression(latent_dim, poly_order, include_sine, include_exp)
 * (`sindy.py:42-77`). */
typedef struct {
  int32_t dim;          /* latent_dim d, 1..SB_MAX_DIM */
  int32_t poly_order;   /* 1..SB_MAX_POLY */
  int32_t include_sine; /* 0/1 */
  int32_t include_exp;  /* 0/1 */
} sb_library;

/* sb_train_step `flags` and the packed fp64 output layout.
 *   out[0]               = sum_{n,i} r[n,i]^2            with r = Θ(x)·Wᵀ − dx   (SB_STEP_LOSS)
 *   out[1]               = n (number of samples reduced, as double)
 *   out[2 .. 2+d*K)      = sum_n r[n,i]·Θ_k(x_n), row-major d×K  (SB_STEP_GRAD; the MSE gradient of
 *                          `train.py:663-664,689` is 2/(n·d) times this)
 *   then K*K doubles     = Gram ΘᵀΘ, row-major                    (SB_STEP_GRAM; `sindy.py:261` restated)
 *   then K*d doubles     = ΘᵀẊ, row-major K×d                     (SB_STEP_B)
 * Sections that are not requested are absent (the following ones move up). Sums, not means, so that
 * shards on several GPUs combine with one all-reduce(sum). */
#define SB_STEP_LOSS 1u
#define SB_STEP_GRAD 2u
#define SB_STEP_GRAM 4u
#define SB_STEP_B 8u

/* dtype tags for the rollout */
#define SB_F32 0
#define SB_F64 1
/* integrators (`model_utils.py:223-255`) */
#define SB_EULER 0
#define SB_RK4 1

int sb_version(void);
const char* sb_last_error(void);

/* Number of kernels this library has launched in this process (all threads, all devices). */
unsigned long long sb_kernel_launches(void);

/* Number of CUDA devices visible (0 if none / driver missing). */
int sb_device_count(void);

/* K = number of library columns; `sindy.py:179-189` get_term_num (extended to degree 5). <0 on error. */
int sb_library_size(const sb_library* lib);
/* Exponent table K×d (row-major) for the polynomial columns; sine rows hold -1 at their variable,
 * exp rows -2 (others 0). Host memory. Mirrors the enumeration of `sindy.py:13-24`. */
int sb_library_exponents(const sb_library* lib, int32_t* out_host);

/* Bytes of device workspace any reducing call below may need for this library. */
int64_t sb_workspace_bytes(const sb_library* lib);
/* Number of doubles sb_train_step writes for `flags`. */
int64_t sb_train_step_out_len(const sb_library* lib, uint32_t flags);

/* Θ(x): `sindy.py:201-203` eval_Theta_at. x (n×d) → theta (n×K). Debug/parity only — the
 * product paths never materialise Θ. */
int sb_theta(const float* x, int64_t n, const sb_library* lib, float* theta, void* stream);

/* h(x) = Θ(x)·Wᵀ with W = Ξ⊙mask (d×K): `sindy.py:79-82` forward. y (n×d). */
int sb_forward(const float* x, int64_t n, const sb_library* lib, const float* w, float* y,
               void* stream);

/* Vector-Jacobian product of sb_forward (what autograd does for `loss.backward()`,
 * `train.py:689`): gw[i,k] = sum_n gy[n,i]·Θ_k(x_n) (fp64, d×K; may be NULL) and
 * gx[n,j] = sum_i gy[n,i] sum_k W[i,k] ∂Θ_k/∂x_j (n×d; may be NULL). */
int sb_backward(const float* x, const float* gy, int64_t n, const sb_library* lib, const float* w,
                double* gw, float* gx, void* workspace, int64_t workspace_bytes, void* stream);

/* Jacobian-vector product J_h(x)·u = W·(J_Θ(x)·u): what `torch.autograd.functional.jvp(regressor, x, u)`
 * computes by double-vjp in `model_utils.py:53-56` and `train.py:503-507`. out (n×d). */
int sb_jvp(const float* x, const float* u, int64_t n, const sb_library* lib, const float* w,
           float* out, void* stream);

/* Vector-Jacobian product of sb_jvp w.r.t. (W, x, u) for cotangent g (n×d):
 *   gw[i,k] = sum_n g[n,i]·(J_Θ(x_n)u_n)_k   (fp64 d×K, may be NULL)
 *   gx      = Hessian-vector term sum_i g_i sum_k W_ik ∂²Θ_k/∂x∂x · u   (n×d, may be NULL)
 *   gu      = J_h(x)ᵀ g                        (n×d, may be NULL)
 * Needed because `symmreg_i` differentiates through its JVPs (`model_utils.py:32,56`). */
int sb_jvp_backward(const float* x, const float* u, const float* g, int64_t n,
                    const sb_library* lib, const float* w, double* gw, float* gx, float* gu,
                    void* workspace, int64_t workspace_bytes, void* stream);

/* Fused train step: one pass over (x, dx) producing the sections selected by `flags` (layout above).
 * Replaces `regressor(x)` + MSELoss + backward of the LBFGS closure (`train.py:645-690`) and the
 * Θ/augmented-matrix build of `solve_SINDy_one_step` (`sindy.py:260-264`). dx may be NULL only if
 * flags == SB_STEP_GRAM. w may be NULL if neither LOSS nor GRAD is requested. */
int sb_train_step(const float* x, const float* dx, int64_t n, const sb_library* lib,
                  const float* w, uint32_t flags, double* out, void* workspace,
                  int64_t workspace_bytes, void* stream);

/* One closure evaluation of the LBFGS / Adam loops without sym-reg (`train.py:645-690`, `:512-527`):
 *   loss = mean((Θ(x)(Ξ⊙mask)ᵀ − dx)²) + w_l1·‖Ξ‖₁      (fp32 scalar, device)
 *   grad = dloss/dΞ = (2/(n·d))·(Σ_n r⊗Θ)⊙mask + w_l1·sign(Ξ)   (fp32 d×K, device)
 * xi is the UNMASKED parameter matrix, mask (d×K fp32, may be NULL) the sparsity mask. packed_out (2+d·K doubles,
 * required) also receives the raw sums of sb_train_step(LOSS|GRAD). For the specialised libraries this is two
 * launches: Ξ⊙mask into the constant bank, then the fused kernel whose last block writes loss and grad. */
int sb_closure(const float* x, const float* dx, int64_t n, const sb_library* lib, const float* xi,
               const float* mask, double w_l1, double* packed_out, float* loss_out, float* grad_out,
               void* workspace, int64_t workspace_bytes, void* stream);

/* sb_closure over samples sharded across `world` GPUs of one node, with the all-reduce INSIDE the kernel: the last
 * block of every rank sends each of its d·K+2 totals as one self-validating 16-byte line {lo32, epoch, hi32, epoch}
 * with a single peer store over NVLink into every rank's symmetric buffer, polls the lines of its own buffer until the
 * epochs of all senders match and adds them in rank order, then writes the GLOBAL loss and gradient (identical bits
 * on every rank) — no collective launch, no fence, one NVLink one-way latency. peer_bufs: host array of `world` device
 * pointers (peer-mapped, e.g. torch symmetric memory), each at least sb_peer_buffer_bytes(lib, world) bytes and
 * zero-filled before the first call; epoch_dev: TWO zero-initialised device uint32 owned by this rank — [0] the epoch
 * counter the kernel advances, [1] a sticky status word. Every rank must make the same sequence of calls. Only the
 * specialised (fused) libraries are supported: SB_ERR_UNSUPPORTED otherwise. packed_out receives the GLOBAL sums.
 * A lost peer makes the kernel give up after $SB_PEER_TIMEOUT_MS (default 30 000 ms) instead of hanging: the sums, loss
 * and gradient of that call are NaN (never a silently partial result), epoch_dev[1] is set to the epoch of the first
 * loss, and from then on sb_fit_step leaves xi, the optimiser state and the resident coefficients untouched — the host
 * checks epoch_dev[1] at its synchronisation points and re-synchronises the ranks before clearing it. */
int sb_closure_peer(const float* x, const float* dx, int64_t n, const sb_library* lib, const float* xi,
                    const float* mask, double w_l1, double* packed_out, float* loss_out, float* grad_out,
                    void* workspace, int64_t workspace_bytes, const void* const* peer_bufs, int world, int rank,
                    uint32_t* epoch_dev, void* stream);
int64_t sb_peer_buffer_bytes(const sb_library* lib, int world);

/* One whole iteration of the reference's Adam loop without sym-reg (`train.py:512-530`: forward, MSELoss, L1,
 * backward, optimizer.step()) as ONE kernel launch for the specialised libraries: the last block of the fused kernel
 * evaluates loss = w_mse·MSE + w_l1·‖Ξ‖₁ and its gradient (as sb_closure, at the parameters BEFORE the update), applies
 * the optimiser update to `xi` in place and packs the new Ξ⊙mask into the constant bank for the next call.
 *   SB_OPT_SGD : Ξ ← Ξ − lr·g
 *   SB_OPT_ADAM: torch.optim.Adam (no weight decay, no amsgrad) in fp32 with the same operation order:
 *                m ← lerp(m, g, 1−β1); v ← β2·v + (1−β2)·g²; Ξ ← Ξ − lr/(1−β1ᵗ) · m / (√v/√(1−β2ᵗ) + eps)
 * opt_state (Adam only): 2·d·K floats [m | v] followed by one uint32 step counter t (all zero before the first step;
 * the kernel advances t). call_flags: SB_FIT_W_RESIDENT promises that the resident slot of the constant bank still holds
 * Ξ⊙mask of THESE parameters — true right after sb_load_w or after the previous sb_fit_step on the same device and
 * stream, provided xi/mask were not modified by the caller and no OTHER fit (sb_fit_step / sb_load_w with other
 * parameters) ran on the device in between; the stateless entry points never touch the resident slot. Without the flag
 * the call packs Ξ⊙mask first (one more launch). peer_bufs/world/rank/epoch_dev as in
 * sb_closure_peer (world ≤ 1: single GPU, peer_bufs/epoch_dev may be NULL): every rank applies the identical update to
 * its replica of Ξ from the identical all-reduced gradient. Libraries without a specialised kernel, or misaligned
 * inputs: SB_ERR_UNSUPPORTED (use sb_closure + the framework's optimiser). */
#define SB_OPT_NONE 0
#define SB_OPT_SGD 1
#define SB_OPT_ADAM 2
#define SB_FIT_W_RESIDENT 1u
typedef struct {
  int32_t kind;  /* SB_OPT_SGD / SB_OPT_ADAM */
  float lr;
  float beta1;   /* Adam; torch defaults 0.9, 0.999, 1e-8 */
  float beta2;
  float eps;
  float w_mse;   /* w_sindy_x */
  float w_l1;    /* w_sindy_reg */
  float w_sym;   /* weight of the linear Lie-derivative regulariser (0 = none) */
  const float* sym_quad; /* device, (d·K)×(d·K) fp32 symmetric H (16-byte aligned) with
                            Σ_v Σ_n ‖J_h(z_n)(v z_n) − v h(z_n)‖² = wᵀHw, w = vec(Ξ⊙mask) row-major (`train.py:503-507`,
                            intended formula; H = Σ_v L_vᵀ(I_d⊗ΘᵀΘ)L_v is a constant of the data set, built once per fit);
                            NULL = no regulariser. Loss and gradient gain w_sym·wᵀHw and w_sym·2Hw⊙mask. */
} sb_fit_options;
int sb_fit_step(const float* x, const float* dx, int64_t n, const sb_library* lib, float* xi, const float* mask,
                const sb_fit_options* opt, float* opt_state, double* packed_out, float* loss_out, float* grad_out,
                void* workspace, int64_t workspace_bytes, const void* const* peer_bufs, int world, int rank,
                uint32_t* epoch_dev, uint32_t call_flags, void* stream);
/* Ξ⊙mask (mask may be NULL) into the resident slot of the constant bank: makes SB_FIT_W_RESIDENT true for the next
 * sb_fit_step after the caller changed xi or mask (e.g. `set_threshold`, `sindy.py:192-195`) or after another fit
 * used the slot. */
int sb_load_w(const sb_library* lib, const float* xi, const float* mask, void* stream);

/* The same epilogue applied to packed sums that were combined across GPUs (all-reduce(sum) of
 * sb_train_step's output): loss_out / grad_out as in sb_closure (either may be NULL). */
int sb_step_epilogue(const double* packed, const sb_library* lib, const float* xi, const float* mask,
                     double w_l1, float* loss_out, float* grad_out, void* stream);

/* Name of the kernel variant sb_train_step would dispatch for this library ("fused_tma<3,5>",
 * "generic" ...). Static string. */
const char* sb_train_step_variant(const sb_library* lib, uint32_t flags);

/* Fused kernels of the symmetry regularisers (config 3, `lv/noise99_eq_isymreg.cfg`), for the libraries
 * sb_symreg_supported() reports (d, poly_order, sin, exp) ∈ {(2,2,0,0), (2,2,0,1), (2,3,0,0), (3,2,0,0), (3,3,0,0)};
 * other libraries: SB_ERR_UNSUPPORTED (the host side then composes sb_forward / sb_jvp / sb_jvp_backward through
 * autograd like the reference composes its tensor ops).
 *  - sb_euler_flow: fx = f(x), the flow map of n_steps explicit-Euler steps x ← x + dt·Θ(x)Wᵀ (`model_utils.py:236-240`
 *    as called from `train.py:669-673`), and — when v is given — jv = J_f(x)·v (`model_utils.py:55-56`,
 *    `jvp(f, x, v_x)[1]`), both (n × d) fp32, one launch.
 *  - sb_euler_flow_backward: for cotangents g_fx, g_jv (either may be NULL) of those outputs: gw (d×K fp64) =
 *    dL/dW, gv (n × d fp32, may be NULL) = dL/dv = J_f(x)ᵀ g_jv, gx (n × d, may be NULL) = dL/dx; one launch
 *    (reverse sweep over the recomputed states, second derivatives of the library included). n_steps ≤ 32.
 *  - sb_symreg_r: the reversed regulariser with precomputed group action (`model_utils.py:126-170`; gx = g(x) (n × d),
 *    jgx = J_g(x) (n × d × d, row-major) as `precompute_symmreg_r` :172-211 provides them): out (fp64, d·K + 1) =
 *    [Σ_n (J_g(x_n)ᵀ r_n)_i Θ_k(x_n) − r_{n,i} Θ_k(g(x_n))  (d×K) | Σ_n ‖r_n‖²],  r_n = J_g(x_n) h(x_n) − h(g(x_n)):
 *    loss = out[d·K]/(n·d) and dL/dW = 2·out[:d·K]/(n·d) per group element, in one streaming pass. */
int sb_symreg_supported(const sb_library* lib);
int sb_euler_flow(const float* x, const float* v, int64_t n, const sb_library* lib, const float* w, float dt,
                  int n_steps, float* fx, float* jv, void* stream);
int sb_euler_flow_backward(const float* x, const float* v, const float* g_fx, const float* g_jv, int64_t n,
                           const sb_library* lib, const float* w, float dt, int n_steps, double* gw, float* gv,
                           float* gx, void* workspace, int64_t workspace_bytes, void* stream);
int sb_symreg_r(const float* x, const float* gx, const float* jgx, int64_t n, const sb_library* lib, const float* w,
                double* out, void* workspace, int64_t workspace_bytes, void* stream);

/* Fixed-step rollout of dx/dt = Θ(x)·Wᵀ for every initial condition in lock-step.
 *  - `model_utils.py:223-255` odeint (dtype SB_F32; method SB_EULER / SB_RK4; record_dx = 0):
 *      states after step s for s = stride, 2·stride, ... are written to x_out[(s/stride − 1), ic, :]
 *      (x0 itself is NOT stored, as `full_traj` there); x_last (n_ics×d, may be NULL) gets the final state.
 *  - `data_utils/ode.py:7-28` solve_ode_batch (dtype SB_F64, SB_RK4, record_dx = 1):
 *      n_steps counts stored rows INCLUDING x0: row s (s % stride == 0) holds x after s steps and
 *      dx_out the RHS there; only n_steps − 1 updates are made.
 * x0, w, outputs are float or double according to `dtype`. Outputs have leading dimension
 * n_rows = rows stored, then n_ics, then d. x_out / dx_out may be NULL. */
int sb_rollout(const void* x0, int64_t n_ics, const sb_library* lib, const void* w, double dt,
               int64_t n_steps, int64_t stride, int method, int dtype, int record_dx,
               void* x_out, void* dx_out, void* x_last, void* stream);

/* Fused rollout and scoring of many models (model selection along a threshold path, Mangan et al. 2017): for every
 * (model m, initial condition n) integrate dx/dt = Θ(x)·W_mᵀ from x0[n] (fp32, SB_EULER / SB_RK4, the operation order of
 * sb_rollout's odeint mode) and, after every `steps_per_row` steps r = 1..n_rows, add
 * Σ_j ((double)x_j − (double)y_obs[r−1, n, j])² (the row sum formed in j order) to sse[m, n] in row order (fp64). A pair
 * stops at the first row whose state has a non-finite component or |x_j| > blowup (blowup ≤ 0: no bound);
 * valid_rows[m, n] = rows compared before that (n_rows if none), sse holds those rows only. The compared states are
 * bit-identical to the rows sb_rollout(x0, W_m, dt, n_rows·steps_per_row, stride = steps_per_row) stores.
 * w: n_models × d × K fp32 (already masked). y_obs: n_rows × n_ics × d (the x_out layout of sb_rollout, x0 excluded).
 * sse, valid_rows: n_models × n_ics. One thread owns a pair: no atomics; a pair's outputs have the same bits alone, in
 * any batch, in any model order and on every repeat. SB_ERR_INVALID for a NULL pointer, n_ics < 0, n_models < 1,
 * steps_per_row < 1, n_rows outside 1..INT32_MAX, an unknown method or dt not > 0 (n_ics = 0 is a no-op);
 * SB_ERR_UNSUPPORTED for a library sb_library_size rejects. */
int sb_rollout_score(const float* x0, int64_t n_ics, const sb_library* lib, const float* w, int n_models, double dt,
                     int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs, float blowup,
                     double* sse, int32_t* valid_rows, void* stream);

/* Gradient of the fused scores (trajectory refit of the candidates): with the arguments of sb_rollout_score, sse and
 * valid_rows are bit-identical to what sb_rollout_score returns, and grad (n_models × d × K fp64) = ∂/∂W_m of
 * Σ_n sse[m, n], the SSE as reported: a pair that stopped after valid_rows[m, n] = v rows contributes the gradient of its
 * sum over rows 1..v (nothing for v = 0). It is the discrete adjoint of the fp32 recurrence that was scored (same step,
 * same right-hand side), so it is exact up to fp32 rounding of the reverse sweep; the per-thread sums are added in fp64
 * every 32 steps. No atomics on values: a model's gradient has the same bits alone, in any batch, in any model order and
 * on every repeat (it may change in the last bits when the ICs are split into different batches).
 * ws: device workspace of at least sb_rollout_score_grad_workspace_bytes(n_ics, lib, n_models, steps_per_row, n_rows)
 * bytes (the state every 32 steps of every pair, fp32, and one fp64 d×K row per model and block of 64 ICs); it need not
 * be initialised. SB_ERR_WORKSPACE if it is shorter; otherwise the status codes of sb_rollout_score, and NULL grad or ws
 * is SB_ERR_INVALID. n_ics = 0 sets grad to 0. The workspace size is negative (a status) for invalid sizes. */
int64_t sb_rollout_score_grad_workspace_bytes(int64_t n_ics, const sb_library* lib, int n_models,
                                              int64_t steps_per_row, int64_t n_rows);
int sb_rollout_score_grad(const float* x0, int64_t n_ics, const sb_library* lib, const float* w, int n_models,
                          double dt, int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs,
                          float blowup, double* sse, int32_t* valid_rows, double* grad, void* ws, int64_t ws_bytes,
                          void* stream);

/* sb_rollout_score with per-model initial conditions (output-error fits that estimate each trajectory's start):
 * x0_per_model = 0 is sb_rollout_score (x0: n_ics × d, shared by all models; the same bits), 1 reads model m's starts
 * from x0 + m·n_ics·d (x0: n_models × n_ics × d). A pair's outputs depend only on its own start, W_m and the data.
 * SB_ERR_INVALID for x0_per_model outside {0, 1}; otherwise the status codes of sb_rollout_score. */
int sb_rollout_score_ics(const float* x0, int x0_per_model, int64_t n_ics, const sb_library* lib, const float* w,
                         int n_models, double dt, int64_t steps_per_row, int64_t n_rows, int method,
                         const float* y_obs, float blowup, double* sse, int32_t* valid_rows, void* stream);

/* sb_rollout_score_grad with per-model initial conditions (x0_per_model as in sb_rollout_score_ics) and the gradient
 * with respect to them: grad_x0 (n_models × n_ics × d fp64) = ∂sse[m, n]/∂x0 of the pair (m, n), the adjoint state after
 * the first step is reversed, widened from fp32. A pair with valid_rows = 0 gets exact zeros. Each element has one
 * writer and no sum, so its bits do not depend on the batch, the model order or how the ICs are split. grad and grad_x0
 * may each be NULL: with grad NULL the kernel keeps no W̄ accumulators and reduces nothing (the start-only variant,
 * same sse / valid_rows / grad_x0 bits). Both NULL, or x0_per_model outside {0, 1}, is SB_ERR_INVALID; the workspace
 * size and the other status codes are those of sb_rollout_score_grad. sb_rollout_score_grad is this call with
 * x0_per_model = 0 and grad_x0 = NULL. */
int sb_rollout_score_grad_ics(const float* x0, int x0_per_model, int64_t n_ics, const sb_library* lib, const float* w,
                              int n_models, double dt, int64_t steps_per_row, int64_t n_rows, int method,
                              const float* y_obs, float blowup, double* sse, int32_t* valid_rows, double* grad,
                              double* grad_x0, void* ws, int64_t ws_bytes, void* stream);

/* Most tangent columns of sb_rollout_score_gn: n_params, plus d when the start blocks are requested. (3,5)'s full
 * d·K = 168 coefficients and 3 starts need 171. */
#define SB_GN_MAX_COLS 176

/* Gauss–Newton information of the fused scores (coefficient standard errors of a trajectory refit, Cov(θ) ≈
 * σ̂²·(JᵀJ)⁻¹): with the arguments of sb_rollout_score_ics, sse and valid_rows are bit-identical to what it returns, and
 * for the n_params coefficients params[m, ·] of each model (int32 indices into the flat d×K W_m, −1 = padding) with
 * J = ∂x_r/∂θ at every compared row r ≤ valid_rows of a pair and E = x_r − y_r:
 *   jtj (n_models × n_params × n_params fp64, symmetric) = Σ_n Σ_r JᵀJ,   jtr (n_models × n_params fp64) = Σ_n Σ_r JᵀE.
 * With jtj_px, jtj_xx and jtr_x (all given or all NULL) the start x0 of each pair is a parameter too, J_x = ∂x_r/∂x0:
 *   jtj_px (n_models × n_ics × n_params × d) = Σ_r JᵀJ_x,  jtj_xx (n_models × n_ics × d × d) = Σ_r J_xᵀJ_x,
 *   jtr_x (n_models × n_ics × d) = Σ_r J_xᵀE,  per pair.
 * J is the tangent-linear of the fp32 recurrence that was scored (same step, same right-hand side), so it is its exact
 * derivative up to fp32 rounding. Rows and columns of padded indices, and every block of a pair with valid_rows = 0,
 * are exact zeros. Each row's products are summed in fp32 over a block's pairs and added to fp64 sums in a fixed order
 * with no atomics on values: a model's outputs have the same bits alone, in any batch, in any model order and on every
 * repeat (for the same n_params and n_ics). It costs about n_params'·2d² + d library sweeps per RK4 stage and pair and
 * n_params'²·d per compared row, n_params' = n_params (+ d).
 * ws: device workspace of at least sb_rollout_score_gn_workspace_bytes(n_ics, lib, n_models, n_params, x0_blocks)
 * bytes (one fp64 row of n_params(n_params+1)/2 + n_params sums per model and block of at most 32 per model); it need
 * not be initialised; SB_ERR_WORKSPACE if it is shorter. SB_ERR_INVALID for the size and pointer errors of
 * sb_rollout_score_ics, n_params < 1, only some of the start outputs given, or an index outside [−1, d·K) (params are
 * read back to the host for this check: the call synchronises the stream); SB_ERR_UNSUPPORTED for n_params (+ d) above
 * SB_GN_MAX_COLS. n_ics = 0 sets jtj and jtr to 0. The workspace size is negative (a status) for invalid sizes. */
int64_t sb_rollout_score_gn_workspace_bytes(int64_t n_ics, const sb_library* lib, int n_models, int n_params,
                                            int x0_blocks);
int sb_rollout_score_gn(const float* x0, int x0_per_model, int64_t n_ics, const sb_library* lib, const float* w,
                        int n_models, const int32_t* params, int n_params, double dt, int64_t steps_per_row,
                        int64_t n_rows, int method, const float* y_obs, float blowup, double* sse,
                        int32_t* valid_rows, double* jtj, double* jtr, double* jtj_px, double* jtj_xx, double* jtr_x,
                        void* ws, int64_t ws_bytes, void* stream);

/* WSINDy weak-form integrals with trigonometric test functions (`sindy.py:332-347,361-362`):
 *   V[j,t]  = dt·sqrt(2/T)·sin((j+1)π t/T),  V'[j,t] = dt·sqrt(2/T)·(j+1)π/T·cos((j+1)π t/T),  t = t_idx·dt
 *   G[traj,j,k] = sum_t V[j,t]·Θ_k(x[traj,t]),   b[traj,j,i] = −sum_t V'[j,t]·x[traj,t,i]
 * x is (n_traj × T × d); test functions are generated on the fly in fp32 with the reference's
 * operation order. G (n_traj×n_test×K) and b (n_traj×n_test×d) are fp64. */
int sb_wsindy_integrals(const float* x, int64_t n_traj, int64_t T, const sb_library* lib, float dt,
                        double t_max, int n_test, double* G, double* b, void* stream);

/* WSINDy weak-form integrals with compactly supported test functions (Messenger & Bortz, Weak SINDy for ODEs, 2021):
 * every test function is the same window of `support` = L samples at its own start
 *   s_j = ⌊j·(T−L)/(n_test−1)⌋ (s_0 = 0 when n_test = 1),
 *   G[traj,j,k] = sum_q phi[q]·Θ_k(x[traj, s_j+q]),   b[traj,j,i] = −sum_q dphi[q]·x[traj, s_j+q, i],  q = 0..L−1.
 * phi, dphi: device arrays of L floats, the rows' values on their support with dt folded in (for the piecewise
 * polynomial family of WSINDyWrapper(test_func_family='poly'): phi[q] = fp32(dt·c·φ_q), dphi[q] = fp32(dt·c·φ'_q),
 * φ_q = (4u(1−u))^p, u = q/(L−1), c = 1/sqrt(dt·Σφ²)). x is (n_traj × T × d); G (n_traj×n_test×K) and b
 * (n_traj×n_test×d) are fp64. Sums run in fp32 over blocks of at most 2048 consecutive support samples, then in fp64;
 * no atomics: G[traj] and b[traj] have the same bits alone, in any batch and on every repeat.
 * SB_ERR_INVALID unless 3 ≤ L ≤ T and 1 ≤ n_test ≤ T − L + 1, or for a NULL pointer (n_traj = 0 is a no-op);
 * SB_ERR_UNSUPPORTED for a library sb_library_size rejects. */
int sb_wsindy_local_integrals(const float* x, int64_t n_traj, int64_t T, const sb_library* lib, const float* phi,
                              const float* dphi, int support, int n_test, double* G, double* b, void* stream);

/* Frozen-MLP chains on the tensor cores (SURVEY §8f-3): the encoder / decoder of the frozen autoencoder
 * (`autoencoder.py:38-66`: Linear [+ BatchNorm in eval mode, folded into the weights by the host] + ReLU, hidden width a
 * multiple of 256, thin first / last layers of width ≤ 8) as evaluated inside `symmreg_i` / `symmreg_f` /
 * `precompute_symmreg_r` (`model_utils.py:8-211`): values, Jacobian-vector products (`jvp(autoencoder.decoder, z, v)`,
 * `autoencoder.py:110-113, 132`) and the transpose products `loss.backward()` needs. Every wide layer is
 *   C = epilogue(A · Bᵀ),  A (m × k), B (n × k) frozen,  epilogue ∈ {0: + bias, 1: ReLU(· + bias), 2: ReLU mask of
 *   another activation tensor R (C = R > 0 ? · : 0)}  — tangents use B = W, R = this layer's value output; cotangents
 *   use B = Wᵀ, R = the layer's value input —
 * computed by one persistent tcgen05 kernel in 3×TF32 (fp32-faithful). Activations are kept in HBM in the PANEL FORMAT
 * the tensor core consumes: sb_mlp_panel_bytes(m, f) bytes for an (m × f) tensor (rows padded to 128; per 128-row tile and
 * 16-feature block a contiguous 16 KB [tf32-hi | lo] pair in the canonical K-major core-matrix layout), so that a
 * layer's epilogue writes the next layer's operand and the operand ring is filled by plain bulk copies.
 *  - sb_mlp_pack_weights: B (n × k) from w: transpose = 0: w is B row-major (B[i][j] = w[i·k + j]); transpose = 1: w is Bᵀ
 *    row-major (B[i][j] = w[j·n + i]). packed: 8·n·k bytes. n a multiple of 256, k a multiple of 256 (≤ 2048).
 *  - sb_mlp_pack_rows / sb_mlp_unpack_rows: (m × f) row-major fp32 ↔ panel format (tests, wide inputs).
 *  - sb_mlp_thin_in: C = epilogue(x · wᵀ [+ bias]), x (m × in_dim ≤ 8) row-major, w (f × in_dim), panel-format output.
 *  - sb_mlp_thin_out: y (m × out_dim ≤ 8, row-major) = A · wᵀ [+ bias], A in panel format, w (out_dim × f).
 *  - sb_mlp_gemm: the wide layer above; bias (n floats) and mask_panel may be NULL as the mode allows.
 *  - sb_mlp_gemm_out: the wide layer with the thin OUTPUT layer fused into its epilogue: y (m × out_dim) = C · w_outᵀ
 *    [+ bias_out], w_out (out_dim × n) row-major; c_panel may be NULL when the wide activations are not needed
 *    afterwards (tangent and cotangent chains). partials: scratch of sb_mlp_partials_bytes(m, n, out_dim) bytes — per
 *    64-column granule the row's partial products, added in granule order by a second tiny launch, so y does not
 *    depend on how tiles were scheduled.
 * All pointers to panel / packed buffers must be 16-byte aligned. */
int64_t sb_mlp_panel_bytes(int64_t m, int f);
int sb_mlp_pack_weights(const float* w, int n, int k, int transpose, void* packed, void* stream);
int sb_mlp_pack_rows(const float* x, int64_t m, int f, void* panel, void* stream);
int sb_mlp_unpack_rows(const void* panel, int64_t m, int f, float* x, void* stream);
int sb_mlp_thin_in(const float* x, int64_t m, int in_dim, const float* w, const float* bias, const void* mask_panel,
                   int f, int mode, void* c_panel, void* stream);
int sb_mlp_thin_out(const void* a_panel, int64_t m, int f, const float* w, const float* bias, int out_dim, float* y,
                    void* stream);
int sb_mlp_gemm(const void* a_panel, int64_t m, int k, const void* w_packed, int n, const float* bias,
                const void* mask_panel, int mode, void* c_panel, void* stream);
int64_t sb_mlp_partials_bytes(int64_t m, int n, int out_dim);
int sb_mlp_gemm_out(const void* a_panel, int64_t m, int k, const void* w_packed, int n, const float* bias,
                    const void* mask_panel, int mode, void* c_panel, const float* w_out, const float* bias_out,
                    int out_dim, void* partials, float* y, void* stream);

/* Debug/profiling aid: while dev_buf (device memory, 16 uint64 per CTA, at least 16·592 words) is set, every fused
 * kernel launched afterwards records %globaltimer stamps of its phases per CTA: 0 entry, 1 first tile landed, 2 end of
 * the sample loop, 3 partial written + ticket taken, and for the last block 4 totals ready, 5 after the peer exchange,
 * 6 end of the epilogue, 7 = SM id, 8 partial rows staged in shared memory, 9 rows summed. NULL switches it off (default). Not thread-safe; tools/trace_fused.py reads it. */
void sb_debug_trace(void* dev_buf);

/* FP32 FMA-pipe peak microbenchmark used for the roofline denominator (not in MEASURED_PEAKS.json):
 * variant 0 = scalar FFMA, 1 = packed FFMA2 (fma.rn.f32x2), 2 = FFMA2 with a constant-bank operand; design probes in the
 * same unit (2 x lane-operations/s): 3 = warp shuffles only, 4 = variant 2 with one SHFL per 4 FFMA2 (FFMA2 counted).
 * Runs on `stream`, writes the achieved TFLOP/s (2 flop per lane-FMA) to *tflops_host. Synchronises. */
int sb_fp32_peak(int variant, int iters, double* tflops_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SINDY_B200_H */
