// sb_common.cuh — shared internals of libsindy_b200.so (not part of the ABI).
//
// Library enumeration follows the reference's `sindy.py:7-30` (SINDyConst/Poly1/Poly2/Poly3/Sine/Exp):
// degree-n monomials over non-decreasing index tuples in lexicographic order, each formed left to right,
// i.e. column(i1..in) = column(i1..i(n-1)) * x[in]. That recurrence (parent column, variable) is the only
// table the kernels need: values, Jacobian-vector and Hessian-vector sweeps all run over it.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include <utility>

#include "../../include/sindy_b200.h"

namespace sb {

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define SB_CUDA_TRY(expr)                                         \
  do {                                                            \
    cudaError_t _e = (expr);                                      \
    if (_e != cudaSuccess) return ::sb::cuda_fail(_e, #expr);     \
  } while (0)

// every kernel launch of the library goes through this check; it also feeds sb_kernel_launches()
void count_launch();
#define SB_LAUNCH_CHECK(name)                                     \
  do {                                                            \
    cudaError_t _e = cudaGetLastError();                          \
    if (_e != cudaSuccess) return ::sb::cuda_fail(_e, name);      \
    ::sb::count_launch();                                         \
  } while (0)

// ---------------------------------------------------------------------------------------------
// runtime library table (kernel parameter of the generic kernels; ~540 bytes)
// ---------------------------------------------------------------------------------------------
struct LibTab {
  int d;       // state dimension
  int K;       // total columns
  int n_poly;  // polynomial columns (1 + d + ...)
  int sine;    // 0/1
  int exp_;    // 0/1
  unsigned char parent[SB_MAX_TERMS];  // parent column of polynomial column k (k > d)
  unsigned char var[SB_MAX_TERMS];     // variable multiplied onto the parent
};

// Number of monomials of degree exactly n in d variables: C(n+d-1, d-1).
constexpr int n_monomials(int d, int n) {
  long long r = 1;
  for (int i = 1; i <= d - 1; ++i) r = r * (n + i) / i;
  return (int)r;
}
constexpr int n_poly_terms(int d, int p) {
  int k = 0;
  for (int n = 0; n <= p; ++n) k += n_monomials(d, n);
  return k;
}

// Validates `lib` and fills `tab`. Returns SB_OK or an error status.
int build_table(const sb_library* lib, LibTab* tab);

// ---------------------------------------------------------------------------------------------
// compile-time library tables for the specialised kernels
// ---------------------------------------------------------------------------------------------
template <int D, int P>
struct PolyTab {
  static constexpr int K = n_poly_terms(D, P);
  int parent[K];
  int var[K];
  int degree[K];
  int block_begin[P + 2];  // first column of each degree block; block_begin[P+1] = K
};

template <int D, int P>
constexpr PolyTab<D, P> make_poly_tab() {
  PolyTab<D, P> t{};
  constexpr int K = PolyTab<D, P>::K;
  int last[K] = {};  // last (largest) variable index of each column's tuple
  t.parent[0] = 0; t.var[0] = 0; t.degree[0] = 0; last[0] = 0;
  t.block_begin[0] = 0;
  t.block_begin[1] = 1;
  int k = 1;
  for (int j = 0; j < D; ++j) { t.parent[k] = 0; t.var[k] = j; t.degree[k] = 1; last[k] = j; ++k; }
  for (int n = 2; n <= P; ++n) {
    t.block_begin[n] = k;
    const int pb = t.block_begin[n - 1], pe = k;
    for (int p = pb; p < pe; ++p)
      for (int j = last[p]; j < D; ++j) { t.parent[k] = p; t.var[k] = j; t.degree[k] = n; last[k] = j; ++k; }
  }
  t.block_begin[P + 1] = k;
  return t;
}

template <int D, int P>
struct Poly {
  static constexpr int K = PolyTab<D, P>::K;
  static constexpr PolyTab<D, P> tab = make_poly_tab<D, P>();
};

// compile-time loop: f(std::integral_constant<int, I>) for I in [B, E)
template <int B, int E, class F>
__host__ __device__ __forceinline__ void static_for(F&& f) {
  if constexpr (B < E) {
    f(std::integral_constant<int, B>{});
    static_for<B + 1, E>(static_cast<F&&>(f));
  }
}

// Θ(x) for a polynomial library, fully unrolled: m[k] = m[parent] * x[var]  (`sindy.py:13-24`)
template <int D, int P, class T>
__device__ __forceinline__ void expand_poly(const T (&x)[D], T (&m)[Poly<D, P>::K]) {
  using L = Poly<D, P>;
  m[0] = T(1);
  static_for<0, D>([&](auto j) { m[1 + j] = x[j]; });
  static_for<1 + D, L::K>([&](auto kc) {
    constexpr int k = kc;
    constexpr int p = L::tab.parent[k];
    constexpr int v = L::tab.var[k];
    m[k] = m[p] * x[v];
  });
}

// Library CODE of the specialised kernels: PC = poly_order + 10·include_exp + 20·include_sine, so that the polynomial
// shapes keep their plain degree (PC = P) and config 3's library (degree 2 + exp) is PC = 12.
template <int D, int PC>
struct LibCode {
  static constexpr int P = PC % 10;
  static constexpr int E = (PC / 10) % 2;
  static constexpr int S = PC / 20;
  static constexpr int NP = Poly<D, P>::K;
  static constexpr int K = NP + D * (S + E);
};
template <int D, int PC>
__host__ __device__ inline bool lib_matches(const LibTab& t) {
  using L = LibCode<D, PC>;
  return t.d == D && t.n_poly == L::NP && (t.sine != 0) == (L::S != 0) && (t.exp_ != 0) == (L::E != 0);
}
// Θ(x) for a library code: the polynomial block, then sin(x_j), then exp(x_j) (`sindy.py:7-30`); sin / exp are
// sinf / expf for float by overload
template <int D, int PC, class T>
__device__ __forceinline__ void expand_lib(const T (&x)[D], T (&m)[LibCode<D, PC>::K]) {
  using L = LibCode<D, PC>;
  if constexpr (L::S == 0 && L::E == 0) {
    expand_poly<D, L::P>(x, m);
  } else {
    T mp[L::NP];
    expand_poly<D, L::P>(x, mp);
    static_for<0, L::NP>([&](auto k) { m[k] = mp[k]; });
    if constexpr (L::S) static_for<0, D>([&](auto j) { m[L::NP + j] = sin(x[j]); });
    if constexpr (L::E) static_for<0, D>([&](auto j) { m[L::NP + D * L::S + j] = exp(x[j]); });
  }
}
// Θ(x) for a runtime table, in the same column order; m holds at least t.K values
template <class T>
__device__ __forceinline__ void expand_table(const LibTab& t, const T* x, T* m) {
  m[0] = T(1);
  for (int j = 0; j < t.d; ++j) m[1 + j] = x[j];
  for (int k = 1 + t.d; k < t.n_poly; ++k) m[k] = m[t.parent[k]] * x[t.var[k]];
  int k = t.n_poly;
  if (t.sine) for (int j = 0; j < t.d; ++j) m[k++] = sin(x[j]);
  if (t.exp_) for (int j = 0; j < t.d; ++j) m[k++] = exp(x[j]);
}

// Value-only reverse sweep of expand_lib: xb += J_Θ(x)ᵀ·mb for the cotangent mb on Θ(x) (consumed: the parents' entries
// receive their children's contributions). m = Θ(x). m_k = m_p·x_v gives mb_p += mb_k·x_v and xb_v += mb_k·m_p.
template <int D, int PC, class T>
__device__ __forceinline__ void reverse_lib(const T (&x)[D], const T (&m)[LibCode<D, PC>::K],
                                            T (&mb)[LibCode<D, PC>::K], T (&xb)[D]) {
  using L = LibCode<D, PC>;
  using Tab = Poly<D, L::P>;
  constexpr int NP = L::NP;
  if constexpr (L::S) static_for<0, D>([&](auto j) { xb[j] = fma(mb[NP + j], cos(x[j]), xb[j]); });
  if constexpr (L::E) static_for<0, D>([&](auto j) { xb[j] = fma(mb[NP + D * L::S + j], m[NP + D * L::S + j], xb[j]); });
  static_for<0, NP - 1 - D>([&](auto qc) {
    constexpr int k = NP - 1 - qc;  // NP-1 down to D+1
    constexpr int p = Tab::tab.parent[k], v = Tab::tab.var[k];
    mb[p] = fma(mb[k], x[v], mb[p]);
    xb[v] = fma(mb[k], m[p], xb[v]);
  });
  static_for<0, D>([&](auto j) { xb[j] += mb[1 + j]; });
}
// the same sweep over a runtime table; m, mb hold t.K values, x, xb t.d
template <class T>
__device__ __forceinline__ void reverse_table(const LibTab& t, const T* x, const T* m, T* mb, T* xb) {
  int k = t.n_poly;
  if (t.sine) for (int j = 0; j < t.d; ++j, ++k) xb[j] = fma(mb[k], cos(x[j]), xb[j]);
  if (t.exp_) for (int j = 0; j < t.d; ++j, ++k) xb[j] = fma(mb[k], m[k], xb[j]);
  for (k = t.n_poly - 1; k > t.d; --k) {
    const int p = t.parent[k], v = t.var[k];
    mb[p] = fma(mb[k], x[v], mb[p]);
    xb[v] = fma(mb[k], m[p], xb[v]);
  }
  for (int j = 0; j < t.d; ++j) xb[j] += mb[1 + j];
}

// ---------------------------------------------------------------------------------------------
// reductions
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Transposed butterfly reduction of V per-lane values across the 32 lanes of a warp with ~V shuffles instead of
// 5·V: at every step a lane keeps one half of its values and trades the other half with its partner. V must be a
// multiple of 32. Afterwards v[0 .. V/32) of lane L hold the warp-wide sums of the original indices
//   i + (L&16 ? V/2 : 0) + (L&8 ? V/4 : 0) + (L&4 ? V/8 : 0) + (L&2 ? V/16 : 0) + (L&1 ? V/32 : 0),  i < V/32.
template <int V, int O = 16>
__device__ __forceinline__ void warp_fold(float (&v)[V], int lane) {
  static_assert(V % 32 == 0, "pad the value count to a multiple of 32");
  if constexpr (O >= 1) {
    constexpr int LIVE = V * O / 16;  // live values halve each step: V, V/2, ..., V/16
    constexpr int H = LIVE / 2;
    const bool up = (lane & O) != 0;
    static_for<0, H>([&](auto ic) {
      constexpr int i = ic;
      const float lo = v[i], hi = v[i + H];
      const float recv = __shfl_xor_sync(0xffffffffu, up ? lo : hi, O);
      v[i] = (up ? hi : lo) + recv;
    });
    warp_fold<V, O / 2>(v, lane);
  }
}
// original index of v[i] (i < V/32) held by `lane` after warp_fold<V>
template <int V>
__device__ __forceinline__ int warp_fold_index(int i, int lane) {
  return i + ((lane & 16) ? V / 2 : 0) + ((lane & 8) ? V / 4 : 0) + ((lane & 4) ? V / 8 : 0) +
         ((lane & 2) ? V / 16 : 0) + ((lane & 1) ? V / 32 : 0);
}

// Workspace header: one ticket counter (must be zero before the first call; every reducing kernel
// resets it before exiting), padded to 256 bytes; partial sums follow.
constexpr int64_t kWsHeaderBytes = 256;

// Grid-size cap used by every reducing kernel (partials per output row).
constexpr int kMaxPartialBlocks = 148 * 4;

// ---------------------------------------------------------------------------------------------
// constant-memory coefficient slots (W = Ξ⊙mask), filled by stream-ordered D2D copies
// ---------------------------------------------------------------------------------------------
constexpr int kConstW = SB_MAX_DIM * SB_MAX_TERMS;  // 2048 floats = 8 KB

// ---------------------------------------------------------------------------------------------
// internal entry points (one per translation unit)
// ---------------------------------------------------------------------------------------------
// generic (runtime-table) path
int generic_theta(const float* x, int64_t n, const LibTab& t, float* theta, cudaStream_t s);
int generic_forward(const float* x, int64_t n, const LibTab& t, const float* w, float* y, cudaStream_t s);
int generic_jvp(const float* x, const float* u, int64_t n, const LibTab& t, const float* w, float* out,
                cudaStream_t s);
int generic_backward(const float* x, const float* gy, int64_t n, const LibTab& t, const float* w,
                     double* gw, float* gx, void* ws, int64_t ws_bytes, cudaStream_t s);
int generic_jvp_backward(const float* x, const float* u, const float* g, int64_t n, const LibTab& t,
                         const float* w, double* gw, float* gx, float* gu, void* ws, int64_t ws_bytes,
                         cudaStream_t s);
int generic_train_step(const float* x, const float* dx, int64_t n, const LibTab& t, const float* w,
                       uint32_t flags, double* out, void* ws, int64_t ws_bytes, cudaStream_t s);
int64_t generic_workspace_bytes(const LibTab& t);

// closure epilogue outputs (loss fp32 scalar, dL/dXi fp32 d×K) and the L1 weight
struct ClosureOut {
  double w_l1;
  float* loss;
  float* grad;
  double w_mse = 1.0;   // weight of the MSE term (w_sindy_x)
};
// optimiser update fused into the closure epilogue of the specialised kernel (sb_fit_step)
struct FitArgs {
  int kind = SB_OPT_NONE;
  float lr = 0.f, beta1 = 0.f, beta2 = 0.f, eps = 0.f;
  float* xi = nullptr;          // parameters, advanced in place
  float* m = nullptr;           // Adam first / second moments (d×K each)
  float* v = nullptr;
  unsigned int* step = nullptr; // Adam step counter (device)
  bool w_resident = false;      // the resident slot already holds Ξ⊙mask (left there by the previous fit step / sb_load_w)
  const float* sym_H = nullptr; // quadratic form of the linear Lie-derivative regulariser ((d·K)² fp32) or NULL
  double w_sym = 0.0;
};
// loss / gradient from (all-reduced) packed sums; one tiny launch
int step_epilogue(const double* packed, const LibTab& t, const float* xi, const float* mask, double w_l1,
                  float* loss_out, float* grad_out, cudaStream_t s);
// W = xi ⊙ mask into `dst` (d×K floats)
int mask_mul(const float* xi, const float* mask, float* dst, int count, cudaStream_t s);

// in-kernel all-reduce over peer-mapped symmetric buffers (one per rank; NVLink P2P). Layout of every buffer:
// [2 parities][world senders][d*K + 2 lines of 16 bytes {lo32, epoch, hi32, epoch}]. `epoch` is a local device
// counter the kernel advances itself (CUDA-graph replay safe).
struct PeerArgs {
  int world = 0;
  int rank = 0;
  double* buf[SB_MAX_PEERS] = {};
  unsigned int* epoch = nullptr;      // [0] epoch counter, [1] sticky status (0 = ok, else the epoch a peer was lost at)
  unsigned int* status = nullptr;     // = epoch + 1
  long long timeout_ticks = 0;        // clock64 ticks a rank waits for its peers before giving up
};

// specialised (compile-time library, register-resident, TMA-staged) fused train step.
// `w` is Ξ; `mask` (may be NULL) is multiplied in while packing W into the constant bank; `co` (may be NULL)
// requests the closure epilogue inside the kernel's last block.
bool fused_supported(const LibTab& t, uint32_t flags);
const char* fused_variant_name(const LibTab& t, uint32_t flags);
int fused_train_step(const float* x, const float* dx, int64_t n, const LibTab& t, const float* w, const float* mask,
                     uint32_t flags, double* out, const ClosureOut* co, const PeerArgs* peer, void* ws,
                     int64_t ws_bytes, cudaStream_t s, const FitArgs* fit = nullptr);
void fused_set_trace(unsigned long long* p);
// Ξ [⊙ mask] into the constant bank of the specialised kernels (one tiny launch)
int fused_load_w(const LibTab& t, const float* xi, const float* mask, cudaStream_t s);
int64_t fused_workspace_bytes(const LibTab& t);
// specialised per-sample forward and dL/dW (cotangent-weighted feature sums) for the same libraries
int fused_forward(const float* x, int64_t n, const LibTab& t, const float* w, float* y, cudaStream_t s);
int fused_weighted_sums(const float* x, const float* g, int64_t n, const LibTab& t, double* out, void* ws,
                        int64_t ws_bytes, cudaStream_t s);

// Gram ΘᵀΘ (K×K fp64) of a polynomial library from power sums; `header` (may be NULL) receives {0, n}
bool moments_supported(const LibTab& t);
int64_t moments_workspace_bytes(const LibTab& t);
int moments_gram(const float* x, int64_t n, const LibTab& t, double* gram_out, double* header, void* ws,
                 int64_t ws_bytes, cudaStream_t s);

// rollout
int rollout(const void* x0, int64_t n_ics, const LibTab& t, const void* w, double dt, int64_t n_steps,
            int64_t stride, int method, int dtype, int record_dx, void* x_out, void* dx_out, void* x_last,
            cudaStream_t s);

// M models × N ICs integrated and scored against observed rows with the rollout's own step and right-hand sides
// (sb_rollout.cu), so the compared states are the ones `rollout` stores; arguments validated by the caller. Model m starts
// from x0 + m·x0_model_stride (0: one start set shared by all models, n_ics·d: one set per model).
int rollout_score(const float* x0, int64_t x0_model_stride, int64_t n_ics, const LibTab& t, const float* w,
                  int n_models, double dt, int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs,
                  float blowup, double* sse, int32_t* valid_rows, cudaStream_t s);
// the same scores, ∂/∂W_m Σ_n sse[m, n] (grad) and ∂sse[m, n]/∂x0 of the pair (grad_x0, n_models × n_ics × d) by the
// discrete adjoint of the scored recurrence; either output may be NULL, not both. Arguments validated by the caller. The
// workspace size is -1 when it does not fit in int64.
int64_t rollout_score_grad_workspace_bytes(int64_t n_ics, const LibTab& t, int n_models, int64_t steps_per_row,
                                           int64_t n_rows);
int rollout_score_grad(const float* x0, int64_t x0_model_stride, int64_t n_ics, const LibTab& t, const float* w,
                       int n_models, double dt, int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs,
                       float blowup, double* sse, int32_t* valid_rows, double* grad, double* grad_x0, void* ws,
                       int64_t ws_bytes, cudaStream_t s);
// the same scores and the Gauss–Newton information of the listed coefficients (params: n_models × n_params indices
// into d×K, −1 padding) and, when jtj_px is given, of each pair's start, from tangent-linear rollouts. Arguments
// validated by the caller (n_params + start columns ≤ SB_GN_MAX_COLS). The workspace size is -1 when it does not fit
// in int64.
int64_t rollout_score_gn_workspace_bytes(int64_t n_ics, const LibTab& t, int n_models, int n_params, int x0_blocks);
int rollout_score_gn(const float* x0, int64_t x0_model_stride, int64_t n_ics, const LibTab& t, const float* w,
                     int n_models, const int32_t* params, int n_params, double dt, int64_t steps_per_row,
                     int64_t n_rows, int method, const float* y_obs, float blowup, double* sse, int32_t* valid_rows,
                     double* jtj, double* jtr, double* jtj_px, double* jtj_xx, double* jtr_x, void* ws,
                     int64_t ws_bytes, cudaStream_t s);

// WSINDy integrals
int wsindy_integrals(const float* x, int64_t n_traj, int64_t T, const LibTab& t, float dt, double t_max,
                     int n_test, double* G, double* b, cudaStream_t s);
// WSINDy integrals with compactly supported test functions (sb_wsindy_local.cu); sizes validated by the caller
int wsindy_local_integrals(const float* x, int64_t n_traj, int64_t T, const LibTab& t, const float* phi,
                           const float* dphi, int L, int n_test, double* G, double* b, cudaStream_t s);

// fused symmetry-regulariser kernels (sb_symreg.cu): Euler flow map with JVP and its reverse sweep, reversed regulariser
bool symreg_supported(const LibTab& t);
int64_t symreg_workspace_bytes(const LibTab& t);
int euler_flow(const float* x, const float* v, int64_t n, const LibTab& t, const float* w, float dt, int n_steps,
               float* fx, float* jv, cudaStream_t s);
int euler_flow_backward(const float* x, const float* v, const float* g_fx, const float* g_jv, int64_t n,
                        const LibTab& t, const float* w, float dt, int n_steps, double* gw, float* gv, float* gx,
                        void* ws, int64_t ws_bytes, cudaStream_t s);
int symreg_r(const float* x, const float* gx, const float* jg, int64_t n, const LibTab& t, const float* w,
             double* out, void* ws, int64_t ws_bytes, cudaStream_t s);

// tensor-core (tcgen05, 3xTF32) WSINDy integrals over many trajectories (sb_wsindy_tc.cu)
bool wsindy_tc_supported(const LibTab& t, int n_test);
int wsindy_integrals_tc(const float* x, int64_t n_traj, int64_t T, const LibTab& t, float dt, double t_max, int n_test,
                        double* G, double* b, cudaStream_t s);

// frozen-MLP chains on the tensor cores (sb_mlp.cu): panel-format activations, 3xTF32 tcgen05 GEMM with fused epilogue
int64_t mlp_panel_bytes(int64_t m, int f);
int mlp_pack_weights(const float* w, int n, int k, int transpose, void* packed, cudaStream_t s);
int mlp_pack_rows(const float* x, int64_t m, int f, void* packed, cudaStream_t s);
int mlp_unpack_rows(const void* packed, int64_t m, int f, float* x, cudaStream_t s);
int mlp_gemm(const void* a_panel, int64_t m, int k, const void* w_packed, int n, const float* bias,
             const void* mask_panel, int mode, void* c_panel, cudaStream_t s);
int64_t mlp_partials_bytes(int64_t m, int n, int out_dim);
int mlp_gemm_out(const void* a_panel, int64_t m, int k, const void* w_packed, int n, const float* bias,
                 const void* mask_panel, int mode, void* c_panel, const float* w_out, const float* bias_out,
                 int out_dim, void* partials, float* y, cudaStream_t s);
int mlp_thin_in(const float* x, int64_t m, int in_dim, const float* w, const float* bias, const void* mask_panel,
                int f, int mode, void* c_panel, cudaStream_t s);
int mlp_thin_out(const void* a_panel, int64_t m, int f, const float* w, const float* bias, int out_dim, float* y,
                 cudaStream_t s);

// FP32 peak microbenchmark
int fp32_peak(int variant, int iters, double* tflops_host, cudaStream_t s);

}  // namespace sb
