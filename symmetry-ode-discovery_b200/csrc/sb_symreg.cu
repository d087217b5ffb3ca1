// sb_symreg.cu — fused kernels of the symmetry regularisers of config 3 (`lv/noise99_eq_isymreg.cfg`) for compile-time
// libraries, polynomial AND with sin / exp columns.
//
//  * sb_euler_flow / sb_euler_flow_backward — the flow map f = n explicit-Euler steps of h(x) = Θ(x)·Wᵀ
//    (`model_utils.py:236-240`, called from `train.py:669-673`) together with its Jacobian-vector product J_f(x)·v
//    (`model_utils.py:55-56`: `jvp(f, x, v_x)`), and the reverse sweep that returns dL/dW, dL/dv [, dL/dx] for cotangents
//    on both outputs. The reference obtains J_f·v by the double-vjp trick through 10 Python Euler steps (two reverse
//    passes with create_graph=True, differentiated a third time by loss.backward()): ~200 small launches per closure.
//    Here one thread carries one sample through all steps: forward = 1 launch, backward = 1 launch (states recomputed
//    and kept in local memory, adjoint recursion with the Hessian-vector term, d×K sums reduced in fp64).
//      x_{s+1} = x_s + dt·W Θ(x_s)                     v_{s+1} = v_s + dt·W J_Θ(x_s) v_s
//      μ_s = μ_{s+1} + dt·J_h(x_s)ᵀ μ_{s+1}            λ_s = λ_{s+1} + dt·J_h(x_s)ᵀ λ_{s+1} + dt·[∂_x(J_h(x_s) v_s)]ᵀ μ_{s+1}
//      dW += dt·(λ_{s+1} ⊗ Θ(x_s) + μ_{s+1} ⊗ J_Θ(x_s) v_s),   dv = μ_0,   dx = λ_0
//  * sb_symreg_r — the reversed regulariser with precomputed group action (`model_utils.py:126-170` with g(x), J_g(x)
//    from `precompute_symmreg_r` :172-211): Σ_n Σ_i (J_g(x_n) h(x_n) − h(g(x_n)))_i² and its d×K gradient sums in ONE
//    streaming pass (two library evaluations and a d×d mat-vec per sample, 4·(2d + d²) bytes per sample).
//
// The library sweeps (value, tangent, reverse) run over the compile-time parent/variable recurrence of sb_common.cuh;
// everything stays in registers except the per-step states of the backward kernel.
#include "sb_common.cuh"

namespace sb {

namespace {

constexpr int kThreads = 128;

template <int D_, int P_, int S_, int E_>
struct Lib {
  static constexpr int D = D_, P = P_, S = S_, E = E_;
  static constexpr int NP = Poly<D, P>::K;
  static constexpr int K = NP + D * (S + E);
  using T = Poly<D, P>;

  __device__ static __forceinline__ void expand(const float (&x)[D], float (&m)[K]) {
    expand_lib<D, P + 10 * E + 20 * S>(x, m);
  }
  // t = J_Θ(x)·u (forward differentiation of the recurrence); cs = cos(x) when S
  __device__ static __forceinline__ void tangent(const float (&x)[D], const float (&u)[D], const float (&m)[K],
                                                 float (&t)[K]) {
    t[0] = 0.f;
    static_for<0, D>([&](auto j) { t[1 + j] = u[j]; });
    static_for<1 + D, NP>([&](auto kc) {
      constexpr int k = kc;
      constexpr int p = T::tab.parent[k], v = T::tab.var[k];
      t[k] = fmaf(t[p], x[v], m[p] * u[v]);
    });
    if constexpr (S) static_for<0, D>([&](auto j) { t[NP + j] = cosf(x[j]) * u[j]; });
    if constexpr (E) static_for<0, D>([&](auto j) { t[NP + D * S + j] = m[NP + D * S + j] * u[j]; });
  }
  // reverse sweep: cotangents mb on Θ(x) and tb on J_Θ(x)·u  ->  xb += ..., ub += ...  (mb, tb are consumed)
  __device__ static __forceinline__ void reverse(const float (&x)[D], const float (&u)[D], const float (&m)[K],
                                                 const float (&t)[K], float (&mb)[K], float (&tb)[K], float (&xb)[D],
                                                 float (&ub)[D]) {
    if constexpr (S) static_for<0, D>([&](auto jc) {
      constexpr int j = jc;
      const float sn = m[NP + j], cs = cosf(x[j]);
      xb[j] += mb[NP + j] * cs - tb[NP + j] * sn * u[j];
      ub[j] += tb[NP + j] * cs;
    });
    if constexpr (E) static_for<0, D>([&](auto jc) {
      constexpr int j = jc;
      constexpr int k = NP + D * S + j;
      xb[j] += mb[k] * m[k] + tb[k] * m[k] * u[j];
      ub[j] += tb[k] * m[k];
    });
    static_for<0, NP - 1 - D>([&](auto qc) {
      constexpr int k = NP - 1 - qc;          // NP-1 down to D+1
      constexpr int p = T::tab.parent[k], v = T::tab.var[k];
      // t_k = t_p x_v + m_p u_v ;  m_k = m_p x_v
      tb[p] = fmaf(tb[k], x[v], tb[p]);
      mb[p] = fmaf(tb[k], u[v], fmaf(mb[k], x[v], mb[p]));
      xb[v] = fmaf(tb[k], t[p], fmaf(mb[k], m[p], xb[v]));
      ub[v] = fmaf(tb[k], m[p], ub[v]);
    });
    static_for<0, D>([&](auto j) { xb[j] += mb[1 + j]; ub[j] += tb[1 + j]; });
  }
};

// ---- block / grid reduction of NV per-thread fp32 values into fp64 totals (ordered, deterministic) ---------------
struct RedArgs {
  double* partial;       // [grid][NV]
  unsigned int* ticket;
  double* out;           // [NV]
};

template <int NV>
__device__ __forceinline__ void reduce_to_out(const float (&v)[NV], const RedArgs& r) {
  constexpr int NW = kThreads / 32;
  __shared__ float red[NW][NV];
  __shared__ int is_last;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  static_for<0, NV>([&](auto e) {
    const float s = warp_sum(v[e]);
    if (lane == 0) red[wid][e] = s;
  });
  __syncthreads();
  double* mine = r.partial + (int64_t)blockIdx.x * NV;
  for (int e = threadIdx.x; e < NV; e += kThreads) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < NW; ++w) s += (double)red[w][e];
    mine[e] = s;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(r.ticket, 1u) == gridDim.x - 1u);
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  for (int e = threadIdx.x; e < NV; e += kThreads) {
    double s = 0.0;
    for (unsigned int b = 0; b < gridDim.x; ++b) s += __ldcg(r.partial + (int64_t)b * NV + e);
    r.out[e] = s;
  }
  if (threadIdx.x == 0) *r.ticket = 0u;
}

// ---- Euler flow: forward ------------------------------------------------------------------------------------------
template <class L>
__global__ void __launch_bounds__(kThreads) euler_flow_fwd_kernel(const float* __restrict__ x,
                                                                  const float* __restrict__ v, int64_t n,
                                                                  const float* __restrict__ w, float dt, int n_steps,
                                                                  float* __restrict__ fx, float* __restrict__ jv) {
  constexpr int D = L::D, K = L::K;
  __shared__ float sw[D * K];
  for (int e = threadIdx.x; e < D * K; e += kThreads) sw[e] = w[e];
  __syncthreads();
  for (int64_t s = (int64_t)blockIdx.x * kThreads + threadIdx.x; s < n; s += (int64_t)gridDim.x * kThreads) {
    float xs[D], vs[D];
    static_for<0, D>([&](auto q) { xs[q] = x[s * D + q]; vs[q] = v ? v[s * D + q] : 0.f; });
    for (int it = 0; it < n_steps; ++it) {
      float m[K], t[K];
      L::expand(xs, m);
      if (v) L::tangent(xs, vs, m, t);
      float h[D], jh[D];
      static_for<0, D>([&](auto ic) {
        constexpr int i = ic;
        float a = 0.f, b = 0.f;
        static_for<0, K>([&](auto k) { a = fmaf(sw[i * K + k], m[k], a); });
        if (v) static_for<0, K>([&](auto k) { b = fmaf(sw[i * K + k], t[k], b); });
        h[i] = a; jh[i] = b;
      });
      // x + dt*f(x) with the product rounded before the sum, like the reference's separate tensor ops
      static_for<0, D>([&](auto q) {
        xs[q] = __fadd_rn(xs[q], __fmul_rn(dt, h[q]));
        vs[q] = __fadd_rn(vs[q], __fmul_rn(dt, jh[q]));
      });
    }
    static_for<0, D>([&](auto q) { fx[s * D + q] = xs[q]; if (jv) jv[s * D + q] = vs[q]; });
  }
}

// ---- Euler flow: backward -----------------------------------------------------------------------------------------
constexpr int kMaxSteps = 32;

template <class L>
__global__ void __launch_bounds__(kThreads) euler_flow_bwd_kernel(const float* __restrict__ x,
                                                                  const float* __restrict__ v,
                                                                  const float* __restrict__ g_fx,
                                                                  const float* __restrict__ g_jv, int64_t n,
                                                                  const float* __restrict__ w, float dt, int n_steps,
                                                                  float* __restrict__ gv, float* __restrict__ gx,
                                                                  RedArgs red) {
  constexpr int D = L::D, K = L::K;
  __shared__ float sw[D * K];
  for (int e = threadIdx.x; e < D * K; e += kThreads) sw[e] = w[e];
  __syncthreads();
  float acc[D * K];
  static_for<0, D * K>([&](auto e) { acc[e] = 0.f; });
  for (int64_t s = (int64_t)blockIdx.x * kThreads + threadIdx.x; s < n; s += (int64_t)gridDim.x * kThreads) {
    float xh[kMaxSteps][D], vh[kMaxSteps][D];    // states BEFORE step it (local memory: indexed by the step)
    float xs[D], vs[D];
    static_for<0, D>([&](auto q) { xs[q] = x[s * D + q]; vs[q] = v ? v[s * D + q] : 0.f; });
    for (int it = 0; it < n_steps; ++it) {
      static_for<0, D>([&](auto q) { xh[it][q] = xs[q]; vh[it][q] = vs[q]; });
      float m[K], t[K];
      L::expand(xs, m);
      L::tangent(xs, vs, m, t);
      static_for<0, D>([&](auto ic) {
        constexpr int i = ic;
        float a = 0.f, b = 0.f;
        static_for<0, K>([&](auto k) { a = fmaf(sw[i * K + k], m[k], a); b = fmaf(sw[i * K + k], t[k], b); });
        xs[i] = __fadd_rn(xs[i], __fmul_rn(dt, a));
        vs[i] = __fadd_rn(vs[i], __fmul_rn(dt, b));
      });
    }
    float lam[D], mu[D];
    static_for<0, D>([&](auto q) {
      lam[q] = g_fx ? g_fx[s * D + q] : 0.f;
      mu[q] = g_jv ? g_jv[s * D + q] : 0.f;
    });
    for (int it = n_steps - 1; it >= 0; --it) {
      static_for<0, D>([&](auto q) { xs[q] = xh[it][q]; vs[q] = vh[it][q]; });
      float m[K], t[K], mb[K], tb[K];
      L::expand(xs, m);
      L::tangent(xs, vs, m, t);
      float dl[D], dm[D];
      static_for<0, D>([&](auto q) { dl[q] = dt * lam[q]; dm[q] = dt * mu[q]; });
      static_for<0, K>([&](auto kc) {
        constexpr int k = kc;
        float a = 0.f, b = 0.f;
        static_for<0, D>([&](auto ic) {
          constexpr int i = ic;
          a = fmaf(dl[i], sw[i * K + k], a);
          b = fmaf(dm[i], sw[i * K + k], b);
          acc[i * K + k] = fmaf(dl[i], m[k], fmaf(dm[i], t[k], acc[i * K + k]));
        });
        mb[k] = a; tb[k] = b;
      });
      float xb[D], ub[D];
      static_for<0, D>([&](auto q) { xb[q] = 0.f; ub[q] = 0.f; });
      L::reverse(xs, vs, m, t, mb, tb, xb, ub);
      static_for<0, D>([&](auto q) { lam[q] += xb[q]; mu[q] += ub[q]; });
    }
    static_for<0, D>([&](auto q) {
      if (gv) gv[s * D + q] = mu[q];
      if (gx) gx[s * D + q] = lam[q];
    });
  }
  reduce_to_out<D * K>(acc, red);
}

// ---- reversed regulariser with precomputed g(x), J_g(x) ----------------------------------------------------------------
template <class L>
__global__ void __launch_bounds__(kThreads) symreg_r_kernel(const float* __restrict__ x, const float* __restrict__ gx,
                                                            const float* __restrict__ jg, int64_t n,
                                                            const float* __restrict__ w, RedArgs red) {
  constexpr int D = L::D, K = L::K;
  __shared__ float sw[D * K];
  for (int e = threadIdx.x; e < D * K; e += kThreads) sw[e] = w[e];
  __syncthreads();
  float acc[D * K + 1];
  static_for<0, D * K + 1>([&](auto e) { acc[e] = 0.f; });
  for (int64_t s = (int64_t)blockIdx.x * kThreads + threadIdx.x; s < n; s += (int64_t)gridDim.x * kThreads) {
    float xs[D], gs[D], J[D][D];
    static_for<0, D>([&](auto q) { xs[q] = x[s * D + q]; gs[q] = gx[s * D + q]; });
    static_for<0, D>([&](auto a) { static_for<0, D>([&](auto b) { J[a][b] = jg[(s * D + a) * D + b]; }); });
    float m[K], mg[K];
    L::expand(xs, m);
    L::expand(gs, mg);
    float h[D], hg[D];
    static_for<0, D>([&](auto ic) {
      constexpr int i = ic;
      float a = 0.f, b = 0.f;
      static_for<0, K>([&](auto k) { a = fmaf(sw[i * K + k], m[k], a); b = fmaf(sw[i * K + k], mg[k], b); });
      h[i] = a; hg[i] = b;
    });
    float r[D], q[D];
    static_for<0, D>([&](auto ac) {
      constexpr int a = ac;
      float p = 0.f;
      static_for<0, D>([&](auto b) { p = fmaf(J[a][b], h[b], p); });
      r[a] = p - hg[a];
      acc[D * K] = fmaf(r[a], r[a], acc[D * K]);
    });
    static_for<0, D>([&](auto ic) {                      // q = J_gᵀ r
      constexpr int i = ic;
      float p = 0.f;
      static_for<0, D>([&](auto a) { p = fmaf(J[a][i], r[a], p); });
      q[i] = p;
    });
    static_for<0, D>([&](auto ic) {
      constexpr int i = ic;
      static_for<0, K>([&](auto k) { acc[i * K + k] = fmaf(q[i], m[k], fmaf(-r[i], mg[k], acc[i * K + k])); });
    });
  }
  reduce_to_out<D * K + 1>(acc, red);
}

int grid_for(int64_t n) {
  int64_t g = (n + kThreads - 1) / kThreads;
  if (g > 148 * 8) g = 148 * 8;
  return g < 1 ? 1 : (int)g;
}

int red_setup(RedArgs* r, int grid, int nv, double* out, void* ws, int64_t ws_bytes) {
  const int64_t need = kWsHeaderBytes + (int64_t)grid * nv * (int64_t)sizeof(double);
  if (ws_bytes < need) {
    set_error("workspace too small: %lld < %lld bytes", (long long)ws_bytes, (long long)need);
    return SB_ERR_WORKSPACE;
  }
  r->ticket = reinterpret_cast<unsigned int*>(ws);
  r->partial = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + kWsHeaderBytes);
  r->out = out;
  return SB_OK;
}

// the specialised libraries: (d, poly_order, sine, exp)
#define SB_SYMREG_SHAPES(X) X(2, 2, 0, 0) X(2, 2, 0, 1) X(2, 3, 0, 0) X(3, 2, 0, 0) X(3, 3, 0, 0)
#define SB_MATCH(D, P, S, E) (t.d == D && t.n_poly == n_poly_terms(D, P) && t.sine == S && t.exp_ == E)

}  // namespace

bool symreg_supported(const LibTab& t) {
#define X(D, P, S, E) if (SB_MATCH(D, P, S, E)) return true;
  SB_SYMREG_SHAPES(X)
#undef X
  return false;
}

int64_t symreg_workspace_bytes(const LibTab& t) {
  return kWsHeaderBytes + (int64_t)148 * 8 * ((int64_t)t.d * t.K + 1) * (int64_t)sizeof(double);
}

int euler_flow(const float* x, const float* v, int64_t n, const LibTab& t, const float* w, float dt, int n_steps,
               float* fx, float* jv, cudaStream_t s) {
#define X(D, P, S, E)                                                                                         \
  if (SB_MATCH(D, P, S, E)) {                                                                                 \
    euler_flow_fwd_kernel<Lib<D, P, S, E>><<<grid_for(n), kThreads, 0, s>>>(x, v, n, w, dt, n_steps, fx, jv); \
    SB_LAUNCH_CHECK("euler_flow_fwd_kernel");                                                                 \
    return SB_OK;                                                                                             \
  }
  SB_SYMREG_SHAPES(X)
#undef X
  set_error("no fused Euler flow for d=%d K=%d", t.d, t.K);
  return SB_ERR_UNSUPPORTED;
}

int euler_flow_backward(const float* x, const float* v, const float* g_fx, const float* g_jv, int64_t n,
                        const LibTab& t, const float* w, float dt, int n_steps, double* gw, float* gv, float* gx,
                        void* ws, int64_t ws_bytes, cudaStream_t s) {
  if (n_steps > kMaxSteps) { set_error("n_steps=%d > %d", n_steps, kMaxSteps); return SB_ERR_UNSUPPORTED; }
  const int grid = grid_for(n);
  RedArgs r{};
  int st = red_setup(&r, grid, t.d * t.K, gw, ws, ws_bytes);
  if (st != SB_OK) return st;
#define X(D, P, S, E)                                                                                      \
  if (SB_MATCH(D, P, S, E)) {                                                                              \
    euler_flow_bwd_kernel<Lib<D, P, S, E>><<<grid, kThreads, 0, s>>>(x, v, g_fx, g_jv, n, w, dt, n_steps, gv, gx, r); \
    SB_LAUNCH_CHECK("euler_flow_bwd_kernel");                                                              \
    return SB_OK;                                                                                          \
  }
  SB_SYMREG_SHAPES(X)
#undef X
  set_error("no fused Euler flow for d=%d K=%d", t.d, t.K);
  return SB_ERR_UNSUPPORTED;
}

int symreg_r(const float* x, const float* gx, const float* jg, int64_t n, const LibTab& t, const float* w,
             double* out, void* ws, int64_t ws_bytes, cudaStream_t s) {
  const int grid = grid_for(n);
  RedArgs r{};
  int st = red_setup(&r, grid, t.d * t.K + 1, out, ws, ws_bytes);
  if (st != SB_OK) return st;
#define X(D, P, S, E)                                                                        \
  if (SB_MATCH(D, P, S, E)) {                                                                \
    symreg_r_kernel<Lib<D, P, S, E>><<<grid, kThreads, 0, s>>>(x, gx, jg, n, w, r);          \
    SB_LAUNCH_CHECK("symreg_r_kernel");                                                      \
    return SB_OK;                                                                            \
  }
  SB_SYMREG_SHAPES(X)
#undef X
  set_error("no fused reversed regulariser for d=%d K=%d", t.d, t.K);
  return SB_ERR_UNSUPPORTED;
}

}  // namespace sb
