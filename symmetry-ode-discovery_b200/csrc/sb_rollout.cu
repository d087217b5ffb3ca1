// sb_rollout.cu — lock-step fixed-step integration of dx/dt = Θ(x)·Wᵀ for a batch of initial conditions (sb_rollout),
// M models × N initial conditions integrated and scored against observed rows in one launch (sb_rollout_score), and
// the gradient of those scores with respect to every model's W by the discrete adjoint (sb_rollout_score_grad).
//
// Two reference functions share the rollout kernels:
//   * `model_utils.py:223-255` odeint(f, x0, t, dt, method, full_traj): torch fp32, Euler or classic RK4,
//     trajectory WITHOUT x0;
//   * `data_utils/ode.py:7-28` solve_ode_batch: NumPy float64 RK4 that also records dx = f(x) at every stored
//     row (row 0 = x0) and makes num_steps-1 updates.
// One thread integrates its initial conditions for all steps: the state, the 4 stage derivatives and the K
// monomials stay in registers; the only HBM traffic is the strided trajectory store (and x0). The update formulas
// reproduce the reference's operation order with explicit round-to-nearest mul/add (no FMA contraction across the
// reference's separate tensor ops), so that fp32 rollouts track torch's and fp64 rollouts track NumPy's to rounding.
//
// Model selection simulates every candidate Ξ of a threshold path from every validation initial condition and compares
// the states with the data. With sb_rollout that is one launch, one HBM trajectory and one reduction per model; the
// scoring kernels instead fold each compared row into an fp64 SSE in registers: the only HBM traffic is x0, the
// observed rows (shared by all models, so L2-resident for cfg-sized data) and two outputs per pair. They run the same
// odeint step and the same right-hand side as the rollout kernel launch_rollout picks for the library, so the states
// they compare are bit-identical to the rows sb_rollout stores. Where W comes from does not enter the arithmetic.
#include <cstdlib>

#include "sb_common.cuh"

namespace sb {

namespace {

constexpr int kThreads = 128;

__constant__ double c_rw[kConstW];  // W as float or double (reinterpreted), 16 KB

template <class T> __device__ __forceinline__ T mul_rn(T a, T b);
template <> __device__ __forceinline__ float mul_rn<float>(float a, float b) { return __fmul_rn(a, b); }
template <> __device__ __forceinline__ double mul_rn<double>(double a, double b) { return __dmul_rn(a, b); }
template <class T> __device__ __forceinline__ T add_rn(T a, T b);
template <> __device__ __forceinline__ float add_rn<float>(float a, float b) { return __fadd_rn(a, b); }
template <> __device__ __forceinline__ double add_rn<double>(double a, double b) { return __dadd_rn(a, b); }
template <class T> __device__ __forceinline__ T div_rn(T a, T b);
template <> __device__ __forceinline__ float div_rn<float>(float a, float b) { return __fdiv_rn(a, b); }
template <> __device__ __forceinline__ double div_rn<double>(double a, double b) { return __ddiv_rn(a, b); }

// ---- fp32 Θ(x)·Wᵀ in packed pairs -------------------------------------------------------------------------------
// W delivery. The coefficient pairs are loop-invariant, so ptxas either keeps all of them in vector registers or, when
// an opaque offset `off` (always 0, unknown to the compiler, different per call site) defeats the hoisting, reloads
// every pair inside the time loop.
//   * One IC per thread (rollout_spec_kernel): W from the constant bank at offset 0, hoisted. For d=3, K=56 that is
//     164 registers and 3 blocks of 128 threads per SM; the opaque offset there (52 registers, 9 blocks per SM) costs
//     one indexed LDCU.64 per packed FMA and was measured SLOWER (73.1 ms against 67.9 for 1e6 ICs x 2000 steps):
//     issue-bound. Inline `ld.const` with immediate addresses is hoisted by ptxas just the same.
//   * NB = 2 ICs per thread (rollout_rk4_multi_kernel): the constant bank with the opaque offset. Every loaded pair
//     feeds NB packed FMAs (uniform-register operands), the thread needs ~100 registers and carries two independent
//     dependency chains.
//   * The scorer: the models are produced on the device (STLSQ), so their W cannot become kernel parameters without a
//     device-to-host copy and a host synchronisation per call, and the per-module constant slot would be shared by
//     concurrent streams. Each block stages its model's W (≤ 168 floats) in shared memory and reads it as float4 (two
//     pairs) with a block-uniform address, so one LDS.128 feeds 2·NB packed FMAs; the opaque offset again keeps ptxas
//     from hoisting the loads into registers it does not have.

// pair kk of output i: W[i][2kk], W[i][2kk+1], K/2 pairs per output
template <int K>
struct ConstW {
  const float2* w2;  // c_rw [+ opaque offset]
  template <int I, int KK> __device__ __forceinline__ float2 pair(float4&) const { return w2[I * (K / 2) + KK]; }
};
// D rows of KQ float4 (K/2 pairs, zero-padded to an even count); q carries the float4 loaded for an even pair to the
// odd pair after it
template <int K>
struct SharedW {
  static constexpr int KQ = (K / 2 + 1) / 2;
  const float4* w4;  // block-staged W [+ opaque offset]
  template <int I, int KK> __device__ __forceinline__ float2 pair(float4& q) const {
    if constexpr (KK % 2 == 0) {
      q = w4[I * KQ + KK / 2];
      return make_float2(q.x, q.y);
    } else {
      return make_float2(q.z, q.w);
    }
  }
};

// f = Θ(x)·Wᵀ for NB states of library code PC (sb_common.cuh LibCode): per state and output, pair kk is accumulated
// with fma.rn.f32x2 into s0 (kk even) or s1 (kk odd), f = (s0.x + s0.y) + (s1.x + s1.y). The monomials are formed in
// column order and each pair is consumed as soon as both its columns exist.
template <int D, int PC, int NB, class W>
__device__ __forceinline__ void eval_pairs(const W& w, const float (&x)[NB][D], float (&f)[NB][D]) {
  using L = LibCode<D, PC>;
  using Tab = Poly<D, L::P>;
  constexpr int NP = L::NP, K = L::K;
  static_assert(K % 2 == 0, "packed pairs");
  float m[NB][K];
  float2 s0[NB][D], s1[NB][D];
  float4 wq[D];
  static_for<0, NB>([&](auto b) {
    static_for<0, D>([&](auto i) { s0[b][i] = make_float2(0.f, 0.f); s1[b][i] = make_float2(0.f, 0.f); });
  });
  static_for<0, K>([&](auto kc) {
    constexpr int k = kc;
    static_for<0, NB>([&](auto bc) {
      constexpr int b = bc;
      if constexpr (k == 0) m[b][0] = 1.f;
      else if constexpr (k <= D) m[b][k] = x[b][k - 1];
      else if constexpr (k < NP) {
        constexpr int pk = Tab::tab.parent[k];
        constexpr int vk = Tab::tab.var[k];
        m[b][k] = m[b][pk] * x[b][vk];
      } else if constexpr (k < NP + D * L::S) m[b][k] = sinf(x[b][k - NP]);
      else m[b][k] = expf(x[b][k - NP - D * L::S]);
    });
    if constexpr (k % 2 == 1) {
      constexpr int kk = k / 2;
      static_for<0, D>([&](auto ic) {
        constexpr int i = ic;
        const float2 wp = w.template pair<i, kk>(wq[i]);
        float2 (&s)[NB][D] = kk % 2 == 0 ? s0 : s1;
        static_for<0, NB>([&](auto b) { s[b][i] = __ffma2_rn(wp, make_float2(m[b][k - 1], m[b][k]), s[b][i]); });
      });
    }
  });
  static_for<0, NB>([&](auto b) {
    static_for<0, D>([&](auto i) { f[b][i] = (s0[b][i].x + s0[b][i].y) + (s1[b][i].x + s1[b][i].y); });
  });
}

// ---- right-hand sides of the one-IC kernels -------------------------------------------------------------------------
// specialised: compile-time library, W from the constant bank
template <int D, int PC, class T>
struct SpecRhs {
  static constexpr int DN = D;
  static constexpr int K = LibCode<D, PC>::K;
  static_assert(K % 2 == 0, "every specialised library has an even K: fp32 evaluates packed pairs only");
  __device__ __forceinline__ int dim() const { return D; }
  // `off` (always 0, opaque, different per call site) only matters in fp64: it keeps ptxas from hoisting coefficient
  // loads out of the time loop into registers it does not have (168 registers + spills -> 136, none)
  __device__ __forceinline__ void eval(const T (&x)[D], T (&f)[D], int off = 0) const {
    if constexpr (std::is_same<T, float>::value) {
      eval_pairs<D, PC, 1>(ConstW<K>{reinterpret_cast<const float2*>(c_rw)},
                           reinterpret_cast<const float (&)[1][D]>(x), reinterpret_cast<float (&)[1][D]>(f));
    } else {
      T m[K];
      expand_lib<D, PC>(x, m);
      const T* w = reinterpret_cast<const T*>(c_rw) + 2 * off;
      static_for<0, D>([&](auto ic) {
        constexpr int i = ic;
        // two partial sums (even / odd columns) keep the dependent chain short
        T s0 = T(0), s1 = T(0);
        static_for<0, K>([&](auto kc) {
          constexpr int k = kc;
          if constexpr (k % 2 == 0) s0 = fma(w[i * K + k], m[k], s0);
          else s1 = fma(w[i * K + k], m[k], s1);
        });
        f[i] = s0 + s1;
      });
    }
  }
};

// generic: runtime table, W from global memory, one fma chain per output
template <class T, int KMAX>
struct GenRhs {
  static constexpr int DN = SB_MAX_DIM;
  const LibTab& t;
  const T* w;
  __device__ __forceinline__ int dim() const { return t.d; }
  __device__ __forceinline__ void eval(const T (&x)[SB_MAX_DIM], T (&f)[SB_MAX_DIM], int = 0) const {
    T m[KMAX];
    expand_table(t, x, m);
    for (int i = 0; i < t.d; ++i) {
      T s = T(0);
      for (int q = 0; q < t.K; ++q) s = fma(__ldg(w + i * t.K + q), m[q], s);
      f[i] = s;
    }
  }
};

// ---- the odeint step ------------------------------------------------------------------------------------------------
// `model_utils.py:236-253`: x + dt*k1, or RK4 with x + dt/2*k1 etc.; the python scalars dt/2, dt/6 are rounded to T once.
// f(y, k, stage) evaluates the right-hand side of the NB states y into k; stage = 0..3 numbers the RK4 evaluations.
template <class T>
struct Odeint {
  T dt, hdt, sdt;
  __device__ __forceinline__ explicit Odeint(double h) : dt((T)h), hdt((T)(h / 2.0)), sdt((T)(h / 6.0)) {}

  template <int NB, int DN, class F>
  __device__ __forceinline__ void step(int method, T (&x)[NB][DN], F&& f) const {
    T k1[NB][DN], k2[NB][DN], k3[NB][DN], k4[NB][DN], xt[NB][DN];
    auto from_x = [&](T (&y)[NB][DN], T h, const T (&k)[NB][DN]) {
      static_for<0, NB>([&](auto b) { static_for<0, DN>([&](auto j) { y[b][j] = add_rn(x[b][j], mul_rn(h, k[b][j])); }); });
    };
    f(x, k1, 0);
    if (method == SB_EULER) {
      from_x(x, dt, k1);
      return;
    }
    from_x(xt, hdt, k1);
    f(xt, k2, 1);
    from_x(xt, hdt, k2);
    f(xt, k3, 2);
    from_x(xt, dt, k3);
    f(xt, k4, 3);
    const T two = T(2);
    static_for<0, NB>([&](auto b) {
      static_for<0, DN>([&](auto j) {
        T acc = add_rn(k1[b][j], mul_rn(two, k2[b][j]));
        acc = add_rn(acc, mul_rn(two, k3[b][j]));
        acc = add_rn(acc, k4[b][j]);
        x[b][j] = add_rn(x[b][j], mul_rn(sdt, acc));
      });
    });
  }
};

// ---- rollout --------------------------------------------------------------------------------------------------------
struct RollArgs {
  const void* x0;
  int64_t n_ics;
  double dt;
  int64_t n_steps;
  int64_t stride;
  int method;
  int record_dx;
  long long opaque;   // always 0, unknown to the compiler: see the W delivery note
  void* x_out;
  void* dx_out;
  void* x_last;
};

template <class RHS, class T>
__device__ __forceinline__ void rollout_body(const RHS& rhs, const RollArgs& a) {
  constexpr int DN = RHS::DN;
  const int d = rhs.dim();
  const int64_t ic = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (ic >= a.n_ics) return;
  const T* x0 = reinterpret_cast<const T*>(a.x0);
  T* xo = reinterpret_cast<T*>(a.x_out);
  T* dxo = reinterpret_cast<T*>(a.dx_out);
  T xs[1][DN];         // the odeint step works on rows of states: here one
  T (&x)[DN] = xs[0];
#pragma unroll
  for (int j = 0; j < DN; ++j) x[j] = (j < d) ? x0[ic * d + j] : T(0);

  const Odeint<T> ode(a.dt);
  const int64_t row_elems = a.n_ics * d;
  auto store = [&](T* base, int64_t row, const T (&v)[DN]) {
#pragma unroll
    for (int j = 0; j < DN; ++j)
      if (j < d) base[row * row_elems + ic * d + j] = v[j];
  };

  if (a.record_dx) {
    // `data_utils/ode.py:14-26`: k_i = dt*f(.), x += (k1 + 2k2 + 2k3 + k4)/6, rows include x0
    T k1[DN], k2[DN], k3[DN], k4[DN], xt[DN];
    const T dt = ode.dt, half = T(0.5), two = T(2), six = T(6);
    int64_t row = 0, until = 0;   // next stored row and steps until it (no 64-bit division in the step loop)
    for (int64_t i = 0; i < a.n_steps; ++i) {
      rhs.eval(x, k1, (int)(i & a.opaque));
      if (until == 0) {
        if (xo) store(xo, row, x);
        if (dxo) store(dxo, row, k1);
        ++row;
        until = a.stride;
      }
      --until;
      if (i == a.n_steps - 1) break;
      if (a.method == SB_EULER) {
#pragma unroll
        for (int j = 0; j < DN; ++j) x[j] = add_rn(x[j], mul_rn(dt, k1[j]));
        continue;
      }
#pragma unroll
      for (int j = 0; j < DN; ++j) { k1[j] = mul_rn(dt, k1[j]); xt[j] = add_rn(x[j], mul_rn(half, k1[j])); }
      rhs.eval(xt, k2, (int)((i + 1) & a.opaque));
#pragma unroll
      for (int j = 0; j < DN; ++j) { k2[j] = mul_rn(dt, k2[j]); xt[j] = add_rn(x[j], mul_rn(half, k2[j])); }
      rhs.eval(xt, k3, (int)((i + 2) & a.opaque));
#pragma unroll
      for (int j = 0; j < DN; ++j) { k3[j] = mul_rn(dt, k3[j]); xt[j] = add_rn(x[j], k3[j]); }
      rhs.eval(xt, k4, (int)((i + 3) & a.opaque));
#pragma unroll
      for (int j = 0; j < DN; ++j) {
        k4[j] = mul_rn(dt, k4[j]);
        T s = add_rn(k1[j], mul_rn(two, k2[j]));
        s = add_rn(s, mul_rn(two, k3[j]));
        s = add_rn(s, k4[j]);
        x[j] = add_rn(x[j], div_rn(s, six));
      }
    }
  } else {
    int64_t row = 0, until = a.stride;   // next stored row and steps until it (no 64-bit division in the step loop)
    for (int64_t s = 1; s <= a.n_steps; ++s) {
      ode.step(a.method, xs, [&](const auto& y, auto& k, int st) { rhs.eval(y[0], k[0], (int)((s + st) & a.opaque)); });
      if (--until == 0) {
        if (xo) store(xo, row, x);
        ++row;
        until = a.stride;
      }
    }
  }
  if (a.x_last) {
    T* xl = reinterpret_cast<T*>(a.x_last);
#pragma unroll
    for (int j = 0; j < DN; ++j)
      if (j < d) xl[ic * d + j] = x[j];
  }
}

template <int D, int P, class T, int S = 0, int E = 0>
__global__ void __launch_bounds__(kThreads) rollout_spec_kernel(RollArgs a) {
  SpecRhs<D, P + 10 * E + 20 * S, T> rhs;
  rollout_body<SpecRhs<D, P + 10 * E + 20 * S, T>, T>(rhs, a);
}

template <class T, int KMAX>
__global__ void __launch_bounds__(kThreads) rollout_gen_kernel(LibTab t, const T* w, RollArgs a) {
  GenRhs<T, KMAX> rhs{t, w};
  rollout_body<GenRhs<T, KMAX>, T>(rhs, a);
}

// Blocks of kMultiThreads = 64 threads (128 initial conditions): with the whole batch resident at once — 1e6 / 8 ICs per
// GPU in the sharded C5 rollout is two thirds of one wave — the SM loads differ by at most one block, and the run time is
// set by the fullest SM: 128-thread blocks gave 489 blocks over 148 SMs = 3 or 4 per SM (+21 % on the slowest, measured
// as 6.58x at 8 GPUs instead of 8x); 64-thread blocks give 6 or 7. The scorer's blocks have the same shape.
constexpr int kMultiThreads = 64;
constexpr int kMultiNB = 2;

// fp32 RK4 (odeint layout) of a polynomial library, NB initial conditions per thread
template <int D, int P, int NB>
__global__ void __launch_bounds__(kMultiThreads) rollout_rk4_multi_kernel(RollArgs a) {
  constexpr int kThreads = kMultiThreads;
  constexpr int K = Poly<D, P>::K;
  const int64_t base = (int64_t)blockIdx.x * (kThreads * NB) + threadIdx.x;
  if (base >= a.n_ics) return;
  const float* x0 = reinterpret_cast<const float*>(a.x0);
  float* xo = reinterpret_cast<float*>(a.x_out);
  float x[NB][D];
  bool live[NB];
  static_for<0, NB>([&](auto bc) {
    constexpr int b = bc;
    const int64_t ic = base + (int64_t)b * kThreads;
    live[b] = ic < a.n_ics;
    static_for<0, D>([&](auto j) { x[b][j] = live[b] ? x0[ic * D + j] : 0.f; });
  });
  const Odeint<float> ode(a.dt);
  const int64_t row_elems = a.n_ics * D;
  int64_t row = 0, until = a.stride;
  for (int64_t s = 1; s <= a.n_steps; ++s) {
    ode.step(SB_RK4, x, [&](const auto& y, auto& k, int st) {
      eval_pairs<D, P, NB>(ConstW<K>{reinterpret_cast<const float2*>(c_rw) + 2 * (int)((s + st) & a.opaque)}, y, k);
    });
    if (--until == 0) {
      if (xo) {
        static_for<0, NB>([&](auto bc) {
          constexpr int b = bc;
          const int64_t ic = base + (int64_t)b * kThreads;
          if (live[b]) static_for<0, D>([&](auto j) { xo[row * row_elems + ic * D + j] = x[b][j]; });
        });
      }
      ++row;
      until = a.stride;
    }
  }
  if (a.x_last) {
    float* xl = reinterpret_cast<float*>(a.x_last);
    static_for<0, NB>([&](auto bc) {
      constexpr int b = bc;
      const int64_t ic = base + (int64_t)b * kThreads;
      if (live[b]) static_for<0, D>([&](auto j) { xl[ic * D + j] = x[b][j]; });
    });
  }
}

// ---- scoring --------------------------------------------------------------------------------------------------------
constexpr int kMaxGridY = 65535;

struct ScoreArgs {
  const float* x0;   // starts of the first model of this launch
  int64_t x0_model_stride;   // elements from one model's starts to the next: 0 (shared) or n_ics·d
  int64_t n_ics;
  double dt;
  int64_t steps_per_row;
  int64_t n_rows;
  const float* y_obs;
  float blowup;
  long long opaque;  // always 0, unknown to the compiler
  const float* w;    // W of the first model of this launch (n_models × d × K)
  double* sse;       // of the first model of this launch
  int32_t* valid;
};

// Compares one state with its observed row: false (and no change) if the state is non-finite or beyond the bound,
// otherwise sse += Σ_j ((double)x_j − (double)y_j)², the row sum formed in j order first.
template <int DN>
__device__ __forceinline__ bool score_row(const float (&x)[DN], int d, const float* y, float blowup, double& sse) {
  bool ok = true;
#pragma unroll
  for (int j = 0; j < DN; ++j)
    if (j < d) ok = ok && isfinite(x[j]) && !(blowup > 0.f && fabsf(x[j]) > blowup);
  if (!ok) return false;
  double r = 0.0;
#pragma unroll
  for (int j = 0; j < DN; ++j)
    if (j < d) {
      const double e = __dadd_rn((double)x[j], -(double)__ldg(y + j));
      r = __dadd_rn(r, __dmul_rn(e, e));
    }
  sse = __dadd_rn(sse, r);
  return true;
}

// grid = (IC blocks, models); NB ICs per thread, W staged in shared memory. The states are those of the rollout kernel
// for the same library: rollout_rk4_multi_kernel (RK4, polynomial) or rollout_spec_kernel (Euler, or (2,2)+exp).
template <int D, int PC, int METHOD>
__global__ void __launch_bounds__(kMultiThreads) rollout_score_spec_kernel(ScoreArgs a) {
  constexpr int kThreads = kMultiThreads, NB = kMultiNB;
  constexpr int K = LibCode<D, PC>::K, KQ = SharedW<K>::KQ;
  __shared__ float4 sw[D * KQ];
  const int64_t model = blockIdx.y;
  {
    const float* wm = a.w + model * (D * K);
    float* s = reinterpret_cast<float*>(sw);
    for (int q = threadIdx.x; q < D * KQ * 4; q += kThreads) {
      const int i = q / (KQ * 4), c = q % (KQ * 4);
      s[q] = c < K ? wm[i * K + c] : 0.f;
    }
  }
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * (kThreads * NB) + threadIdx.x;
  if (base >= a.n_ics) return;
  const float* x0 = a.x0 + model * a.x0_model_stride;
  float x[NB][D];
  bool track[NB];
  double sse[NB];
  int64_t valid[NB];
  static_for<0, NB>([&](auto bc) {
    constexpr int b = bc;
    const int64_t ic = base + (int64_t)b * kThreads;
    track[b] = ic < a.n_ics;
    sse[b] = 0.0;
    valid[b] = a.n_rows;
    static_for<0, D>([&](auto j) { x[b][j] = track[b] ? x0[ic * D + j] : 0.f; });
  });
  const bool live1 = track[1];
  const Odeint<float> ode(a.dt);
  const int64_t row_elems = a.n_ics * D;
  int64_t row = 0, until = a.steps_per_row;
  for (int64_t s = 1;; ++s) {
    ode.step(METHOD, x, [&](const auto& y, auto& k, int st) {
      eval_pairs<D, PC, NB>(SharedW<K>{sw + (int)((s + st) & a.opaque)}, y, k);
    });
    if (--until == 0) {
      const float* y = a.y_obs + row * row_elems;
      static_for<0, NB>([&](auto bc) {
        constexpr int b = bc;
        const int64_t ic = base + (int64_t)b * kThreads;
        if (track[b] && !score_row<D>(x[b], D, y + ic * D, a.blowup, sse[b])) { track[b] = false; valid[b] = row; }
      });
      ++row;
      until = a.steps_per_row;
      if (row == a.n_rows || !(track[0] || track[1])) break;
    }
  }
  static_for<0, NB>([&](auto bc) {
    constexpr int b = bc;
    const int64_t ic = base + (int64_t)b * kThreads;
    if (b == 0 || live1) {
      a.sse[model * a.n_ics + ic] = sse[b];
      a.valid[model * a.n_ics + ic] = (int32_t)valid[b];
    }
  });
}

// Runtime-table library: GenRhs with the model's W, one IC per thread, as rollout_gen_kernel.
template <int KMAX>
__global__ void __launch_bounds__(kThreads) rollout_score_gen_kernel(LibTab t, int method, ScoreArgs a) {
  constexpr int DN = SB_MAX_DIM;
  const int64_t ic = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (ic >= a.n_ics) return;
  const int64_t model = blockIdx.y;
  const int d = t.d;
  const GenRhs<float, KMAX> rhs{t, a.w + model * d * t.K};
  const float* x0 = a.x0 + model * a.x0_model_stride;
  float x[1][DN];
#pragma unroll
  for (int j = 0; j < DN; ++j) x[0][j] = (j < d) ? x0[ic * d + j] : 0.f;
  const Odeint<float> ode(a.dt);
  double sse = 0.0;
  int64_t valid = a.n_rows, row = 0, until = a.steps_per_row;
  for (;;) {
    ode.step(method, x, [&](const auto& y, auto& k, int) { rhs.eval(y[0], k[0]); });
    if (--until == 0) {
      if (!score_row<DN>(x[0], d, a.y_obs + (row * a.n_ics + ic) * d, a.blowup, sse)) { valid = row; break; }
      if (++row == a.n_rows) break;
      until = a.steps_per_row;
    }
  }
  a.sse[model * a.n_ics + ic] = sse;
  a.valid[model * a.n_ics + ic] = (int32_t)valid;
}

// ---- gradient of the scores -----------------------------------------------------------------------------------------
// ∂/∂W_m Σ_n sse[m, n] by the discrete adjoint of the fp32 recurrence the scorer executes. One thread owns one (model,
// IC) pair; grid = (IC blocks, models), W staged per block as the scorer stages it.
//   forward:  the scorer's loop (same step, same right-hand side, same row test), so sse / valid are its bits; the state
//             at every step c·kCkpt is stored to the workspace, [checkpoint][model][ic][d].
//   backward: the pair's objective ends at step S = valid·steps_per_row. Segments [c·kCkpt, (c+1)·kCkpt) ∩ [0, S) are
//             walked last to first: the segment's step-start states are recomputed from its checkpoint into a
//             per-thread array, then each step is reversed, its stages recomputed from its step-start state (nothing is
//             stored per stage). RK4, x' = x + sdt·(((k1 + 2k2) + 2k3) + k4), k_s = h(y_s): with a = sdt·λ,
//             k̄4 = a, k̄3 = k̄2 = 2a, k̄1 = a; for s = 4..1, ȳ_s = J_h(y_s)ᵀk̄_s and W̄ += k̄_s ⊗ Θ(y_s), ȳ_s enters λ and
//             k̄_{s−1} (times dt, hdt, hdt). Every compared row adds 2(x_r − y_r) to λ. Euler is the one-stage case.
//   sums:     W̄ in d·K fp32 registers per thread, added to an fp64 row per warp in shared memory at every segment end
//             (a warp-shuffle sum in fixed order), so an fp32 sum spans at most kCkpt steps; the warps' rows are added in
//             warp order into one fp64 partial row per (model, IC block), and grad_sum_kernel adds those in block order.
// Nothing depends on which other models share the launch: a model's gradient has the same bits alone, in any batch and
// any model order, on every repeat (not across IC batch splits, which regroup the sums).
//   starts:   λ after step 1 is reversed is ∂sse/∂x0 of the pair; it is written, widened to fp64, when grad_x0 is wanted.
//             One writer per element and no sum, so those bits do not depend on the batch, the model order or the IC
//             split. A pair with valid_rows = 0 reverses no step and writes exact zeros.
//   WG:       false drops everything that exists only for W̄ (the d·K accumulators, the shared rows, the segment-end
//             warp sums and the partial rows): the start-only variant for a caller that keeps W fixed.
constexpr int kCkpt = 32;             // checkpoint interval: kCkpt + 1 states per thread in local memory
constexpr int kGradThreads = kMultiThreads;
constexpr int kGradWarps = kGradThreads / 32;

struct GradArgs {
  ScoreArgs s;         // this launch's models, as the scorer gets them
  int64_t n_models;    // models of the whole call (checkpoint layout)
  int64_t model0;      // first model of this launch
  float* ckpt;         // [checkpoint][model][ic][d]
  double* partial;     // [model][IC block][d·K], from this launch's first model (WG only)
  double* grad_x0;     // [model][ic][d], from this launch's first model; NULL: not wanted
};

// specialised library: W from the block-staged shared copy (SharedW rows of KQ float4)
template <int D, int PC>
struct SpecGrad {
  static constexpr bool kStatic = true;
  static constexpr int DN = D, K = LibCode<D, PC>::K, ACC = D * K, KQ = SharedW<K>::KQ;
  static constexpr int THL = 1;   // Θ row of jac: in shared memory
  const float4* sw;
  __device__ __forceinline__ int dim() const { return D; }
  __device__ __forceinline__ int dk() const { return D * K; }
  __device__ __forceinline__ void eval(const float (&y)[D], float (&k)[D], int off) const {
    eval_pairs<D, PC, 1>(SharedW<K>{sw + off}, reinterpret_cast<const float (&)[1][D]>(y),
                         reinterpret_cast<float (&)[1][D]>(k));
  }
  // xb = J_h(y)ᵀu = J_Θ(y)ᵀ(Wᵀu);  acc += u ⊗ Θ(y) when WG
  template <bool WG, int NA>
  __device__ __forceinline__ void vjp(const float (&y)[D], const float (&u)[D], float (&xb)[D], float (&acc)[NA],
                                      int off) const {
    const float* w = reinterpret_cast<const float*>(sw + off);
    float m[K], mb[K];
    expand_lib<D, PC>(y, m);
    static_for<0, K>([&](auto kc) {
      constexpr int k = kc;
      float s = 0.f;
      static_for<0, D>([&](auto ic) {
        constexpr int i = ic;
        s = fmaf(w[i * KQ * 4 + k], u[i], s);
        if constexpr (WG) acc[i * K + k] = fmaf(u[i], m[k], acc[i * K + k]);
      });
      mb[k] = s;
    });
    static_for<0, D>([&](auto j) { xb[j] = 0.f; });
    reverse_lib<D, PC>(y, m, mb, xb);
  }
  // J_h(y) row by row, row i = J_Θ(y)ᵀW_i (one reverse sweep each), and Θ(y) into th (a per-thread shared row). The
  // sweeps read Θ back from that row: K values held in registers through d sweeps spill at (3,5)
  __device__ __forceinline__ void jac(const float (&y)[D], float (&jh)[D][D], float* th, int off) const {
    const float* w = reinterpret_cast<const float*>(sw + off);
    {
      float m[K];
      expand_lib<D, PC>(y, m);
      static_for<0, K>([&](auto k) { th[k] = m[k]; });
    }
    asm volatile("" ::: "memory");   // no store-to-load forwarding: the sweeps load Θ from shared memory
    const float (&m)[K] = *reinterpret_cast<const float (*)[K]>(th);
    // one sweep at a time: unrolled, the d independent sweeps are interleaved with d·K cotangents live
#pragma unroll 1
    for (int i = 0; i < D; ++i) {
      float mb[K], xb[D];
      static_for<0, K>([&](auto k) { mb[k] = w[i * KQ * 4 + k]; });
      static_for<0, D>([&](auto j) { xb[j] = 0.f; });
      reverse_lib<D, PC>(y, m, mb, xb);
      static_for<0, D>([&](auto ic) {
        if (ic == i) static_for<0, D>([&](auto j) { jh[ic][j] = xb[j]; });
      });
    }
  }
};

// runtime-table library: GenRhs with the model's W in global memory
template <int KMAX>
struct GenGrad {
  static constexpr bool kStatic = false;
  static constexpr int DN = SB_MAX_DIM, ACC = SB_MAX_DIM * KMAX;
  static constexpr int THL = KMAX;   // Θ row of jac: per-thread local array
  const LibTab& t;
  const float* w;
  __device__ __forceinline__ int dim() const { return t.d; }
  __device__ __forceinline__ int dk() const { return t.d * t.K; }
  __device__ __forceinline__ void eval(const float (&y)[DN], float (&k)[DN], int) const {
    GenRhs<float, KMAX>{t, w}.eval(y, k);
  }
  template <bool WG, int NA>
  __device__ __forceinline__ void vjp(const float (&y)[DN], const float (&u)[DN], float (&xb)[DN], float (&acc)[NA],
                                      int) const {
    float m[KMAX], mb[KMAX];
    expand_table(t, y, m);
    for (int k = 0; k < t.K; ++k) {
      float s = 0.f;
      for (int i = 0; i < t.d; ++i) {
        s = fmaf(__ldg(w + i * t.K + k), u[i], s);
        if constexpr (WG) acc[i * t.K + k] = fmaf(u[i], m[k], acc[i * t.K + k]);
      }
      mb[k] = s;
    }
#pragma unroll
    for (int j = 0; j < DN; ++j) xb[j] = 0.f;
    reverse_table(t, y, m, mb, xb);
  }
  __device__ __forceinline__ void jac(const float (&y)[DN], float (&jh)[DN][DN], float* th, int) const {
    expand_table(t, y, th);
    float mb[KMAX], xb[DN];
    for (int i = 0; i < t.d; ++i) {
      for (int k = 0; k < t.K; ++k) mb[k] = __ldg(w + i * t.K + k);
#pragma unroll
      for (int j = 0; j < DN; ++j) xb[j] = 0.f;
      reverse_table(t, y, th, mb, xb);
      // jh is in local memory here (DN = SB_MAX_DIM): index the row directly
#pragma unroll
      for (int j = 0; j < DN; ++j) jh[i][j] = xb[j];
    }
  }
};

__device__ __forceinline__ int64_t warp_max(int64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const int64_t u = __shfl_xor_sync(0xffffffffu, (long long)v, o);
    v = u > v ? u : v;
  }
  return v;
}

// with WG every thread of the block takes part (warp shuffles, block barrier), including those past the last IC
template <bool WG, class G>
__device__ __forceinline__ void grad_body(const G& g, int method, const GradArgs& a, double* sacc) {
  constexpr int DN = G::DN;
  const int d = g.dim(), dk = g.dk();
  const ScoreArgs& sa = a.s;
  const int64_t model = blockIdx.y, N = sa.n_ics, spr = sa.steps_per_row;
  const int64_t ic = (int64_t)blockIdx.x * kGradThreads + threadIdx.x;
  const bool live = ic < N;
  const int64_t ck_stride = a.n_models * N * d;
  float* ck = a.ckpt + ((a.model0 + model) * N + (live ? ic : 0)) * d;
  const Odeint<float> ode(sa.dt);
  auto step = [&](float (&x)[1][DN], int64_t s) {
    ode.step(method, x, [&](const auto& y, auto& k, int st) { g.eval(y[0], k[0], (int)((s + st) & sa.opaque)); });
  };

  // ---- forward: the scorer's loop, with checkpoints ----
  float x[1][DN];
#pragma unroll
  for (int j = 0; j < DN; ++j) x[0][j] = (live && j < d) ? sa.x0[model * sa.x0_model_stride + ic * d + j] : 0.f;
  int64_t valid = 0;
  if (live) {
    double sse = 0.0;
    valid = sa.n_rows;
    int64_t row = 0, until = spr, tock = 0, c = 0;
    for (int64_t s = 1;; ++s) {
      if (tock == 0) {                              // the state after step s − 1 = c·kCkpt
#pragma unroll
        for (int j = 0; j < DN; ++j)
          if (j < d) ck[c * ck_stride + j] = x[0][j];
        ++c;
        tock = kCkpt;
      }
      --tock;
      step(x, s);
      if (--until == 0) {
        if (!score_row<DN>(x[0], d, sa.y_obs + (row * N + ic) * d, sa.blowup, sse)) { valid = row; break; }
        if (++row == sa.n_rows) break;
        until = spr;
      }
    }
    sa.sse[model * N + ic] = sse;
    sa.valid[model * N + ic] = (int32_t)valid;
  }

  // ---- backward over the segments of [0, S) ----
  const int64_t S = valid * spr;
  const int64_t n_seg = WG ? warp_max((S + kCkpt - 1) / kCkpt) : (S + kCkpt - 1) / kCkpt;
  float acc[WG ? G::ACC : 1];
  if constexpr (!WG) {
  } else if constexpr (G::kStatic) {
    static_for<0, G::ACC>([&](auto e) { acc[e] = 0.f; });
  } else {
    for (int e = 0; e < dk; ++e) acc[e] = 0.f;
  }
  float lam[DN];
#pragma unroll
  for (int j = 0; j < DN; ++j) lam[j] = 0.f;
  float seg[kCkpt + 1][DN];
  double* mine = sacc + (threadIdx.x >> 5) * G::ACC;
  const bool lane0 = (threadIdx.x & 31) == 0;
  for (int64_t c = n_seg - 1; c >= 0; --c) {
    const int64_t s0 = c * kCkpt;
    const int n = S > s0 ? (int)(S - s0 < kCkpt ? S - s0 : kCkpt) : 0;
    if (n > 0) {
#pragma unroll
      for (int j = 0; j < DN; ++j) x[0][j] = j < d ? ck[c * ck_stride + j] : 0.f;
#pragma unroll
      for (int j = 0; j < DN; ++j) seg[0][j] = x[0][j];
      for (int q = 1; q <= n; ++q) {
        step(x, s0 + q);
#pragma unroll
        for (int j = 0; j < DN; ++j) seg[q][j] = x[0][j];
      }
      int64_t r_until = (s0 + n) % spr, row = (s0 + n) / spr;   // steps back to the next compared row, its number
      for (int q = n; q >= 1; --q) {
        if (r_until == 0) {                          // λ += ∂/∂x_s of ‖x_s − y_row‖²
          const float* y = sa.y_obs + ((row - 1) * N + ic) * d;
#pragma unroll
          for (int j = 0; j < DN; ++j)
            if (j < d) lam[j] += 2.f * (seg[q][j] - __ldg(y + j));
          --row;
          r_until = spr;
        }
        --r_until;
        const int off = (int)((s0 + q) & sa.opaque);
        float y1[DN];
#pragma unroll
        for (int j = 0; j < DN; ++j) y1[j] = seg[q - 1][j];
        float xb[DN];
        if (method == SB_EULER) {
          float u[DN];
#pragma unroll
          for (int j = 0; j < DN; ++j) u[j] = ode.dt * lam[j];
          g.template vjp<WG>(y1, u, xb, acc, off);
#pragma unroll
          for (int j = 0; j < DN; ++j) lam[j] += xb[j];
          continue;
        }
        // the stages y_1..y_4 of Odeint::step, recomputed bit for bit
        float ys[4][DN], k[DN];
#pragma unroll
        for (int j = 0; j < DN; ++j) ys[0][j] = y1[j];
        g.eval(y1, k, off);
#pragma unroll
        for (int j = 0; j < DN; ++j) ys[1][j] = add_rn(y1[j], mul_rn(ode.hdt, k[j]));
        g.eval(ys[1], k, off);
#pragma unroll
        for (int j = 0; j < DN; ++j) ys[2][j] = add_rn(y1[j], mul_rn(ode.hdt, k[j]));
        g.eval(ys[2], k, off);
#pragma unroll
        for (int j = 0; j < DN; ++j) ys[3][j] = add_rn(y1[j], mul_rn(ode.dt, k[j]));
        float av[DN];
#pragma unroll
        for (int j = 0; j < DN; ++j) { av[j] = ode.sdt * lam[j]; k[j] = av[j]; }   // k̄4 = sdt·λ
        // one copy of the stage sweep: a library's vjp inlined four times does not fit the register file at d·K = 168
#pragma unroll 1
        for (int st = 3; st >= 0; --st) {
          float ysd[DN];
#pragma unroll
          for (int j = 0; j < DN; ++j) ysd[j] = ys[st][j];
          g.template vjp<WG>(ysd, k, xb, acc, off);
          const float route = st == 3 ? ode.dt : ode.hdt, base = st == 1 ? 1.f : 2.f;
#pragma unroll
          for (int j = 0; j < DN; ++j) { lam[j] += xb[j]; k[j] = base * av[j] + route * xb[j]; }   // k̄_{st}
        }
      }
    }
    // segment end: fp32 sums into the warp's fp64 row
    if constexpr (!WG) {
    } else if constexpr (G::kStatic) {
      static_for<0, G::ACC>([&](auto e) {
        const double v = warp_sum((double)acc[e]);
        if (lane0) mine[e] += v;
        acc[e] = 0.f;
      });
    } else {
      for (int e = 0; e < dk; ++e) {
        const double v = warp_sum((double)acc[e]);
        if (lane0) mine[e] += v;
        acc[e] = 0.f;
      }
    }
  }
  if (a.grad_x0 && live) {
    double* gx = a.grad_x0 + (model * N + ic) * d;
#pragma unroll
    for (int j = 0; j < DN; ++j)
      if (j < d) gx[j] = (double)lam[j];
  }
  if constexpr (WG) {
    __syncthreads();
    double* part = a.partial + (model * gridDim.x + blockIdx.x) * dk;
    for (int e = threadIdx.x; e < dk; e += kGradThreads) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < kGradWarps; ++w) v += sacc[w * G::ACC + e];
      part[e] = v;
    }
  }
}

template <int D, int PC, int METHOD, bool WG>
__global__ void __launch_bounds__(kGradThreads) rollout_grad_spec_kernel(GradArgs a) {
  using G = SpecGrad<D, PC>;
  constexpr int K = G::K, KQ = G::KQ, NS = WG ? kGradWarps * G::ACC : 1;
  __shared__ float4 sw[D * KQ];
  __shared__ double sacc[NS];
  {
    const float* wm = a.s.w + (int64_t)blockIdx.y * (D * K);
    float* s = reinterpret_cast<float*>(sw);
    for (int q = threadIdx.x; q < D * KQ * 4; q += kGradThreads) {
      const int i = q / (KQ * 4), c = q % (KQ * 4);
      s[q] = c < K ? wm[i * K + c] : 0.f;
    }
    if constexpr (WG)
      for (int q = threadIdx.x; q < NS; q += kGradThreads) sacc[q] = 0.0;
  }
  __syncthreads();
  grad_body<WG>(G{sw}, METHOD, a, sacc);
}

template <int KMAX, bool WG>
__global__ void __launch_bounds__(kGradThreads) rollout_grad_gen_kernel(LibTab t, int method, GradArgs a) {
  using G = GenGrad<KMAX>;
  constexpr int NS = WG ? kGradWarps * G::ACC : 1;
  __shared__ double sacc[NS];
  if constexpr (WG) {
    for (int q = threadIdx.x; q < NS; q += kGradThreads) sacc[q] = 0.0;
    __syncthreads();
  }
  grad_body<WG>(G{t, a.s.w + (int64_t)blockIdx.y * t.d * t.K}, method, a, sacc);
}

// grad[m, e] = Σ_b partial[m, b, e] in block order
__global__ void __launch_bounds__(256) grad_sum_kernel(const double* partial, int64_t n_blocks, int dk, int64_t n,
                                                       double* grad) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const int64_t m = i / dk, e = i % dk;
  const double* p = partial + m * n_blocks * dk + e;
  double v = 0.0;
  for (int64_t b = 0; b < n_blocks; ++b) v += p[b * dk];
  grad[i] = v;
}

// ---- Gauss–Newton information of the scores -------------------------------------------------------------------------
// For the listed coefficients θ of each model (indices into the flat d×K W, −1 = padding) and optionally each pair's
// start: J = ∂x_r/∂(θ, x0) at every compared row r of the pair, F_θθ = Σ_pairs Σ_r JθᵀJθ, g_θ = Σ JθᵀE (E = x_r − y_r),
// and per pair F_θx = Σ_r JθᵀJx, F_xx = Σ_r JxᵀJx, g_x = Σ_r JxᵀE. J is carried forward with the states: the tangent-
// linear of the same fp32 recurrence the scorer runs (not of the continuous sensitivity equation), in Odeint::step's
// stage order,
//   S' = S + sdt·(((K1 + 2K2) + 2K3) + K4),  K_s = J_h(y_s)·S_s + E(Θ(y_s)),  S_1 = S, S_2 = S + hdt·K1, ...
// where coefficient (i, k) has the source column e_i·Θ_k(y_s) and a start column none; S(0) = [0 | I_d]. J_h(y_s) is
// formed from d value-only reverse sweeps of the library (row i = J_Θᵀ W_i), Θ(y_s) goes to a per-thread shared row.
//   layout:  grid = (IC-group blocks, models). A block holds G pairs × T chunks of C directions: thread (g, t)
//            integrates pair g's state (repeated across its chunks) and directions t·C .. t·C + C − 1 of
//            P' = n_params + (d if start blocks). The primal is the scorer's loop, so sse / valid are its bits.
//   rows:    at each compared row every thread writes its d × C slice of J and chunk 0 the residual to shared memory
//            (a pair that has stopped, or is past the last IC, writes zeros, so it adds exact zeros); after a barrier
//            each thread adds, for the entries it owns, the fp32 sum over the block's pairs (in pair order) of that
//            row's products to an fp64 accumulator in shared memory: the upper triangle of F_θθ and g_θ, and the per-pair
//            blocks. So no fp32 sum spans more than one row.
//   sums:    a block walks IC groups blockIdx.x, blockIdx.x + gridDim.x, ... in order; gridDim.x depends only on n_ics
//            and P', never on the number of models. Its θ sums go to one fp64 row per (model, block), gn_sum_kernel adds
//            those in block order. The per-pair blocks have one writer each. A model's outputs have the same bits
//            alone, in any batch, in any model order and on every repeat (for the same n_params).
// tangent directions per thread: 8, or 4 for a specialised library of K ≥ 32 columns ((3,5): 255 registers and 644
// bytes of spill stores at 8, none at 4)
template <int K> constexpr int gn_chunk() { return K >= 32 ? 4 : 8; }
constexpr int kGnC = 8;               // the runtime-table kernels
constexpr int kGnThreads = 128;       // block target: G = max(1, kGnThreads / T) pairs of T chunks
constexpr int kGnMaxBlocks = 32;      // IC-group blocks per model
constexpr int kGnMaxCols = SB_GN_MAX_COLS;
static_assert(kGnMaxCols % 8 == 0, "whole chunks");

struct GnArgs {
  ScoreArgs s;            // this launch's models, as the scorer gets them
  const int32_t* params;  // [model][P], from this launch's first model
  int P, X, T, G;         // listed coefficients, start columns (d or 0), chunks per pair, pairs per block
  int64_t n_groups;       // ⌈n_ics / G⌉
  double* partial;        // [model][block][P(P+1)/2 + P], from this launch's first model
  double* jtj_px;         // [model][ic][P][d], from this launch's first model (X only)
  double* jtj_xx;         // [model][ic][d][d]
  double* jtr_x;          // [model][ic][d]
};

// shared memory of one block: [θ sums: P(P+1)/2 + P fp64][pair sums: G·(P·d + d² + d) fp64 when X]
// [J slices: G·d·T·C fp32][residuals: G·d fp32][Θ rows: threads·(K|1) fp32, specialised libraries only]
__host__ __device__ inline int64_t gn_tri(int P) { return (int64_t)P * (P + 1) / 2; }
__host__ __device__ inline int64_t gn_pair_elems(int P, int d) { return (int64_t)P * d + d * d + d; }

template <int C, class G>
__device__ __forceinline__ void gn_body(const G& g, int method, const GnArgs& a, int K) {
  extern __shared__ double gn_smem[];
  constexpr int DN = G::DN;
  const int d = g.dim(), P = a.P, NG = a.G, nt = blockDim.x, tid = threadIdx.x;
  const int gp = tid / a.T, ch = tid % a.T, cols = a.T * C;
  const int tri = (int)gn_tri(P), PE = (int)gn_pair_elems(P, d);   // < 2^31 below SB_GN_MAX_COLS
  const ScoreArgs& sa = a.s;
  const int64_t model = blockIdx.y, N = sa.n_ics, spr = sa.steps_per_row;
  double* acc = gn_smem;
  double* pacc = acc + tri + P;
  float* jsh = reinterpret_cast<float*>(pacc + (a.X ? NG * PE : 0));
  float* esh = jsh + NG * d * cols;
  float* th;
  float thl[G::THL];
  if constexpr (G::kStatic) th = esh + NG * d + tid * (K | 1);
  else th = thl;
  for (int e = tid; e < tri + P; e += nt) acc[e] = 0.0;
  if (a.X)
    for (int e = tid; e < NG * PE; e += nt) pacc[e] = 0.0;

  // this thread's directions: code = component << 16 | column of a listed coefficient, −1 for a start column or padding
  const int32_t* prm = a.params + model * P;
  int code[C];
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const int q = ch * C + c;
    const int p = q < P ? prm[q] : -1;
    code[c] = p < 0 ? -1 : (p / K) << 16 | (p % K);
  }
  const Odeint<float> ode(sa.dt);
  const int n_stage = method == SB_EULER ? 1 : 4;
  float* Jg = jsh + gp * d * cols;

  for (int64_t grp = blockIdx.x; grp < a.n_groups; grp += gridDim.x) {
    const int64_t ic = grp * NG + gp;
    const bool live = ic < N;
    float x[DN], S[C][DN];
#pragma unroll
    for (int j = 0; j < DN; ++j) x[j] = (live && j < d) ? sa.x0[model * sa.x0_model_stride + ic * d + j] : 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) {
      const int q = ch * C + c - P;   // start column q: S(0) = e_q
#pragma unroll
      for (int j = 0; j < DN; ++j) S[c][j] = (a.X && q == j) ? 1.f : 0.f;
    }
    bool track = live;
    double sse = 0.0;
    int64_t valid = sa.n_rows, row = 0, s = 0;
    for (;;) {
      if (track) {
        for (int64_t q = 0; q < spr; ++q) {
          const int off = (int)(++s & sa.opaque);
          float acc_t[C][DN], dy[C][DN], y[DN], k[DN], kacc[DN], jh[DN][DN];
#pragma unroll
          for (int j = 0; j < DN; ++j) y[j] = x[j];
#pragma unroll
          for (int c = 0; c < C; ++c)
#pragma unroll
            for (int j = 0; j < DN; ++j) dy[c][j] = S[c][j];
          // one copy of the stage: J_h and the library sweeps inlined four times do not fit the register file at (3,5)
#pragma unroll 1
          for (int st = 0; st < n_stage; ++st) {
            g.jac(y, jh, th, off);
            g.eval(y, k, off);
            const float wgt = (st == 1 || st == 2) ? 2.f : 1.f;
            const float hn = st == 2 ? ode.dt : ode.hdt;   // from this stage to the next stage's state
#pragma unroll
            for (int c = 0; c < C; ++c) {
              const int comp = code[c] >> 16;   // −1: no source
              const float src = th[code[c] < 0 ? 0 : code[c] & 0xffff];
              float v[DN];
#pragma unroll
              for (int i = 0; i < DN; ++i) {
                v[i] = i == comp ? src : 0.f;
#pragma unroll
                for (int j = 0; j < DN; ++j)
                  if (i < d && j < d) v[i] = fmaf(jh[i][j], dy[c][j], v[i]);
              }
#pragma unroll
              for (int i = 0; i < DN; ++i) {
                acc_t[c][i] = st == 0 ? v[i] : fmaf(wgt, v[i], acc_t[c][i]);
                dy[c][i] = fmaf(hn, v[i], S[c][i]);
              }
            }
            // the primal: Odeint::step's operations in its order
#pragma unroll
            for (int j = 0; j < DN; ++j) {
              kacc[j] = st == 0 ? k[j] : add_rn(kacc[j], st == 3 ? k[j] : mul_rn(2.f, k[j]));
              y[j] = add_rn(x[j], mul_rn(hn, k[j]));
            }
          }
          const float h = method == SB_EULER ? ode.dt : ode.sdt;
#pragma unroll
          for (int j = 0; j < DN; ++j) {
            x[j] = add_rn(x[j], mul_rn(h, kacc[j]));
#pragma unroll
            for (int c = 0; c < C; ++c) S[c][j] = fmaf(h, acc_t[c][j], S[c][j]);
          }
        }
        if (!score_row<DN>(x, d, sa.y_obs + (row * N + ic) * d, sa.blowup, sse)) { track = false; valid = row; }
      }
      // this row's slice of J and the residual
      for (int i = 0; i < d; ++i) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
          float v = 0.f;
#pragma unroll
          for (int j = 0; j < DN; ++j)
            if (j == i) v = S[c][j];
          Jg[i * cols + ch * C + c] = track ? v : 0.f;
        }
      }
      if (ch == 0) {
        const float* yr = sa.y_obs + (row * N + (live ? ic : 0)) * d;
#pragma unroll
        for (int j = 0; j < DN; ++j)
          if (j < d) esh[gp * d + j] = track ? x[j] - __ldg(yr + j) : 0.f;
      }
      const int any = __syncthreads_or(track);
      // F_θθ upper triangle (row-major: row a holds b = a..P−1) and g_θ
      {
        int ra = 0, cb = tid;
        while (cb >= P && ra < P) { ++ra; cb += ra - P; }
        for (int e = tid; e < tri; e += nt) {
          float v = 0.f;
          for (int q = 0; q < NG; ++q)
            for (int i = 0; i < d; ++i) {
              const float* r = jsh + (q * d + i) * cols;
              v = fmaf(r[ra], r[cb], v);
            }
          acc[e] += (double)v;
          cb += nt;
          while (cb >= P && ra < P) { ++ra; cb += ra - P; }
        }
        for (int e = tid; e < P; e += nt) {
          float v = 0.f;
          for (int q = 0; q < NG; ++q)
            for (int i = 0; i < d; ++i) v = fmaf(jsh[(q * d + i) * cols + e], esh[q * d + i], v);
          acc[tri + e] += (double)v;
        }
      }
      if (a.X) {
        for (int e = tid; e < NG * PE; e += nt) {
          const int q = e / PE, r = e - q * PE;
          const float* Jq = jsh + q * d * cols;
          int c1, c2 = -1;   // column pair, or c2 = −1: the residual
          if (r < P * d) { c1 = r / d; c2 = P + r % d; }
          else if (r < P * d + d * d) { c1 = P + (r - P * d) / d; c2 = P + (r - P * d) % d; }
          else c1 = P + r - P * d - d * d;
          float v = 0.f;
          for (int i = 0; i < d; ++i) v = fmaf(Jq[i * cols + c1], c2 < 0 ? esh[q * d + i] : Jq[i * cols + c2], v);
          pacc[e] += (double)v;
        }
      }
      __syncthreads();
      if (++row == sa.n_rows || !any) break;
    }
    if (live && ch == 0) {
      sa.sse[model * N + ic] = sse;
      sa.valid[model * N + ic] = (int32_t)valid;
    }
    if (a.X) {   // the group's per-pair blocks, by the threads that own them (so no barrier)
      for (int e = tid; e < NG * PE; e += nt) {
        const int q = e / PE, r = e - q * PE;
        const int64_t icq = grp * NG + q, pr = model * N + icq;
        if (icq < N) {
          if (r < P * d) a.jtj_px[pr * P * d + r] = prm[r / d] < 0 ? 0.0 : pacc[e];
          else if (r < P * d + d * d) a.jtj_xx[pr * d * d + r - P * d] = pacc[e];
          else a.jtr_x[pr * d + r - P * d - d * d] = pacc[e];
        }
        pacc[e] = 0.0;
      }
    }
  }
  double* part = a.partial + (model * gridDim.x + blockIdx.x) * (tri + P);
  for (int e = tid; e < tri + P; e += nt) part[e] = acc[e];
}

template <int D, int PC, int METHOD>
__global__ void __launch_bounds__(kGnThreads, 1) rollout_gn_spec_kernel(GnArgs a) {
  using G = SpecGrad<D, PC>;
  constexpr int K = G::K, KQ = G::KQ;
  __shared__ float4 sw[D * KQ];
  {
    const float* wm = a.s.w + (int64_t)blockIdx.y * (D * K);
    float* s = reinterpret_cast<float*>(sw);
    for (int q = threadIdx.x; q < D * KQ * 4; q += blockDim.x) {
      const int i = q / (KQ * 4), c = q % (KQ * 4);
      s[q] = c < K ? wm[i * K + c] : 0.f;
    }
  }
  __syncthreads();
  gn_body<gn_chunk<K>()>(G{sw}, METHOD, a, K);
}

template <int KMAX>
__global__ void __launch_bounds__(kGnThreads) rollout_gn_gen_kernel(LibTab t, int method, GnArgs a) {
  gn_body<kGnC>(GenGrad<KMAX>{t, a.s.w + (int64_t)blockIdx.y * t.d * t.K}, method, a, t.K);
}

// jtj[m] (P × P, both triangles from the same sums) and jtr[m]: Σ_b partial[m, b, ·] in block order; rows and columns of
// padded indices are exact zeros
__global__ void __launch_bounds__(256) gn_sum_kernel(const double* partial, int64_t n_blocks, int P,
                                                     const int32_t* params, int64_t n, double* jtj, double* jtr) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const int64_t per = (int64_t)P * P + P, tri = gn_tri(P), m = i / per, r = i % per;
  const int32_t* prm = params + m * P;
  int64_t e;
  bool dead;
  if (r < (int64_t)P * P) {
    const int a = (int)(r / P), b = (int)(r % P), lo = a < b ? a : b, hi = a < b ? b : a;
    e = (int64_t)lo * P - (int64_t)lo * (lo - 1) / 2 + (hi - lo);
    dead = prm[a] < 0 || prm[b] < 0;
  } else {
    e = tri + (r - (int64_t)P * P);
    dead = prm[r - (int64_t)P * P] < 0;
  }
  double v = 0.0;
  if (!dead) {
    const double* p = partial + m * n_blocks * (tri + P) + e;
    for (int64_t b = 0; b < n_blocks; ++b) v += p[b * (tri + P)];
  }
  if (r < (int64_t)P * P) jtj[m * P * P + r] = v;
  else jtr[m * P + r - (int64_t)P * P] = v;
}

// ---- launch ---------------------------------------------------------------------------------------------------------
// The specialised libraries as (D, library code PC): the polynomials and, for config 3 (Lotka-Volterra in canonical
// coordinates, `data_utils/lotka.py:33-41`), degree 2 + exp. Everything else runs on the runtime table.
#define SB_SPEC_SHAPES(X) X(2, 2) X(2, 3) X(3, 2) X(3, 3) X(3, 5) X(2, 12)

// SB_ROLLOUT_MULTI=0 selects the one-initial-condition-per-thread kernel for the fp32 RK4 rollout (A/B, bitwise test)
bool rollout_multi_enabled() {
  const char* e = getenv("SB_ROLLOUT_MULTI");
  return !(e && e[0] == '0');
}

template <int D, int PC, class T>
int launch_rollout_spec(const void* w, const RollArgs& a, cudaStream_t s) {
  using L = LibCode<D, PC>;
  SB_CUDA_TRY(cudaMemcpyToSymbolAsync(c_rw, w, sizeof(T) * D * L::K, 0, cudaMemcpyDeviceToDevice, s));
  if constexpr (std::is_same<T, float>::value && L::S == 0 && L::E == 0) {
    if (a.method == SB_RK4 && !a.record_dx && rollout_multi_enabled()) {
      const unsigned grid = (unsigned)((a.n_ics + kMultiNB * kMultiThreads - 1) / (kMultiNB * kMultiThreads));
      rollout_rk4_multi_kernel<D, L::P, kMultiNB><<<grid, kMultiThreads, 0, s>>>(a);
      SB_LAUNCH_CHECK("rollout_rk4_multi_kernel");
      return SB_OK;
    }
  }
  const unsigned grid = (unsigned)((a.n_ics + kThreads - 1) / kThreads);
  rollout_spec_kernel<D, L::P, T, L::S, L::E><<<grid, kThreads, 0, s>>>(a);
  SB_LAUNCH_CHECK("rollout_spec_kernel");
  return SB_OK;
}

template <class T>
int launch_rollout(const LibTab& t, const void* w, const RollArgs& a, cudaStream_t s) {
#define X(D, PC) \
  if (lib_matches<D, PC>(t)) return launch_rollout_spec<D, PC, T>(w, a, s);
  SB_SPEC_SHAPES(X)
#undef X
  const unsigned grid = (unsigned)((a.n_ics + kThreads - 1) / kThreads);
  if (t.K <= 16) rollout_gen_kernel<T, 16><<<grid, kThreads, 0, s>>>(t, reinterpret_cast<const T*>(w), a);
  else if (t.K <= 64) rollout_gen_kernel<T, 64><<<grid, kThreads, 0, s>>>(t, reinterpret_cast<const T*>(w), a);
  else rollout_gen_kernel<T, 256><<<grid, kThreads, 0, s>>>(t, reinterpret_cast<const T*>(w), a);
  SB_LAUNCH_CHECK("rollout_gen_kernel");
  return SB_OK;
}

template <int D, int PC>
int launch_score_spec(const ScoreArgs& a, int method, int n_models, cudaStream_t s) {
  const unsigned gx = (unsigned)((a.n_ics + kMultiThreads * kMultiNB - 1) / (kMultiThreads * kMultiNB));
  const dim3 grid(gx, (unsigned)n_models);
  if (method == SB_EULER) rollout_score_spec_kernel<D, PC, SB_EULER><<<grid, kMultiThreads, 0, s>>>(a);
  else rollout_score_spec_kernel<D, PC, SB_RK4><<<grid, kMultiThreads, 0, s>>>(a);
  SB_LAUNCH_CHECK("rollout_score_spec_kernel");
  return SB_OK;
}

int launch_score(const LibTab& t, const ScoreArgs& a, int method, int n_models, cudaStream_t s) {
#define X(D, PC) \
  if (lib_matches<D, PC>(t)) return launch_score_spec<D, PC>(a, method, n_models, s);
  SB_SPEC_SHAPES(X)
#undef X
  const dim3 grid((unsigned)((a.n_ics + kThreads - 1) / kThreads), (unsigned)n_models);
  if (t.K <= 16) rollout_score_gen_kernel<16><<<grid, kThreads, 0, s>>>(t, method, a);
  else if (t.K <= 64) rollout_score_gen_kernel<64><<<grid, kThreads, 0, s>>>(t, method, a);
  else rollout_score_gen_kernel<256><<<grid, kThreads, 0, s>>>(t, method, a);
  SB_LAUNCH_CHECK("rollout_score_gen_kernel");
  return SB_OK;
}

int64_t grad_blocks(int64_t n_ics) { return (n_ics + kGradThreads - 1) / kGradThreads; }

template <int D, int PC, bool WG>
int launch_grad_spec(const GradArgs& a, int method, int n_models, cudaStream_t s) {
  const dim3 grid((unsigned)grad_blocks(a.s.n_ics), (unsigned)n_models);
  if (method == SB_EULER) rollout_grad_spec_kernel<D, PC, SB_EULER, WG><<<grid, kGradThreads, 0, s>>>(a);
  else rollout_grad_spec_kernel<D, PC, SB_RK4, WG><<<grid, kGradThreads, 0, s>>>(a);
  SB_LAUNCH_CHECK("rollout_grad_spec_kernel");
  return SB_OK;
}

template <bool WG>
int launch_grad(const LibTab& t, const GradArgs& a, int method, int n_models, cudaStream_t s) {
#define X(D, PC) \
  if (lib_matches<D, PC>(t)) return launch_grad_spec<D, PC, WG>(a, method, n_models, s);
  SB_SPEC_SHAPES(X)
#undef X
  const dim3 grid((unsigned)grad_blocks(a.s.n_ics), (unsigned)n_models);
  if (t.K <= 16) rollout_grad_gen_kernel<16, WG><<<grid, kGradThreads, 0, s>>>(t, method, a);
  else if (t.K <= 64) rollout_grad_gen_kernel<64, WG><<<grid, kGradThreads, 0, s>>>(t, method, a);
  else rollout_grad_gen_kernel<256, WG><<<grid, kGradThreads, 0, s>>>(t, method, a);
  SB_LAUNCH_CHECK("rollout_grad_gen_kernel");
  return SB_OK;
}

// The Gauss–Newton block shape and shared memory for P listed coefficients and X start columns, as gn_body lays it out
struct GnShape {
  int T, G, threads;
  int64_t n_groups, blocks, smem;
};
GnShape gn_shape(int64_t n_ics, const LibTab& t, int P, int X, bool spec) {
  GnShape g;
  const int C = spec && t.K >= 32 ? 4 : kGnC;   // gn_chunk
  g.T = (P + X + C - 1) / C;
  g.G = kGnThreads / g.T > 1 ? kGnThreads / g.T : 1;
  g.threads = g.G * g.T;
  g.n_groups = (n_ics + g.G - 1) / g.G;
  g.blocks = g.n_groups < kGnMaxBlocks ? g.n_groups : kGnMaxBlocks;
  g.smem = 8 * (gn_tri(P) + P + (X ? g.G * gn_pair_elems(P, t.d) : 0)) +
           4 * ((int64_t)g.G * t.d * g.T * C + g.G * t.d + (spec ? (int64_t)g.threads * (t.K | 1) : 0));
  return g;
}

bool gn_spec(const LibTab& t) {
#define X(D, PC) \
  if (lib_matches<D, PC>(t)) return true;
  SB_SPEC_SHAPES(X)
#undef X
  return false;
}

template <class Kern, class... Args>
int launch_gn_kernel(Kern kern, const GnShape& g, int n_models, cudaStream_t s, Args... args) {
  // always: the default dynamic limit is 48 KB less the kernel's static shared memory
  SB_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
  kern<<<dim3((unsigned)g.blocks, (unsigned)n_models), g.threads, (size_t)g.smem, s>>>(args...);
  SB_LAUNCH_CHECK("rollout_gn_kernel");
  return SB_OK;
}

template <int D, int PC>
int launch_gn_spec(const GnArgs& a, const GnShape& g, int method, int n_models, cudaStream_t s) {
  if (method == SB_EULER) return launch_gn_kernel(rollout_gn_spec_kernel<D, PC, SB_EULER>, g, n_models, s, a);
  return launch_gn_kernel(rollout_gn_spec_kernel<D, PC, SB_RK4>, g, n_models, s, a);
}

int launch_gn(const LibTab& t, const GnArgs& a, const GnShape& g, int method, int n_models, cudaStream_t s) {
#define X(D, PC) \
  if (lib_matches<D, PC>(t)) return launch_gn_spec<D, PC>(a, g, method, n_models, s);
  SB_SPEC_SHAPES(X)
#undef X
  if (t.K <= 16) return launch_gn_kernel(rollout_gn_gen_kernel<16>, g, n_models, s, t, method, a);
  if (t.K <= 64) return launch_gn_kernel(rollout_gn_gen_kernel<64>, g, n_models, s, t, method, a);
  return launch_gn_kernel(rollout_gn_gen_kernel<256>, g, n_models, s, t, method, a);
}

// workspace: [partial rows: n_models × IC blocks × d·K fp64, padded to 256 bytes][checkpoints: n_ckpt × n_models ×
// n_ics × d fp32], n_ckpt = ⌈n_rows·steps_per_row / kCkpt⌉
struct GradLayout {
  int64_t partial_bytes, ckpt_bytes;
};
bool grad_layout(int64_t n_ics, const LibTab& t, int n_models, int64_t steps_per_row, int64_t n_rows, GradLayout* L) {
  int64_t steps, rows_el, part, ck;
  if (__builtin_mul_overflow(n_rows, steps_per_row, &steps)) return false;
  const int64_t n_ckpt = (steps - 1) / kCkpt + 1;
  if (__builtin_mul_overflow(grad_blocks(n_ics), (int64_t)n_models, &part)) return false;
  if (__builtin_mul_overflow(part, (int64_t)(t.d * t.K) * 8, &part)) return false;
  if (__builtin_mul_overflow((int64_t)n_models * n_ics, (int64_t)t.d * 4, &rows_el)) return false;
  if (__builtin_mul_overflow(rows_el, n_ckpt, &ck)) return false;
  part = (part + 255) / 256 * 256;
  if (part > INT64_MAX - ck) return false;
  L->partial_bytes = part;
  L->ckpt_bytes = ck;
  return true;
}

}  // namespace

int64_t rollout_score_grad_workspace_bytes(int64_t n_ics, const LibTab& t, int n_models, int64_t steps_per_row,
                                           int64_t n_rows) {
  GradLayout L;
  if (!grad_layout(n_ics, t, n_models, steps_per_row, n_rows, &L)) return -1;
  return L.partial_bytes + L.ckpt_bytes;
}

int rollout_score_grad(const float* x0, int64_t x0_model_stride, int64_t n_ics, const LibTab& t, const float* w,
                       int n_models, double dt, int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs,
                       float blowup, double* sse, int32_t* valid_rows, double* grad, double* grad_x0, void* ws,
                       int64_t ws_bytes, cudaStream_t s) {
  GradLayout L;
  if (!grad_layout(n_ics, t, n_models, steps_per_row, n_rows, &L)) {
    set_error("rollout_score_grad workspace size overflows int64");
    return SB_ERR_INVALID;
  }
  if (ws_bytes < L.partial_bytes + L.ckpt_bytes) {
    set_error("workspace too small: %lld < %lld bytes", (long long)ws_bytes,
              (long long)(L.partial_bytes + L.ckpt_bytes));
    return SB_ERR_WORKSPACE;
  }
  const int dk = t.d * t.K;
  const int64_t nblk = grad_blocks(n_ics);
  double* partial = reinterpret_cast<double*>(ws);
  GradArgs a{};
  a.s.x0_model_stride = x0_model_stride;
  a.s.n_ics = n_ics; a.s.dt = dt; a.s.steps_per_row = steps_per_row; a.s.n_rows = n_rows;
  a.s.y_obs = y_obs; a.s.blowup = blowup; a.s.opaque = 0;
  a.n_models = n_models;
  a.ckpt = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + L.partial_bytes);
  // more models than gridDim.y allows: further launches on the same stream
  for (int m0 = 0; m0 < n_models; m0 += kMaxGridY) {
    const int nm = n_models - m0 < kMaxGridY ? n_models - m0 : kMaxGridY;
    a.s.x0 = x0 + (int64_t)m0 * x0_model_stride;
    a.s.w = w + (int64_t)m0 * dk;
    a.s.sse = sse + (int64_t)m0 * n_ics;
    a.s.valid = valid_rows + (int64_t)m0 * n_ics;
    a.model0 = m0;
    a.partial = partial + (int64_t)m0 * nblk * dk;
    a.grad_x0 = grad_x0 ? grad_x0 + (int64_t)m0 * n_ics * t.d : nullptr;
    const int st = grad ? launch_grad<true>(t, a, method, nm, s) : launch_grad<false>(t, a, method, nm, s);
    if (st != SB_OK) return st;
  }
  if (!grad) return SB_OK;
  const int64_t n = (int64_t)n_models * dk;
  grad_sum_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(partial, nblk, dk, n, grad);
  SB_LAUNCH_CHECK("grad_sum_kernel");
  return SB_OK;
}

// workspace: one fp64 row of P(P+1)/2 + P θ sums per (model, IC-group block)
int64_t rollout_score_gn_workspace_bytes(int64_t n_ics, const LibTab& t, int n_models, int n_params, int x0_blocks) {
  const GnShape g = gn_shape(n_ics, t, n_params, x0_blocks ? t.d : 0, gn_spec(t));
  int64_t b;
  if (__builtin_mul_overflow((int64_t)n_models * g.blocks, (gn_tri(n_params) + n_params) * 8, &b)) return -1;
  return b;
}

int rollout_score_gn(const float* x0, int64_t x0_model_stride, int64_t n_ics, const LibTab& t, const float* w,
                     int n_models, const int32_t* params, int n_params, double dt, int64_t steps_per_row,
                     int64_t n_rows, int method, const float* y_obs, float blowup, double* sse, int32_t* valid_rows,
                     double* jtj, double* jtr, double* jtj_px, double* jtj_xx, double* jtr_x, void* ws,
                     int64_t ws_bytes, cudaStream_t s) {
  const int X = jtj_px ? t.d : 0;
  const int64_t need = rollout_score_gn_workspace_bytes(n_ics, t, n_models, n_params, X != 0);
  if (need < 0) {
    set_error("rollout_score_gn workspace size overflows int64");
    return SB_ERR_INVALID;
  }
  if (ws_bytes < need) {
    set_error("workspace too small: %lld < %lld bytes", (long long)ws_bytes, (long long)need);
    return SB_ERR_WORKSPACE;
  }
  const GnShape g = gn_shape(n_ics, t, n_params, X, gn_spec(t));
  int dev = 0, smem_max = 0;
  SB_CUDA_TRY(cudaGetDevice(&dev));
  SB_CUDA_TRY(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  if (g.smem + 1024 > smem_max) {
    set_error("rollout_score_gn needs %lld bytes of shared memory per block, the device has %d", (long long)g.smem,
              smem_max);
    return SB_ERR_UNSUPPORTED;
  }
  const int64_t per = gn_tri(n_params) + n_params;
  double* partial = reinterpret_cast<double*>(ws);
  GnArgs a{};
  a.s.x0_model_stride = x0_model_stride;
  a.s.n_ics = n_ics; a.s.dt = dt; a.s.steps_per_row = steps_per_row; a.s.n_rows = n_rows;
  a.s.y_obs = y_obs; a.s.blowup = blowup; a.s.opaque = 0;
  a.P = n_params; a.X = X; a.T = g.T; a.G = g.G; a.n_groups = g.n_groups;
  // more models than gridDim.y allows: further launches on the same stream
  for (int m0 = 0; m0 < n_models; m0 += kMaxGridY) {
    const int nm = n_models - m0 < kMaxGridY ? n_models - m0 : kMaxGridY;
    a.s.x0 = x0 + (int64_t)m0 * x0_model_stride;
    a.s.w = w + (int64_t)m0 * t.d * t.K;
    a.s.sse = sse + (int64_t)m0 * n_ics;
    a.s.valid = valid_rows + (int64_t)m0 * n_ics;
    a.params = params + (int64_t)m0 * n_params;
    a.partial = partial + (int64_t)m0 * g.blocks * per;
    if (X) {
      a.jtj_px = jtj_px + (int64_t)m0 * n_ics * n_params * X;
      a.jtj_xx = jtj_xx + (int64_t)m0 * n_ics * X * X;
      a.jtr_x = jtr_x + (int64_t)m0 * n_ics * X;
    }
    const int st = launch_gn(t, a, g, method, nm, s);
    if (st != SB_OK) return st;
  }
  const int64_t n = (int64_t)n_models * ((int64_t)n_params * n_params + n_params);
  gn_sum_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(partial, g.blocks, n_params, params, n, jtj, jtr);
  SB_LAUNCH_CHECK("gn_sum_kernel");
  return SB_OK;
}

int rollout(const void* x0, int64_t n_ics, const LibTab& t, const void* w, double dt, int64_t n_steps,
            int64_t stride, int method, int dtype, int record_dx, void* x_out, void* dx_out, void* x_last,
            cudaStream_t s) {
  RollArgs a{};
  a.x0 = x0; a.n_ics = n_ics; a.dt = dt; a.n_steps = n_steps; a.stride = stride; a.method = method;
  a.record_dx = record_dx; a.opaque = 0; a.x_out = x_out; a.dx_out = dx_out; a.x_last = x_last;
  if (dtype == SB_F32) return launch_rollout<float>(t, w, a, s);
  return launch_rollout<double>(t, w, a, s);
}

int rollout_score(const float* x0, int64_t x0_model_stride, int64_t n_ics, const LibTab& t, const float* w,
                  int n_models, double dt, int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs,
                  float blowup, double* sse, int32_t* valid_rows, cudaStream_t s) {
  ScoreArgs a{};
  a.x0_model_stride = x0_model_stride; a.n_ics = n_ics; a.dt = dt; a.steps_per_row = steps_per_row; a.n_rows = n_rows; a.y_obs = y_obs;
  a.blowup = blowup; a.opaque = 0;
  // more models than gridDim.y allows: further launches on the same stream
  for (int m0 = 0; m0 < n_models; m0 += kMaxGridY) {
    const int nm = n_models - m0 < kMaxGridY ? n_models - m0 : kMaxGridY;
    a.x0 = x0 + (int64_t)m0 * x0_model_stride;
    a.w = w + (int64_t)m0 * t.d * t.K;
    a.sse = sse + (int64_t)m0 * n_ics;
    a.valid = valid_rows + (int64_t)m0 * n_ics;
    const int st = launch_score(t, a, method, nm, s);
    if (st != SB_OK) return st;
  }
  return SB_OK;
}

}  // namespace sb
