// sb_rollout.cu — lock-step fixed-step integration of dx/dt = Θ(x)·Wᵀ for a batch of initial conditions (sb_rollout),
// and M models × N initial conditions integrated and scored against observed rows in one launch (sb_rollout_score).
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
  const float* x0;
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
    static_for<0, D>([&](auto j) { x[b][j] = track[b] ? a.x0[ic * D + j] : 0.f; });
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
  float x[1][DN];
#pragma unroll
  for (int j = 0; j < DN; ++j) x[0][j] = (j < d) ? a.x0[ic * d + j] : 0.f;
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

}  // namespace

int rollout(const void* x0, int64_t n_ics, const LibTab& t, const void* w, double dt, int64_t n_steps,
            int64_t stride, int method, int dtype, int record_dx, void* x_out, void* dx_out, void* x_last,
            cudaStream_t s) {
  RollArgs a{};
  a.x0 = x0; a.n_ics = n_ics; a.dt = dt; a.n_steps = n_steps; a.stride = stride; a.method = method;
  a.record_dx = record_dx; a.opaque = 0; a.x_out = x_out; a.dx_out = dx_out; a.x_last = x_last;
  if (dtype == SB_F32) return launch_rollout<float>(t, w, a, s);
  return launch_rollout<double>(t, w, a, s);
}

int rollout_score(const float* x0, int64_t n_ics, const LibTab& t, const float* w, int n_models, double dt,
                  int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs, float blowup, double* sse,
                  int32_t* valid_rows, cudaStream_t s) {
  ScoreArgs a{};
  a.x0 = x0; a.n_ics = n_ics; a.dt = dt; a.steps_per_row = steps_per_row; a.n_rows = n_rows; a.y_obs = y_obs;
  a.blowup = blowup; a.opaque = 0;
  // more models than gridDim.y allows: further launches on the same stream
  for (int m0 = 0; m0 < n_models; m0 += kMaxGridY) {
    const int nm = n_models - m0 < kMaxGridY ? n_models - m0 : kMaxGridY;
    a.w = w + (int64_t)m0 * t.d * t.K;
    a.sse = sse + (int64_t)m0 * n_ics;
    a.valid = valid_rows + (int64_t)m0 * n_ics;
    const int st = launch_score(t, a, method, nm, s);
    if (st != SB_OK) return st;
  }
  return SB_OK;
}

}  // namespace sb
