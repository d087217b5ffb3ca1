// sb_rollout_score.cu — M models × N initial conditions integrated in one launch and scored against observed rows.
//
// Model selection simulates every candidate Ξ of a threshold path from every validation initial condition and compares
// the states with the data. With sb_rollout that is one launch, one HBM trajectory and one reduction per model; here a
// thread integrates its (model, IC) pairs and folds each compared row into an fp64 SSE in registers: the only HBM
// traffic is x0, the observed rows (shared by all models, so L2-resident for cfg-sized data) and two outputs per pair.
//
// Bit identity with sb_rollout (odeint mode, fp32): the states compared are the states sb_rollout stores. Every kernel
// below repeats the operation order of the kernel launch_rollout (sb_rollout.cu) dispatches to for the same library —
// the same monomial recurrence, the same explicit round-to-nearest update formulas, and for the specialised shapes the
// same packed-FMA pairs accumulated alternately into two partial sums; for the runtime-table path one fma chain per
// output. Where W comes from does not enter the arithmetic.
//
// W delivery: the coefficients are produced on the device (STLSQ), so they cannot become kernel parameters without a
// device-to-host copy and a host synchronisation per call, and a per-module __constant__ slot would be shared by
// concurrent streams. Each block of the specialised kernels stages its model's W (≤ 168 floats) in shared memory and
// reads it as float4 (two packed pairs) with a block-uniform address, so one LDS.128 feeds 2·NB packed FMAs. As in
// rollout_rk4_multi_kernel, an opaque zero offset per call site keeps ptxas from hoisting the loop-invariant loads into
// registers it does not have.
#include "sb_common.cuh"

namespace sb {

namespace {

constexpr int kScoreThreads = 64;  // two ICs per thread: 128 ICs per block, as rollout_rk4_multi_kernel
constexpr int kScoreNB = 2;
constexpr int kGenThreads = 128;   // runtime-table path: one IC per thread, as rollout_gen_kernel
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

// Θ(x)·Wᵀ for NB states of a specialised library (code PC: sb_common.cuh LibCode), W from shared memory laid out as
// D rows of KQ float4 (K/2 pairs, zero-padded to an even count). Per state and output the pairs are accumulated in the
// order of SpecRhs / eval_multi (sb_rollout.cu): pair kk into s0 (kk even) or s1 (kk odd), f = (s0.x+s0.y)+(s1.x+s1.y).
template <int D, int PC, int NB>
__device__ __forceinline__ void eval_score(const float4* sw, const float (&x)[NB][D], float (&f)[NB][D], int off) {
  using L = LibCode<D, PC>;
  constexpr int NP = L::NP, K = L::K, KQ = (K / 2 + 1) / 2;
  static_assert(K % 2 == 0, "packed pairs");
  using Tab = Poly<D, L::P>;
  const float4* w4 = sw + off;
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
      } else if constexpr (k < NP + D * L::S) m[b][k] = sin(x[b][k - NP]);  // sinf / expf by overload, as SpecRhs
      else m[b][k] = exp(x[b][k - NP - D * L::S]);
    });
    if constexpr (k % 2 == 1) {
      constexpr int kk = k / 2;
      static_for<0, D>([&](auto ic) {
        constexpr int i = ic;
        if constexpr (kk % 2 == 0) wq[i] = w4[i * KQ + kk / 2];
        const float2 w = (kk % 2 == 0) ? make_float2(wq[i].x, wq[i].y) : make_float2(wq[i].z, wq[i].w);
        static_for<0, NB>([&](auto bc) {
          constexpr int b = bc;
          const float2 m2 = make_float2(m[b][k - 1], m[b][k]);
          if constexpr (kk % 2 == 0) s0[b][i] = __ffma2_rn(w, m2, s0[b][i]);
          else s1[b][i] = __ffma2_rn(w, m2, s1[b][i]);
        });
      });
    }
  });
  static_for<0, NB>([&](auto b) {
    static_for<0, D>([&](auto i) { f[b][i] = (s0[b][i].x + s0[b][i].y) + (s1[b][i].x + s1[b][i].y); });
  });
}

// grid = (IC blocks, models); NB = 2 ICs per thread. METHOD: SB_EULER (rollout_spec_kernel's odeint branch) or SB_RK4
// (rollout_rk4_multi_kernel); both are the same formulas per IC.
template <int D, int PC, int METHOD>
__global__ void __launch_bounds__(kScoreThreads) rollout_score_spec_kernel(ScoreArgs a) {
  constexpr int NB = kScoreNB;
  constexpr int K = LibCode<D, PC>::K, KQ = (K / 2 + 1) / 2;
  __shared__ float4 sw[D * KQ];
  const int64_t model = blockIdx.y;
  {
    const float* wm = a.w + model * (D * K);
    float* s = reinterpret_cast<float*>(sw);
    for (int q = threadIdx.x; q < D * KQ * 4; q += kScoreThreads) {
      const int i = q / (KQ * 4), c = q % (KQ * 4);
      s[q] = c < K ? wm[i * K + c] : 0.f;
    }
  }
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * (kScoreThreads * NB) + threadIdx.x;
  if (base >= a.n_ics) return;
  float x[NB][D], k1[NB][D], k2[NB][D], k3[NB][D], k4[NB][D], xt[NB][D];
  bool track[NB];
  double sse[NB];
  int64_t valid[NB];
  static_for<0, NB>([&](auto bc) {
    constexpr int b = bc;
    const int64_t ic = base + (int64_t)b * kScoreThreads;
    track[b] = ic < a.n_ics;
    sse[b] = 0.0;
    valid[b] = a.n_rows;
    static_for<0, D>([&](auto j) { x[b][j] = track[b] ? a.x0[ic * D + j] : 0.f; });
  });
  const bool live1 = track[1];
  const float dt = (float)a.dt, hdt = (float)(a.dt / 2.0), sdt = (float)(a.dt / 6.0), two = 2.f;
  const int64_t row_elems = a.n_ics * D;
  int64_t row = 0, until = a.steps_per_row;
  for (int64_t s = 1;; ++s) {
    eval_score<D, PC, NB>(sw, x, k1, (int)(s & a.opaque));
    if constexpr (METHOD == SB_EULER) {
      static_for<0, NB>([&](auto b) { static_for<0, D>([&](auto j) { x[b][j] = __fadd_rn(x[b][j], __fmul_rn(dt, k1[b][j])); }); });
    } else {
      static_for<0, NB>([&](auto b) { static_for<0, D>([&](auto j) { xt[b][j] = __fadd_rn(x[b][j], __fmul_rn(hdt, k1[b][j])); }); });
      eval_score<D, PC, NB>(sw, xt, k2, (int)((s + 1) & a.opaque));
      static_for<0, NB>([&](auto b) { static_for<0, D>([&](auto j) { xt[b][j] = __fadd_rn(x[b][j], __fmul_rn(hdt, k2[b][j])); }); });
      eval_score<D, PC, NB>(sw, xt, k3, (int)((s + 2) & a.opaque));
      static_for<0, NB>([&](auto b) { static_for<0, D>([&](auto j) { xt[b][j] = __fadd_rn(x[b][j], __fmul_rn(dt, k3[b][j])); }); });
      eval_score<D, PC, NB>(sw, xt, k4, (int)((s + 3) & a.opaque));
      static_for<0, NB>([&](auto b) {
        static_for<0, D>([&](auto j) {
          float acc = __fadd_rn(k1[b][j], __fmul_rn(two, k2[b][j]));
          acc = __fadd_rn(acc, __fmul_rn(two, k3[b][j]));
          acc = __fadd_rn(acc, k4[b][j]);
          x[b][j] = __fadd_rn(x[b][j], __fmul_rn(sdt, acc));
        });
      });
    }
    if (--until == 0) {
      const float* y = a.y_obs + row * row_elems;
      static_for<0, NB>([&](auto bc) {
        constexpr int b = bc;
        const int64_t ic = base + (int64_t)b * kScoreThreads;
        if (track[b] && !score_row<D>(x[b], D, y + ic * D, a.blowup, sse[b])) { track[b] = false; valid[b] = row; }
      });
      ++row;
      until = a.steps_per_row;
      if (row == a.n_rows || !(track[0] || track[1])) break;
    }
  }
  static_for<0, NB>([&](auto bc) {
    constexpr int b = bc;
    const int64_t ic = base + (int64_t)b * kScoreThreads;
    if (b == 0 || live1) {
      a.sse[model * a.n_ics + ic] = sse[b];
      a.valid[model * a.n_ics + ic] = (int32_t)valid[b];
    }
  });
}

// Runtime-table library: GenRhs of sb_rollout.cu (one fma chain per output, W from global memory), one IC per thread.
template <int KMAX>
__global__ void __launch_bounds__(kGenThreads) rollout_score_gen_kernel(LibTab t, int method, ScoreArgs a) {
  constexpr int DN = SB_MAX_DIM;
  const int64_t ic = (int64_t)blockIdx.x * kGenThreads + threadIdx.x;
  if (ic >= a.n_ics) return;
  const int64_t model = blockIdx.y;
  const int d = t.d;
  const float* w = a.w + model * d * t.K;
  auto eval = [&](const float (&xs)[DN], float (&f)[DN]) {
    float m[KMAX];
    m[0] = 1.f;
    for (int j = 0; j < d; ++j) m[1 + j] = xs[j];
    for (int k = 1 + d; k < t.n_poly; ++k) m[k] = m[t.parent[k]] * xs[t.var[k]];
    int k = t.n_poly;
    if (t.sine) for (int j = 0; j < d; ++j) m[k++] = sin(xs[j]);
    if (t.exp_) for (int j = 0; j < d; ++j) m[k++] = exp(xs[j]);
    for (int i = 0; i < d; ++i) {
      float s = 0.f;
      for (int q = 0; q < t.K; ++q) s = fma(__ldg(w + i * t.K + q), m[q], s);
      f[i] = s;
    }
  };
  float x[DN], k1[DN], k2[DN], k3[DN], k4[DN], xt[DN];
#pragma unroll
  for (int j = 0; j < DN; ++j) x[j] = (j < d) ? a.x0[ic * d + j] : 0.f;
  const float dt = (float)a.dt, hdt = (float)(a.dt / 2.0), sdt = (float)(a.dt / 6.0), two = 2.f;
  double sse = 0.0;
  int64_t valid = a.n_rows, row = 0, until = a.steps_per_row;
  for (;;) {
    eval(x, k1);
    if (method == SB_EULER) {
#pragma unroll
      for (int j = 0; j < DN; ++j) x[j] = __fadd_rn(x[j], __fmul_rn(dt, k1[j]));
    } else {
#pragma unroll
      for (int j = 0; j < DN; ++j) xt[j] = __fadd_rn(x[j], __fmul_rn(hdt, k1[j]));
      eval(xt, k2);
#pragma unroll
      for (int j = 0; j < DN; ++j) xt[j] = __fadd_rn(x[j], __fmul_rn(hdt, k2[j]));
      eval(xt, k3);
#pragma unroll
      for (int j = 0; j < DN; ++j) xt[j] = __fadd_rn(x[j], __fmul_rn(dt, k3[j]));
      eval(xt, k4);
#pragma unroll
      for (int j = 0; j < DN; ++j) {
        float acc = __fadd_rn(k1[j], __fmul_rn(two, k2[j]));
        acc = __fadd_rn(acc, __fmul_rn(two, k3[j]));
        acc = __fadd_rn(acc, k4[j]);
        x[j] = __fadd_rn(x[j], __fmul_rn(sdt, acc));
      }
    }
    if (--until == 0) {
      if (!score_row<DN>(x, d, a.y_obs + (row * a.n_ics + ic) * d, a.blowup, sse)) { valid = row; break; }
      if (++row == a.n_rows) break;
      until = a.steps_per_row;
    }
  }
  a.sse[model * a.n_ics + ic] = sse;
  a.valid[model * a.n_ics + ic] = (int32_t)valid;
}

template <int D, int PC>
int launch_spec(const ScoreArgs& a, int method, int n_models, cudaStream_t s) {
  const unsigned gx = (unsigned)((a.n_ics + kScoreThreads * kScoreNB - 1) / (kScoreThreads * kScoreNB));
  const dim3 grid(gx, (unsigned)n_models);
  if (method == SB_EULER) rollout_score_spec_kernel<D, PC, SB_EULER><<<grid, kScoreThreads, 0, s>>>(a);
  else rollout_score_spec_kernel<D, PC, SB_RK4><<<grid, kScoreThreads, 0, s>>>(a);
  SB_LAUNCH_CHECK("rollout_score_spec_kernel");
  return SB_OK;
}

int launch_score(const LibTab& t, const ScoreArgs& a, int method, int n_models, cudaStream_t s) {
  // the libraries launch_rollout (sb_rollout.cu) specialises, with their PC codes; everything else: runtime table
#define SB_SCORE_SPEC(D, PC) \
  if (lib_matches<D, PC>(t)) return launch_spec<D, PC>(a, method, n_models, s);
  SB_SCORE_SPEC(2, 2) SB_SCORE_SPEC(2, 3) SB_SCORE_SPEC(3, 2) SB_SCORE_SPEC(3, 3) SB_SCORE_SPEC(3, 5)
  SB_SCORE_SPEC(2, 12)
#undef SB_SCORE_SPEC
  const dim3 grid((unsigned)((a.n_ics + kGenThreads - 1) / kGenThreads), (unsigned)n_models);
  if (t.K <= 16) rollout_score_gen_kernel<16><<<grid, kGenThreads, 0, s>>>(t, method, a);
  else if (t.K <= 64) rollout_score_gen_kernel<64><<<grid, kGenThreads, 0, s>>>(t, method, a);
  else rollout_score_gen_kernel<256><<<grid, kGenThreads, 0, s>>>(t, method, a);
  SB_LAUNCH_CHECK("rollout_score_gen_kernel");
  return SB_OK;
}

}  // namespace

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
