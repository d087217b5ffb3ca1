// sb_generic.cu — runtime-table kernels that cover EVERY supported library (dim <= 8, poly_order <= 5,
// optional sin/exp columns, K <= 256). One thread owns one sample; the library row lives in a per-thread
// local array that is filled by the parent/variable recurrence. These kernels are the parity-complete
// path; the hot shapes are served by the register-resident specialisations in sb_fused.cu / sb_rollout.cu.
//
// Reductions ("rows" kernel): out[row, k] = sum_n L_row(n) * F_k(n). blockIdx.y selects the row, so a thread
// never holds more than K accumulators:
//   train step : rows = d residual rows (L = r_i, also sum r_i^2) [+ K Gram rows (L = Θ_a)] [+ d rows (L = dx_i)]
//   backward   : rows = d (L = gy_i, F = Θ)                         -> dL/dW      (`train.py:689`)
//   jvp bwd    : rows = d (L = g_i,  F = J_Θ(x)u)                   -> dL/dW of the JVP (`model_utils.py:56`)
// Per-thread sums are fp32, everything across threads is fp64; the last block to finish (ticket counter)
// adds the per-block partials in index order, so results are run-to-run deterministic.
#include "sb_common.cuh"

namespace sb {

namespace {

constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------------------
// per-sample sweeps over the library recurrence
// ------------------------------------------------------------------------------------------------
template <int KMAX>
__device__ __forceinline__ void load_x(const float* __restrict__ x, int64_t s, int d, float* xv) {
#pragma unroll
  for (int j = 0; j < SB_MAX_DIM; ++j)
    if (j < d) xv[j] = __ldg(x + s * d + j);
}

// tt = J_Θ(x)·u by forward differentiation of the recurrence
template <int KMAX>
__device__ __forceinline__ void tangent(const LibTab& t, const float* xv, const float* uv, const float* m,
                                        float* tt) {
  tt[0] = 0.f;
  for (int j = 0; j < t.d; ++j) tt[1 + j] = uv[j];
  for (int k = 1 + t.d; k < t.n_poly; ++k) {
    const int p = t.parent[k], v = t.var[k];
    tt[k] = tt[p] * xv[v] + m[p] * uv[v];
  }
  int k = t.n_poly;
  if (t.sine) for (int j = 0; j < t.d; ++j) tt[k++] = cosf(xv[j]) * uv[j];
  if (t.exp_) for (int j = 0; j < t.d; ++j, ++k) tt[k] = m[k] * uv[j];
}

template <int KMAX>
__device__ __forceinline__ float dot_w(const float* __restrict__ w, int i, int K, const float* f) {
  float acc = 0.f;
  for (int k = 0; k < K; ++k) acc = fmaf(__ldg(w + i * K + k), f[k], acc);
  return acc;
}

// ------------------------------------------------------------------------------------------------
// per-sample map kernels
// ------------------------------------------------------------------------------------------------
template <int KMAX>
__global__ void __launch_bounds__(kThreads) theta_kernel(LibTab t, const float* __restrict__ x, int64_t n,
                                                         float* __restrict__ theta) {
  float m[KMAX], xv[SB_MAX_DIM];
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
    load_x<KMAX>(x, s, t.d, xv);
    expand_table(t, xv, m);
    for (int k = 0; k < t.K; ++k) theta[s * t.K + k] = m[k];
  }
}

template <int KMAX>
__global__ void __launch_bounds__(kThreads) forward_kernel(LibTab t, const float* __restrict__ x, int64_t n,
                                                           const float* __restrict__ w, float* __restrict__ y) {
  float m[KMAX], xv[SB_MAX_DIM];
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
    load_x<KMAX>(x, s, t.d, xv);
    expand_table(t, xv, m);
    for (int i = 0; i < t.d; ++i) y[s * t.d + i] = dot_w<KMAX>(w, i, t.K, m);
  }
}

template <int KMAX>
__global__ void __launch_bounds__(kThreads) jvp_kernel(LibTab t, const float* __restrict__ x,
                                                       const float* __restrict__ u, int64_t n,
                                                       const float* __restrict__ w, float* __restrict__ out) {
  float m[KMAX], tt[KMAX], xv[SB_MAX_DIM], uv[SB_MAX_DIM];
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
    load_x<KMAX>(x, s, t.d, xv);
    load_x<KMAX>(u, s, t.d, uv);
    expand_table(t, xv, m);
    tangent<KMAX>(t, xv, uv, m, tt);
    for (int i = 0; i < t.d; ++i) out[s * t.d + i] = dot_w<KMAX>(w, i, t.K, tt);
  }
}

// gx = J_h(x)^T gy: reverse sweep with mbar initialised to c_k = sum_i gy_i W_ik
template <int KMAX>
__global__ void __launch_bounds__(kThreads) backward_x_kernel(LibTab t, const float* __restrict__ x,
                                                              const float* __restrict__ gy, int64_t n,
                                                              const float* __restrict__ w,
                                                              float* __restrict__ gx) {
  float m[KMAX], mb[KMAX], xv[SB_MAX_DIM], gv[SB_MAX_DIM], xb[SB_MAX_DIM];
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
    load_x<KMAX>(x, s, t.d, xv);
    load_x<KMAX>(gy, s, t.d, gv);
    expand_table(t, xv, m);
    for (int k = 0; k < t.K; ++k) {
      float c = 0.f;
      for (int i = 0; i < t.d; ++i) c = fmaf(gv[i], __ldg(w + i * t.K + k), c);
      mb[k] = c;
    }
    for (int j = 0; j < t.d; ++j) xb[j] = 0.f;
    for (int k = t.n_poly - 1; k > t.d; --k) {
      const int p = t.parent[k], v = t.var[k];
      mb[p] = fmaf(mb[k], xv[v], mb[p]);
      xb[v] = fmaf(mb[k], m[p], xb[v]);
    }
    for (int j = 0; j < t.d; ++j) xb[j] += mb[1 + j];
    int k = t.n_poly;
    if (t.sine) for (int j = 0; j < t.d; ++j, ++k) xb[j] = fmaf(mb[k], cosf(xv[j]), xb[j]);
    if (t.exp_) for (int j = 0; j < t.d; ++j, ++k) xb[j] = fmaf(mb[k], m[k], xb[j]);
    for (int j = 0; j < t.d; ++j) gx[s * t.d + j] = xb[j];
  }
}

// cotangents of out = W·(J_Θ(x)u) w.r.t. x (Hessian-vector term) and u (= J_h^T g)
template <int KMAX>
__global__ void __launch_bounds__(kThreads) jvp_backward_xu_kernel(LibTab t, const float* __restrict__ x,
                                                                   const float* __restrict__ u,
                                                                   const float* __restrict__ g, int64_t n,
                                                                   const float* __restrict__ w,
                                                                   float* __restrict__ gx,
                                                                   float* __restrict__ gu) {
  float m[KMAX], tt[KMAX], tb[KMAX], mb[KMAX];
  float xv[SB_MAX_DIM], uv[SB_MAX_DIM], gv[SB_MAX_DIM], xb[SB_MAX_DIM], ub[SB_MAX_DIM];
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (int64_t)gridDim.x * blockDim.x) {
    load_x<KMAX>(x, s, t.d, xv);
    load_x<KMAX>(u, s, t.d, uv);
    load_x<KMAX>(g, s, t.d, gv);
    expand_table(t, xv, m);
    tangent<KMAX>(t, xv, uv, m, tt);
    for (int k = 0; k < t.K; ++k) {
      float c = 0.f;
      for (int i = 0; i < t.d; ++i) c = fmaf(gv[i], __ldg(w + i * t.K + k), c);
      tb[k] = c;
      mb[k] = 0.f;
    }
    for (int j = 0; j < t.d; ++j) { xb[j] = 0.f; ub[j] = 0.f; }
    for (int k = t.n_poly - 1; k > t.d; --k) {
      const int p = t.parent[k], v = t.var[k];
      // tt[k] = tt[p]*x[v] + m[p]*u[v]
      tb[p] = fmaf(tb[k], xv[v], tb[p]);
      xb[v] = fmaf(tb[k], tt[p], xb[v]);
      mb[p] = fmaf(tb[k], uv[v], mb[p]);
      ub[v] = fmaf(tb[k], m[p], ub[v]);
      // m[k] = m[p]*x[v]
      mb[p] = fmaf(mb[k], xv[v], mb[p]);
      xb[v] = fmaf(mb[k], m[p], xb[v]);
    }
    for (int j = 0; j < t.d; ++j) { ub[j] += tb[1 + j]; xb[j] += mb[1 + j]; }
    int k = t.n_poly;
    if (t.sine)
      for (int j = 0; j < t.d; ++j, ++k) {
        ub[j] = fmaf(tb[k], cosf(xv[j]), ub[j]);
        xb[j] = fmaf(-tb[k] * m[k], uv[j], xb[j]);  // m[k] = sin(x_j)
      }
    if (t.exp_)
      for (int j = 0; j < t.d; ++j, ++k) {
        ub[j] = fmaf(tb[k], m[k], ub[j]);
        xb[j] = fmaf(tb[k] * m[k], uv[j], xb[j]);
      }
    if (gx) for (int j = 0; j < t.d; ++j) gx[s * t.d + j] = xb[j];
    if (gu) for (int j = 0; j < t.d; ++j) gu[s * t.d + j] = ub[j];
  }
}

// ------------------------------------------------------------------------------------------------
// rows (reduction) kernel
// ------------------------------------------------------------------------------------------------
enum { MODE_STEP = 0, MODE_BWD = 1, MODE_JVPBWD = 2 };

struct RowsArgs {
  const float* x;
  const float* a;   // STEP: dx   BWD: gy   JVPBWD: u
  const float* b;   // JVPBWD: g
  const float* w;
  int64_t n;
  uint32_t flags;   // STEP only
  int n_rows;
  int nbx;
  double* partial;  // [n_rows][nbx][K+1]
  unsigned int* ticket;
  double* out;
};

// row -> (kind, index): kind 0 = residual / cotangent row i, 1 = Gram row a, 2 = b row i
__device__ __forceinline__ void decode_row(int row, int d, int K, uint32_t flags, int mode, int& kind, int& idx) {
  if (mode != MODE_STEP) { kind = 0; idx = row; return; }
  int r = row;
  if (flags & (SB_STEP_LOSS | SB_STEP_GRAD)) {
    if (r < d) { kind = 0; idx = r; return; }
    r -= d;
  }
  if (flags & SB_STEP_GRAM) {
    if (r < K) { kind = 1; idx = r; return; }
    r -= K;
  }
  kind = 2; idx = r;
}

template <int KMAX, int MODE>
__global__ void __launch_bounds__(kThreads) rows_kernel(LibTab t, RowsArgs a) {
  constexpr int NW = kThreads / 32;
  __shared__ float red[NW][KMAX + 1];
  __shared__ int is_last;

  float m[KMAX], acc[KMAX];
  float tt[MODE == MODE_JVPBWD ? KMAX : 1];
  float xv[SB_MAX_DIM], uv[SB_MAX_DIM];
  const int d = t.d, K = t.K;
  int kind, idx;
  decode_row(blockIdx.y, d, K, a.flags, MODE, kind, idx);
  const bool want_acc = !(MODE == MODE_STEP && kind == 0 && !(a.flags & SB_STEP_GRAD));

  for (int k = 0; k < K; ++k) acc[k] = 0.f;
  float lacc = 0.f;

  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < a.n; s += (int64_t)a.nbx * blockDim.x) {
    load_x<KMAX>(a.x, s, d, xv);
    expand_table(t, xv, m);
    float L;
    const float* feat = m;
    if (MODE == MODE_STEP) {
      if (kind == 0) {
        L = dot_w<KMAX>(a.w, idx, K, m) - __ldg(a.a + s * d + idx);
        lacc = fmaf(L, L, lacc);
      } else if (kind == 1) {
        L = m[idx];
      } else {
        L = __ldg(a.a + s * d + idx);
      }
    } else if (MODE == MODE_BWD) {
      L = __ldg(a.a + s * d + idx);
    } else {
      load_x<KMAX>(a.a, s, d, uv);
      tangent<KMAX>(t, xv, uv, m, tt);
      feat = tt;
      L = __ldg(a.b + s * d + idx);
    }
    if (want_acc)
      for (int k = 0; k < K; ++k) acc[k] = fmaf(L, feat[k], acc[k]);
  }

  // block reduction: warp shuffles (fp32) then fp64 across warps
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int k = 0; k < K; ++k) {
    float v = warp_sum(acc[k]);
    if (lane == 0) red[wid][k] = v;
  }
  {
    float v = warp_sum(lacc);
    if (lane == 0) red[wid][K] = v;
  }
  __syncthreads();
  double* my_partial = a.partial + ((int64_t)blockIdx.y * a.nbx + blockIdx.x) * (K + 1);
  for (int k = threadIdx.x; k <= K; k += blockDim.x) {
    double v = 0.0;
#pragma unroll
    for (int wq = 0; wq < NW; ++wq) v += (double)red[wq][k];
    my_partial[k] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int total = gridDim.x * gridDim.y;
    is_last = (atomicAdd(a.ticket, 1u) == total - 1u);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();

  // final, ordered reduction over blockIdx.x by the last block
  const int n_rows = a.n_rows;
  for (int e = threadIdx.x; e < n_rows * K; e += blockDim.x) {
    const int row = e / K, k = e % K;
    int rk, ri;
    decode_row(row, d, K, a.flags, MODE, rk, ri);
    if (MODE == MODE_STEP && rk == 0 && !(a.flags & SB_STEP_GRAD)) continue;
    const double* p = a.partial + (int64_t)row * a.nbx * (K + 1) + k;
    double v = 0.0;
    for (int bx = 0; bx < a.nbx; ++bx) v += p[(int64_t)bx * (K + 1)];
    if (MODE != MODE_STEP) {
      a.out[ri * K + k] = v;
    } else {
      int64_t off = 2;
      if (rk == 0) { a.out[off + ri * K + k] = v; continue; }
      if (a.flags & SB_STEP_GRAD) off += (int64_t)d * K;
      if (rk == 1) { a.out[off + (int64_t)ri * K + k] = v; continue; }
      if (a.flags & SB_STEP_GRAM) off += (int64_t)K * K;
      a.out[off + (int64_t)k * d + ri] = v;
    }
  }
  if (MODE == MODE_STEP && threadIdx.x == 0) {
    double loss = 0.0;
    if (a.flags & (SB_STEP_LOSS | SB_STEP_GRAD))
      for (int i = 0; i < d; ++i)
        for (int bx = 0; bx < a.nbx; ++bx) loss += a.partial[((int64_t)i * a.nbx + bx) * (K + 1) + K];
    a.out[0] = loss;
    a.out[1] = (double)a.n;
  }
  if (threadIdx.x == 0) *a.ticket = 0u;
}

inline int map_grid(int64_t n) {
  int64_t b = (n + kThreads - 1) / kThreads;
  if (b < 1) b = 1;
  if (b > 148 * 8) b = 148 * 8;
  return (int)b;
}

inline int rows_nbx(int64_t n, int n_rows) {
  int64_t by_n = (n + kThreads - 1) / kThreads;
  int64_t cap = (kMaxPartialBlocks + n_rows - 1) / n_rows;
  if (cap < 1) cap = 1;
  int64_t b = by_n < cap ? by_n : cap;
  return (int)(b < 1 ? 1 : b);
}

inline int max_rows(const LibTab& t) { return 2 * t.d + t.K; }

// picks the local-array size class
#define SB_KMAX_DISPATCH(K, CALL)            \
  do {                                       \
    if ((K) <= 16) { CALL(16); }             \
    else if ((K) <= 64) { CALL(64); }        \
    else { CALL(256); }                      \
  } while (0)

template <int MODE>
int launch_rows(const LibTab& t, RowsArgs a, void* ws, int64_t ws_bytes, cudaStream_t s) {
  a.nbx = rows_nbx(a.n, a.n_rows);
  const int64_t need = kWsHeaderBytes + (int64_t)a.n_rows * a.nbx * (t.K + 1) * (int64_t)sizeof(double);
  if (ws_bytes < need) {
    set_error("workspace too small: %lld < %lld bytes", (long long)ws_bytes, (long long)need);
    return SB_ERR_WORKSPACE;
  }
  a.ticket = reinterpret_cast<unsigned int*>(ws);
  a.partial = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + kWsHeaderBytes);
  dim3 grid(a.nbx, a.n_rows);
#define CALL(KM) rows_kernel<KM, MODE><<<grid, kThreads, 0, s>>>(t, a)
  SB_KMAX_DISPATCH(t.K, CALL);
#undef CALL
  SB_LAUNCH_CHECK("rows_kernel");
  return SB_OK;
}

// loss = Σr²/(n·d) + w_l1·‖Ξ‖₁ ; grad = 2/(n·d)·(Σ r⊗Θ)⊙mask + w_l1·sign(Ξ)   (`train.py:663-664,680-683,689`)
__global__ void __launch_bounds__(kThreads) epilogue_kernel(const double* __restrict__ packed, int d, int K,
                                                            const float* __restrict__ xi,
                                                            const float* __restrict__ mask, double w_l1,
                                                            float* __restrict__ loss_out,
                                                            float* __restrict__ grad_out) {
  __shared__ double l1w[kThreads / 32];
  const double n = packed[1];
  const double denom = (n > 0.0 ? n : 1.0) * d;
  double l1 = 0.0;
  for (int e = threadIdx.x; e < d * K; e += blockDim.x) {
    const float v = xi[e];
    const float mk = mask ? mask[e] : 1.f;
    l1 += fabs((double)v);
    if (grad_out) {
      const double sgn = (v > 0.f) ? 1.0 : ((v < 0.f) ? -1.0 : 0.0);
      grad_out[e] = (float)(packed[2 + e] * (2.0 / denom) * (double)mk + w_l1 * sgn);
    }
  }
  l1 = warp_sum(l1);
  if ((threadIdx.x & 31) == 0) l1w[threadIdx.x >> 5] = l1;
  __syncthreads();
  if (threadIdx.x == 0 && loss_out) {
    double t = 0.0;
    for (int wq = 0; wq < kThreads / 32; ++wq) t += l1w[wq];
    *loss_out = (float)(packed[0] / denom + w_l1 * t);
  }
}

__global__ void mask_mul_kernel(const float* __restrict__ xi, const float* __restrict__ mask, float* __restrict__ dst,
                                int count) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < count) dst[t] = mask ? xi[t] * mask[t] : xi[t];
}

}  // namespace

int step_epilogue(const double* packed, const LibTab& t, const float* xi, const float* mask, double w_l1,
                  float* loss_out, float* grad_out, cudaStream_t s) {
  epilogue_kernel<<<1, kThreads, 0, s>>>(packed, t.d, t.K, xi, mask, w_l1, loss_out, grad_out);
  SB_LAUNCH_CHECK("epilogue_kernel");
  return SB_OK;
}

int mask_mul(const float* xi, const float* mask, float* dst, int count, cudaStream_t s) {
  mask_mul_kernel<<<(count + 255) / 256, 256, 0, s>>>(xi, mask, dst, count);
  SB_LAUNCH_CHECK("mask_mul_kernel");
  return SB_OK;
}

int64_t generic_workspace_bytes(const LibTab& t) {
  // worst case over row counts r in [1, 2d+K]: r * ceil(cap/r) <= cap + r; plus a d×K fp32 scratch for Ξ⊙mask
  const int64_t r = max_rows(t);
  return kWsHeaderBytes + (int64_t)(kMaxPartialBlocks + r) * (t.K + 1) * (int64_t)sizeof(double) +
         (int64_t)t.d * t.K * (int64_t)sizeof(float) + 256;
}

int generic_theta(const float* x, int64_t n, const LibTab& t, float* theta, cudaStream_t s) {
#define CALL(KM) theta_kernel<KM><<<map_grid(n), kThreads, 0, s>>>(t, x, n, theta)
  SB_KMAX_DISPATCH(t.K, CALL);
#undef CALL
  SB_LAUNCH_CHECK("theta_kernel");
  return SB_OK;
}

int generic_forward(const float* x, int64_t n, const LibTab& t, const float* w, float* y, cudaStream_t s) {
#define CALL(KM) forward_kernel<KM><<<map_grid(n), kThreads, 0, s>>>(t, x, n, w, y)
  SB_KMAX_DISPATCH(t.K, CALL);
#undef CALL
  SB_LAUNCH_CHECK("forward_kernel");
  return SB_OK;
}

int generic_jvp(const float* x, const float* u, int64_t n, const LibTab& t, const float* w, float* out,
                cudaStream_t s) {
#define CALL(KM) jvp_kernel<KM><<<map_grid(n), kThreads, 0, s>>>(t, x, u, n, w, out)
  SB_KMAX_DISPATCH(t.K, CALL);
#undef CALL
  SB_LAUNCH_CHECK("jvp_kernel");
  return SB_OK;
}

int generic_backward(const float* x, const float* gy, int64_t n, const LibTab& t, const float* w, double* gw,
                     float* gx, void* ws, int64_t ws_bytes, cudaStream_t s) {
  if (gw) {
    RowsArgs a{};
    a.x = x; a.a = gy; a.w = w; a.n = n; a.flags = 0; a.n_rows = t.d; a.out = gw;
    int st = launch_rows<MODE_BWD>(t, a, ws, ws_bytes, s);
    if (st != SB_OK) return st;
  }
  if (gx && n > 0) {
#define CALL(KM) backward_x_kernel<KM><<<map_grid(n), kThreads, 0, s>>>(t, x, gy, n, w, gx)
    SB_KMAX_DISPATCH(t.K, CALL);
#undef CALL
    SB_LAUNCH_CHECK("backward_x_kernel");
  }
  return SB_OK;
}

int generic_jvp_backward(const float* x, const float* u, const float* g, int64_t n, const LibTab& t,
                         const float* w, double* gw, float* gx, float* gu, void* ws, int64_t ws_bytes,
                         cudaStream_t s) {
  if (gw) {
    RowsArgs a{};
    a.x = x; a.a = u; a.b = g; a.w = w; a.n = n; a.flags = 0; a.n_rows = t.d; a.out = gw;
    int st = launch_rows<MODE_JVPBWD>(t, a, ws, ws_bytes, s);
    if (st != SB_OK) return st;
  }
  if ((gx || gu) && n > 0) {
#define CALL(KM) jvp_backward_xu_kernel<KM><<<map_grid(n), kThreads, 0, s>>>(t, x, u, g, n, w, gx, gu)
    SB_KMAX_DISPATCH(t.K, CALL);
#undef CALL
    SB_LAUNCH_CHECK("jvp_backward_xu_kernel");
  }
  return SB_OK;
}

int generic_train_step(const float* x, const float* dx, int64_t n, const LibTab& t, const float* w,
                       uint32_t flags, double* out, void* ws, int64_t ws_bytes, cudaStream_t s) {
  RowsArgs a{};
  a.x = x; a.a = dx; a.w = w; a.n = n; a.flags = flags; a.out = out;
  a.n_rows = 0;
  if (flags & (SB_STEP_LOSS | SB_STEP_GRAD)) a.n_rows += t.d;
  if (flags & SB_STEP_GRAM) a.n_rows += t.K;
  if (flags & SB_STEP_B) a.n_rows += t.d;
  return launch_rows<MODE_STEP>(t, a, ws, ws_bytes, s);
}

}  // namespace sb
