// sb_wsindy_local.cu — WSINDy weak-form integrals with compactly supported piecewise-polynomial test functions.
//
// Every test function is the same window of `L` samples shifted to its own integer start s_j = ⌊j·(T−L)/(n_test−1)⌋:
//   G[r,j,k] = Σ_q phi[q]·Θ_k(x[r, s_j+q]),   b[r,j,i] = −Σ_q dphi[q]·x[r, s_j+q, i],   q = 0..L−1
// with the host-built fp32 tables phi, dphi (include/sindy_b200.h). The job is a strided correlation of [Θ(x) | x]
// with one fixed filter pair, so a sample costs only the ov = L·n_test/T windows that cover it (about 2 at the
// default support) instead of all n_test rows of the global trigonometric family (sb_wsindy.cu).
//
// Work decomposition: one warp owns one (trajectory, window) output row for the whole support. Its lanes take the
// samples q ≡ lane (mod 32) — consecutive lanes read consecutive samples, so the loads of x and of the tables are
// coalesced — expand Θ(x) in registers and accumulate phi·Θ and dphi·x with packed FFMA2 into per-lane fp32
// partials. After every block of 2048 support samples the partials are folded across the warp (transposed
// butterfly, ~V shuffles for V values) and added into fp64 totals; lane-exclusive fp64 totals are written at the end.
// No atomics, no cross-warp reduction: the result of a row depends only on (x[r], j, L, tables), so G[r] has the same
// bits whether trajectory r is computed alone, in any batch, or on a repeat.
//
// Θ is re-expanded for every window that covers a sample (ov times) instead of being staged once in shared memory:
// reading a staged row back costs at least 2 shared-memory wavefronts per warp per column pair, against one FFMA2
// issue slot per column pair and K−1−d multiplications per re-expansion (an SM issues 4 warp instructions per clock but
// serves one shared-memory wavefront), so staging would make the kernel shared-memory-bound.
//
// Libraries with a compile-time specialisation (LibCode<D, PC>, register-resident Θ and accumulators) are listed in
// the dispatcher; every other library sb_library_size accepts takes the runtime-table kernel below (the same
// decomposition with Θ and the accumulators in local memory), selected by the library alone.
#include "sb_common.cuh"

namespace sb {

namespace {

constexpr int kWarps = 4;        // rows per CTA (one warp each)
constexpr int kBlock = 2048;     // support samples per fp32 partial sum

struct WlArgs {
  const float* x;     // n_traj × T × d
  int64_t n_traj;
  int64_t T;
  const float* phi;   // L
  const float* dphi;  // L
  int L;
  int n_test;
  double* G;          // n_traj × n_test × K
  double* b;          // n_traj × n_test × d
};

__device__ __forceinline__ int64_t window_start(int64_t j, const WlArgs& a) {
  return a.n_test == 1 ? 0 : (j * (a.T - a.L)) / (a.n_test - 1);
}

template <int D, int PC>
struct WlCfg {
  static constexpr int K = LibCode<D, PC>::K;
  static constexpr int NC = K + D;                    // columns: Θ_0..Θ_{K−1}, then x_0..x_{D−1}
  static constexpr int NP = (NC + 1) / 2;             // column pairs (one FFMA2 each)
  static constexpr int VF = (2 * NP + 31) / 32 * 32;  // folded values per row, padded to a multiple of 32
  static constexpr int NO = VF / 32;                  // totals per lane after the fold
};

template <int D, int PC>
__global__ void __launch_bounds__(32 * kWarps) wsindy_local_kernel(WlArgs a) {
  using C = WlCfg<D, PC>;
  const int lane = threadIdx.x & 31;
  const int64_t n_rows = a.n_traj * a.n_test;
  for (int64_t row = (int64_t)blockIdx.x * kWarps + (threadIdx.x >> 5); row < n_rows;
       row += (int64_t)gridDim.x * kWarps) {
    const int64_t r = row / a.n_test, j = row - r * a.n_test;
    const float* xs = a.x + (r * a.T + window_start(j, a)) * D;
    double tot[C::NO];
    static_for<0, C::NO>([&](auto i) { tot[i] = 0.0; });
    for (int q0 = 0; q0 < a.L; q0 += kBlock) {
      const int q1 = a.L - q0 < kBlock ? a.L : q0 + kBlock;
      float2 acc[C::NP];
      static_for<0, C::NP>([&](auto c) { acc[c] = make_float2(0.f, 0.f); });
#pragma unroll 2
      for (int q = q0 + lane; q < q1; q += 32) {
        float xv[D];
        static_for<0, D>([&](auto i) { xv[i] = __ldg(xs + (int64_t)q * D + i); });
        const float w = __ldg(a.phi + q), wd = __ldg(a.dphi + q);
        float m[C::K];
        expand_lib<D, PC>(xv, m);
        static_for<0, C::NP>([&](auto pc) {
          constexpr int c0 = 2 * pc, c1 = 2 * pc + 1;
          float v0, v1, w0, w1;
          if constexpr (c0 < C::K) { v0 = m[c0]; w0 = w; } else { v0 = xv[c0 - C::K]; w0 = wd; }
          if constexpr (c1 < C::K) { v1 = m[c1]; w1 = w; }
          else if constexpr (c1 < C::NC) { v1 = xv[c1 - C::K]; w1 = wd; }
          else { v1 = 0.f; w1 = 0.f; }
          acc[pc] = __ffma2_rn(make_float2(w0, w1), make_float2(v0, v1), acc[pc]);
        });
      }
      float v[C::VF];
      static_for<0, C::VF>([&](auto c) {
        if constexpr (c < 2 * C::NP) v[c] = (c & 1) ? acc[c / 2].y : acc[c / 2].x;
        else v[c] = 0.f;
      });
      warp_fold<C::VF>(v, lane);
      static_for<0, C::NO>([&](auto i) { tot[i] += (double)v[i]; });
    }
    static_for<0, C::NO>([&](auto i) {
      const int c = warp_fold_index<C::VF>(i, lane);
      if (c < C::K) a.G[row * C::K + c] = tot[i];
      else if (c < C::NC) a.b[row * D + (c - C::K)] = -tot[i];
    });
  }
}

// Any library: the same rows, blocks and summation structure with a runtime Θ table (expand_table, as in
// sb_wsindy.cu) and per-column warp sums instead of the fold.
template <int KMAX>
__global__ void __launch_bounds__(32 * kWarps) wsindy_local_generic_kernel(LibTab t, WlArgs a) {
  __shared__ double tot[kWarps][KMAX + SB_MAX_DIM];
  const int d = t.d, K = t.K;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  double* wt = tot[wid];
  const int64_t n_rows = a.n_traj * a.n_test;
  for (int64_t row0 = (int64_t)blockIdx.x * kWarps; row0 < n_rows; row0 += (int64_t)gridDim.x * kWarps) {
    const int64_t row = row0 + wid;
    if (row < n_rows) {   // warp-uniform
      const int64_t r = row / a.n_test, j = row - r * a.n_test;
      const float* xs = a.x + (r * a.T + window_start(j, a)) * d;
      for (int c = lane; c < K + d; c += 32) wt[c] = 0.0;
      for (int q0 = 0; q0 < a.L; q0 += kBlock) {
        const int q1 = a.L - q0 < kBlock ? a.L : q0 + kBlock;
        float m[KMAX], acc[KMAX], accb[SB_MAX_DIM], xv[SB_MAX_DIM];
        for (int k = 0; k < K; ++k) acc[k] = 0.f;
#pragma unroll
        for (int i = 0; i < SB_MAX_DIM; ++i) accb[i] = 0.f;
        for (int q = q0 + lane; q < q1; q += 32) {
#pragma unroll
          for (int i = 0; i < SB_MAX_DIM; ++i)
            if (i < d) xv[i] = __ldg(xs + (int64_t)q * d + i);
          const float w = __ldg(a.phi + q), wd = __ldg(a.dphi + q);
          expand_table(t, xv, m);
          for (int c = 0; c < K; ++c) acc[c] = fmaf(w, m[c], acc[c]);
#pragma unroll
          for (int i = 0; i < SB_MAX_DIM; ++i)
            if (i < d) accb[i] = fmaf(wd, xv[i], accb[i]);
        }
        for (int c = 0; c < K; ++c) {
          const float s = warp_sum(acc[c]);
          if (lane == (c & 31)) wt[c] += (double)s;
        }
#pragma unroll
        for (int i = 0; i < SB_MAX_DIM; ++i) {
          if (i < d) {
            const float s = warp_sum(accb[i]);
            if (lane == ((K + i) & 31)) wt[K + i] += (double)s;
          }
        }
      }
      __syncwarp();
      for (int c = lane; c < K + d; c += 32) {
        if (c < K) a.G[row * K + c] = wt[c];
        else a.b[row * d + (c - K)] = -wt[c];
      }
      __syncwarp();
    }
  }
}

}  // namespace

int wsindy_local_integrals(const float* x, int64_t n_traj, int64_t T, const LibTab& t, const float* phi,
                           const float* dphi, int L, int n_test, double* G, double* b, cudaStream_t s) {
  WlArgs a{};
  a.x = x; a.n_traj = n_traj; a.T = T; a.phi = phi; a.dphi = dphi; a.L = L; a.n_test = n_test; a.G = G; a.b = b;
  const int64_t n_ctas = (n_traj * n_test + kWarps - 1) / kWarps;
  const unsigned grid = (unsigned)(n_ctas < (1ll << 30) ? n_ctas : (1ll << 30));   // the kernels stride over the rest
#define X(D, PC)                                                                \
  if (lib_matches<D, PC>(t)) {                                                  \
    wsindy_local_kernel<D, PC><<<grid, 32 * kWarps, 0, s>>>(a);                 \
    SB_LAUNCH_CHECK("wsindy_local_kernel");                                     \
    return SB_OK;                                                               \
  }
  X(2, 2) X(2, 3) X(3, 2) X(3, 3) X(3, 5)
#undef X
  if (t.K <= 16) wsindy_local_generic_kernel<16><<<grid, 32 * kWarps, 0, s>>>(t, a);
  else if (t.K <= 64) wsindy_local_generic_kernel<64><<<grid, 32 * kWarps, 0, s>>>(t, a);
  else wsindy_local_generic_kernel<256><<<grid, 32 * kWarps, 0, s>>>(t, a);
  SB_LAUNCH_CHECK("wsindy_local_generic_kernel");
  return SB_OK;
}

}  // namespace sb
