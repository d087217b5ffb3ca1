// sb_wsindy.cu — WSINDy weak-form integrals with trigonometric test functions.
//
// Reference: `sindy.py:332-347` builds V[j,t] = dt·sqrt(2/T)·sin((j+1)πt/T) and V'[j,t] as dense (n_test × T)
// fp32 matrices and `sindy.py:361-362` forms G = V·Θ(x), b = −V'·x with two GEMMs. Reading V would cost
// 8·n_test bytes per time sample against 4·d for x, so here the test functions are generated on the fly, in
// fp32 and with the reference's operation order (every intermediate rounded, no FMA contraction), and Θ is
// expanded in registers. blockIdx.x = test function j, blockIdx.y = trajectory: a thread accumulates the K
// entries G[j,:] and the d entries b[j,:] over its time samples; fp64 across threads; one block owns one
// output row, so there is no cross-block reduction and the result is deterministic.
//
// At scale (many trajectories on one uniform grid — SURVEY §8a a10, §8e) the job is a batched contraction
// G_r = V·Θ(x_r), b_r = −V'·x_r with V, V' SHARED by all trajectories r, and the kernel above is the wrong shape: it
// re-expands Θ and re-reads x once per test function (50×) and pays one sincosf per (sample, test function).
// `wsindy_batched_kernel<D,P>` is a register-tiled SIMT GEMM with generated operands instead:
//   * a CTA owns NB trajectories for their whole length and walks the time axis in tiles of 64 samples;
//   * per tile, V and V' (64 samples × 64 test-function slots) are generated ONCE for all NB trajectories into shared
//     memory: one accurately seeded sincosf per (test function, 32-sample segment), then the rotation recurrence
//     (sin,cos)(φ+δ) = (s·cδ + c·sδ, c·cδ − s·sδ) — 4 FMAs per value instead of a sincosf, error <= 32·eps per segment;
//   * x tiles arrive by cp.async one tile ahead; Θ(x) is expanded once per sample (K−1−d multiplications) into shared
//     memory, with x repeated behind it so that b = −V'·x is just more columns;
//   * thread (ty, tx) keeps the 8 test functions 8ty..8ty+7 × one chunk of column pairs of ONE trajectory in registers:
//     every product is a packed FFMA2 of a broadcast pair (V_j, V_j) / (V'_j, V'_j), stored ready in shared memory, with
//     a column pair — 2 LDS.128 + CW2 LDS.64 per 8·CW2 FFMA2;
//   * a thread owns its output entries exclusively: partial sums are flushed into the fp64 outputs every 32 tiles
//     (fp32 accumulation runs over at most 2048 samples), no cross-thread reduction, no atomics, deterministic.
// Algorithmic cost per time sample: (K−1−d) + 2·n_test·(K+d) flop (test functions amortised over the batch) against
// 4·d bytes => FP32-bound by two orders of magnitude (d=2,K=10: 1207 flop / 8 B; d=3,K=56: 5952 flop / 12 B).
#include <cstdlib>

#include "sb_common.cuh"
#include "sb_tma.cuh"

namespace sb {

namespace {

constexpr int kThreads = 256;

struct WsArgs {
  const float* x;   // n_traj × T × d
  int64_t T;
  float dt_f;       // fp32(dt): `self.dt = self.t[1] - self.t[0]`
  float tmax_f;     // fp32(t_max)
  float c1_f;       // fp32(sqrt(2 / t_max))
  int n_test;
  double* G;        // n_traj × n_test × K
  double* b;        // n_traj × n_test × d
};

template <int KMAX>
__global__ void __launch_bounds__(kThreads) wsindy_kernel(LibTab t, WsArgs a) {
  constexpr int NW = kThreads / 32;
  __shared__ float red[NW][KMAX + SB_MAX_DIM];
  const int d = t.d, K = t.K;
  const int j = blockIdx.x;
  const int64_t traj = blockIdx.y;
  const float* xt = a.x + traj * a.T * d;

  float m[KMAX], acc[KMAX], accb[SB_MAX_DIM], xv[SB_MAX_DIM];
  for (int k = 0; k < K; ++k) acc[k] = 0.f;
#pragma unroll
  for (int q = 0; q < SB_MAX_DIM; ++q) accb[q] = 0.f;

  const float pi_f = 3.14159265358979323846f;       // fp32(torch.pi) == fp32(np.pi)
  const float kf = (float)(j + 1);
  const float kpi = __fmul_rn(kf, pi_f);             // k * pi
  // derivative prefactor: ((sqrt(2/T) * k) * pi) / T
  const float dpre = __fdiv_rn(__fmul_rn(__fmul_rn(a.c1_f, kf), pi_f), a.tmax_f);

  for (int64_t ti = threadIdx.x; ti < a.T; ti += kThreads) {
    const float tt = __fmul_rn((float)ti, a.dt_f);                  // torch.arange(n) * dt
    const float arg = __fdiv_rn(__fmul_rn(kpi, tt), a.tmax_f);      // k*pi*t / t_max
    float sn, cs;
    sincosf(arg, &sn, &cs);
    const float v = __fmul_rn(a.dt_f, __fmul_rn(a.c1_f, sn));       // V  = dt * (c1 * sin)
    const float vd = __fmul_rn(a.dt_f, __fmul_rn(dpre, cs));        // V' = dt * (dpre * cos)
#pragma unroll
    for (int q = 0; q < SB_MAX_DIM; ++q)
      if (q < d) xv[q] = __ldg(xt + ti * d + q);
    expand_table(t, xv, m);
    for (int q = 0; q < K; ++q) acc[q] = fmaf(v, m[q], acc[q]);
#pragma unroll
    for (int q = 0; q < SB_MAX_DIM; ++q)
      if (q < d) accb[q] = fmaf(vd, xv[q], accb[q]);
  }

  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int q = 0; q < K; ++q) {
    const float s = warp_sum(acc[q]);
    if (lane == 0) red[wid][q] = s;
  }
#pragma unroll
  for (int q = 0; q < SB_MAX_DIM; ++q) {
    if (q < d) {
      const float s = warp_sum(accb[q]);
      if (lane == 0) red[wid][K + q] = s;
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < K + d; e += kThreads) {
    double s = 0.0;
#pragma unroll
    for (int wq = 0; wq < NW; ++wq) s += (double)red[wq][e];
    if (e < K) a.G[(traj * a.n_test + j) * K + e] = s;
    else a.b[(traj * a.n_test + j) * d + (e - K)] = -s;
  }
}

// ---- batched kernel ---------------------------------------------------------------------------------------------
// Shared-memory row of one (trajectory, sample): [Θ_0 .. Θ_{K-1} | pad to even | x_0 .. x_{d-1} | pad to even | zeros up
// to kChunks·2·CW2]. The x copy at the end makes b = −V'·x just more columns of the same contraction: a column pair
// never mixes a G column (operand V) with a b column (operand V'), so every product is a packed FFMA2 of a broadcast
// pair (V_j, V_j) or (V'_j, V'_j) with a column pair.
template <int D, int P>
struct WbCfg {
  static constexpr int K = Poly<D, P>::K;
  static constexpr int KE = (K + 1) & ~1;                           // Θ columns, padded to even
  static constexpr int DE = (D + 1) & ~1;                           // x columns, padded to even
  static constexpr int kPairs = (KE + DE) / 2;
  static constexpr int kChunks = kPairs <= 8 ? 1 : (kPairs <= 16 ? 2 : 4);   // column chunks per trajectory
  static constexpr int CW2 = (((kPairs + kChunks - 1) / kChunks) + 1) & ~1;  // column pairs per chunk (= per thread), even
  static constexpr int KP = kChunks * CW2 * 2;                      // floats per shared-memory row (multiple of 4)
  static constexpr int kThreads = 128;                              // 8 row groups (ty) × 16 (trajectory, chunk) (tx)
  static constexpr int kRows = 8;                                   // test functions per thread
  static constexpr int NB = 16 / kChunks;                           // trajectories per CTA
  static constexpr int TT = 64;                                     // samples per tile
  static constexpr int MJ = 64;                                     // test-function slots (n_test <= 64)
  static constexpr int kFlush = 32;                                 // tiles between flushes of the fp32 accumulators
  static constexpr int kXTile = NB * TT * D;                        // floats of x per tile (double-buffered, cp.async)
  static constexpr size_t kSmem = (size_t)(2 * TT * MJ + NB * TT * KP + 2 * kXTile) * sizeof(float);
  static constexpr int kMinBlocks = 2;   // shared memory (~96 KB per CTA) allows two CTAs per SM anyway
};

__device__ __forceinline__ void cp_async4(void* dst_smem, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Test-function tiles: value of (sample t, slot j) at float offset ((t·2 + h)·8 + ty)·4 + e with j = 8·ty + 4·h + e, so
// that the 8 row groups of a warp read 128 contiguous bytes per LDS.128 (one wavefront, 4 tx broadcast).
__device__ __forceinline__ int wb_v_index(int t, int j) { return ((t * 2 + ((j >> 2) & 1)) * 8 + (j >> 3)) * 4 + (j & 3); }

// the contraction of one tile for one thread; kLast: this thread's chunk holds the b columns (operand V' from column KE on)
template <int D, int P, bool kLast>
__device__ __forceinline__ void wb_contract(const float* __restrict__ th, const float4* __restrict__ vs,
                                            const float4* __restrict__ vd,
                                            float2 (&acc)[WbCfg<D, P>::kRows][WbCfg<D, P>::CW2]) {
  using C = WbCfg<D, P>;
#pragma unroll 2
  for (int t = 0; t < C::TT; ++t) {
    float2 th2[C::CW2];
    static_for<0, C::CW2 / 2>([&](auto c) {
      const float4 q = *reinterpret_cast<const float4*>(th + t * C::KP + 4 * c);
      th2[2 * c] = make_float2(q.x, q.y);
      th2[2 * c + 1] = make_float2(q.z, q.w);
    });
    const float4 va = vs[(t * 2 + 0) * 8], vb = vs[(t * 2 + 1) * 8];
    const float v[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
    float dv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if constexpr (kLast) {
      const float4 da = vd[(t * 2 + 0) * 8], db = vd[(t * 2 + 1) * 8];
      dv[0] = da.x; dv[1] = da.y; dv[2] = da.z; dv[3] = da.w; dv[4] = db.x; dv[5] = db.y; dv[6] = db.z; dv[7] = db.w;
    }
    static_for<0, C::kRows>([&](auto rc) {
      constexpr int r = rc;
      const float2 v2 = make_float2(v[r], v[r]);
      static_for<0, C::CW2>([&](auto cc) {
        constexpr int c = cc;
        constexpr bool is_b = kLast && ((C::kChunks - 1) * C::CW2 * 2 + 2 * c >= C::KE);
        if constexpr (is_b) acc[r][c] = __ffma2_rn(make_float2(dv[r], dv[r]), th2[c], acc[r][c]);
        else acc[r][c] = __ffma2_rn(v2, th2[c], acc[r][c]);
      });
    });
  }
}

template <int D, int P>
__global__ void __launch_bounds__(WbCfg<D, P>::kThreads, WbCfg<D, P>::kMinBlocks)
wsindy_batched_kernel(WsArgs a, int64_t n_traj) {
  using C = WbCfg<D, P>;
  extern __shared__ __align__(16) float wsm[];
  float* Vs = wsm;                                 // [TT][2][8][4]
  float* Vd = Vs + C::TT * C::MJ;
  float* Th = Vd + C::TT * C::MJ;                  // [NB][TT][KP]
  float* Xs = Th + C::NB * C::TT * C::KP;          // [2][NB][TT][D]
  const int tid = threadIdx.x;
  const int ty = tid & 7, tx = tid >> 3;           // a warp = 8 ty × 4 consecutive tx
  const int chunk = tx / C::NB, tr = tx % C::NB;   // NB ∈ {16, 8, 4}: the chunk is warp-uniform
  const int64_t traj0 = (int64_t)blockIdx.x * C::NB;
  const int64_t my_traj = traj0 + tr;
  const bool live = my_traj < n_traj;

  // generator role: test function gj, segment gs of 32 samples inside every tile
  const int gj = tid & 63, gs = tid >> 6;
  const float pi_f = 3.14159265358979323846f;
  const float kf = (float)(gj + 1);
  const float kpi = __fmul_rn(kf, pi_f);
  const float dpre = __fdiv_rn(__fmul_rn(__fmul_rn(a.c1_f, kf), pi_f), a.tmax_f);
  float cdel, sdel;                                 // rotation by one time step, from the exact phase increment
  {
    double sd, cd;
    sincos((double)(gj + 1) * 3.14159265358979323846 * (double)a.dt_f / (double)a.tmax_f, &sd, &cd);
    cdel = (float)cd; sdel = (float)sd;
  }

  float2 acc[C::kRows][C::CW2];
  static_for<0, C::kRows>([&](auto r) { static_for<0, C::CW2>([&](auto c) { acc[r][c] = make_float2(0.f, 0.f); }); });
  bool first_flush = true;

  // A thread owns its output entries: partial sums go straight into the fp64 outputs (read-modify-write, no atomics).
  // The accumulators are parked in the (idle) Θ tile first and walked by a rolled loop: updating 8·CW2·2 doubles
  // straight from registers makes ptxas keep all the loads in flight at once and costs the kernel ~100 registers.
  static_assert((size_t)C::kThreads * C::kRows * C::CW2 * 2 <= (size_t)C::NB * C::TT * C::KP, "Θ tile too small to park in");
  auto flush = [&]() {
    float2* park = reinterpret_cast<float2*>(Th);
    static_for<0, C::kRows>([&](auto rc) {
      static_for<0, C::CW2>([&](auto cc) {
        park[(rc * C::CW2 + cc) * C::kThreads + tid] = acc[rc][cc];
        acc[rc][cc] = make_float2(0.f, 0.f);
      });
    });
    if (live) {
#pragma unroll 8
      for (int e = 0; e < C::kRows * C::CW2; ++e) {
        const int r = e / C::CW2, c2 = e % C::CW2;
        const int j = C::kRows * ty + r;
        if (j >= a.n_test) continue;
        const float2 v = park[e * C::kThreads + tid];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int col = chunk * 2 * C::CW2 + 2 * c2 + h;            // column of the shared-memory row
          const double val = (double)(h ? v.y : v.x);
          if (col < C::K) {
            double* g = a.G + ((int64_t)my_traj * a.n_test + j) * C::K + col;
            *g = (first_flush ? 0.0 : *g) + val;
          } else if (col >= C::KE && col < C::KE + D) {
            double* bb = a.b + ((int64_t)my_traj * a.n_test + j) * D + (col - C::KE);
            *bb = (first_flush ? 0.0 : *bb) - val;
          }
        }
      }
    }
    first_flush = false;
    __syncthreads();   // the parked values are consumed before the next tile's expansion overwrites the Θ tile
  };

  const int64_t n_tiles = (a.T + C::TT - 1) / C::TT;
  // x of tile `tile` -> buffer `buf` with 4-byte asynchronous copies (no registers held across the contraction):
  // element e of the tile = (trajectory e / (TT·D), offset e % (TT·D) inside the trajectory's contiguous tile)
  auto prefetch_x = [&](int64_t tile, int buf) {
    const int64_t t0 = tile * C::TT;
    float* dst = Xs + (size_t)buf * C::kXTile;
    const int valid = (int)((a.T - t0 < C::TT ? a.T - t0 : C::TT) * D);   // floats of a trajectory's tile inside [0, T)
#pragma unroll 4
    for (int e = tid; e < C::kXTile; e += C::kThreads) {
      const int er = e / (C::TT * D), rest = e % (C::TT * D);
      if (traj0 + er < n_traj && rest < valid) cp_async4(dst + e, a.x + ((traj0 + er) * a.T + t0) * D + rest);
      else dst[e] = 0.f;
    }
    cp_async_commit();
  };
  prefetch_x(0, 0);

  for (int64_t tile = 0; tile < n_tiles; ++tile) {
    const int64_t t0 = tile * C::TT;
    const int buf = (int)(tile & 1);
    // ---- generate V, V' for the tile: 64 slots × 2 segments of 32 samples ----
    {
      const int64_t ts = t0 + 32 * gs;
      float sn = 0.f, cs = 0.f;
      if (gj < a.n_test) {
        const float tt = __fmul_rn((float)ts, a.dt_f);                 // the reference's rounding order for the seed
        sincosf(__fdiv_rn(__fmul_rn(kpi, tt), a.tmax_f), &sn, &cs);
      }
#pragma unroll 8
      for (int q = 0; q < 32; ++q) {
        const bool in = (gj < a.n_test) && (ts + q < a.T);
        const int o = wb_v_index(32 * gs + q, gj);
        Vs[o] = in ? __fmul_rn(a.dt_f, __fmul_rn(a.c1_f, sn)) : 0.f;
        Vd[o] = in ? __fmul_rn(a.dt_f, __fmul_rn(dpre, cs)) : 0.f;
        const float s2 = fmaf(sn, cdel, cs * sdel);
        cs = fmaf(cs, cdel, -sn * sdel);
        sn = s2;
      }
    }
    // ---- x of this tile has landed; start fetching the next one; expand Θ(x) for NB trajectories × TT samples ----
    cp_async_wait_all();
    __syncthreads();
    if (tile + 1 < n_tiles) prefetch_x(tile + 1, buf ^ 1);
    {
      const float* xsrc = Xs + (size_t)buf * C::kXTile;
#pragma unroll 1
      for (int row = tid; row < C::NB * C::TT; row += C::kThreads) {
        float xs[D], m[C::K];
        static_for<0, D>([&](auto q) { xs[q] = xsrc[row * D + q]; });
        expand_poly<D, P>(xs, m);
        float4* dst = reinterpret_cast<float4*>(Th + (size_t)row * C::KP);
        static_for<0, C::KP / 4>([&](auto qc) {       // 16-byte stores: 8 consecutive rows hit 8 distinct bank groups
          constexpr int q4 = qc;
          float v[4];
          static_for<0, 4>([&](auto ec) {
            constexpr int c = 4 * q4 + ec;
            if constexpr (c < C::K) v[ec] = m[c];
            else if constexpr (c >= C::KE && c < C::KE + D) v[ec] = xs[c - C::KE];
            else v[ec] = 0.f;
          });
          dst[q4] = make_float4(v[0], v[1], v[2], v[3]);
        });
      }
    }
    __syncthreads();
    // ---- contract: 8 test functions × CW2 column pairs of one trajectory per thread ----
    {
      const float* th = Th + (size_t)tr * C::TT * C::KP + chunk * C::CW2 * 2;
      const float4* vs4 = reinterpret_cast<const float4*>(Vs) + ty;
      const float4* vd4 = reinterpret_cast<const float4*>(Vd) + ty;
      if (chunk == C::kChunks - 1) wb_contract<D, P, true>(th, vs4, vd4, acc);
      else wb_contract<D, P, false>(th, vs4, vd4, acc);
    }
    __syncthreads();
    if ((tile + 1) % C::kFlush == 0 || tile + 1 == n_tiles) flush();   // the only call site: the lambda is inlined
  }
}

template <int D, int P>
int launch_batched(const WsArgs& a, int64_t n_traj, cudaStream_t s) {
  using C = WbCfg<D, P>;
  static_assert((C::kChunks - 1) * C::CW2 * 2 <= C::KE, "the b columns must sit in the last chunk");
  static_assert(C::KP >= C::KE + C::DE, "row too short");
  auto kern = wsindy_batched_kernel<D, P>;
  static bool attr_set[64] = {false};
  int dev = 0;
  SB_CUDA_TRY(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    SB_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::kSmem));
    attr_set[dev] = true;
  }
  const int64_t grid = (n_traj + C::NB - 1) / C::NB;
  kern<<<(unsigned)grid, C::kThreads, C::kSmem, s>>>(a, n_traj);
  SB_LAUNCH_CHECK("wsindy_batched_kernel");
  return SB_OK;
}

}  // namespace

// Trajectory batches from this size on take the batched kernel (below it the per-test-function kernel has more blocks)
constexpr int64_t kBatchedMinTraj = 8;

int wsindy_integrals(const float* x, int64_t n_traj, int64_t T, const LibTab& t, float dt, double t_max,
                     int n_test, double* G, double* b, cudaStream_t s) {
  WsArgs a{};
  a.x = x; a.T = T; a.dt_f = dt; a.tmax_f = (float)t_max; a.c1_f = (float)sqrt(2.0 / t_max);
  a.n_test = n_test; a.G = G; a.b = b;
  const bool poly = !t.sine && !t.exp_;
  // batches take the tensor-core kernel (sb_wsindy_tc.cu: 1.25-2.2x the CUDA-core batched kernel below, measured);
  // SB_WSINDY_TC=0 selects the CUDA-core kernel (A/B, and the more accurate of the two: 1e-6 against 1.5e-5 on G)
  // Which kernel: a batched kernel (tensor-core or CUDA-core) needs a full wave of CTAs whatever the batch size — 0.8-1.2
  // ms at T = 8000 — while the per-(test function, trajectory) kernel costs 3.6 / 4.9 / 9.1 / 29 us per trajectory at
  // K = 6 / 10 / 20 / 56 (tools/time_wsindy_small.py): below ≈ min(200, 1700/K) trajectories the simple kernel wins (8
  // trajectories at K = 10: 0.06 against 0.78 ms). SB_WSINDY_TC overrides: 1 = tensor-core kernel from 8 trajectories on,
  // 0 = CUDA-core batched kernel, s = per-test-function kernel.
  const char* e = getenv("SB_WSINDY_TC");
  const bool force_simple = e && e[0] == 's';
  const bool force_batched = e && (e[0] == '0' || e[0] == '1');
  int64_t batched_min = 1700 / (t.K > 0 ? t.K : 1);
  if (batched_min > 200) batched_min = 200;
  if (batched_min < kBatchedMinTraj || force_batched) batched_min = kBatchedMinTraj;
  if (!force_simple) {
    if (!(e && e[0] == '0') && T > 0 && n_traj >= batched_min && wsindy_tc_supported(t, n_test))
      return wsindy_integrals_tc(x, n_traj, T, t, dt, t_max, n_test, G, b, s);
  }
  if (!force_simple && poly && T > 0 && n_test <= 64 && n_traj >= batched_min && n_traj <= (int64_t)0x7fffffff * 4) {
#define X(D, P) if (t.d == D && t.n_poly == n_poly_terms(D, P)) return launch_batched<D, P>(a, n_traj, s);
    X(2, 2) X(2, 3) X(3, 2) X(3, 3) X(3, 5)
#undef X
  }
  // per-(test function, trajectory) blocks; gridDim.y is capped at 65535: walk the batch in slices
  for (int64_t r0 = 0; r0 < n_traj; r0 += 65535) {
    const int64_t nr = n_traj - r0 < 65535 ? n_traj - r0 : 65535;
    WsArgs q = a;
    q.x = x + r0 * T * t.d;
    q.G = G + r0 * n_test * t.K;
    q.b = b + r0 * n_test * t.d;
    dim3 grid((unsigned)n_test, (unsigned)nr);
    if (t.K <= 16) wsindy_kernel<16><<<grid, kThreads, 0, s>>>(t, q);
    else if (t.K <= 64) wsindy_kernel<64><<<grid, kThreads, 0, s>>>(t, q);
    else wsindy_kernel<256><<<grid, kThreads, 0, s>>>(t, q);
    SB_LAUNCH_CHECK("wsindy_kernel");
  }
  return SB_OK;
}

}  // namespace sb
