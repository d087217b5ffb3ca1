// sb_api.cu — the extern "C" surface declared in include/sindy_b200.h: argument validation,
// library-table construction and dispatch between the specialised and the generic kernels.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "sb_common.cuh"

namespace sb {

static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return SB_ERR_CUDA;
}

int build_table(const sb_library* lib, LibTab* tab) {
  if (!lib) { set_error("library is NULL"); return SB_ERR_INVALID; }
  const int d = lib->dim, p = lib->poly_order;
  if (d < 1 || d > SB_MAX_DIM) { set_error("dim=%d outside 1..%d", d, SB_MAX_DIM); return SB_ERR_UNSUPPORTED; }
  if (p < 1 || p > SB_MAX_POLY) { set_error("poly_order=%d outside 1..%d", p, SB_MAX_POLY); return SB_ERR_UNSUPPORTED; }
  const int n_poly = n_poly_terms(d, p);
  const int K = n_poly + (lib->include_sine ? d : 0) + (lib->include_exp ? d : 0);
  if (K > SB_MAX_TERMS) { set_error("library has %d columns, max %d", K, SB_MAX_TERMS); return SB_ERR_UNSUPPORTED; }
  memset(tab, 0, sizeof(*tab));
  tab->d = d; tab->K = K; tab->n_poly = n_poly;
  tab->sine = lib->include_sine ? 1 : 0; tab->exp_ = lib->include_exp ? 1 : 0;
  // same recurrence as make_poly_tab (children of parent p are p*x_j for j >= last variable of p)
  int last[SB_MAX_TERMS];
  int k = 0;
  tab->parent[k] = 0; tab->var[k] = 0; last[k] = 0; ++k;
  int prev_begin = k;
  for (int j = 0; j < d; ++j) { tab->parent[k] = 0; tab->var[k] = (unsigned char)j; last[k] = j; ++k; }
  for (int n = 2; n <= p; ++n) {
    const int pb = prev_begin, pe = k;
    prev_begin = k;
    for (int q = pb; q < pe; ++q)
      for (int j = last[q]; j < d; ++j) { tab->parent[k] = (unsigned char)q; tab->var[k] = (unsigned char)j; last[k] = j; ++k; }
  }
  if (k != n_poly) { set_error("internal: enumerated %d polynomial terms, expected %d", k, n_poly); return SB_ERR_INVALID; }
  return SB_OK;
}

static int check_ptr(const void* p, const char* name) {
  if (!p) { set_error("%s is NULL", name); return SB_ERR_INVALID; }
  return SB_OK;
}

}  // namespace sb

using namespace sb;

#define SB_TRY(expr) do { int _s = (expr); if (_s != SB_OK) return _s; } while (0)

extern "C" {

int sb_version(void) { return 100; }

const char* sb_last_error(void) { return g_err; }

unsigned long long sb_kernel_launches(void) { return g_launches.load(std::memory_order_relaxed); }

int sb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int sb_library_size(const sb_library* lib) {
  LibTab t;
  int s = build_table(lib, &t);
  return s == SB_OK ? t.K : s;
}

int sb_library_exponents(const sb_library* lib, int32_t* out) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  SB_TRY(check_ptr(out, "out_host"));
  memset(out, 0, sizeof(int32_t) * (size_t)t.K * t.d);
  for (int k = 1; k < t.n_poly; ++k) {
    for (int j = 0; j < t.d; ++j) out[k * t.d + j] = out[t.parent[k] * t.d + j];
    out[k * t.d + t.var[k]] += 1;
  }
  int k = t.n_poly;
  if (t.sine) for (int j = 0; j < t.d; ++j, ++k) out[k * t.d + j] = -1;
  if (t.exp_) for (int j = 0; j < t.d; ++j, ++k) out[k * t.d + j] = -2;
  return SB_OK;
}

int64_t sb_workspace_bytes(const sb_library* lib) {
  LibTab t;
  int s = build_table(lib, &t);
  if (s != SB_OK) return s;
  int64_t a = generic_workspace_bytes(t), b = fused_workspace_bytes(t), c = moments_workspace_bytes(t);
  if (b > a) a = b;
  if (c > a) a = c;
  const int64_t e = symreg_workspace_bytes(t);
  return e > a ? e : a;
}

int64_t sb_train_step_out_len(const sb_library* lib, uint32_t flags) {
  LibTab t;
  int s = build_table(lib, &t);
  if (s != SB_OK) return s;
  int64_t len = 2;
  if (flags & SB_STEP_GRAD) len += (int64_t)t.d * t.K;
  if (flags & SB_STEP_GRAM) len += (int64_t)t.K * t.K;
  if (flags & SB_STEP_B) len += (int64_t)t.K * t.d;
  return len;
}

int sb_theta(const float* x, int64_t n, const sb_library* lib, float* theta, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0) { set_error("n=%lld < 0", (long long)n); return SB_ERR_INVALID; }
  if (n == 0) return SB_OK;
  SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(theta, "theta"));
  return generic_theta(x, n, t, theta, (cudaStream_t)stream);
}

int sb_forward(const float* x, int64_t n, const sb_library* lib, const float* w, float* y, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0) { set_error("n=%lld < 0", (long long)n); return SB_ERR_INVALID; }
  if (n == 0) return SB_OK;
  SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(w, "w")); SB_TRY(check_ptr(y, "y"));
  if (fused_supported(t, SB_STEP_LOSS | SB_STEP_GRAD)) return fused_forward(x, n, t, w, y, (cudaStream_t)stream);
  return generic_forward(x, n, t, w, y, (cudaStream_t)stream);
}

int sb_jvp(const float* x, const float* u, int64_t n, const sb_library* lib, const float* w, float* out,
           void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0) { set_error("n=%lld < 0", (long long)n); return SB_ERR_INVALID; }
  if (n == 0) return SB_OK;
  SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(u, "u")); SB_TRY(check_ptr(w, "w")); SB_TRY(check_ptr(out, "out"));
  return generic_jvp(x, u, n, t, w, out, (cudaStream_t)stream);
}

int sb_backward(const float* x, const float* gy, int64_t n, const sb_library* lib, const float* w,
                double* gw, float* gx, void* ws, int64_t ws_bytes, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0) { set_error("n=%lld < 0", (long long)n); return SB_ERR_INVALID; }
  if (!gw && !gx) return SB_OK;
  if (n > 0) { SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(gy, "gy")); }
  if (gx) SB_TRY(check_ptr(w, "w"));
  if (gw) SB_TRY(check_ptr(ws, "workspace"));
  const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(gy)) & 15u) == 0;
  if (gw && n > 0 && aligned && fused_supported(t, SB_STEP_LOSS | SB_STEP_GRAD)) {
    // dL/dW through the TMA-staged fused kernel (the cotangent plays the role of dx); gx, if wanted, per sample
    SB_TRY(fused_weighted_sums(x, gy, n, t, gw, ws, ws_bytes, (cudaStream_t)stream));
    if (!gx) return SB_OK;
    return generic_backward(x, gy, n, t, w, nullptr, gx, ws, ws_bytes, (cudaStream_t)stream);
  }
  return generic_backward(x, gy, n, t, w, gw, gx, ws, ws_bytes, (cudaStream_t)stream);
}

int sb_jvp_backward(const float* x, const float* u, const float* g, int64_t n, const sb_library* lib,
                    const float* w, double* gw, float* gx, float* gu, void* ws, int64_t ws_bytes,
                    void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0) { set_error("n=%lld < 0", (long long)n); return SB_ERR_INVALID; }
  if (!gw && !gx && !gu) return SB_OK;
  if (n > 0) { SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(u, "u")); SB_TRY(check_ptr(g, "g")); }
  if (gx || gu) SB_TRY(check_ptr(w, "w"));
  if (gw) SB_TRY(check_ptr(ws, "workspace"));
  return generic_jvp_backward(x, u, g, n, t, w, gw, gx, gu, ws, ws_bytes, (cudaStream_t)stream);
}

static int step_args_ok(const float* x, const float* dx, int64_t n, const float* w, uint32_t flags,
                        double* out, void* ws) {
  if (n < 0) { set_error("n=%lld < 0", (long long)n); return SB_ERR_INVALID; }
  if (flags == 0 || (flags & ~(SB_STEP_LOSS | SB_STEP_GRAD | SB_STEP_GRAM | SB_STEP_B))) {
    set_error("bad flags 0x%x", flags); return SB_ERR_INVALID;
  }
  SB_TRY(check_ptr(out, "out")); SB_TRY(check_ptr(ws, "workspace"));
  if (n > 0) SB_TRY(check_ptr(x, "x"));
  if (n > 0 && (flags & (SB_STEP_LOSS | SB_STEP_GRAD | SB_STEP_B))) SB_TRY(check_ptr(dx, "dx"));
  if (flags & (SB_STEP_LOSS | SB_STEP_GRAD)) SB_TRY(check_ptr(w, "w"));
  return SB_OK;
}

int sb_train_step(const float* x, const float* dx, int64_t n, const sb_library* lib, const float* w,
                  uint32_t flags, double* out, void* ws, int64_t ws_bytes, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  SB_TRY(step_args_ok(x, dx, n, w, flags, out, ws));
  // the TMA-staged kernels need 16-byte aligned, contiguous x / dx
  const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dx)) & 15u) == 0;
  cudaStream_t s = (cudaStream_t)stream;
  const uint32_t rest = flags & ~SB_STEP_GRAM;   // sections served by the fused residual / ΘᵀẊ kernels
  const bool gram = (flags & SB_STEP_GRAM) != 0;
  // The power-sum Gram rounds x^(α_k+α_l) once per sample instead of multiplying the two rounded columns; those
  // rounding errors are unbiased and average out like eps/sqrt(n), but on small ill-conditioned batches they are
  // amplified by cond(ΘᵀΘ). Below this sample count the exact-product generic rows are used (and are fast enough).
  const char* env_min = getenv("SB_MOMENTS_MIN_SAMPLES");
  const int64_t moments_min = env_min ? atoll(env_min) : (int64_t)1 << 20;
  const bool spec = n > 0 && aligned && (!rest || fused_supported(t, rest)) &&
                    (!gram || (moments_supported(t) && n >= moments_min));
  if (!spec) return generic_train_step(x, dx, n, t, w, flags, out, ws, ws_bytes, s);
  if (rest) SB_TRY(fused_train_step(x, dx, n, t, w, nullptr, flags, out, nullptr, nullptr, ws, ws_bytes, s));  // GRAM bit only shifts the ΘᵀẊ offset
  if (gram) {
    double* g_out = out + 2 + ((flags & SB_STEP_GRAD) ? (int64_t)t.d * t.K : 0);
    SB_TRY(moments_gram(x, n, t, g_out, rest ? nullptr : out, ws, ws_bytes, s));
  }
  return SB_OK;
}

int sb_closure(const float* x, const float* dx, int64_t n, const sb_library* lib, const float* xi, const float* mask,
               double w_l1, double* packed_out, float* loss_out, float* grad_out, void* ws, int64_t ws_bytes,
               void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  const uint32_t flags = SB_STEP_LOSS | SB_STEP_GRAD;
  SB_TRY(step_args_ok(x, dx, n, xi, flags, packed_out, ws));
  SB_TRY(check_ptr(loss_out, "loss_out")); SB_TRY(check_ptr(grad_out, "grad_out"));
  cudaStream_t s = (cudaStream_t)stream;
  const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dx)) & 15u) == 0;
  if (n > 0 && aligned && fused_supported(t, flags)) {
    ClosureOut co{w_l1, loss_out, grad_out};
    return fused_train_step(x, dx, n, t, xi, mask, flags, packed_out, &co, nullptr, ws, ws_bytes, s);
  }
  // generic path: W = Ξ⊙mask in the workspace tail, residual rows, then the epilogue launch
  const int64_t need = generic_workspace_bytes(t);
  if (ws_bytes < need) { set_error("workspace too small: %lld < %lld bytes", (long long)ws_bytes, (long long)need); return SB_ERR_WORKSPACE; }
  float* wm = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + need - (int64_t)t.d * t.K * (int64_t)sizeof(float));
  SB_TRY(mask_mul(xi, mask, wm, t.d * t.K, s));
  SB_TRY(generic_train_step(x, dx, n, t, wm, flags, packed_out, ws, ws_bytes, s));
  return step_epilogue(packed_out, t, xi, mask, w_l1, loss_out, grad_out, s);
}

// clock64 ticks a rank waits for its peers: $SB_PEER_TIMEOUT_MS (default 30 s) at the SM clock of the current device.
// Long enough for lazy module loads, graph captures or a checkpoint on another rank; short enough not to wedge the GPU.
static long long peer_timeout_ticks() {
  double ms = 30000.0;
  if (const char* e = getenv("SB_PEER_TIMEOUT_MS")) { const double v = atof(e); if (v > 0.0) ms = v; }
  int dev = 0, khz = 1965000;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev);
  return (long long)(ms * (double)khz);
}

int64_t sb_peer_buffer_bytes(const sb_library* lib, int world) {
  LibTab t;
  int s = build_table(lib, &t);
  if (s != SB_OK) return s;
  if (world < 1 || world > SB_MAX_PEERS) return SB_ERR_INVALID;
  return (int64_t)2 * world * ((int64_t)t.d * t.K + 2) * 16;   // [2 parities][world senders][d*K+2 lines of 16 B]
}

int sb_closure_peer(const float* x, const float* dx, int64_t n, const sb_library* lib, const float* xi,
                    const float* mask, double w_l1, double* packed_out, float* loss_out, float* grad_out, void* ws,
                    int64_t ws_bytes, const void* const* peer_bufs, int world, int rank, uint32_t* epoch_dev,
                    void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  const uint32_t flags = SB_STEP_LOSS | SB_STEP_GRAD;
  SB_TRY(step_args_ok(x, dx, n, xi, flags, packed_out, ws));
  SB_TRY(check_ptr(loss_out, "loss_out")); SB_TRY(check_ptr(grad_out, "grad_out"));
  SB_TRY(check_ptr(peer_bufs, "peer_bufs")); SB_TRY(check_ptr(epoch_dev, "epoch_dev"));
  if (world < 2 || world > SB_MAX_PEERS || rank < 0 || rank >= world) {
    set_error("bad world/rank %d/%d (2..%d ranks)", world, rank, SB_MAX_PEERS); return SB_ERR_INVALID;
  }
  const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dx)) & 15u) == 0;
  if (!aligned || !fused_supported(t, flags)) {
    set_error("sb_closure_peer needs a specialised library and 16-byte aligned inputs"); return SB_ERR_UNSUPPORTED;
  }
  PeerArgs pa;
  pa.world = world; pa.rank = rank; pa.epoch = epoch_dev; pa.status = epoch_dev + 1;
  pa.timeout_ticks = peer_timeout_ticks();
  for (int r = 0; r < world; ++r) {
    if (!peer_bufs[r]) { set_error("peer_bufs[%d] is NULL", r); return SB_ERR_INVALID; }
    pa.buf[r] = reinterpret_cast<double*>(const_cast<void*>(peer_bufs[r]));
  }
  ClosureOut co{w_l1, loss_out, grad_out};
  // n == 0 on a rank is legal (it still takes part in the exchange)
  return fused_train_step(x, dx, n, t, xi, mask, flags, packed_out, &co, &pa, ws, ws_bytes, (cudaStream_t)stream);
}

int sb_fit_step(const float* x, const float* dx, int64_t n, const sb_library* lib, float* xi, const float* mask,
                const sb_fit_options* opt, float* opt_state, double* packed_out, float* loss_out, float* grad_out,
                void* ws, int64_t ws_bytes, const void* const* peer_bufs, int world, int rank, uint32_t* epoch_dev,
                uint32_t call_flags, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  const uint32_t flags = SB_STEP_LOSS | SB_STEP_GRAD;
  SB_TRY(step_args_ok(x, dx, n, xi, flags, packed_out, ws));
  SB_TRY(check_ptr(opt, "opt"));
  if (opt->kind != SB_OPT_SGD && opt->kind != SB_OPT_ADAM) { set_error("unknown optimiser kind %d", opt->kind); return SB_ERR_INVALID; }
  if (opt->kind == SB_OPT_ADAM) SB_TRY(check_ptr(opt_state, "opt_state"));
  if (call_flags & ~SB_FIT_W_RESIDENT) { set_error("bad call_flags 0x%x", call_flags); return SB_ERR_INVALID; }
  const bool aligned = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dx)) & 15u) == 0;
  if (!aligned || !fused_supported(t, flags)) {
    set_error("sb_fit_step needs a specialised library and 16-byte aligned inputs"); return SB_ERR_UNSUPPORTED;
  }
  PeerArgs pa;
  if (world > 1) {
    SB_TRY(check_ptr(peer_bufs, "peer_bufs")); SB_TRY(check_ptr(epoch_dev, "epoch_dev"));
    if (world > SB_MAX_PEERS || rank < 0 || rank >= world) {
      set_error("bad world/rank %d/%d (max %d ranks)", world, rank, SB_MAX_PEERS); return SB_ERR_INVALID;
    }
    pa.world = world; pa.rank = rank; pa.epoch = epoch_dev; pa.status = epoch_dev + 1;
    pa.timeout_ticks = peer_timeout_ticks();
    for (int r = 0; r < world; ++r) {
      if (!peer_bufs[r]) { set_error("peer_bufs[%d] is NULL", r); return SB_ERR_INVALID; }
      pa.buf[r] = reinterpret_cast<double*>(const_cast<void*>(peer_bufs[r]));
    }
  } else if (n == 0) {
    set_error("sb_fit_step: no samples"); return SB_ERR_INVALID;
  }
  ClosureOut co{(double)opt->w_l1, loss_out, grad_out, (double)opt->w_mse};
  FitArgs fa;
  fa.kind = opt->kind; fa.lr = opt->lr; fa.beta1 = opt->beta1; fa.beta2 = opt->beta2; fa.eps = opt->eps;
  fa.xi = xi;
  if (opt->kind == SB_OPT_ADAM) {
    const int dk = t.d * t.K;
    fa.m = opt_state; fa.v = opt_state + dk; fa.step = reinterpret_cast<unsigned int*>(opt_state + 2 * dk);
  }
  fa.w_resident = (call_flags & SB_FIT_W_RESIDENT) != 0;
  if (opt->sym_quad && opt->w_sym != 0.f) {
    if (reinterpret_cast<uintptr_t>(opt->sym_quad) & 15u) { set_error("sym_quad must be 16-byte aligned"); return SB_ERR_INVALID; }
    fa.sym_H = opt->sym_quad; fa.w_sym = (double)opt->w_sym;
  }
  return fused_train_step(x, dx, n, t, xi, mask, flags, packed_out, &co, world > 1 ? &pa : nullptr, ws, ws_bytes,
                          (cudaStream_t)stream, &fa);
}

int sb_load_w(const sb_library* lib, const float* xi, const float* mask, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  SB_TRY(check_ptr(xi, "xi"));
  if (!fused_supported(t, SB_STEP_LOSS | SB_STEP_GRAD)) {
    set_error("sb_load_w: no specialised kernel for this library"); return SB_ERR_UNSUPPORTED;
  }
  return fused_load_w(t, xi, mask, (cudaStream_t)stream);
}

int sb_step_epilogue(const double* packed, const sb_library* lib, const float* xi, const float* mask, double w_l1,
                     float* loss_out, float* grad_out, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  SB_TRY(check_ptr(packed, "packed")); SB_TRY(check_ptr(xi, "xi"));
  if (!loss_out && !grad_out) return SB_OK;
  return step_epilogue(packed, t, xi, mask, w_l1, loss_out, grad_out, (cudaStream_t)stream);
}

const char* sb_train_step_variant(const sb_library* lib, uint32_t flags) {
  LibTab t;
  if (build_table(lib, &t) != SB_OK) return "unsupported";
  const uint32_t rest = flags & ~SB_STEP_GRAM;
  const bool gram = (flags & SB_STEP_GRAM) != 0;
  if ((rest && !fused_supported(t, rest)) || (gram && !moments_supported(t))) return "generic";
  if (!rest) return "moments";
  return fused_variant_name(t, rest);
}

int sb_rollout(const void* x0, int64_t n_ics, const sb_library* lib, const void* w, double dt,
               int64_t n_steps, int64_t stride, int method, int dtype, int record_dx, void* x_out,
               void* dx_out, void* x_last, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n_ics < 0 || n_steps < 0 || stride < 1) {
    set_error("bad rollout sizes n_ics=%lld n_steps=%lld stride=%lld", (long long)n_ics, (long long)n_steps,
              (long long)stride);
    return SB_ERR_INVALID;
  }
  if (method != SB_EULER && method != SB_RK4) { set_error("unknown method %d", method); return SB_ERR_INVALID; }
  if (dtype != SB_F32 && dtype != SB_F64) { set_error("unknown dtype %d", dtype); return SB_ERR_INVALID; }
  if (n_ics == 0) return SB_OK;
  SB_TRY(check_ptr(x0, "x0")); SB_TRY(check_ptr(w, "w"));
  return rollout(x0, n_ics, t, w, dt, n_steps, stride, method, dtype, record_dx, x_out, dx_out, x_last,
                 (cudaStream_t)stream);
}

int sb_rollout_score(const float* x0, int64_t n_ics, const sb_library* lib, const float* w, int n_models, double dt,
                     int64_t steps_per_row, int64_t n_rows, int method, const float* y_obs, float blowup,
                     double* sse, int32_t* valid_rows, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n_ics < 0 || n_models < 1 || steps_per_row < 1 || n_rows < 1 || n_rows > INT32_MAX ||
      steps_per_row > INT64_MAX / n_rows) {
    set_error("bad rollout_score sizes n_ics=%lld n_models=%d steps_per_row=%lld n_rows=%lld", (long long)n_ics,
              n_models, (long long)steps_per_row, (long long)n_rows);
    return SB_ERR_INVALID;
  }
  if (method != SB_EULER && method != SB_RK4) { set_error("unknown method %d", method); return SB_ERR_INVALID; }
  if (!(dt > 0.0)) { set_error("dt=%g is not positive", dt); return SB_ERR_INVALID; }
  SB_TRY(check_ptr(x0, "x0")); SB_TRY(check_ptr(w, "w")); SB_TRY(check_ptr(y_obs, "y_obs"));
  SB_TRY(check_ptr(sse, "sse")); SB_TRY(check_ptr(valid_rows, "valid_rows"));
  if (n_ics == 0) return SB_OK;
  return rollout_score(x0, n_ics, t, w, n_models, dt, steps_per_row, n_rows, method, y_obs, blowup, sse, valid_rows,
                       (cudaStream_t)stream);
}

int sb_wsindy_integrals(const float* x, int64_t n_traj, int64_t T, const sb_library* lib, float dt,
                        double t_max, int n_test, double* G, double* b, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n_traj < 0 || T < 0 || n_test < 1 || n_test > 1024) {
    set_error("bad wsindy sizes n_traj=%lld T=%lld n_test=%d", (long long)n_traj, (long long)T, n_test);
    return SB_ERR_INVALID;
  }
  if (n_traj == 0) return SB_OK;
  SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(G, "G")); SB_TRY(check_ptr(b, "b"));
  return wsindy_integrals(x, n_traj, T, t, dt, t_max, n_test, G, b, (cudaStream_t)stream);
}

int sb_wsindy_local_integrals(const float* x, int64_t n_traj, int64_t T, const sb_library* lib, const float* phi,
                              const float* dphi, int support, int n_test, double* G, double* b, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  // 3 <= L <= T, 1 <= n_test <= T - L + 1 (distinct starts), and j·(T − L) must fit in int64 for every start
  if (n_traj < 0 || support < 3 || T < support || n_test < 1 || n_test > T - support + 1 ||
      (n_test > 1 && T - support > INT64_MAX / (n_test - 1))) {
    set_error("bad wsindy_local sizes n_traj=%lld T=%lld support=%d n_test=%d", (long long)n_traj, (long long)T,
              support, n_test);
    return SB_ERR_INVALID;
  }
  if (n_traj == 0) return SB_OK;
  SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(phi, "phi")); SB_TRY(check_ptr(dphi, "dphi"));
  SB_TRY(check_ptr(G, "G")); SB_TRY(check_ptr(b, "b"));
  return wsindy_local_integrals(x, n_traj, T, t, phi, dphi, support, n_test, G, b, (cudaStream_t)stream);
}

int sb_symreg_supported(const sb_library* lib) {
  LibTab t;
  if (build_table(lib, &t) != SB_OK) return 0;
  return symreg_supported(t) ? 1 : 0;
}

int sb_euler_flow(const float* x, const float* v, int64_t n, const sb_library* lib, const float* w, float dt,
                  int n_steps, float* fx, float* jv, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0 || n_steps < 0) { set_error("bad sizes n=%lld n_steps=%d", (long long)n, n_steps); return SB_ERR_INVALID; }
  if (n == 0) return SB_OK;
  SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(w, "w")); SB_TRY(check_ptr(fx, "fx"));
  if (jv && !v) { set_error("jv requested without v"); return SB_ERR_INVALID; }
  return euler_flow(x, v, n, t, w, dt, n_steps, fx, jv, (cudaStream_t)stream);
}

int sb_euler_flow_backward(const float* x, const float* v, const float* g_fx, const float* g_jv, int64_t n,
                           const sb_library* lib, const float* w, float dt, int n_steps, double* gw, float* gv,
                           float* gx, void* ws, int64_t ws_bytes, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0 || n_steps < 0) { set_error("bad sizes n=%lld n_steps=%d", (long long)n, n_steps); return SB_ERR_INVALID; }
  SB_TRY(check_ptr(w, "w")); SB_TRY(check_ptr(gw, "gw")); SB_TRY(check_ptr(ws, "workspace"));
  if (n > 0) SB_TRY(check_ptr(x, "x"));
  return euler_flow_backward(x, v, g_fx, g_jv, n, t, w, dt, n_steps, gw, gv, gx, ws, ws_bytes, (cudaStream_t)stream);
}

int sb_symreg_r(const float* x, const float* gx, const float* jgx, int64_t n, const sb_library* lib, const float* w,
                double* out, void* ws, int64_t ws_bytes, void* stream) {
  LibTab t;
  SB_TRY(build_table(lib, &t));
  if (n < 0) { set_error("bad size n=%lld", (long long)n); return SB_ERR_INVALID; }
  SB_TRY(check_ptr(w, "w")); SB_TRY(check_ptr(out, "out")); SB_TRY(check_ptr(ws, "workspace"));
  if (n > 0) { SB_TRY(check_ptr(x, "x")); SB_TRY(check_ptr(gx, "gx")); SB_TRY(check_ptr(jgx, "jgx")); }
  return symreg_r(x, gx, jgx, n, t, w, out, ws, ws_bytes, (cudaStream_t)stream);
}

static int check_16(const void* p, const char* name) {
  if (!p) { set_error("%s is NULL", name); return SB_ERR_INVALID; }
  if (reinterpret_cast<uintptr_t>(p) & 15u) { set_error("%s must be 16-byte aligned", name); return SB_ERR_INVALID; }
  return SB_OK;
}

int64_t sb_mlp_panel_bytes(int64_t m, int f) { return (m < 0 || f <= 0) ? 0 : mlp_panel_bytes(m, f); }

int sb_mlp_pack_weights(const float* w, int n, int k, int transpose, void* packed, void* stream) {
  SB_TRY(check_ptr(w, "w")); SB_TRY(check_16(packed, "packed"));
  return mlp_pack_weights(w, n, k, transpose, packed, (cudaStream_t)stream);
}

int sb_mlp_pack_rows(const float* x, int64_t m, int f, void* panel, void* stream) {
  if (m < 0) { set_error("bad size m=%lld", (long long)m); return SB_ERR_INVALID; }
  SB_TRY(check_16(panel, "panel"));
  if (m > 0) SB_TRY(check_16(x, "x"));
  return mlp_pack_rows(x, m, f, panel, (cudaStream_t)stream);
}

int sb_mlp_unpack_rows(const void* panel, int64_t m, int f, float* x, void* stream) {
  if (m < 0) { set_error("bad size m=%lld", (long long)m); return SB_ERR_INVALID; }
  SB_TRY(check_16(panel, "panel"));
  if (m > 0) SB_TRY(check_16(x, "x"));
  return mlp_unpack_rows(panel, m, f, x, (cudaStream_t)stream);
}

int sb_mlp_gemm(const void* a_panel, int64_t m, int k, const void* w_packed, int n, const float* bias,
                const void* mask_panel, int mode, void* c_panel, void* stream) {
  if (m < 0) { set_error("bad size m=%lld", (long long)m); return SB_ERR_INVALID; }
  SB_TRY(check_16(a_panel, "a_panel")); SB_TRY(check_16(w_packed, "w_packed")); SB_TRY(check_16(c_panel, "c_panel"));
  if (bias) SB_TRY(check_16(bias, "bias"));
  if (mask_panel) SB_TRY(check_16(mask_panel, "mask_panel"));
  return mlp_gemm(a_panel, m, k, w_packed, n, bias, mask_panel, mode, c_panel, (cudaStream_t)stream);
}

int64_t sb_mlp_partials_bytes(int64_t m, int n, int out_dim) {
  return (m < 0 || n <= 0 || out_dim <= 0) ? 0 : mlp_partials_bytes(m, n, out_dim);
}

int sb_mlp_gemm_out(const void* a_panel, int64_t m, int k, const void* w_packed, int n, const float* bias,
                    const void* mask_panel, int mode, void* c_panel, const float* w_out, const float* bias_out,
                    int out_dim, void* partials, float* y, void* stream) {
  if (m < 0) { set_error("bad size m=%lld", (long long)m); return SB_ERR_INVALID; }
  SB_TRY(check_16(a_panel, "a_panel")); SB_TRY(check_16(w_packed, "w_packed")); SB_TRY(check_16(w_out, "w_out"));
  if (c_panel) SB_TRY(check_16(c_panel, "c_panel"));
  if (bias) SB_TRY(check_16(bias, "bias"));
  if (mask_panel) SB_TRY(check_16(mask_panel, "mask_panel"));
  if (m > 0) { SB_TRY(check_ptr(partials, "partials")); SB_TRY(check_ptr(y, "y")); }
  return mlp_gemm_out(a_panel, m, k, w_packed, n, bias, mask_panel, mode, c_panel, w_out, bias_out, out_dim, partials, y,
                      (cudaStream_t)stream);
}

int sb_mlp_thin_in(const float* x, int64_t m, int in_dim, const float* w, const float* bias, const void* mask_panel,
                   int f, int mode, void* c_panel, void* stream) {
  if (m < 0) { set_error("bad size m=%lld", (long long)m); return SB_ERR_INVALID; }
  SB_TRY(check_ptr(w, "w")); SB_TRY(check_16(c_panel, "c_panel"));
  if (m > 0) SB_TRY(check_ptr(x, "x"));
  if (mask_panel) SB_TRY(check_16(mask_panel, "mask_panel"));
  return mlp_thin_in(x, m, in_dim, w, bias, mask_panel, f, mode, c_panel, (cudaStream_t)stream);
}

int sb_mlp_thin_out(const void* a_panel, int64_t m, int f, const float* w, const float* bias, int out_dim, float* y,
                    void* stream) {
  if (m < 0) { set_error("bad size m=%lld", (long long)m); return SB_ERR_INVALID; }
  SB_TRY(check_16(a_panel, "a_panel")); SB_TRY(check_ptr(w, "w"));
  if (m > 0) SB_TRY(check_ptr(y, "y"));
  return mlp_thin_out(a_panel, m, f, w, bias, out_dim, y, (cudaStream_t)stream);
}

void sb_debug_trace(void* dev_buf) { fused_set_trace(reinterpret_cast<unsigned long long*>(dev_buf)); }

int sb_fp32_peak(int variant, int iters, double* tflops_host, void* stream) {
  SB_TRY(check_ptr(tflops_host, "tflops_host"));
  if (variant < 0 || variant > 4 || iters < 1) { set_error("bad variant/iters"); return SB_ERR_INVALID; }
  return fp32_peak(variant, iters, tflops_host, (cudaStream_t)stream);
}

}  // extern "C"
