"""ctypes binding of libsindy_b200.so (C ABI in include/sindy_b200.h).

PyTorch is used only as the owner of device memory and streams: every wrapper takes CUDA tensors, passes raw
device pointers plus the current stream, and returns freshly allocated CUDA tensors. There is no CPU path:
importing this module never needs a GPU, but every compute call raises ``RuntimeError`` if the shared library
is missing or the tensors are not on a CUDA device.
"""
from __future__ import annotations

import ctypes
import math
import os
import threading
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint32, c_void_p
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

_PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG_DIR, "libsindy_b200.so")

SB_STEP_LOSS, SB_STEP_GRAD, SB_STEP_GRAM, SB_STEP_B = 1, 2, 4, 8
SB_F32, SB_F64 = 0, 1
SB_EULER, SB_RK4 = 0, 1
SB_MAX_DIM, SB_MAX_POLY, SB_MAX_TERMS = 8, 5, 256
SB_OPT_NONE, SB_OPT_SGD, SB_OPT_ADAM = 0, 1, 2
SB_FIT_W_RESIDENT = 1


class _CLibrary(ctypes.Structure):
    _fields_ = [("dim", c_int32), ("poly_order", c_int32), ("include_sine", c_int32), ("include_exp", c_int32)]


class _CFitOptions(ctypes.Structure):
    _fields_ = [("kind", c_int32), ("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("eps", c_float),
                ("w_mse", c_float), ("w_l1", c_float), ("w_sym", c_float), ("sym_quad", c_void_p)]


# every symbol include/sindy_b200.h declares: name -> (restype, argtypes)
_SIGNATURES = {
    "sb_version": (c_int, []),
    "sb_last_error": (c_char_p, []),
    "sb_device_count": (c_int, []),
    "sb_kernel_launches": (ctypes.c_ulonglong, []),
    "sb_library_size": (c_int, [POINTER(_CLibrary)]),
    "sb_library_exponents": (c_int, [POINTER(_CLibrary), POINTER(c_int32)]),
    "sb_workspace_bytes": (c_int64, [POINTER(_CLibrary)]),
    "sb_train_step_out_len": (c_int64, [POINTER(_CLibrary), c_uint32]),
    "sb_theta": (c_int, [c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p]),
    "sb_forward": (c_int, [c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p, c_void_p]),
    "sb_backward": (c_int, [c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p, c_void_p,
                            c_void_p, c_int64, c_void_p]),
    "sb_jvp": (c_int, [c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p, c_void_p]),
    "sb_jvp_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "sb_train_step": (c_int, [c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_uint32, c_void_p,
                              c_void_p, c_int64, c_void_p]),
    "sb_closure": (c_int, [c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p, c_double, c_void_p,
                           c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "sb_closure_peer": (c_int, [c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p, c_double, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_int64, POINTER(c_void_p), c_int, c_int, c_void_p,
                                c_void_p]),
    "sb_peer_buffer_bytes": (c_int64, [POINTER(_CLibrary), c_int]),
    "sb_fit_step": (c_int, [c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p,
                            POINTER(_CFitOptions), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                            POINTER(c_void_p), c_int, c_int, c_void_p, c_uint32, c_void_p]),
    "sb_load_w": (c_int, [POINTER(_CLibrary), c_void_p, c_void_p, c_void_p]),
    "sb_step_epilogue": (c_int, [c_void_p, POINTER(_CLibrary), c_void_p, c_void_p, c_double, c_void_p, c_void_p,
                                 c_void_p]),
    "sb_train_step_variant": (c_char_p, [POINTER(_CLibrary), c_uint32]),
    "sb_rollout": (c_int, [c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_double, c_int64, c_int64, c_int,
                           c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sb_rollout_score": (c_int, [c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_int, c_double, c_int64, c_int64,
                                 c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p]),
    "sb_rollout_score_grad_workspace_bytes": (c_int64, [c_int64, POINTER(_CLibrary), c_int, c_int64, c_int64]),
    "sb_rollout_score_grad": (c_int, [c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_int, c_double, c_int64,
                                      c_int64, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                      c_void_p]),
    "sb_rollout_score_ics": (c_int, [c_void_p, c_int, c_int64, POINTER(_CLibrary), c_void_p, c_int, c_double, c_int64,
                                     c_int64, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p]),
    "sb_rollout_score_grad_ics": (c_int, [c_void_p, c_int, c_int64, POINTER(_CLibrary), c_void_p, c_int, c_double,
                                          c_int64, c_int64, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_int64, c_void_p]),
    "sb_rollout_score_gn_workspace_bytes": (c_int64, [c_int64, POINTER(_CLibrary), c_int, c_int, c_int]),
    "sb_rollout_score_gn": (c_int, [c_void_p, c_int, c_int64, POINTER(_CLibrary), c_void_p, c_int, c_void_p, c_int,
                                    c_double, c_int64, c_int64, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "sb_wsindy_integrals": (c_int, [c_void_p, c_int64, c_int64, POINTER(_CLibrary), c_float, c_double, c_int,
                                    c_void_p, c_void_p, c_void_p]),
    "sb_wsindy_local_integrals": (c_int, [c_void_p, c_int64, c_int64, POINTER(_CLibrary), c_void_p, c_void_p, c_int,
                                          c_int, c_void_p, c_void_p, c_void_p]),
    "sb_symreg_supported": (c_int, [POINTER(_CLibrary)]),
    "sb_euler_flow": (c_int, [c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_float, c_int, c_void_p,
                              c_void_p, c_void_p]),
    "sb_euler_flow_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p,
                                       c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "sb_symreg_r": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, POINTER(_CLibrary), c_void_p, c_void_p, c_void_p,
                            c_int64, c_void_p]),
    "sb_mlp_panel_bytes": (c_int64, [c_int64, c_int]),
    "sb_mlp_pack_weights": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "sb_mlp_pack_rows": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "sb_mlp_unpack_rows": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "sb_mlp_thin_in": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p,
                               c_void_p]),
    "sb_mlp_thin_out": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "sb_mlp_gemm": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                            c_void_p]),
    "sb_mlp_partials_bytes": (c_int64, [c_int64, c_int, c_int]),
    "sb_mlp_gemm_out": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "sb_debug_trace": (None, [c_void_p]),
    "sb_fp32_peak": (c_int, [c_int, c_int, POINTER(c_double), c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_lib_lock = threading.Lock()


def load() -> ctypes.CDLL:
    """Load libsindy_b200.so (once). Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} not found: build it with `python __graft_entry__.py` (or `make -C "
                    f"{os.path.join(_PKG_DIR, 'csrc')}`). There is no CPU fallback.")
            lib = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


class SindyB200Error(RuntimeError):
    pass


def _check(status: int, what: str) -> None:
    if status != 0:
        msg = load().sb_last_error().decode("utf-8", "replace")
        raise SindyB200Error(f"{what} failed with status {status}: {msg}")


@dataclass(frozen=True)
class Library:
    """The function library Θ of SINDyRegression(latent_dim, poly_order, include_sine, include_exp)."""
    dim: int
    poly_order: int
    include_sine: bool = False
    include_exp: bool = False

    def c(self) -> _CLibrary:
        return _CLibrary(int(self.dim), int(self.poly_order), int(bool(self.include_sine)), int(bool(self.include_exp)))

    @property
    def K(self) -> int:
        k = load().sb_library_size(ctypes.byref(self.c()))
        if k < 0:
            _check(k, "sb_library_size")
        return k

    def exponents(self) -> torch.Tensor:
        k, d = self.K, self.dim
        buf = (c_int32 * (k * d))()
        _check(load().sb_library_exponents(ctypes.byref(self.c()), buf), "sb_library_exponents")
        return torch.tensor(list(buf), dtype=torch.int32).view(k, d)

    def workspace_bytes(self) -> int:
        b = load().sb_workspace_bytes(ctypes.byref(self.c()))
        if b < 0:
            _check(int(b), "sb_workspace_bytes")
        return int(b)

    def step_out_len(self, flags: int) -> int:
        return int(load().sb_train_step_out_len(ctypes.byref(self.c()), flags))


def device_count() -> int:
    return int(load().sb_device_count())


def kernel_launches() -> int:
    """Kernels launched by libsindy_b200.so in this process so far."""
    return int(load().sb_kernel_launches())


# ---------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------
_workspaces = {}


def _require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(f"sindy_b200: `{name}` is on {t.device}; the B200 path has no CPU fallback")


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    _require_cuda(t, name)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _stream(dev: torch.device) -> int:
    return int(torch.cuda.current_stream(dev).cuda_stream)


def _workspace(lib: Library, dev: torch.device) -> torch.Tensor:
    """Zero-initialised scratch (ticket counter + per-block partials), one per (device, stream, library)."""
    key = (dev.index, _stream(dev), lib)
    ws = _workspaces.get(key)
    if ws is None:
        ws = torch.zeros(lib.workspace_bytes(), dtype=torch.uint8, device=dev)
        _workspaces[key] = ws
    return ws


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _flat(x: torch.Tensor, d: int, name: str) -> torch.Tensor:
    if x.shape[-1] != d:
        raise ValueError(f"`{name}` has last dimension {x.shape[-1]}, library expects {d}")
    return x.reshape(-1, d)


# ---------------------------------------------------------------------------------------------------------
# compute entry points
# ---------------------------------------------------------------------------------------------------------
def theta(x: torch.Tensor, lib: Library) -> torch.Tensor:
    """Θ(x): (..., d) -> (..., K). Debug / parity only."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    out = torch.empty(xf.shape[0], lib.K, dtype=torch.float32, device=xf.device)
    with torch.cuda.device(xf.device):
        _check(load().sb_theta(xf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()), out.data_ptr(),
                               _stream(xf.device)), "sb_theta")
    return out.view(*x.shape[:-1], lib.K)


def forward(x: torch.Tensor, w: torch.Tensor, lib: Library) -> torch.Tensor:
    """h(x) = Θ(x) Wᵀ, W = Ξ⊙mask (d×K)."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    w = _f32c(w, "w")
    out = torch.empty_like(xf)
    with torch.cuda.device(xf.device):
        _check(load().sb_forward(xf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()), w.data_ptr(), out.data_ptr(),
                                 _stream(xf.device)), "sb_forward")
    return out.view(x.shape)


def backward(x: torch.Tensor, gy: torch.Tensor, w: torch.Tensor, lib: Library, need_gw: bool = True,
             need_gx: bool = False) -> Tuple[Optional[torch.Tensor], Optional[torch.Tensor]]:
    """(gw fp64 d×K, gx fp32 like x) for cotangent gy of forward()."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    gf = _flat(_f32c(gy, "gy"), lib.dim, "gy")
    w = _f32c(w, "w")
    dev = xf.device
    gw = torch.empty(lib.dim, lib.K, dtype=torch.float64, device=dev) if need_gw else None
    gx = torch.empty_like(xf) if need_gx else None
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_backward(xf.data_ptr(), gf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()), w.data_ptr(),
                                  _ptr(gw), _ptr(gx), ws.data_ptr(), ws.numel(), _stream(dev)), "sb_backward")
    return gw, (gx.view(x.shape) if gx is not None else None)


def jvp(x: torch.Tensor, u: torch.Tensor, w: torch.Tensor, lib: Library) -> torch.Tensor:
    """J_h(x)·u."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    uf = _flat(_f32c(u, "u"), lib.dim, "u")
    w = _f32c(w, "w")
    out = torch.empty_like(xf)
    with torch.cuda.device(xf.device):
        _check(load().sb_jvp(xf.data_ptr(), uf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()), w.data_ptr(),
                             out.data_ptr(), _stream(xf.device)), "sb_jvp")
    return out.view(x.shape)


def jvp_backward(x: torch.Tensor, u: torch.Tensor, g: torch.Tensor, w: torch.Tensor, lib: Library,
                 need_gw: bool = True, need_gx: bool = True, need_gu: bool = True):
    """Cotangents of jvp() w.r.t. (W [fp64], x, u) for cotangent g."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    uf = _flat(_f32c(u, "u"), lib.dim, "u")
    gf = _flat(_f32c(g, "g"), lib.dim, "g")
    w = _f32c(w, "w")
    dev = xf.device
    gw = torch.empty(lib.dim, lib.K, dtype=torch.float64, device=dev) if need_gw else None
    gx = torch.empty_like(xf) if need_gx else None
    gu = torch.empty_like(xf) if need_gu else None
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_jvp_backward(xf.data_ptr(), uf.data_ptr(), gf.data_ptr(), xf.shape[0],
                                      ctypes.byref(lib.c()), w.data_ptr(), _ptr(gw), _ptr(gx), _ptr(gu),
                                      ws.data_ptr(), ws.numel(), _stream(dev)), "sb_jvp_backward")
    return gw, (gx.view(x.shape) if gx is not None else None), (gu.view(x.shape) if gu is not None else None)


def train_step(x: torch.Tensor, dx: Optional[torch.Tensor], w: Optional[torch.Tensor], lib: Library,
               flags: int = SB_STEP_LOSS | SB_STEP_GRAD, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Fused pass over (x, dx); returns the packed fp64 vector described in include/sindy_b200.h."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    dxf = _flat(_f32c(dx, "dx"), lib.dim, "dx") if dx is not None else None
    if dxf is not None and dxf.shape[0] != xf.shape[0]:
        raise ValueError("x and dx have different numbers of samples")
    wf = _f32c(w, "w") if w is not None else None
    dev = xf.device
    n_out = lib.step_out_len(flags)
    if out is None:
        out = torch.empty(n_out, dtype=torch.float64, device=dev)
    elif out.numel() < n_out or out.dtype != torch.float64 or not out.is_cuda:
        raise ValueError("`out` must be a CUDA float64 tensor with at least step_out_len(flags) elements")
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_train_step(xf.data_ptr(), _ptr(dxf), xf.shape[0], ctypes.byref(lib.c()), _ptr(wf), flags,
                                    out.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)), "sb_train_step")
    return out


def closure(x: torch.Tensor, dx: torch.Tensor, xi: torch.Tensor, mask: Optional[torch.Tensor], lib: Library,
            w_l1: float = 0.0, packed: Optional[torch.Tensor] = None, loss: Optional[torch.Tensor] = None,
            grad: Optional[torch.Tensor] = None):
    """One closure evaluation (`train.py:645-690` without sym-reg): returns (loss fp32 scalar tensor, dL/dΞ fp32
    (d×K), packed fp64 sums). xi is the unmasked parameter matrix. Output tensors may be passed in for reuse
    (CUDA-graph friendly)."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    dxf = _flat(_f32c(dx, "dx"), lib.dim, "dx")
    xi = _f32c(xi, "xi")
    mk = _f32c(mask, "mask") if mask is not None else None
    dev = xf.device
    d, K = lib.dim, lib.K
    if packed is None:
        packed = torch.empty(2 + d * K, dtype=torch.float64, device=dev)
    if loss is None:
        loss = torch.empty((), dtype=torch.float32, device=dev)
    if grad is None:
        grad = torch.empty(d, K, dtype=torch.float32, device=dev)
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_closure(xf.data_ptr(), dxf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()), xi.data_ptr(),
                                 _ptr(mk), float(w_l1), packed.data_ptr(), loss.data_ptr(), grad.data_ptr(),
                                 ws.data_ptr(), ws.numel(), _stream(dev)), "sb_closure")
    return loss, grad, packed


def peer_buffer_bytes(lib: Library, world: int) -> int:
    b = int(load().sb_peer_buffer_bytes(ctypes.byref(lib.c()), int(world)))
    if b < 0:
        _check(b, "sb_peer_buffer_bytes")
    return b


def closure_peer(x: torch.Tensor, dx: torch.Tensor, xi: torch.Tensor, mask: Optional[torch.Tensor], lib: Library,
                 peer_ptrs, rank: int, epoch: torch.Tensor, w_l1: float = 0.0, packed: Optional[torch.Tensor] = None,
                 loss: Optional[torch.Tensor] = None, grad: Optional[torch.Tensor] = None):
    """closure() over samples sharded across GPUs with the all-reduce inside the kernel (peer stores over NVLink).
    peer_ptrs: device pointers of every rank's symmetric buffer (index = rank); epoch: this rank's CUDA uint32
    counter (zero before the first call). Returns the GLOBAL (loss, dL/dΞ, packed sums), identical on all ranks."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    dxf = _flat(_f32c(dx, "dx"), lib.dim, "dx")
    xi = _f32c(xi, "xi")
    mk = _f32c(mask, "mask") if mask is not None else None
    dev = xf.device
    d, K = lib.dim, lib.K
    if packed is None:
        packed = torch.empty(2 + d * K, dtype=torch.float64, device=dev)
    if loss is None:
        loss = torch.empty((), dtype=torch.float32, device=dev)
    if grad is None:
        grad = torch.empty(d, K, dtype=torch.float32, device=dev)
    world = len(peer_ptrs)
    arr = (c_void_p * world)(*[int(p) for p in peer_ptrs])
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_closure_peer(xf.data_ptr(), dxf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()), xi.data_ptr(),
                                      _ptr(mk), float(w_l1), packed.data_ptr(), loss.data_ptr(), grad.data_ptr(),
                                      ws.data_ptr(), ws.numel(), arr, world, int(rank), epoch.data_ptr(),
                                      _stream(dev)), "sb_closure_peer")
    return loss, grad, packed


def fit_state(lib: Library, device) -> torch.Tensor:
    """Zeroed Adam state of sb_fit_step: [m (d×K) | v (d×K) | step counter] as 2·d·K+1 32-bit words."""
    return torch.zeros(2 * lib.dim * lib.K + 1, dtype=torch.float32, device=device)


# The RESIDENT coefficient slot of the one-launch iteration (include/sindy_b200.h): sb_fit_step reads Ξ⊙mask from it and
# its epilogue writes the next one back; the stateless calls (forward, closure, STLSQ passes) use the scratch slot and
# never touch it. Only another FIT on the same device can: every load_w bumps a per-device generation and returns it; a
# stepper compares it with the generation it last saw before each launch / graph replay and re-packs on a mismatch
# (FitStepper._own_slot, train._adam_fused_epochs) — xi and mask live in the stepper's own memory, so that is always
# possible and costs one tiny launch.
_slot_lock = threading.Lock()
_slot_generation = {}   # device index -> counter bumped by every load of the resident slot


def bump_slot_generation(device) -> int:
    idx = torch.device(device).index or 0
    with _slot_lock:
        g = _slot_generation.get(idx, 0) + 1
        _slot_generation[idx] = g
        return g


def slot_generation(device) -> int:
    idx = torch.device(device).index or 0
    with _slot_lock:
        return _slot_generation.get(idx, 0)


def load_w(xi: torch.Tensor, mask: Optional[torch.Tensor], lib: Library) -> int:
    """Ξ⊙mask into the resident slot of the constant bank (makes SB_FIT_W_RESIDENT true). Returns the slot's new
    generation: whoever loaded it last owns it."""
    xi = _f32c(xi, "xi")
    mk = _f32c(mask, "mask") if mask is not None else None
    with torch.cuda.device(xi.device):
        _check(load().sb_load_w(ctypes.byref(lib.c()), xi.data_ptr(), _ptr(mk), _stream(xi.device)), "sb_load_w")
    return bump_slot_generation(xi.device)


def fit_step(x: torch.Tensor, dx: torch.Tensor, xi: torch.Tensor, mask: Optional[torch.Tensor], lib: Library,
             kind: str = "adam", lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, w_mse: float = 1.0,
             w_l1: float = 0.0, state: Optional[torch.Tensor] = None, w_resident: bool = False,
             packed: Optional[torch.Tensor] = None, loss: Optional[torch.Tensor] = None,
             grad: Optional[torch.Tensor] = None, peer_ptrs=None, rank: int = 0,
             epoch: Optional[torch.Tensor] = None, sym_quad: Optional[torch.Tensor] = None, w_sym: float = 0.0):
    """One iteration of the Adam (or SGD) loop `train.py:512-530` in ONE launch: loss and dL/dΞ at the current
    parameters, then `xi` (fp32 CUDA, contiguous) is advanced IN PLACE. Returns (loss, grad, packed). `state`
    = fit_state(lib) for Adam. With peer_ptrs the samples are sharded over the ranks (see closure_peer).
    sym_quad (symreg.quadratic_form) adds w_sym × the linear Lie-derivative regulariser of the data set.
    w_resident=False packs Ξ⊙mask into the resident slot first (and takes the slot over: its generation is bumped)."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    dxf = _flat(_f32c(dx, "dx"), lib.dim, "dx")
    if xf.data_ptr() % 16:       # the TMA-staged kernel needs 16-byte aligned inputs (a view at an odd offset)
        xf = xf.clone()
    if dxf.data_ptr() % 16:
        dxf = dxf.clone()
    _require_cuda(xi, "xi")
    if xi.dtype != torch.float32 or not xi.is_contiguous():
        raise ValueError("`xi` is updated in place: it must be a contiguous float32 CUDA tensor")
    mk = _f32c(mask, "mask") if mask is not None else None
    kinds = {"sgd": SB_OPT_SGD, "adam": SB_OPT_ADAM}
    if kind not in kinds:
        raise ValueError(f"unknown optimiser {kind!r}")
    if kind == "adam" and (state is None or state.numel() < 2 * lib.dim * lib.K + 1 or not state.is_cuda):
        raise ValueError("Adam needs `state` = fit_state(lib, device)")
    dev = xf.device
    d, K = lib.dim, lib.K
    if packed is None:
        packed = torch.empty(2 + d * K, dtype=torch.float64, device=dev)
    if loss is None:
        loss = torch.empty((), dtype=torch.float32, device=dev)
    if grad is None:
        grad = torch.empty(d, K, dtype=torch.float32, device=dev)
    if sym_quad is not None:
        dk = lib.dim * lib.K
        if (not sym_quad.is_cuda or sym_quad.dtype != torch.float32 or not sym_quad.is_contiguous()
                or tuple(sym_quad.shape) != (dk, dk)):
            raise ValueError("`sym_quad` must be a contiguous CUDA float32 (d·K, d·K) matrix (symreg.quadratic_form)")
    opt = _CFitOptions(kinds[kind], float(lr), float(betas[0]), float(betas[1]), float(eps), float(w_mse), float(w_l1),
                       float(w_sym) if sym_quad is not None else 0.0, _ptr(sym_quad))
    world = len(peer_ptrs) if peer_ptrs else 1
    arr = (c_void_p * world)(*[int(p) for p in peer_ptrs]) if world > 1 else None
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_fit_step(xf.data_ptr(), dxf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()), xi.data_ptr(),
                                  _ptr(mk), ctypes.byref(opt), _ptr(state), packed.data_ptr(), loss.data_ptr(),
                                  grad.data_ptr(), ws.data_ptr(), ws.numel(), arr, world, int(rank), _ptr(epoch),
                                  SB_FIT_W_RESIDENT if w_resident else 0, _stream(dev)), "sb_fit_step")
    if not w_resident:
        bump_slot_generation(dev)
    return loss, grad, packed


def step_epilogue(packed: torch.Tensor, xi: torch.Tensor, mask: Optional[torch.Tensor], lib: Library,
                  w_l1: float = 0.0, loss: Optional[torch.Tensor] = None, grad: Optional[torch.Tensor] = None):
    """loss and dL/dΞ from packed sums that were all-reduced over the ranks (one launch)."""
    if not packed.is_cuda or packed.dtype != torch.float64:
        raise RuntimeError("sindy_b200: `packed` must be a CUDA float64 tensor")
    xi = _f32c(xi, "xi")
    mk = _f32c(mask, "mask") if mask is not None else None
    dev = packed.device
    if loss is None:
        loss = torch.empty((), dtype=torch.float32, device=dev)
    if grad is None:
        grad = torch.empty(lib.dim, lib.K, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _check(load().sb_step_epilogue(packed.data_ptr(), ctypes.byref(lib.c()), xi.data_ptr(), _ptr(mk), float(w_l1),
                                       loss.data_ptr(), grad.data_ptr(), _stream(dev)), "sb_step_epilogue")
    return loss, grad


def train_step_variant(lib: Library, flags: int = SB_STEP_LOSS | SB_STEP_GRAD) -> str:
    return load().sb_train_step_variant(ctypes.byref(lib.c()), flags).decode()


def unpack_step(out: torch.Tensor, lib: Library, flags: int) -> dict:
    """Split the packed train-step vector into named views."""
    d, K = lib.dim, lib.K
    res = {"sum_sq": out[0], "n": out[1]}
    off = 2
    if flags & SB_STEP_GRAD:
        res["grad_raw"] = out[off:off + d * K].view(d, K)
        off += d * K
    if flags & SB_STEP_GRAM:
        res["gram"] = out[off:off + K * K].view(K, K)
        off += K * K
    if flags & SB_STEP_B:
        res["b"] = out[off:off + K * d].view(K, d)
    return res


def rollout(x0: torch.Tensor, w: torch.Tensor, lib: Library, dt: float, n_steps: int, stride: int = 1,
            method: str = "rk4", record_dx: bool = False, want_traj: bool = True, want_last: bool = True):
    """Batched fixed-step integration; dtype follows x0 (float32 or float64). See sb_rollout in the header."""
    _require_cuda(x0, "x0")
    if x0.dtype not in (torch.float32, torch.float64):
        x0 = x0.float()
    dtype = SB_F32 if x0.dtype == torch.float32 else SB_F64
    x0f = _flat(x0.contiguous(), lib.dim, "x0")
    w = w.to(device=x0f.device, dtype=x0f.dtype).contiguous()
    meth = {"euler": SB_EULER, "rk4": SB_RK4}.get(method)
    if meth is None:
        raise ValueError("Unrecognized ODEInt method.")
    n_ics, d = x0f.shape
    dev = x0f.device
    if record_dx:
        n_rows = (n_steps + stride - 1) // stride if n_steps > 0 else 0
    else:
        n_rows = n_steps // stride
    x_out = torch.empty(n_rows, n_ics, d, dtype=x0f.dtype, device=dev) if want_traj else None
    dx_out = torch.empty(n_rows, n_ics, d, dtype=x0f.dtype, device=dev) if (want_traj and record_dx) else None
    x_last = torch.empty(n_ics, d, dtype=x0f.dtype, device=dev) if want_last else None
    with torch.cuda.device(dev):
        _check(load().sb_rollout(x0f.data_ptr(), n_ics, ctypes.byref(lib.c()), w.data_ptr(), float(dt),
                                 int(n_steps), int(stride), meth, dtype, int(bool(record_dx)), _ptr(x_out),
                                 _ptr(dx_out), _ptr(x_last), _stream(dev)), "sb_rollout")
    return x_out, dx_out, x_last


def _score_args(x0, W, lib, dt, steps_per_row, y_obs, method, blowup):
    """The argument checks and conversions shared by rollout_score and rollout_score_grad. x0 is (N, d), shared by all
    models, or (M, N, d), one start set per model; returns x0 as (N, d) or (M, N, d) and whether it is per model."""
    x0 = _f32c(x0, "x0")
    per_model = x0.dim() == 3
    x0f = x0 if per_model else _flat(x0, lib.dim, "x0")
    n_ics, d = x0f.shape[-2:]
    dev = x0f.device
    W = _f32c(W, "W")
    if W.dim() == 2:
        W = W.unsqueeze(0)
    if W.dim() != 3 or W.shape[1:] != (d, lib.K):
        raise ValueError(f"W has shape {tuple(W.shape)}, expected (n_models, {d}, {lib.K})")
    if per_model and (d != lib.dim or x0f.shape[0] != W.shape[0]):
        raise ValueError(f"per-model x0 has shape {tuple(x0f.shape)}, expected ({W.shape[0]}, n_ics, {lib.dim})")
    y = _f32c(y_obs, "y_obs")
    if y.dim() != 3 or y.shape[1:] != (n_ics, d) or y.shape[0] < 1:
        raise ValueError(f"y_obs has shape {tuple(y.shape)}, expected (n_rows >= 1, {n_ics}, {d})")
    if W.device != dev or y.device != dev:
        raise ValueError("x0, W and y_obs must be on one device")
    meth = {"euler": SB_EULER, "rk4": SB_RK4}.get(method)
    if meth is None:
        raise ValueError("Unrecognized ODEInt method.")
    if isinstance(steps_per_row, bool) or int(steps_per_row) != steps_per_row or steps_per_row < 1:
        raise ValueError(f"steps_per_row must be a positive integer, got {steps_per_row!r}")
    if not (math.isfinite(dt) and dt > 0):
        raise ValueError(f"dt must be positive, got {dt}")
    if blowup is not None and not blowup > 0:
        raise ValueError(f"blowup must be positive or None, got {blowup}")
    return x0f, per_model, W, y, meth, dev


def rollout_score(x0: torch.Tensor, W: torch.Tensor, lib: Library, dt: float, steps_per_row: int, y_obs: torch.Tensor,
                  method: str = "rk4", blowup: Optional[float] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Every model W[m] (M × d × K, already masked; one d × K model is M = 1) integrated in fp32 from every initial
    condition x0 (N × d, or M × N × d: model m starts from x0[m]) and compared with y_obs (n_rows × N × d: the states
    after steps_per_row, 2·steps_per_row, ... steps). Returns sse (M × N fp64, summed over the rows compared) and
    valid_rows (M × N int32: rows compared before the first non-finite state or |x_j| > blowup; n_rows if none). The
    compared states are bit-identical to rollout(x0[m], W[m], lib, dt, n_rows·steps_per_row, stride=steps_per_row,
    method). See sb_rollout_score_ics."""
    x0f, per_model, W, y, meth, dev = _score_args(x0, W, lib, dt, steps_per_row, y_obs, method, blowup)
    n_ics = x0f.shape[-2]
    n_models = W.shape[0]
    sse = torch.empty(n_models, n_ics, dtype=torch.float64, device=dev)
    valid = torch.empty(n_models, n_ics, dtype=torch.int32, device=dev)
    if n_models == 0 or n_ics == 0:
        return sse, valid
    with torch.cuda.device(dev):
        _check(load().sb_rollout_score_ics(x0f.data_ptr(), int(per_model), n_ics, ctypes.byref(lib.c()), W.data_ptr(),
                                           n_models, float(dt), int(steps_per_row), y.shape[0], meth, y.data_ptr(),
                                           0.0 if blowup is None else float(blowup), sse.data_ptr(), valid.data_ptr(),
                                           _stream(dev)), "sb_rollout_score_ics")
    return sse, valid


def rollout_score_grad(x0: torch.Tensor, W: torch.Tensor, lib: Library, dt: float, steps_per_row: int,
                       y_obs: torch.Tensor, method: str = "rk4", blowup: Optional[float] = None, x0_grad: bool = False,
                       w_grad: bool = True):
    """rollout_score and the gradient of its scores: returns (sse, valid_rows, grad) with sse / valid_rows
    bit-identical to rollout_score's and grad (M × d × K fp64) = ∂/∂W[m] of sse[m].sum(), each pair's SSE over the rows
    it compared (discrete adjoint of the fp32 recurrence). With x0_grad it returns (sse, valid_rows, grad, grad_x0),
    grad_x0 (M × N × d fp64) = ∂sse[m, n]/∂x0 of the pair (x0 shared or per model as in rollout_score); w_grad=False
    then gives grad = None and runs the start-only kernel variant. See sb_rollout_score_grad_ics."""
    if not (w_grad or x0_grad):
        raise ValueError("rollout_score_grad needs w_grad or x0_grad")
    x0f, per_model, W, y, meth, dev = _score_args(x0, W, lib, dt, steps_per_row, y_obs, method, blowup)
    n_ics, d = x0f.shape[-2:]
    n_models = W.shape[0]
    sse = torch.empty(n_models, n_ics, dtype=torch.float64, device=dev)
    valid = torch.empty(n_models, n_ics, dtype=torch.int32, device=dev)
    grad = torch.zeros(n_models, d, lib.K, dtype=torch.float64, device=dev) if w_grad else None
    gx0 = torch.zeros(n_models, n_ics, d, dtype=torch.float64, device=dev) if x0_grad else None
    done = (sse, valid, grad, gx0) if x0_grad else (sse, valid, grad)
    if n_models == 0 or n_ics == 0:
        return done
    sl = load()
    nb = int(sl.sb_rollout_score_grad_workspace_bytes(n_ics, ctypes.byref(lib.c()), n_models, int(steps_per_row),
                                                      y.shape[0]))
    if nb < 0:
        _check(nb, "sb_rollout_score_grad_workspace_bytes")
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _check(sl.sb_rollout_score_grad_ics(x0f.data_ptr(), int(per_model), n_ics, ctypes.byref(lib.c()), W.data_ptr(),
                                            n_models, float(dt), int(steps_per_row), y.shape[0], meth, y.data_ptr(),
                                            0.0 if blowup is None else float(blowup), sse.data_ptr(), valid.data_ptr(),
                                            _ptr(grad), _ptr(gx0), ws.data_ptr(), nb, _stream(dev)),
               "sb_rollout_score_grad_ics")
    return done


# most tangent columns of rollout_score_gn (SB_GN_MAX_COLS): n_params, plus d with x0_blocks
GN_MAX_COLS = 176


def rollout_score_gn(x0: torch.Tensor, W: torch.Tensor, params: torch.Tensor, lib: Library, dt: float,
                     steps_per_row: int, y_obs: torch.Tensor, method: str = "rk4", blowup: Optional[float] = None,
                     x0_blocks: bool = False):
    """rollout_score and the Gauss–Newton information of its scores. params (M × P int, or P for every model): indices
    into the flat d×K W[m] of the coefficients θ, −1 = padding. With J = ∂x_r/∂θ at every compared row of a pair (the
    tangent-linear of the fp32 recurrence that was scored) and E = x_r − y_r, returns a dict of sse / valid_rows
    (bit-identical to rollout_score's), jtj (M × P × P fp64) = Σ_pairs Σ_r JᵀJ and jtr (M × P fp64) = Σ JᵀE; padded
    rows and columns are exact zeros. x0_blocks=True also treats each pair's start as a parameter, J_x = ∂x_r/∂x0, and
    adds jtj_px (M × N × P × d) = Σ_r JᵀJ_x, jtj_xx (M × N × d × d) = Σ_r J_xᵀJ_x and jtr_x (M × N × d) = Σ_r J_xᵀE,
    per pair. P (+ d with x0_blocks) is at most GN_MAX_COLS. See sb_rollout_score_gn."""
    x0f, per_model, W, y, meth, dev = _score_args(x0, W, lib, dt, steps_per_row, y_obs, method, blowup)
    n_ics, d = x0f.shape[-2:]
    n_models = W.shape[0]
    if not isinstance(x0_blocks, bool):
        raise ValueError(f"x0_blocks must be True or False, got {x0_blocks!r}")
    prm = torch.as_tensor(params)
    if prm.is_floating_point() or prm.dtype == torch.bool or prm.is_complex():
        raise ValueError(f"params must be an integer tensor, got {prm.dtype}")
    if prm.dim() == 1:
        prm = prm.unsqueeze(0).expand(n_models, -1)
    if prm.dim() != 2 or prm.shape[0] != n_models or prm.shape[1] < 1:
        raise ValueError(f"params has shape {tuple(prm.shape)}, expected ({n_models}, n_params >= 1)")
    P = prm.shape[1]
    cols = P + (d if x0_blocks else 0)
    if cols > GN_MAX_COLS:
        raise ValueError(f"{P} parameters{' and ' + str(d) + ' start columns' if x0_blocks else ''} exceed the "
                         f"{GN_MAX_COLS} tangent columns of rollout_score_gn")
    if prm.numel() and (int(prm.min()) < -1 or int(prm.max()) >= d * lib.K):
        raise ValueError(f"params must lie in [-1, {d * lib.K}), got [{int(prm.min())}, {int(prm.max())}]")
    prm = prm.to(device=dev, dtype=torch.int32).contiguous()
    f64 = dict(dtype=torch.float64, device=dev)
    out = {"sse": torch.empty(n_models, n_ics, **f64),
           "valid_rows": torch.empty(n_models, n_ics, dtype=torch.int32, device=dev),
           "jtj": torch.zeros(n_models, P, P, **f64), "jtr": torch.zeros(n_models, P, **f64)}
    if x0_blocks:
        out.update(jtj_px=torch.zeros(n_models, n_ics, P, d, **f64), jtj_xx=torch.zeros(n_models, n_ics, d, d, **f64),
                   jtr_x=torch.zeros(n_models, n_ics, d, **f64))
    if n_models == 0 or n_ics == 0:
        return out
    sl = load()
    nb = int(sl.sb_rollout_score_gn_workspace_bytes(n_ics, ctypes.byref(lib.c()), n_models, P, int(x0_blocks)))
    if nb < 0:
        _check(nb, "sb_rollout_score_gn_workspace_bytes")
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _check(sl.sb_rollout_score_gn(x0f.data_ptr(), int(per_model), n_ics, ctypes.byref(lib.c()), W.data_ptr(),
                                      n_models, prm.data_ptr(), P, float(dt), int(steps_per_row), y.shape[0], meth,
                                      y.data_ptr(), 0.0 if blowup is None else float(blowup), out["sse"].data_ptr(),
                                      out["valid_rows"].data_ptr(), out["jtj"].data_ptr(), out["jtr"].data_ptr(),
                                      _ptr(out.get("jtj_px")), _ptr(out.get("jtj_xx")), _ptr(out.get("jtr_x")),
                                      ws.data_ptr(), nb, _stream(dev)), "sb_rollout_score_gn")
    return out


def wsindy_integrals(x: torch.Tensor, lib: Library, dt: float, t_max: float, n_test: int = 50):
    """G (n_traj×n_test×K) and b (n_traj×n_test×d), fp64, for x of shape (n_traj, T, d) or (T, d)."""
    xf = _f32c(x, "x")
    single = xf.dim() == 2
    if single:
        xf = xf.unsqueeze(0)
    n_traj, T, d = xf.shape
    if d != lib.dim:
        raise ValueError(f"x has last dimension {d}, library expects {lib.dim}")
    dev = xf.device
    G = torch.empty(n_traj, n_test, lib.K, dtype=torch.float64, device=dev)
    b = torch.empty(n_traj, n_test, d, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _check(load().sb_wsindy_integrals(xf.data_ptr(), n_traj, T, ctypes.byref(lib.c()), float(dt), float(t_max),
                                          int(n_test), G.data_ptr(), b.data_ptr(), _stream(dev)),
               "sb_wsindy_integrals")
    return (G[0], b[0]) if single else (G, b)


def wsindy_local_integrals(x: torch.Tensor, lib: Library, phi: torch.Tensor, dphi: torch.Tensor, n_test: int):
    """G (n_traj×n_test×K) and b (n_traj×n_test×d), fp64, for x of shape (n_traj, T, d) or (T, d), with the compactly
    supported test functions whose values on their support are phi, dphi (1-D, `support` = len(phi) floats on x's
    device; starts s_j = ⌊j·(T−L)/(n_test−1)⌋). See sb_wsindy_local_integrals in include/sindy_b200.h."""
    xf = _f32c(x, "x")
    ph = _f32c(phi, "phi").reshape(-1)
    dph = _f32c(dphi, "dphi").reshape(-1)
    if ph.numel() != dph.numel():
        raise ValueError(f"phi has {ph.numel()} values, dphi {dph.numel()}")
    if ph.device != xf.device or dph.device != xf.device:
        raise ValueError("phi and dphi must be on the device of x")
    single = xf.dim() == 2
    if single:
        xf = xf.unsqueeze(0)
    n_traj, T, d = xf.shape
    if d != lib.dim:
        raise ValueError(f"x has last dimension {d}, library expects {lib.dim}")
    dev = xf.device
    G = torch.empty(n_traj, n_test, lib.K, dtype=torch.float64, device=dev)
    b = torch.empty(n_traj, n_test, d, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _check(load().sb_wsindy_local_integrals(xf.data_ptr(), n_traj, T, ctypes.byref(lib.c()), ph.data_ptr(),
                                                dph.data_ptr(), ph.numel(), int(n_test), G.data_ptr(), b.data_ptr(),
                                                _stream(dev)), "sb_wsindy_local_integrals")
    return (G[0], b[0]) if single else (G, b)


def symreg_supported(lib: Library) -> bool:
    """True if the fused Euler-flow / reversed-regulariser kernels exist for this library."""
    return bool(load().sb_symreg_supported(ctypes.byref(lib.c())))


# Longest flow euler_flow_backward accepts: the backward kernel keeps every step's state in a fixed per-thread array
# (`kMaxSteps` in csrc/sb_symreg.cu) and returns SB_ERR_UNSUPPORTED beyond it. The forward has no limit.
EULER_FLOW_MAX_STEPS = 32


def euler_flow(x: torch.Tensor, v: Optional[torch.Tensor], w: torch.Tensor, lib: Library, dt: float, n_steps: int):
    """fx = n_steps explicit-Euler steps of h(x) = Θ(x)Wᵀ from x (`model_utils.py:236-240`) and, with v, jv = J_f(x)·v
    (`model_utils.py:55-56`), one launch. Shapes of x are kept; returns (fx, jv or None)."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    vf = _flat(_f32c(v, "v"), lib.dim, "v") if v is not None else None
    wf = _f32c(w, "w")
    fx = torch.empty_like(xf)
    jv = torch.empty_like(xf) if vf is not None else None
    with torch.cuda.device(xf.device):
        _check(load().sb_euler_flow(xf.data_ptr(), _ptr(vf), xf.shape[0], ctypes.byref(lib.c()), wf.data_ptr(),
                                    float(dt), int(n_steps), fx.data_ptr(), _ptr(jv), _stream(xf.device)),
               "sb_euler_flow")
    return fx.view(x.shape), (jv.view(x.shape) if jv is not None else None)


def euler_flow_backward(x, v, g_fx, g_jv, w, lib: Library, dt: float, n_steps: int, need_gv=True, need_gx=False):
    """Reverse sweep of euler_flow: (gw (d×K fp64), gv or None, gx or None) for cotangents g_fx / g_jv (either None)."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    vf = _flat(_f32c(v, "v"), lib.dim, "v") if v is not None else None
    gf = _flat(_f32c(g_fx, "g_fx"), lib.dim, "g_fx") if g_fx is not None else None
    gj = _flat(_f32c(g_jv, "g_jv"), lib.dim, "g_jv") if g_jv is not None else None
    wf = _f32c(w, "w")
    dev = xf.device
    gw = torch.empty(lib.dim, lib.K, dtype=torch.float64, device=dev)
    gv = torch.empty_like(xf) if (need_gv and vf is not None) else None
    gx = torch.empty_like(xf) if need_gx else None
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_euler_flow_backward(xf.data_ptr(), _ptr(vf), _ptr(gf), _ptr(gj), xf.shape[0],
                                             ctypes.byref(lib.c()), wf.data_ptr(), float(dt), int(n_steps),
                                             gw.data_ptr(), _ptr(gv), _ptr(gx), ws.data_ptr(), ws.numel(),
                                             _stream(dev)), "sb_euler_flow_backward")
    return gw, (gv.view(x.shape) if gv is not None else None), (gx.view(x.shape) if gx is not None else None)


def symreg_r(x: torch.Tensor, gx: torch.Tensor, jgx: torch.Tensor, w: torch.Tensor, lib: Library) -> torch.Tensor:
    """Packed fp64 sums of the reversed regulariser for one group element: out[:d·K] = gradient sums (d×K), out[d·K] =
    Σ‖J_g(x)h(x) − h(g(x))‖² (`model_utils.py:126-170`); one streaming launch."""
    xf = _flat(_f32c(x, "x"), lib.dim, "x")
    gf = _flat(_f32c(gx, "gx"), lib.dim, "gx")
    jf = _f32c(jgx, "jgx").reshape(-1, lib.dim, lib.dim)
    if gf.shape[0] != xf.shape[0] or jf.shape[0] != xf.shape[0]:
        raise ValueError("x, gx and jgx must describe the same samples")
    wf = _f32c(w, "w")
    dev = xf.device
    out = torch.empty(lib.dim * lib.K + 1, dtype=torch.float64, device=dev)
    ws = _workspace(lib, dev)
    with torch.cuda.device(dev):
        _check(load().sb_symreg_r(xf.data_ptr(), gf.data_ptr(), jf.data_ptr(), xf.shape[0], ctypes.byref(lib.c()),
                                  wf.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev)),
               "sb_symreg_r")
    return out


def fp32_peak(variant: int = 1, iters: int = 4096, device: Optional[torch.device] = None) -> float:
    """Measured FP32 FMA-pipe peak in TFLOP/s (0 = FFMA, 1 = FFMA2, 2 = FFMA2 with constant operand)."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
    val = c_double(0.0)
    with torch.cuda.device(dev):
        _check(load().sb_fp32_peak(int(variant), int(iters), ctypes.byref(val), _stream(dev)), "sb_fp32_peak")
    return float(val.value)
