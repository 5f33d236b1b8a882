"""ctypes binding of libcpz.so (include/cpz.h). This is the ONLY compute path of the package: there is no CPU
fallback, and every call raises `CpzError` when the library or a B200-class device is missing."""
from __future__ import annotations

import ctypes as C
import os
import weakref
from typing import Optional

import numpy as np

from .desc import CClosureDesc, CClosureUvtDesc, CModelDesc, ClosureDesc, ClosureUvtDesc, ModelDesc

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcpz.so")

EXPORTS = [
    "cpz_version", "cpz_last_error", "cpz_device_count", "cpz_sizeof_model_desc", "cpz_sizeof_closure_desc", "cpz_ctx_create", "cpz_ctx_destroy", "cpz_ctx_set_allreduce",
    "cpz_ctx_synchronize", "cpz_ctx_stream", "cpz_ctx_launch_count", "cpz_ctx_nonfinite_count", "cpz_model_create", "cpz_model_destroy",
    "cpz_model_n_params", "cpz_model_n_saved", "cpz_model_describe", "cpz_set_theta", "cpz_get_theta", "cpz_model_set_time", "cpz_rhs",
    "cpz_rhs_dev", "cpz_rhs_vjp", "cpz_rhs_vjp_dev", "cpz_predict_flux", "cpz_predict_flux_dev", "cpz_solve", "cpz_solve_dev", "cpz_loss_grad", "cpz_loss_grad_dev", "cpz_train_step",
    "cpz_train_step_dev", "cpz_set_mpp_params", "cpz_get_mpp_params", "cpz_loss_grad_mpp", "cpz_loss_grad_mpp_dev", "cpz_adam_get_state", "cpz_adam_set_state", "cpz_closure_step", "cpz_closure_step_dev",
    "cpz_sizeof_closure_uvt_desc", "cpz_closure_step_uvt", "cpz_closure_step_uvt_dev",
]

ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p)


ERR_INVALID, ERR_CUDA, ERR_NONFINITE, ERR_COLLECTIVE = -1, -2, -3, -4


class CpzError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libcpz error {code}: {msg}")
        self.code = code


_lib = None


def lib() -> C.CDLL:
    """Load libcpz.so (built in-tree by __graft_entry__.build()). Fails loudly when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CpzError(-2, f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
                           "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    fp, vp, sz, i32, f32 = C.POINTER(C.c_float), C.c_void_p, C.c_size_t, C.c_int32, C.c_float
    L.cpz_version.restype = C.c_int
    L.cpz_last_error.restype = C.c_char_p
    L.cpz_device_count.argtypes = [C.POINTER(C.c_int)]
    L.cpz_ctx_create.argtypes = [C.c_int, vp, C.POINTER(vp)]
    L.cpz_ctx_destroy.argtypes = [vp]
    L.cpz_ctx_set_allreduce.argtypes = [vp, ALLREDUCE_FN, vp, C.c_int, C.c_int]
    L.cpz_ctx_synchronize.argtypes = [vp]
    L.cpz_ctx_stream.argtypes = [vp, C.POINTER(vp)]
    L.cpz_ctx_launch_count.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.cpz_ctx_nonfinite_count.argtypes = [vp, C.POINTER(C.c_uint64)]
    L.cpz_model_create.argtypes = [vp, C.POINTER(CModelDesc), C.POINTER(vp)]
    L.cpz_model_destroy.argtypes = [vp]
    L.cpz_model_n_params.argtypes = [vp, C.POINTER(sz)]
    L.cpz_model_n_saved.argtypes = [vp, C.POINTER(i32)]
    L.cpz_model_describe.argtypes = [vp, C.c_char_p, sz]
    L.cpz_set_theta.argtypes = [vp, vp, sz]
    L.cpz_get_theta.argtypes = [vp, vp, sz]
    L.cpz_model_set_time.argtypes = [vp, i32, f32, f32, i32, i32, i32, i32]
    for name in ("cpz_rhs", "cpz_rhs_dev", "cpz_predict_flux", "cpz_predict_flux_dev"):
        getattr(L, name).argtypes = [vp, vp, vp, vp, f32, vp, sz]
    for name in ("cpz_rhs_vjp", "cpz_rhs_vjp_dev"):
        getattr(L, name).argtypes = [vp, vp, vp, vp, f32, vp, vp, vp, vp, sz]
    for name in ("cpz_solve", "cpz_solve_dev"):
        getattr(L, name).argtypes = [vp, vp, vp, vp, vp, sz]
    for name in ("cpz_loss_grad", "cpz_loss_grad_dev"):
        getattr(L, name).argtypes = [vp, vp, vp, vp, vp, sz, vp, vp, vp]
    for name in ("cpz_loss_grad_mpp", "cpz_loss_grad_mpp_dev"):
        getattr(L, name).argtypes = [vp, vp, vp, vp, vp, sz, vp, vp, vp, vp]
    L.cpz_set_mpp_params.argtypes = [vp, vp]
    L.cpz_get_mpp_params.argtypes = [vp, vp]
    for name in ("cpz_train_step", "cpz_train_step_dev"):
        getattr(L, name).argtypes = [vp, vp, vp, vp, vp, sz, vp, f32, f32, f32, f32, vp]
    L.cpz_adam_get_state.argtypes = [vp, vp, vp, vp, sz]
    L.cpz_adam_set_state.argtypes = [vp, vp, vp, vp, sz]
    for name in ("cpz_closure_step", "cpz_closure_step_dev"):
        getattr(L, name).argtypes = [vp, C.POINTER(CClosureDesc), vp, vp, vp, vp]
    for name in ("cpz_closure_step_uvt", "cpz_closure_step_uvt_dev"):
        getattr(L, name).argtypes = [vp, C.POINTER(CClosureUvtDesc), vp, vp, vp, vp, vp]
    for name in EXPORTS:
        if name not in ("cpz_last_error", "cpz_sizeof_model_desc", "cpz_sizeof_closure_desc", "cpz_sizeof_closure_uvt_desc"):
            getattr(L, name).restype = C.c_int
    L.cpz_sizeof_model_desc.restype = C.c_size_t
    L.cpz_sizeof_closure_desc.restype = C.c_size_t
    L.cpz_sizeof_closure_uvt_desc.restype = C.c_size_t
    if (L.cpz_sizeof_model_desc() != C.sizeof(CModelDesc) or L.cpz_sizeof_closure_desc() != C.sizeof(CClosureDesc)
            or L.cpz_sizeof_closure_uvt_desc() != C.sizeof(CClosureUvtDesc)):
        raise CpzError(-1, "ABI mismatch between desc.py and libcpz.so (rebuild the library)")
    _lib = L
    return L


def _check(rc: int) -> None:
    if rc != 0:
        raise CpzError(rc, lib().cpz_last_error().decode(errors="replace"))


def device_count() -> int:
    n = C.c_int(0)
    _check(lib().cpz_device_count(C.byref(n)))
    return n.value


def _np(a, shape=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None:
        assert a.shape == tuple(shape), (a.shape, shape)
    return a


def _ptr(a) -> Optional[int]:
    """Host numpy array or torch tensor (host or device) -> raw address; None -> NULL."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
        return a.ctypes.data
    if isinstance(a, int):
        return a
    # torch tensor
    assert a.is_contiguous() and str(a.dtype) == "torch.float32", (a.dtype, a.is_contiguous())
    return a.data_ptr()


class Context:
    """One CUDA device + stream (cpz_ctx). `stream` is a raw cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream)."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self._h = C.c_void_p()
        _check(lib().cpz_ctx_create(device, C.c_void_p(stream) if stream else None, C.byref(self._h)))
        self.device = device
        self._ar_cb = None
        self._models = weakref.WeakSet()  # models must be destroyed before their context

    def set_allreduce(self, fn, rank: int, world_size: int) -> None:
        """fn(dev_ptr:int, n_floats:int, stream:int) -> None must sum the device buffer over all ranks in place."""
        def tramp(user, buf, n, stream):
            try:
                fn(buf, n, stream)
                return 0
            except Exception as e:  # noqa: BLE001 - the error crosses a C boundary as a status code
                import traceback
                traceback.print_exc()
                return 1
        self._ar_cb = ALLREDUCE_FN(tramp)
        _check(lib().cpz_ctx_set_allreduce(self._h, self._ar_cb, None, rank, world_size))

    def synchronize(self) -> None:
        _check(lib().cpz_ctx_synchronize(self._h))

    @property
    def stream(self) -> int:
        s = C.c_void_p()
        _check(lib().cpz_ctx_stream(self._h, C.byref(s)))
        return s.value or 0

    @property
    def launch_count(self) -> int:
        n = C.c_uint64(0)
        _check(lib().cpz_ctx_launch_count(self._h, C.byref(n)))
        return n.value

    @property
    def nonfinite_count(self) -> int:
        """Non-finite values seen so far in final frames / losses (synchronises the stream); see CPZ_ERR_NONFINITE."""
        n = C.c_uint64(0)
        _check(lib().cpz_ctx_nonfinite_count(self._h, C.byref(n)))
        return n.value

    def close(self) -> None:
        if self._h:
            for m in list(self._models):
                m.close()
            lib().cpz_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class Model:
    """cpz_model: one NDE (description + theta + ADAM state) on a Context."""

    def __init__(self, ctx: Context, desc: ModelDesc, theta: Optional[np.ndarray] = None):
        self.ctx = ctx
        self.desc = desc
        self._c = desc.to_c()
        self._h = C.c_void_p()
        _check(lib().cpz_model_create(ctx._h, C.byref(self._c), C.byref(self._h)))
        ctx._models.add(self)
        p = C.c_size_t(0)
        _check(lib().cpz_model_n_params(self._h, C.byref(p)))
        self.P = p.value
        assert self.P == desc.n_params
        if theta is not None:
            self.set_theta(theta)

    # -- parameters
    def set_theta(self, theta) -> None:
        th = _np(theta, (self.P,))
        _check(lib().cpz_set_theta(self._h, _ptr(th), self.P))

    def get_theta(self) -> np.ndarray:
        th = np.empty(self.P, dtype=np.float32)
        _check(lib().cpz_get_theta(self._h, _ptr(th), self.P))
        return th

    def set_time(self, integrator=None, dt=None, t0=None, n_steps=None, n_substeps=None, save_stride=None, ckpt_stride=None):
        from .desc import INTEGRATOR
        d = self.desc
        for k, v in dict(integrator=integrator, dt=dt, t0=t0, n_steps=n_steps, n_substeps=n_substeps,
                         save_stride=save_stride, ckpt_stride=ckpt_stride).items():
            if v is not None:
                setattr(d, k, v)
        _check(lib().cpz_model_set_time(self._h, INTEGRATOR[d.integrator], d.dt, d.t0, d.n_steps, d.n_substeps,
                                        d.save_stride, d.ckpt_stride))

    def describe(self) -> str:
        buf = C.create_string_buffer(8192)
        _check(lib().cpz_model_describe(self._h, buf, 8192))
        return buf.value.decode()

    @property
    def n_saved(self) -> int:
        n = C.c_int32(0)
        _check(lib().cpz_model_n_saved(self._h, C.byref(n)))
        return n.value

    # -- host-pointer flavour (numpy in / numpy out)
    def rhs(self, x, bcs, t: float = 0.0, Q=None) -> np.ndarray:
        x = _np(x)
        ncol = x.shape[0]
        bcs = _np(bcs, (ncol, self.desc.n_bc))
        Q = None if Q is None else _np(Q, (ncol,))
        out = np.empty_like(x)
        _check(lib().cpz_rhs(self._h, _ptr(x), _ptr(bcs), _ptr(Q), float(t), _ptr(out), ncol))
        return out

    def rhs_vjp(self, x, bcs, dxdt_bar, t: float = 0.0, Q=None, want_x: bool = True, want_theta: bool = True,
                want_mpp: bool = False):
        """Pullback of rhs() at x for the cotangent dxdt_bar [ncol, S] — cpz_rhs_vjp. Returns (x_bar [ncol, S],
        theta_bar [P], mpp_bar [5] wrt (nu0, nu_m, dRi, Ric, Pr)); an output that is not wanted is None."""
        x = _np(x)
        ncol = x.shape[0]
        bcs = _np(bcs, (ncol, self.desc.n_bc))
        ybar = _np(dxdt_bar, x.shape)
        Q = None if Q is None else _np(Q, (ncol,))
        xb = np.empty_like(x) if want_x else None
        tb = np.empty(self.P, dtype=np.float32) if want_theta else None
        pb = np.empty(5, dtype=np.float32) if want_mpp else None
        _check(lib().cpz_rhs_vjp(self._h, _ptr(x), _ptr(bcs), _ptr(Q), float(t), _ptr(ybar), _ptr(xb), _ptr(tb), _ptr(pb),
                                 ncol))
        return xb, tb, pb

    def predict_flux(self, x, bcs, t: float = 0.0, Q=None) -> np.ndarray:
        """Total face fluxes [ncol, n_fields, Nz+1] (scaled) of one RHS evaluation — cpz_predict_flux."""
        x = _np(x)
        ncol = x.shape[0]
        bcs = _np(bcs, (ncol, self.desc.n_bc))
        Q = None if Q is None else _np(Q, (ncol,))
        out = np.empty((ncol, self.desc.n_fields, self.desc.Nz + 1), dtype=np.float32)
        _check(lib().cpz_predict_flux(self._h, _ptr(x), _ptr(bcs), _ptr(Q), float(t), _ptr(out), ncol))
        return out

    def solve(self, x0, bcs, Q=None, out: Optional[np.ndarray] = None) -> np.ndarray:
        x0 = _np(x0)
        ncol = x0.shape[0]
        bcs = _np(bcs, (ncol, self.desc.n_bc))
        Q = None if Q is None else _np(Q, (ncol,))
        if out is None:
            out = np.empty((ncol, self.n_saved, self.desc.S), dtype=np.float32)
        _check(lib().cpz_solve(self._h, _ptr(x0), _ptr(bcs), _ptr(Q), _ptr(out), ncol))
        return out

    def loss_grad(self, x0, bcs, targets, loss_w, Q=None, want_grad: bool = True):
        x0 = _np(x0)
        ncol = x0.shape[0]
        bcs = _np(bcs, (ncol, self.desc.n_bc))
        targets = _np(targets, (ncol, self.n_saved, self.desc.S))
        Q = None if Q is None else _np(Q, (ncol,))
        w = _np(loss_w, (6,))
        loss = np.zeros(7, dtype=np.float32)
        grad = np.zeros(self.P, dtype=np.float32) if want_grad else None
        _check(lib().cpz_loss_grad(self._h, _ptr(x0), _ptr(bcs), _ptr(Q), _ptr(targets), ncol, _ptr(w), _ptr(loss),
                                   _ptr(grad)))
        return loss, grad

    def loss_grad_mpp(self, x0, bcs, targets, loss_w, Q=None, want_theta_grad: bool = False):
        """(loss[7], d loss/d(nu0, nu_m, dRi, Ric, Pr) [5], theta gradient or None) — cpz_loss_grad_mpp."""
        x0 = _np(x0)
        ncol = x0.shape[0]
        bcs = _np(bcs, (ncol, self.desc.n_bc))
        targets = _np(targets, (ncol, self.n_saved, self.desc.S))
        Q = None if Q is None else _np(Q, (ncol,))
        w = _np(loss_w, (6,))
        loss = np.zeros(7, dtype=np.float32)
        gp = np.zeros(5, dtype=np.float32)
        gt = np.zeros(self.P, dtype=np.float32) if (want_theta_grad and self.P > 0) else None
        _check(lib().cpz_loss_grad_mpp(self._h, _ptr(x0), _ptr(bcs), _ptr(Q), _ptr(targets), ncol, _ptr(w), _ptr(loss),
                                       _ptr(gt), _ptr(gp)))
        return loss, gp, gt

    def set_mpp_params(self, nu0, nu_m, dRi, Ric, Pr) -> None:
        p = np.array([nu0, nu_m, dRi, Ric, Pr], dtype=np.float32)
        _check(lib().cpz_set_mpp_params(self._h, _ptr(p)))
        d = self.desc
        d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr = (float(v) for v in p)

    def mpp_params(self) -> np.ndarray:
        p = np.zeros(5, dtype=np.float32)
        _check(lib().cpz_get_mpp_params(self._h, _ptr(p)))
        return p

    def train_step(self, x0, bcs, targets, loss_w, lr, beta1=0.9, beta2=0.999, eps=1e-8, Q=None) -> np.ndarray:
        x0 = _np(x0)
        ncol = x0.shape[0]
        bcs = _np(bcs, (ncol, self.desc.n_bc))
        targets = _np(targets, (ncol, self.n_saved, self.desc.S))
        Q = None if Q is None else _np(Q, (ncol,))
        w = _np(loss_w, (6,))
        loss = np.zeros(7, dtype=np.float32)
        _check(lib().cpz_train_step(self._h, _ptr(x0), _ptr(bcs), _ptr(Q), _ptr(targets), ncol, _ptr(w), float(lr),
                                    float(beta1), float(beta2), float(eps), _ptr(loss)))
        return loss

    def adam_state(self):
        mt = np.empty(self.P, dtype=np.float32)
        vt = np.empty(self.P, dtype=np.float32)
        bp = np.empty(2, dtype=np.float32)
        _check(lib().cpz_adam_get_state(self._h, _ptr(mt), _ptr(vt), _ptr(bp), self.P))
        return mt, vt, bp

    def set_adam_state(self, mt, vt, beta_pow) -> None:
        _check(lib().cpz_adam_set_state(self._h, _ptr(_np(mt, (self.P,))), _ptr(_np(vt, (self.P,))),
                                        _ptr(_np(beta_pow, (2,))), self.P))

    def reset_adam_state(self) -> None:
        """Zero moments and uninitialised beta powers: the next train_step starts a fresh Flux.ADAM."""
        z = np.zeros(self.P, dtype=np.float32)
        self.set_adam_state(z, z, np.zeros(2, dtype=np.float32))

    def closure_step(self, cdesc: ClosureDesc, T, y):
        T = _np(T, (cdesc.Nz, cdesc.Ny, cdesc.Nx))
        y = _np(y, (cdesc.Ny,))
        forcing = np.empty_like(T)
        T_out = np.empty_like(T)
        c = cdesc.to_c()
        _check(lib().cpz_closure_step(self._h, C.byref(c), _ptr(T), _ptr(y), _ptr(forcing), _ptr(T_out)))
        return forcing, T_out

    def closure_step_uvt(self, cdesc: ClosureUvtDesc, u, v, T):
        """One host-model step of the embedded u/v/T NDE: (dz_flux [3,Nz,Ny,Nx], uvT' [3,Nz,Ny,Nx]); fields are [Nz,Ny,Nx]."""
        shp = (cdesc.Nz, cdesc.Ny, cdesc.Nx)
        u, v, T = _np(u, shp), _np(v, shp), _np(T, shp)
        dzf = np.empty((3,) + shp, dtype=np.float32)
        out = np.empty((3,) + shp, dtype=np.float32)
        c = cdesc.to_c()
        _check(lib().cpz_closure_step_uvt(self._h, C.byref(c), _ptr(u), _ptr(v), _ptr(T), _ptr(dzf), _ptr(out)))
        return dzf, out

    # -- device-pointer flavour (torch CUDA tensors or raw addresses; enqueued on the context's stream, no sync)
    def rhs_dev(self, x, bcs, out, t: float = 0.0, Q=None, ncol: Optional[int] = None) -> None:
        ncol = ncol if ncol is not None else x.shape[0]
        _check(lib().cpz_rhs_dev(self._h, _ptr(x), _ptr(bcs), _ptr(Q), float(t), _ptr(out), ncol))

    def rhs_vjp_dev(self, x, bcs, dxdt_bar, x_bar=None, theta_bar=None, mpp_bar=None, t: float = 0.0, Q=None,
                    ncol: Optional[int] = None) -> None:
        """cpz_rhs_vjp_dev: the outputs given (x_bar [ncol, S], theta_bar [P], mpp_bar [5]) are overwritten."""
        ncol = ncol if ncol is not None else x.shape[0]
        _check(lib().cpz_rhs_vjp_dev(self._h, _ptr(x), _ptr(bcs), _ptr(Q), float(t), _ptr(dxdt_bar), _ptr(x_bar),
                                     _ptr(theta_bar), _ptr(mpp_bar), ncol))

    def solve_dev(self, x0, bcs, traj, Q=None, ncol: Optional[int] = None) -> None:
        ncol = ncol if ncol is not None else x0.shape[0]
        _check(lib().cpz_solve_dev(self._h, _ptr(x0), _ptr(bcs), _ptr(Q), _ptr(traj), ncol))

    def loss_grad_dev(self, x0, bcs, targets, loss_w, loss_out, grad_out, Q=None, ncol: Optional[int] = None) -> None:
        ncol = ncol if ncol is not None else x0.shape[0]
        w = _np(loss_w, (6,))
        _check(lib().cpz_loss_grad_dev(self._h, _ptr(x0), _ptr(bcs), _ptr(Q), _ptr(targets), ncol, _ptr(w),
                                       _ptr(loss_out), _ptr(grad_out)))

    def train_step_dev(self, x0, bcs, targets, loss_w, lr, beta1=0.9, beta2=0.999, eps=1e-8, Q=None,
                       ncol: Optional[int] = None) -> np.ndarray:
        ncol = ncol if ncol is not None else x0.shape[0]
        w = _np(loss_w, (6,))
        loss = np.zeros(7, dtype=np.float32)
        _check(lib().cpz_train_step_dev(self._h, _ptr(x0), _ptr(bcs), _ptr(Q), _ptr(targets), ncol, _ptr(w), float(lr),
                                        float(beta1), float(beta2), float(eps), _ptr(loss)))
        return loss

    def closure_step_dev(self, cdesc: ClosureDesc, T, y, forcing, T_out) -> None:
        c = cdesc.to_c()
        _check(lib().cpz_closure_step_dev(self._h, C.byref(c), _ptr(T), _ptr(y), _ptr(forcing), _ptr(T_out)))

    def closure_step_uvt_dev(self, cdesc: ClosureUvtDesc, u, v, T, dz_flux, uvT_out) -> None:
        c = cdesc.to_c()
        _check(lib().cpz_closure_step_uvt_dev(self._h, C.byref(c), _ptr(u), _ptr(v), _ptr(T), _ptr(dz_flux), _ptr(uvT_out)))

    def close(self) -> None:
        if self._h:
            lib().cpz_model_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass
