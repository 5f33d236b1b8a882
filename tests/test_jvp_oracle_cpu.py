"""The FP64 reference of the pushforwards (cpz_rhs_jvp, cpz_solve_jvp): torch.func.jvp of the unchanged oracle (oracle/nde.py
rhs and solve). Checked against reverse mode by the dot-product identity <J v, w> = <v, J^T w> on every model the GPU tests
use, and against central differences on a smooth model. Central differences are no oracle on the relu, convective-adjustment
and mPP models (kinks, the CA switch and the steep Richardson-number step put them 1e-1 .. 5 off the tangent at steps of
1e-4 .. 1e-6), hence the duality. No GPU needed."""
import numpy as np
import pytest
import torch

from cpz_b200 import synthetic as syn
from cpz_b200.desc import (FLAG_CA, FLAG_DIURNAL, FLAG_IMPLICIT_DIFFUSION as IMP, FLAG_MPP, FLAG_SMOOTH_RI, FLAG_ZERO_WEIGHTS,
                           RHS_INFER, RHS_TRAIN)
from oracle import nde
from test_rhs_gpu import UVT_CASES


def mpp_allowed(d):
    """Where cpz_loss_grad_mpp (and so an mpp tangent) is accepted."""
    return d.n_fields == 3 and (d.has(FLAG_MPP) or d.variant == RHS_INFER) and not d.has(FLAG_SMOOTH_RI)


def p_of(d, dtype=torch.float64):
    return torch.tensor([float(np.float32(v)) for v in (d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr)], dtype=dtype)


def _tangent_call(fn, d, theta, x, xd, thd, pd, dtype):
    """(primal, tangent) of fn(theta, x, p) by torch.func.jvp; a None tangent is zero. p is the model's mPP constants when
    pd is given, else absent (the constants of the description)."""
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    th, xt = conv(theta), conv(x)
    thd = torch.zeros_like(th) if thd is None else conv(thd)
    xd = torch.zeros_like(xt) if xd is None else conv(xd)
    if pd is None:
        out, tan = torch.func.jvp(lambda a, b: fn(a, b, None), (th, xt), (thd, xd))
    else:
        out, tan = torch.func.jvp(fn, (th, xt, p_of(d, dtype)), (thd, xd, conv(pd)))
    return out.detach().numpy(), tan.detach().numpy()


def oracle_rhs_jvp(d, theta, x, bcs, xd=None, thd=None, pd=None, t=0.0, Q=None, dtype=torch.float64):
    """(f, f_dot) of nde.rhs at x for the tangents (x_dot, theta_dot, mpp_dot)."""
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    b, q = conv(bcs), None if Q is None else conv(Q)
    return _tangent_call(lambda th, x_, p: nde.rhs(d, th, x_, b, t, q, p_mpp=p), d, theta, x, xd, thd, pd, dtype)


def oracle_solve_jvp(d, theta, x0, bcs, xd=None, thd=None, pd=None, Q=None, dtype=torch.float64):
    """(traj, traj_dot) of nde.solve at x0 for the tangents (x0_dot, theta_dot, mpp_dot)."""
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    b, q = conv(bcs), None if Q is None else conv(Q)
    return _tangent_call(lambda th, x_, p: nde.solve(d, th, x_, b, q, mpp=p), d, theta, x0, xd, thd, pd, dtype)


def tangents_of(d, ncol, seed=5, with_p=None):
    """Random tangents (x_dot [ncol, S], theta_dot [P] or None, mpp_dot [5] or None); mpp_dot scaled to each parameter."""
    rng = np.random.default_rng(seed)
    xd = rng.standard_normal((ncol, d.S)).astype(np.float32)
    thd = rng.standard_normal(d.n_params).astype(np.float32) if d.n_params > 0 else None
    with_p = mpp_allowed(d) if with_p is None else with_p
    pd = None
    if with_p:
        pd = (rng.standard_normal(5) * 0.1 * np.abs([d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr])).astype(np.float32)
    return xd, thd, pd


def theta_of(d, scale=1.0):
    return syn.theta_random(d, scale=scale) if d.n_params > 0 else np.zeros(0, dtype=np.float32)


# ---- the models of the GPU tests (test_rhs_jvp_gpu.py, test_solve_jvp_gpu.py), at a few columns
def _uvt(variant, flags, **kw):
    return lambda: syn.wind_mixing_desc(variant=variant, flags=flags, **kw)


def _fc(ca, mpp, implicit=False, **kw):
    def mk():
        d = syn.free_convection_desc(ca=ca, mpp=mpp, **kw)
        if implicit:
            d.flags |= IMP
        return d
    return mk


def _nets(width, acts, variant=RHS_TRAIN, flags=0, **kw):
    def mk():
        d = syn.wind_mixing_desc(variant=variant, flags=flags, net=None, **kw)
        d.nets = [syn.NetDesc([d.S] + list(width) + [d.Nz - 1], list(acts)) for _ in range(3)]
        return d
    return mk


RHS_MODELS = {f"uvt_{v}_{f}": _uvt(v, f) for v, f in UVT_CASES}
RHS_MODELS.update({
    "mish40": _nets([40], ["mish", "identity"]),
    "tanh40": _nets([40], ["tanh", "identity"]),
    "nn_free": _uvt(RHS_TRAIN, FLAG_MPP, net=None),
    "fc": _fc(False, False),
    "fc_ca": _fc(True, False),
    "fc_ca_mpp": _fc(True, True),
    "uvt_Nz16": _uvt(RHS_TRAIN, None, Nz=16),
    "fc_Nz64": _fc(True, False, Nz=64),
    "uvt_implicit": _uvt(RHS_INFER, FLAG_MPP | FLAG_CA | IMP, n_substeps=1),
    "fc_implicit": _fc(True, True, implicit=True, n_substeps=1),
})

SOLVE_MODELS = {
    "tc_mish": _uvt(RHS_TRAIN, None, n_steps=12, save_stride=4, ckpt_stride=4),
    "relu": _nets([50, 20], ["relu", "relu", "identity"], n_steps=12, save_stride=4, ckpt_stride=4),
    "implicit_mpp": _uvt(RHS_INFER, FLAG_MPP | FLAG_ZERO_WEIGHTS | IMP, n_steps=12, save_stride=3, ckpt_stride=4, n_substeps=1),
    "diurnal": _uvt(RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=12, save_stride=4, ckpt_stride=4),
    "final_frame_only": _uvt(RHS_TRAIN, None, n_steps=10, save_stride=0, ckpt_stride=4),
    "infer_mpp_ca": _uvt(RHS_INFER, FLAG_MPP | FLAG_CA, n_steps=12, save_stride=1, ckpt_stride=9),
    "streamed": _nets([128], ["relu", "identity"], variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=8, save_stride=2,
                      ckpt_stride=4),
    "rk4": _uvt(RHS_TRAIN, FLAG_MPP, n_steps=12, save_stride=4, ckpt_stride=4, integrator="rk4"),
    "euler": _uvt(RHS_INFER, FLAG_MPP | FLAG_CA, n_steps=12, save_stride=4, ckpt_stride=4, integrator="euler"),
    "fc_ca": _fc(True, False, n_steps=12, save_stride=4, ckpt_stride=4),
    "fc_ca_mpp": _fc(True, True, n_steps=12, save_stride=4, ckpt_stride=4),
    "fc_implicit": _fc(True, True, implicit=True, n_steps=12, save_stride=4, ckpt_stride=4, n_substeps=1),
    "nn_free": _uvt(RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS, n_steps=12, save_stride=4, ckpt_stride=4, net=None),
}


def _dot_identity(kind, d, ncol, t=0.37, diurnal=False):
    theta = theta_of(d)
    x, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol) if diurnal else None
    xd, thd, pd = tangents_of(d, ncol)
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=torch.float64))
    if kind == "rhs":
        _, jv = oracle_rhs_jvp(d, theta, x, bcs, xd, thd, pd, t=t, Q=Q)
    else:
        _, jv = oracle_solve_jvp(d, theta, x, bcs, xd, thd, pd, Q=Q)
    w = np.random.default_rng(3).standard_normal(jv.shape)
    xt, th = conv(x).requires_grad_(True), conv(theta).requires_grad_(True)
    p = p_of(d).requires_grad_(True) if pd is not None else None
    b, q = conv(bcs), None if Q is None else conv(Q)
    f = nde.rhs(d, th, xt, b, t, q, p_mpp=p) if kind == "rhs" else nde.solve(d, th, xt, b, q, mpp=p)
    leaves = [xt, th] + ([p] if p is not None else [])
    g = torch.autograd.grad(f, leaves, grad_outputs=conv(w), allow_unused=True)
    g = [np.zeros(l.shape) if gi is None else gi.numpy() for gi, l in zip(g, leaves)]
    lhs = float(np.sum(jv * w))
    rhs = float(np.sum(g[0] * xd) + (np.sum(g[1] * thd) if thd is not None else 0.0) + (np.sum(g[2] * pd) if pd is not None else 0.0))
    scale = np.linalg.norm(jv) * np.linalg.norm(w)
    return abs(lhs - rhs) / scale, lhs, rhs


@pytest.mark.parametrize("name", list(RHS_MODELS))
def test_oracle_rhs_jvp_dot_identity(name):
    d = RHS_MODELS[name]()
    e, lhs, rhs = _dot_identity("rhs", d, 3, diurnal=d.has(FLAG_DIURNAL))
    assert e <= 1e-10, (name, e, lhs, rhs)


@pytest.mark.parametrize("name", list(SOLVE_MODELS))
def test_oracle_solve_jvp_dot_identity(name):
    d = SOLVE_MODELS[name]()
    e, lhs, rhs = _dot_identity("solve", d, 2, diurnal=d.has(FLAG_DIURNAL))
    assert e <= 1e-10, (name, e, lhs, rhs)


@pytest.mark.parametrize("kind", ["rhs", "solve"])
def test_oracle_jvp_matches_central_differences_on_a_smooth_model(kind):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=0, Nz=16, n_steps=4, save_stride=2, ckpt_stride=2, n_substeps=2)
    ncol = 3
    theta = syn.theta_random(d, scale=0.3).astype(np.float64)
    x, bcs = syn.columns(d, ncol)
    x, bcs = x.astype(np.float64), bcs.astype(np.float64)
    xd, thd, _ = tangents_of(d, ncol, with_p=False)
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=torch.float64))

    def f(s):
        with torch.no_grad():
            th, xs = conv(theta + s * thd), conv(x + s * xd)
            out = nde.rhs(d, th, xs, conv(bcs), 0.37) if kind == "rhs" else nde.solve(d, th, xs, conv(bcs))
            return out.numpy()

    jv = (oracle_rhs_jvp(d, theta, x, bcs, xd, thd, t=0.37) if kind == "rhs" else oracle_solve_jvp(d, theta, x, bcs, xd, thd))[1]
    eps = 1e-6
    fd = (f(eps) - f(-eps)) / (2 * eps)
    e = np.linalg.norm(jv - fd) / np.linalg.norm(jv)
    assert e <= 1e-6, e
