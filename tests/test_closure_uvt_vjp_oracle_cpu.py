"""The FP64 reference of the u/v/T closure-step pullback (torch.autograd of oracle/nde.py: closure_step_uvt, with the five mPP
parameters as autograd leaves) against central finite differences of the same oracle, without a GPU. The GPU pullback
(cpz_closure_step_uvt_vjp, tests/test_closure_uvt_vjp_gpu.py) is compared with this reference."""
import copy

import numpy as np
import pytest
import torch

from cpz_b200 import synthetic as syn
from cpz_b200.desc import ClosureUvtDesc, RHS_INFER
from oracle import nde

MPP_NAMES = ("nu0", "nu_m", "dRi", "Ric", "Pr")


def _c32_or_tensor(v):
    """nde._c32, but a torch tensor passes through: lets the mPP parameters be autograd leaves of the unchanged oracle."""
    return v if torch.is_tensor(v) else float(np.float32(v))


def oracle_closure_uvt(d, theta, cd, u, v, T, p):
    """nde.closure_step_uvt with the mPP parameters p = (nu0, nu_m, dRi, Ric, Pr) given as tensors (all inputs tensors)."""
    dd = copy.copy(d)
    for i, k in enumerate(MPP_NAMES):
        setattr(dd, k, p[i])
    saved = nde._c32
    nde._c32 = _c32_or_tensor
    try:
        return nde.closure_step_uvt(dd, theta, cd, u, v, T)
    finally:
        nde._c32 = saved


def mpp_of(d, dtype=torch.float64):
    return torch.tensor([float(np.float32(getattr(d, k))) for k in MPP_NAMES], dtype=dtype)


def oracle_closure_uvt_vjp(d, theta, cd, u, v, T, dzf_bar, uvT_bar, dtype=torch.float64):
    """(uvT_bar_in [3,Nz,Ny,Nx], theta_bar [P], mpp_bar [5]) = autograd of the oracle step for the cotangents dzf_bar and
    uvT_bar ([3,Nz,Ny,Nx] each, None = zero)."""
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    xs = [conv(a).requires_grad_(True) for a in (u, v, T)]
    th = conv(theta).requires_grad_(True)
    p = mpp_of(d, dtype).requires_grad_(True)
    dzf, out = oracle_closure_uvt(d, th, cd, *xs, p)
    L = 0.0
    if dzf_bar is not None:
        L = L + (dzf * conv(dzf_bar)).sum()
    if uvT_bar is not None:
        L = L + (out * conv(uvT_bar)).sum()
    g = torch.autograd.grad(L, xs + [th, p], allow_unused=True)
    g = [torch.zeros_like(l) if gi is None else gi for gi, l in zip(g, xs + [th, p])]
    return torch.stack(g[:3]).detach().numpy(), g[3].detach().numpy(), g[4].detach().numpy()


@pytest.mark.parametrize("ca", [False, True])
def test_closure_uvt_vjp_reference_matches_finite_differences(ca):
    """Directional derivatives in u, v, T, theta and p on a 4 x 2 x 32 field: the smooth (mish) production nets and random
    directions keep the differences away from the convective-adjustment switch and from the step's other branches."""
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    theta = syn.theta_random(d, scale=0.5)
    nx, ny = 4, 2
    u, v, T = syn.uvt_fields(d, nx, ny, unstable_every=3 if ca else 0)
    cd = ClosureUvtDesc(Nx=nx, Ny=ny, Nz=32, dz=d.H / 32, dt=60.0, uw_top=-1e-4, vw_top=2e-5, wT_top=3e-5, convective_adjustment=ca)
    rng = np.random.default_rng(11)
    fb = rng.standard_normal((3, 32, ny, nx))
    ob = rng.standard_normal((3, 32, ny, nx))
    xb, tb, pb = oracle_closure_uvt_vjp(d, theta, cd, u, v, T, fb, ob)
    t64 = (lambda a: torch.tensor(np.asarray(a), dtype=torch.float64))
    base = [t64(a) for a in (u, v, T)] + [t64(theta), mpp_of(d)]

    def L(args):
        with torch.no_grad():
            dzf, out = oracle_closure_uvt(d, args[3], cd, args[0], args[1], args[2], args[4])
            return float((dzf * t64(fb)).sum() + (out * t64(ob)).sum())

    grads = [xb[0], xb[1], xb[2], tb, pb]
    for i, name in enumerate(("u", "v", "T", "theta", "p")):
        x = base[i]
        dirn = torch.tensor(rng.standard_normal(x.shape), dtype=torch.float64)
        # the fields move by O(1e-3) (their vertical differences are small: Ri is strongly nonlinear in them); theta and p
        # relative to their size (p spans 1e-4 .. 1)
        dirn = dirn * (1e-3 if name in ("u", "v", "T") else (x.abs() + (1e-3 if name == "theta" else 0.0)))
        h = {"theta": 1e-6, "p": 1e-4}.get(name, 1e-5)
        plus, minus = list(base), list(base)
        plus[i], minus[i] = x + h * dirn, x - h * dirn
        fd = (L(plus) - L(minus)) / (2 * h)
        terms = torch.tensor(grads[i]) * dirn
        ad = float(terms.sum())
        # relative to the sum of the magnitudes of the terms: a directional derivative can cancel far below its terms
        err = abs(fd - ad) / max(float(terms.abs().sum()), 1e-30)
        print(f"closure_uvt vjp reference ca={ca} {name}: autograd {ad:.6e} central difference {fd:.6e} rel err {err:.1e}")
        assert err <= 1e-5, (name, ad, fd)
    assert np.abs(pb).max() > 0 and np.abs(tb).max() > 0
