"""The FP64 reference of the gyre closure-step pullback (torch.autograd of the unchanged oracle/nde.py: closure_step) against
central finite differences of the same oracle, without a GPU. The GPU pullback (cpz_closure_step_vjp,
tests/test_closure_vjp_gpu.py) is compared with this reference."""
import numpy as np
import pytest
import torch

from cpz_b200 import synthetic as syn
from cpz_b200.desc import ClosureDesc
from oracle import nde


def gyre_inputs(nx, ny, seed=4000):
    """syn.gyre_field with every third column turned upside down (statically unstable), so that the adjustment acts."""
    T, y = syn.gyre_field(nx, ny, 32, seed=seed)
    T[:, :, ::3] = T[::-1, :, ::3]
    return np.ascontiguousarray(T), y


def oracle_closure_vjp(d, theta, cd, T, y, forcing_bar, T_out_bar, dtype=torch.float64):
    """(T_bar [Nz,Ny,Nx], theta_bar [P]) = autograd of the oracle step for the cotangents forcing_bar and T_out_bar
    ([Nz,Ny,Nx] each, None = zero)."""
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    Tt = conv(T).requires_grad_(True)
    th = conv(theta).requires_grad_(True)
    forcing, T_out = nde.closure_step(d, th, cd, Tt, conv(y))
    L = 0.0
    if forcing_bar is not None:
        L = L + (forcing * conv(forcing_bar)).sum()
    if T_out_bar is not None:
        L = L + (T_out * conv(T_out_bar)).sum()
    g = torch.autograd.grad(L, [Tt, th], allow_unused=True)
    g = [torch.zeros_like(l) if gi is None else gi for gi, l in zip(g, [Tt, th])]
    return g[0].detach().numpy(), g[1].detach().numpy()


@pytest.mark.parametrize("which", ["forcing_bar", "T_out_bar"])
def test_closure_vjp_reference_matches_finite_differences(which):
    """Directional derivatives in T and theta on a 4 x 2 x 32 gyre field with a third of the columns inverted. The smooth
    (mish) net and random directions of size 1e-6 keep the differences away from the convective-adjustment switch. Each
    cotangent is checked on its own: the forcing path's part of T_bar is some 1e-7 of the T' path's (the forcing is O(1e-6)),
    so with both given a difference quotient could not see it."""
    from cpz_b200.desc import NetDesc
    d = syn.free_convection_desc(ca=False, net=None)
    d.nets = [NetDesc([32, 64, 64, 31], ["mish", "mish", "identity"])]
    theta = syn.theta_random(d, scale=1.0)
    nx, ny = 4, 2
    T, y = gyre_inputs(nx, ny)
    cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
    rng = np.random.default_rng(11)
    fb = rng.standard_normal((32, ny, nx)) if which == "forcing_bar" else None
    ob = rng.standard_normal((32, ny, nx)) if which == "T_out_bar" else None
    Tb, tb = oracle_closure_vjp(d, theta, cd, T, y, fb, ob)
    t64 = (lambda a: torch.tensor(np.asarray(a), dtype=torch.float64))
    base = [t64(T), t64(theta)]

    def L(args):
        with torch.no_grad():
            forcing, T_out = nde.closure_step(d, args[1], cd, args[0], t64(y))
            return float((forcing * t64(fb)).sum() if fb is not None else (T_out * t64(ob)).sum())

    with torch.no_grad():
        _, T_out = nde.closure_step(d, base[1], cd, base[0], t64(y))
    assert (T_out - base[0]).abs().max() > 1e-3  # the adjustment acts
    grads = [Tb, tb]
    for i, name in enumerate(("T", "theta")):
        if name == "theta" and fb is None:
            assert np.all(tb == 0)  # theta reaches the forcing only
            continue
        x = base[i]
        dirn = torch.tensor(rng.standard_normal(x.shape), dtype=torch.float64)
        dirn = dirn * (1.0 if name == "T" else (x.abs() + 1e-3))
        h = 1e-6
        plus, minus = list(base), list(base)
        plus[i], minus[i] = x + h * dirn, x - h * dirn
        fd = (L(plus) - L(minus)) / (2 * h)
        terms = torch.tensor(grads[i]) * dirn
        ad = float(terms.sum())
        # relative to the sum of the magnitudes of the terms: a directional derivative can cancel far below its terms
        err = abs(fd - ad) / max(float(terms.abs().sum()), 1e-30)
        print(f"closure vjp reference {which} {name}: autograd {ad:.6e} central difference {fd:.6e} rel err {err:.1e}")
        assert err <= 1e-5, (name, ad, fd)
