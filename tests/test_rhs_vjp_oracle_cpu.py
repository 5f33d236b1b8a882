"""The FP64 reference of the RHS pullback (test_rhs_vjp_gpu.oracle_rhs_vjp: torch.autograd of oracle/nde.py rhs) agrees with
central finite differences of nde.rhs. No GPU needed."""
import numpy as np
import pytest
import torch

from cpz_b200 import synthetic as syn
from cpz_b200.desc import FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_TRAIN
from oracle import nde
from test_rhs_vjp_gpu import oracle_rhs_vjp, ybar_of


def _fd_directional(d, theta, x, bcs, ybar, dx, dth, dp, eps):
    """ybar . (f(z + eps v) - f(z - eps v)) / (2 eps) for a direction v = (dx, dth, dp) in (x, theta, p) space."""
    p0 = np.array([np.float32(v) for v in (d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr)], dtype=np.float64)
    t = lambda a: torch.tensor(a, dtype=torch.float64)

    def f(s):
        with torch.no_grad():
            return nde.rhs(d, t(theta + s * dth), t(x + s * dx), t(bcs), 0.3, None, p_mpp=t(p0 + s * dp)).numpy()

    return float(np.sum(ybar * (f(eps) - f(-eps))) / (2 * eps))


@pytest.mark.parametrize("model", ["uvT", "T_only"])
def test_oracle_vjp_matches_finite_differences(model):
    if model == "uvT":
        d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, net="uvT_small", Nz=16)
    else:
        d = syn.free_convection_desc(ca=True, mpp=True, Nz=16)
    ncol = 6
    theta = syn.theta_random(d, scale=1.0).astype(np.float64)
    x, bcs = syn.columns(d, ncol)
    x, bcs = x.astype(np.float64), bcs.astype(np.float64)
    ybar = ybar_of(d, ncol).astype(np.float64)
    xb, tb, pb = oracle_rhs_vjp(d, theta, x, bcs, ybar, t=0.3, want_mpp=True)
    rng = np.random.default_rng(11)
    for _ in range(3):
        dx, dth, dp = rng.standard_normal(x.shape), rng.standard_normal(theta.shape), rng.standard_normal(5)
        dp *= np.abs(np.array([d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr]))  # steps relative to each parameter's size
        for v in ((dx, 0 * dth, 0 * dp), (0 * dx, dth, 0 * dp), (0 * dx, 0 * dth, dp)):
            fd = _fd_directional(d, theta, x, bcs, ybar, *v, eps=1e-7)
            ad = float(np.sum(xb * v[0]) + np.sum(tb * v[1]) + np.sum(pb * v[2]))
            assert abs(ad - fd) <= 1e-6 * max(abs(fd), 1.0), (model, ad, fd)
