"""The FP64 reference of the solve pullback (test_solve_vjp_gpu.oracle_solve_vjp: torch.autograd of oracle/nde.py solve)
agrees with central finite differences of <solve, traj_bar>. No GPU needed."""
import numpy as np
import pytest
import torch

from cpz_b200 import synthetic as syn
from cpz_b200.desc import FLAG_IMPLICIT_DIFFUSION as IMP, FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN
from oracle import nde
from test_solve_vjp_gpu import oracle_solve_vjp, tbar_of


def _fd_directional(d, theta, x0, bcs, tbar, dx, dth, dp, eps):
    """<tbar, (solve(z + eps v) - solve(z - eps v)) / (2 eps)> for a direction v = (dx, dth, dp) in (x0, theta, p) space."""
    p0 = np.array([np.float32(v) for v in (d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr)], dtype=np.float64)
    t = lambda a: torch.tensor(a, dtype=torch.float64)

    def f(s):
        with torch.no_grad():
            return nde.solve(d, t(theta + s * dth), t(x0 + s * dx), t(bcs), None, mpp=t(p0 + s * dp)).numpy()

    return float(np.sum(tbar * (f(eps) - f(-eps))) / (2 * eps))


@pytest.mark.parametrize("implicit", [False, True])
def test_oracle_solve_vjp_matches_finite_differences(implicit):
    if implicit:
        d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | IMP, Nz=16, n_steps=4, save_stride=2,
                                 ckpt_stride=2, n_substeps=1)
    else:
        d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, Nz=16, n_steps=4, save_stride=2,
                                 ckpt_stride=2, n_substeps=2)
    ncol = 4
    theta = syn.theta_random(d, scale=0.3).astype(np.float64)
    x0, bcs = syn.columns(d, ncol)
    x0, bcs = x0.astype(np.float64), bcs.astype(np.float64)
    n_saved = d.n_steps // d.save_stride + 1
    tbar = tbar_of(d, ncol, n_saved).astype(np.float64)
    xb, tb, pb = oracle_solve_vjp(d, theta, x0, bcs, tbar, want_mpp=True)
    rng = np.random.default_rng(12)
    for _ in range(2):
        dx, dth, dp = rng.standard_normal(x0.shape), rng.standard_normal(theta.shape), rng.standard_normal(5)
        dp *= np.abs(np.array([d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr]))  # steps relative to each parameter's size
        for v in ((dx, 0 * dth, 0 * dp), (0 * dx, dth, 0 * dp), (0 * dx, 0 * dth, dp)):
            fd = _fd_directional(d, theta, x0, bcs, tbar, *v, eps=1e-7)
            ad = float(np.sum(xb * v[0]) + np.sum(tb * v[1]) + np.sum(pb * v[2]))
            assert abs(ad - fd) <= 1e-6 * max(abs(fd), 1.0), (implicit, ad, fd)
