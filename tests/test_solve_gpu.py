"""S2/S6 parity: fixed-step forward solve, CUDA vs FP64 oracle. Tolerance 1e-4 (relative, inf-norm) on profiles."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import FLAG_CA, FLAG_DIURNAL, FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN
from util import assert_blocks, field_blocks, oracle_solve, rel_inf

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _check(ctx, d, theta, ncol, use_q=False):
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol) if use_q else None
    m = engine.Model(ctx, d, theta)
    got = m.solve(x0, bcs, Q=Q)
    m.close()
    ref = oracle_solve(d, theta, x0, bcs, Q)
    ref32 = oracle_solve(d, theta, x0, bcs, Q, dtype=torch.float32)
    assert got.shape == ref.shape
    err, floor = rel_inf(got, ref), rel_inf(ref32, ref)
    err_final = rel_inf(got[:, -1], ref[:, -1])
    print(f"solve {d.integrator} steps={d.n_steps}x{d.n_substeps} ncol={ncol}: cuda {err:.2e} (final {err_final:.2e}) fp32-oracle {floor:.2e}")
    assert np.isfinite(got).all()
    assert err <= TOL, (err, floor)
    assert_blocks("solve", got, ref, ref32, field_blocks(d), TOL)
    return got


@pytest.mark.parametrize("integrator", ["euler", "rk4", "tsit5"])
def test_solve_integrators(ctx, integrator):
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=48, save_stride=4, integrator=integrator)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 45)


def test_solve_frame0_is_initial_condition_and_final_only(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=24, save_stride=8)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, 33)
    m = engine.Model(ctx, d, th)
    tr = m.solve(x0, bcs)
    assert tr.shape == (33, 4, 96)
    np.testing.assert_array_equal(tr[:, 0], x0)
    m.set_time(save_stride=0)
    fin = m.solve(x0, bcs)
    assert fin.shape == (33, 1, 96)
    np.testing.assert_array_equal(fin[:, 0], tr[:, -1])
    m.close()


def test_solve_train_variant_diurnal(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=36, save_stride=9)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 40, use_q=True)


def test_solve_infer_convective_adjustment(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=36, save_stride=9)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 40)


@pytest.mark.parametrize("ca", [False, True])
def test_solve_free_convection(ctx, ca):
    d = syn.free_convection_desc(ca=ca, n_steps=45, save_stride=9)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 70)


def test_solve_long_horizon_config2_slice(ctx):
    """A 64-column slice of BASELINE config 2 (1152 steps, all frames saved) against the FP64 oracle."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=1152, save_stride=1)
    th = syn.theta_init(d, scale=1e-5)
    _check(ctx, d, th, 64)


def test_solve_deterministic_and_sharding_invariant(ctx):
    """Forward results are bitwise identical regardless of how columns are split (SURVEY 8e)."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=16, save_stride=4)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, 96)
    m = engine.Model(ctx, d, th)
    full = m.solve(x0, bcs)
    again = m.solve(x0, bcs)
    np.testing.assert_array_equal(full, again)
    parts = np.concatenate([m.solve(x0[:40], bcs[:40]), m.solve(x0[40:], bcs[40:])])
    np.testing.assert_array_equal(full, parts)
    m.close()
