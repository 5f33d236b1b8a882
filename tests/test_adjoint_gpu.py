"""S3/S4 parity: loss, exact discrete-adjoint gradient, fused ADAM step — CUDA (through the C ABI) vs the FP64 oracle
(torch autograd through the unrolled fixed-step solve). Tolerance 1e-4 relative (norm-wise) on loss and gradient."""
import os

import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import (FLAG_CA, FLAG_DIURNAL, FLAG_MPP, FLAG_SMOOTH_NN, FLAG_SMOOTH_RI, FLAG_ZERO_WEIGHTS, RHS_INFER,
                           RHS_TRAIN)
from oracle import nde
from util import assert_blocks, fp32_spread, oracle_loss_grad, oracle_solve, rel_inf, t64, theta_blocks, ulp_nudge

pytestmark = pytest.mark.gpu
TOL = 1e-4
W_GRAD = np.array([0.7, 0.7, 1.0, 3e-3, 3e-3, 5e-3], dtype=np.float32)
W_T = np.array([0, 0, 1.0, 0, 0, 0], dtype=np.float32)


def _targets(d, th, x0, bcs, Q=None, seed=0):
    """the oracle's solution with a perturbed theta (SURVEY 8d 'Targets')"""
    rng = np.random.default_rng(seed)
    th2 = (th * (1 + 0.3 * rng.standard_normal(th.shape))).astype(np.float32)
    return oracle_solve(d, th2, x0, bcs, Q).astype(np.float32)


def _check(ctx, d, th, ncol, w, use_q=False, th_target=None):
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol) if use_q else None
    tgt = _targets(d, th if th_target is None else th_target, x0, bcs, Q)
    m = engine.Model(ctx, d, th)
    loss, grad = m.loss_grad(x0, bcs, tgt, w, Q=Q)
    loss_only, none = m.loss_grad(x0, bcs, tgt, w, Q=Q, want_grad=False)
    m.close()
    tot, comps, g = oracle_loss_grad(d, th, x0, bcs, tgt, w, Q)
    tot32, comps32, g32 = oracle_loss_grad(d, th, x0, bcs, tgt, w, Q, dtype=torch.float32)
    e_l = abs(loss[6] - tot) / abs(tot)
    e_c = np.abs(loss[:6] - comps).max() / abs(tot)
    e_g = np.linalg.norm(grad - g) / np.linalg.norm(g)
    e_gi = rel_inf(grad, g)
    f_g = np.linalg.norm(g32 - g) / np.linalg.norm(g)
    print(f"adjoint variant={d.variant} flags={d.flags} {d.integrator} steps={d.n_steps}x{d.n_substeps} ckpt={d.ckpt_stride} ncol={ncol}: "
          f"loss {e_l:.2e} comps {e_c:.2e} grad L2 {e_g:.2e} inf {e_gi:.2e} (fp32-oracle grad {f_g:.2e}) |g|={np.linalg.norm(g):.3e}")
    assert none is None
    assert np.isfinite(grad).all() and np.linalg.norm(g) > 0
    assert e_l <= TOL and e_c <= TOL, (e_l, e_c)
    # 1e-4, except where the FP32 restatement of the oracle itself is noisier than that (non-smooth RHS: relu kinks and
    # the min(0,.) / stability switches flip under rounding); there the CUDA result must be at least as close to the
    # FP64 oracle as the FP32 oracle is.
    assert e_g <= max(TOL, f_g), (e_g, f_g)
    spread = fp32_spread(lambda s: oracle_loss_grad(d, th, ulp_nudge(x0, s), bcs, tgt, w, Q, dtype=torch.float32)[2])
    assert_blocks("grad", grad, g, g32, theta_blocks(d), TOL, norm="l2", spread=spread)
    assert abs(loss_only[6] - tot) / abs(tot) <= TOL
    return loss, grad


@pytest.mark.parametrize("ckpt", [1, 4, 9])
def test_grad_train_rhs_checkpoint_strides(ctx, ckpt):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=18, save_stride=9, ckpt_stride=ckpt)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 45, W_GRAD)


@pytest.mark.parametrize("integrator", ["euler", "rk4"])
def test_grad_other_integrators(ctx, integrator):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=3, ckpt_stride=3, integrator=integrator)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 33, W_GRAD)


def test_grad_reference_initial_weights(ctx):
    """weights/1e5 (train_NDE.jl:105-107): gradient still matches in the regime training starts from."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=18, save_stride=9, ckpt_stride=9)
    _check(ctx, d, syn.theta_init(d), 64, W_GRAD, th_target=syn.theta_random(d, scale=0.3))


def test_grad_profile_loss_only_weights(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=9, save_stride=3, ckpt_stride=3)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 40, np.array([1, 1, 1, 0, 0, 0], dtype=np.float32))


def test_grad_diurnal(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=12, save_stride=4, ckpt_stride=4)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 40, W_GRAD, use_q=True)


@pytest.mark.parametrize("smooth", [FLAG_SMOOTH_NN, FLAG_SMOOTH_RI, FLAG_SMOOTH_NN | FLAG_SMOOTH_RI])
@pytest.mark.parametrize("ncol", [9, 40])
def test_grad_smoothing_filters(ctx, smooth, ncol):
    """smooth_NN / smooth_Ri (NDE_training.jl:98-102,121-123): the reference trains with them; their VJP is the transposed
    3-point filter. Both batches fit one wave of 4-column tiles (train_tile), so both run the 4-column-tile adjoint; the
    32-column-tile adjoint is test_grad_smoothing_filters_32_column_tiles.
    smooth_Ri averages Richardson numbers that are unbounded where the shear vanishes (+-1e6 next to O(1) values), which in
    FP32 is ill-conditioned whenever the tanh step is sharp: with the default nu_- = 0.1 the FP32 restatement of the oracle
    itself misses the FP64 gradient by 1500 % after 12 steps. The case below (nu_- = 0.01, 4 steps) is one where FP32 is
    meaningful (FP32-oracle floor 1e-6 .. 3e-5); the FP32-oracle floors are printed and bound the comparison as elsewhere."""
    _smoothing_case(ctx, smooth, ncol)


@pytest.mark.parametrize("smooth", [FLAG_SMOOTH_NN, FLAG_SMOOTH_RI, FLAG_SMOOTH_NN | FLAG_SMOOTH_RI])
def test_grad_smoothing_filters_32_column_tiles(ctx, smooth, monkeypatch):
    """The same filters on the 32-column-tile adjoint (CPZ_SMALL_NCOL=0 turns the small tiles off)."""
    monkeypatch.setenv("CPZ_SMALL_NCOL", "0")
    _smoothing_case(ctx, smooth, 40)


def _smoothing_case(ctx, smooth, ncol):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | smooth, n_steps=4, save_stride=2, ckpt_stride=2,
                             nu_m=0.01)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, ncol)
    tgt = _targets(d, th, x0, bcs)
    m = engine.Model(ctx, d, th)
    loss, grad = m.loss_grad(x0, bcs, tgt, W_GRAD)
    m.close()
    tot, comps, g = oracle_loss_grad(d, th, x0, bcs, tgt, W_GRAD)
    tot32, _, g32 = oracle_loss_grad(d, th, x0, bcs, tgt, W_GRAD, dtype=torch.float32)
    f_l, f_g = abs(tot32 - tot) / abs(tot), np.linalg.norm(g32 - g) / np.linalg.norm(g)
    e_l, e_g = abs(loss[6] - tot) / abs(tot), np.linalg.norm(grad - g) / np.linalg.norm(g)
    tiles = "32-column tiles" if os.environ.get("CPZ_SMALL_NCOL") == "0" else "4-column tiles"
    print(f"smoothing flags {smooth} ncol {ncol} ({tiles}): loss {e_l:.2e} (fp32-oracle {f_l:.2e})  grad {e_g:.2e} (fp32-oracle {f_g:.2e})")
    assert e_l <= max(TOL, 3 * f_l) and e_g <= max(TOL, 3 * f_g)
    # the filters matter: the unfiltered model's gradient is a different vector
    d0 = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, n_steps=4, save_stride=2, ckpt_stride=2, nu_m=0.01)
    g0 = oracle_loss_grad(d0, th, x0, bcs, tgt, W_GRAD)[2]
    assert np.linalg.norm(g0 - g) / np.linalg.norm(g) > 10 * max(e_g, 1e-5)


def test_grad_infer_rhs_with_convective_adjustment(ctx):
    """Q5: the trainable mPP + CA combination (a11's nu_T rule)."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=12, save_stride=4, ckpt_stride=4)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 40, W_GRAD)


@pytest.mark.parametrize("ca", [False, True])
def test_grad_free_convection(ctx, ca):
    d = syn.free_convection_desc(ca=ca, n_steps=18, save_stride=9, ckpt_stride=9)
    _check(ctx, d, syn.theta_random(d, scale=0.3), 70, W_T)


def test_grad_ragged_tiles_and_sharding(ctx):
    """Gradients over a column set equal the column-count-weighted mean of the gradients of its shards (what the
    allreduce of [grad*n; sums; n] computes) — SURVEY 8e."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=6, save_stride=3, ckpt_stride=3)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, 75)
    tgt = _targets(d, th, x0, bcs)
    m = engine.Model(ctx, d, th)
    l_all, g_all = m.loss_grad(x0, bcs, tgt, W_GRAD)
    l_a, g_a = m.loss_grad(x0[:31], bcs[:31], tgt[:31], W_GRAD)
    l_b, g_b = m.loss_grad(x0[31:], bcs[31:], tgt[31:], W_GRAD)
    m.close()
    g_mix = (31 * g_a + 44 * g_b) / 75
    l_mix = (31 * l_a + 44 * l_b) / 75
    assert np.linalg.norm(g_mix - g_all) / np.linalg.norm(g_all) <= 1e-5
    assert np.abs(l_mix - l_all).max() / abs(l_all[6]) <= 1e-5


def test_train_step_matches_flux_adam(ctx):
    """cpz_train_step = loss_grad + Flux-0.11 ADAM. The loss/gradient are checked against the oracle above; here the
    optimiser arithmetic is checked by feeding the oracle's ADAM the engine's own gradient (the first ADAM steps move
    every parameter by ~lr*sign(g), so gradient components below FP32 noise would otherwise dominate the comparison)."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=9, save_stride=3, ckpt_stride=3)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, 40)
    tgt = _targets(d, th, x0, bcs)
    m = engine.Model(ctx, d, th)
    lr = 3e-4
    theta = t64(th); mt = torch.zeros_like(theta); vt = torch.zeros_like(theta); bp = (0.9, 0.999)
    for it in range(3):
        l_pre, g_gpu = m.loss_grad(x0, bcs, tgt, W_GRAD)
        loss = m.train_step(x0, bcs, tgt, W_GRAD, lr)
        np.testing.assert_allclose(loss, l_pre, rtol=1e-6)  # the callback sees the loss BEFORE the update
        tot, comps, g = oracle_loss_grad(d, theta.numpy(), x0, bcs, tgt, W_GRAD)
        assert abs(loss[6] - tot) / abs(tot) <= TOL
        g32 = oracle_loss_grad(d, theta.numpy(), x0, bcs, tgt, W_GRAD, dtype=torch.float32)[2]
        floor = np.linalg.norm(g32 - g) / np.linalg.norm(g)
        assert np.linalg.norm(g_gpu - g) / np.linalg.norm(g) <= max(TOL, floor)  # same rule as _check
        theta, mt, vt, bp = nde.adam_step(theta, t64(g_gpu), mt, vt, bp, lr)
        got = m.get_theta()
        err = np.abs(got - theta.numpy()).max() / lr
        print(f"train_step iter {it}: loss {loss[6]:.6e}, max |dtheta error|/lr = {err:.2e}")
        assert err <= 1e-3
        theta = t64(got)  # continue from the engine's FP32 theta
    mt_d, vt_d, bp_d = m.adam_state()
    assert abs(bp_d[0] - 0.9 ** 4) < 1e-6 and abs(bp_d[1] - 0.999 ** 4) < 1e-6
    assert np.linalg.norm(mt_d - mt.numpy()) / np.linalg.norm(mt.numpy()) <= 1e-5
    assert np.linalg.norm(vt_d - vt.numpy()) / np.linalg.norm(vt.numpy()) <= 1e-4
    # resume from saved optimiser state reproduces the next step (checkpoint/resume of data_writing.jl:28-78)
    m2 = engine.Model(ctx, d, m.get_theta())
    m2.set_adam_state(mt_d, vt_d, bp_d)
    l1 = m.train_step(x0, bcs, tgt, W_GRAD, lr)
    l2 = m2.train_step(x0, bcs, tgt, W_GRAD, lr)
    np.testing.assert_allclose(m.get_theta(), m2.get_theta(), rtol=0, atol=1e-9)
    np.testing.assert_allclose(l1, l2, rtol=1e-6)
    m.close(); m2.close()


def test_training_reduces_loss(ctx):
    """A short ADAM run from the reference's initialisation (weights/1e5) lowers the loss."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=18, save_stride=9, ckpt_stride=9)
    th0 = syn.theta_init(d)
    x0, bcs = syn.columns(d, 64)
    tgt = _targets(d, syn.theta_random(d, scale=0.3), x0, bcs)
    m = engine.Model(ctx, d, th0)
    losses = [m.train_step(x0, bcs, tgt, W_GRAD, 1e-3)[6] for _ in range(12)]
    m.close()
    print("losses", losses[0], losses[-1])
    assert losses[-1] < losses[0]


def test_grad_stored_stage_tendencies_match_recompute(ctx, monkeypatch):
    """The tcgen05 forward pass hands its stage tendencies k_i to the reverse sweep; with CPZ_NO_KSTORE the adjoint
    recomputes them in FP32 SIMT. Both must give the same loss and (to FP32 noise) the same gradient."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=18, save_stride=9, ckpt_stride=3)
    th = syn.theta_random(d, scale=0.3)
    ncol = 77
    x0, bcs = syn.columns(d, ncol, seed=5)
    tgt = np.ascontiguousarray(np.repeat(x0[:, None, :], d.n_saved, axis=1)) * np.float32(0.9)
    w = np.array([1, 1, 1, 5e-3, 5e-3, 5e-3], dtype=np.float32)
    monkeypatch.setenv("CPZ_NO_TC_ADJ", "1")  # the FP32 SIMT adjoint (the tensor-core adjoint has its own tests)
    m = engine.Model(ctx, d, th)
    assert "tcgen05" in m.describe()
    l1, g1 = m.loss_grad(x0, bcs, tgt, w)
    monkeypatch.setenv("CPZ_NO_KSTORE", "1")
    l2, g2 = m.loss_grad(x0, bcs, tgt, w)
    m.close()
    assert np.all(np.isfinite(g1)) and np.linalg.norm(g1) > 0
    assert abs(l1[6] - l2[6]) <= 1e-6 * abs(l2[6])
    assert np.linalg.norm(g1 - g2) <= 2e-5 * np.linalg.norm(g2)
