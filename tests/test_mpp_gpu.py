"""8f-3: gradient of the training loss wrt the five modified-Pacanowski-Philander parameters p = (nu0, nu_m, dRi, Ric, Pr)
(wind_mixing/src/diffusivity_parameter_optimisation.jl:1-33,150-197), CUDA through cpz_loss_grad_mpp vs FP64 autograd of
the oracle, plus the host mirror of optimise_modified_pacanowski_philander."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn, wind_mixing as wm
from cpz_b200.desc import FLAG_CA, FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN
from cpz_b200.ocean_parameterizations import ZeroMeanUnitVarianceScaling
from oracle import nde
from util import (assert_blocks, fp32_spread, mpp_blocks, mpp_scale, oracle_loss_grad, oracle_solve, rel_inf, t32, t64,
                  theta_blocks, ulp_nudge)

pytestmark = pytest.mark.gpu
W = np.array([0.7, 0.7, 1.0, 3e-3, 3e-3, 5e-3], dtype=np.float32)
TRUTH = dict(nu_m=0.07, Ric=0.3, Pr=1.3, dRi=0.15, nu0=2e-4)


def _case(variant, flags, net, ncol, n_steps=12):
    d = syn.wind_mixing_desc(variant=variant, flags=flags, net=net, n_steps=n_steps, save_stride=4, ckpt_stride=4)
    th = syn.theta_random(d, scale=0.3) if net else np.zeros(0, dtype=np.float32)
    x0, bcs = syn.columns(d, ncol)
    d_true = syn.wind_mixing_desc(variant=variant, flags=flags, net=net, n_steps=n_steps, save_stride=4, ckpt_stride=4,
                                  n_substeps=d.n_substeps, **TRUTH)
    tgt = oracle_solve(d_true, th, x0, bcs).astype(np.float32)
    return d, th, x0, bcs, tgt


def _spread(d, th, x0, bcs, tgt):
    """FP32-oracle mPP-parameter gradients at ulp-nudged x0 (util.fp32_spread)."""
    return fp32_spread(lambda s: nde.loss_grad_mpp(d, t32(th), t32(ulp_nudge(x0, s)), t32(bcs), None, t32(tgt), W)[1]
                       .numpy().astype(np.float64))


def _errors(d, gp, g, g32, spread):
    """The reference optimises p .* (1 ./ p_initial) (diffusivity_parameter_optimisation.jl:41-52), so the gradient the
    optimiser sees is g_i * p_i: the norm-wise error is taken in that space (tolerance 1e-4, north star). Each parameter is
    also held on its own to max(1e-4, 3 x its FP32-oracle error), which the norm-wise error cannot see (d/d(nu0) is 0.4 % of
    the scaled norm); d/d(nu0) is a sum of many small terms of both signs over the weakly-diffusive faces and d/d(dRi) runs
    through the tanh step, so their floors include FP32-oracle runs at ulp-nudged x0 (util.assert_blocks)."""
    p = mpp_scale(d)
    e_s = np.linalg.norm((gp - g) * p) / np.linalg.norm(g * p)
    f_s = np.linalg.norm((g32 - g) * p) / np.linalg.norm(g * p)
    assert_blocks("mPP-parameter gradient", gp * p, g * p, g32 * p, mpp_blocks(), 1e-4, k=3.0,
                  spread=lambda: [r * p for r in spread()])
    return e_s, f_s, np.abs(gp - g) / np.abs(g), np.abs(g32 - g) / np.abs(g)


@pytest.mark.parametrize("ncol", [9, 70, 5000])
@pytest.mark.parametrize("variant,flags", [(RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS), (RHS_INFER, FLAG_MPP | FLAG_CA)])
def test_mpp_parameter_gradient_nn_free(ctx, ncol, variant, flags):
    """`DE` (NN-free): 4-column tiles (9), 16-column tiles (70 -> 5 tiles) and 32-column tiles (5000) of the adjoint."""
    if ncol > 1000 and variant == RHS_INFER:
        pytest.skip("one large case is enough")
    d, th, x0, bcs, tgt = _case(variant, flags, None, ncol, n_steps=12 if ncol < 1000 else 4)
    m = engine.Model(ctx, d, th)
    loss, gp, gt = m.loss_grad_mpp(x0, bcs, tgt, W)
    loss_only, _ = m.loss_grad(x0, bcs, tgt, W, want_grad=False)
    m.close()
    tot, g = nde.loss_grad_mpp(d, t64(th), t64(x0), t64(bcs), None, t64(tgt), W)
    tot32, g32 = nde.loss_grad_mpp(d, t32(th), t32(x0), t32(bcs), None, t32(tgt), W)
    g, g32 = g.numpy(), g32.numpy().astype(np.float64)
    e_s, f_s, e, fl = _errors(d, gp, g, g32, _spread(d, th, x0, bcs, tgt))
    print(f"mPP-parameter gradient variant={variant} ncol={ncol}: loss {abs(loss[6] - float(tot)) / abs(float(tot)):.2e}  scaled-space L2 {e_s:.2e} "
          f"(fp32-oracle {f_s:.2e})  per parameter (nu0,nu_m,dRi,Ric,Pr) {np.array2string(e, precision=1)}  fp32-oracle {np.array2string(fl, precision=1)}")
    assert gt is None
    assert abs(loss[6] - float(tot)) / abs(float(tot)) <= 1e-4
    np.testing.assert_allclose(loss_only, loss, rtol=1e-5, atol=1e-10)
    assert e_s <= max(1e-4, 3 * f_s), (e_s, f_s)


def test_mpp_parameter_gradient_with_nets(ctx):
    """The same five derivatives of the full NDE (three nets), together with the theta gradient, in one reverse sweep."""
    d, th, x0, bcs, tgt = _case(RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS, "uvT_small", 40)
    m = engine.Model(ctx, d, th)
    loss, gp, gt = m.loss_grad_mpp(x0, bcs, tgt, W, want_theta_grad=True)
    loss2, gt2 = m.loss_grad(x0, bcs, tgt, W)
    m.close()
    tot, g = nde.loss_grad_mpp(d, t64(th), t64(x0), t64(bcs), None, t64(tgt), W)
    _, g32 = nde.loss_grad_mpp(d, t32(th), t32(x0), t32(bcs), None, t32(tgt), W)
    _, _, g_th = oracle_loss_grad(d, th, x0, bcs, tgt, W)
    g_th32 = oracle_loss_grad(d, th, x0, bcs, tgt, W, dtype=torch.float32)[2]
    e_s, f_s, e, fl = _errors(d, gp, g.numpy(), g32.numpy().astype(np.float64), _spread(d, th, x0, bcs, tgt))
    e_th, f_th = np.linalg.norm(gt - g_th) / np.linalg.norm(g_th), np.linalg.norm(g_th32 - g_th) / np.linalg.norm(g_th)
    print(f"NDE with nets: mPP-parameter scaled-space L2 {e_s:.2e} (fp32-oracle {f_s:.2e}) per parameter {np.array2string(e, precision=1)}  "
          f"theta gradient {e_th:.2e} (fp32-oracle {f_th:.2e})")
    assert e_s <= max(1e-4, 3 * f_s) and e_th <= max(1e-4, 3 * f_th)
    spread = fp32_spread(lambda s: oracle_loss_grad(d, th, ulp_nudge(x0, s), bcs, tgt, W, dtype=torch.float32)[2])
    assert_blocks("theta gradient", gt, g_th, g_th32, theta_blocks(d), 1e-4, k=3.0, norm="l2", spread=spread)
    # gt comes from the FP32 SIMT reverse sweep (it carries the five parameter accumulators), gt2 from the tensor-core adjoint
    assert np.linalg.norm(gt - gt2) / np.linalg.norm(gt2) <= max(1e-4, f_th)


def test_set_get_mpp_params(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    x, bcs = syn.columns(d, 20)
    m = engine.Model(ctx, d, np.zeros(0, dtype=np.float32))
    np.testing.assert_allclose(m.mpp_params(), [d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr], rtol=1e-7)
    m.set_mpp_params(2e-4, 0.07, 0.15, 0.3, 1.3)
    got = m.rhs(x, bcs)
    d2 = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None, **TRUTH)
    from util import oracle_rhs
    assert rel_inf(got, oracle_rhs(d2, np.zeros(0, dtype=np.float32), x, bcs)) <= 1e-5
    with pytest.raises(engine.CpzError):
        m.set_mpp_params(1e-4, 0.1, 0.0, 0.25, 1.0)  # dRi = 0
    m.close()


def test_optimise_modified_pacanowski_philander_host_mirror(ctx):
    """Synthetic 'LES' generated by the base closure with other parameters; the box-constrained L-BFGS of the host mirror
    (scaled parameters, loss fractions) must lower the loss and move nu_m, Ric, Pr towards the truth."""
    names = ("u", "v", "T", "uw", "vw", "wT")
    sc = {k: ZeroMeanUnitVarianceScaling(mu=syn.MU[i], sigma=syn.SIGMA[i]) for i, k in enumerate(names)}
    n_frames = 37
    d_true = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None, n_steps=n_frames - 1, save_stride=1, n_substeps=3, nu_m=0.06, Ric=0.32, Pr=1.4,
                                  tau=(n_frames - 1) * 600.0, dt=1.0 / (n_frames - 1))
    x0, bcs = syn.columns(d_true, 18)
    uvT = oracle_solve(d_true, np.zeros(0, dtype=np.float32), x0, bcs).astype(np.float32)
    data = wm.ProfileData(uvT, np.arange(n_frames) * 600.0, bcs, sc, np.linspace(-256.0, 0.0, 33))
    rec = wm.TrainingRecord()
    fit, rec = wm.optimise_modified_pacanowski_philander(data, range(0, n_frames, 4), "Tsit5", 25, train_gradient=True,
                                                         training_fractions={"T": 0.8, "∂T∂z": 0.8, "profile": 0.5}, ctx=ctx,
                                                         n_substeps=3, record=rec)
    print("fitted", fit, "loss", rec.totals[0], "->", min(rec.totals))
    assert min(rec.totals) < 0.2 * rec.totals[0]
    assert abs(fit["nu_m"] - 0.06) < abs(0.1 - 0.06) and abs(fit["Pr"] - 1.4) < abs(1.0 - 1.4)
