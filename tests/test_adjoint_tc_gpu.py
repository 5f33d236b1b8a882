"""N1 (discrete adjoint) on tensor cores: cpz_loss_grad of the production u/v/T nets through solve_tc_kernel<AUX> ->
adjoint_tc_kernel -> wgrad_tc_kernel (csrc/cpz_adjoint_tc.cuh) against the FP64 oracle (torch autograd through the unrolled
fixed-step solve, NDE_training.jl:290-333), against the FP32 SIMT adjoint (CPZ_NO_TC_ADJ=1), and against itself under the
other record-segment / contraction policies. Tolerance 1e-4 relative (norm-wise) on loss and gradient vs the oracle."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import FLAG_CA, FLAG_DIURNAL, FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN
from util import assert_blocks, fp32_spread, oracle_loss_grad, oracle_solve, theta_blocks, ulp_nudge

pytestmark = pytest.mark.gpu
TOL = 1e-4
W_GRAD = np.array([0.7, 0.7, 1.0, 3e-3, 3e-3, 5e-3], dtype=np.float32)


def _problem(d, ncol, use_q=False, seed=0):
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol) if use_q else None
    rng = np.random.default_rng(seed)
    th2 = (th * (1 + 0.3 * rng.standard_normal(th.shape))).astype(np.float32)
    tgt = oracle_solve(d, th2, x0, bcs, Q).astype(np.float32)
    return th, x0, bcs, Q, tgt


def _rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


CASES = {
    "train": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=18, save_stride=9, ckpt_stride=9), 45, False),
    "train_one_column": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4), 1, False),
    "train_ragged_4_tiles": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=3, ckpt_stride=4), 100, False),
    "train_no_shift": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP, n_steps=12, save_stride=4, ckpt_stride=4), 40, False),
    "train_nn_only": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_ZERO_WEIGHTS, n_steps=12, save_stride=4, ckpt_stride=4, n_substeps=1), 40, False),
    "train_ca_only": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_CA | FLAG_ZERO_WEIGHTS, n_steps=12, save_stride=4, ckpt_stride=4), 40, False),
    "train_diurnal": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=12, save_stride=4, ckpt_stride=4), 40, True),
    "infer_ca": (lambda: syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=12, save_stride=4, ckpt_stride=4), 40, False),
    "rk4": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=3, ckpt_stride=3, integrator="rk4"), 33, False),
    "euler": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=3, ckpt_stride=3, integrator="euler"), 33, False),
    "last_frame_only": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=10, save_stride=0, ckpt_stride=4), 40, False),
    "steps_not_a_multiple_of_the_stride": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=20, save_stride=5, ckpt_stride=9), 40, False),
}


@pytest.mark.parametrize("split", ["0", "1"])
@pytest.mark.parametrize("case", list(CASES))
def test_tc_adjoint_matches_the_oracle(ctx, case, split, monkeypatch):
    """split = 0: two column groups per CTA (what batches above 74 tiles run); split = 1: one group per CTA, two CTAs per tile
    (the library's choice for these small batches)."""
    mk, ncol, use_q = CASES[case]
    d = mk()
    th, x0, bcs, Q, tgt = _problem(d, ncol, use_q)
    monkeypatch.setenv("CPZ_TC_SPLIT", split)
    m = engine.Model(ctx, d, th)
    assert "adjoint kernels: tcgen05" in m.describe()
    loss, grad = m.loss_grad(x0, bcs, tgt, W_GRAD, Q=Q)
    monkeypatch.setenv("CPZ_NO_TC_ADJ", "1")
    loss_s, grad_s = m.loss_grad(x0, bcs, tgt, W_GRAD, Q=Q)
    m.close()
    tot, comps, g = oracle_loss_grad(d, th, x0, bcs, tgt, W_GRAD, Q)
    g32 = oracle_loss_grad(d, th, x0, bcs, tgt, W_GRAD, Q, dtype=torch.float32)[2]
    e_l, e_c, e_g, e_s, f_g = abs(loss[6] - tot) / abs(tot), np.abs(loss[:6] - comps).max() / abs(tot), _rel(grad, g), _rel(grad_s, g), _rel(g32, g)
    print(f"tc adjoint {case} split={split}: loss {e_l:.2e} comps {e_c:.2e} grad {e_g:.2e} (fp32 simt adjoint {e_s:.2e}, fp32 oracle {f_g:.2e}; tc vs simt {_rel(grad, grad_s):.2e})")
    assert np.isfinite(grad).all() and np.linalg.norm(g) > 0
    assert e_l <= TOL and e_c <= TOL
    assert e_g <= max(TOL, f_g) and e_s <= max(TOL, f_g)
    spread = fp32_spread(lambda s: oracle_loss_grad(d, th, ulp_nudge(x0, s), bcs, tgt, W_GRAD, Q, dtype=torch.float32)[2])
    assert_blocks("tc adjoint grad", grad, g, g32, theta_blocks(d), TOL, norm="l2", spread=spread)
    assert_blocks("fp32 simt adjoint grad", grad_s, g, g32, theta_blocks(d), TOL, norm="l2", spread=spread)
    assert abs(loss[6] - loss_s[6]) <= 1e-5 * abs(loss_s[6])


@pytest.mark.parametrize("aux_gb", ["0", "0.004", None])
@pytest.mark.parametrize("ckpt", [1, 4, 9])
def test_record_segments_do_not_change_the_gradient(ctx, ckpt, aux_gb, monkeypatch):
    """The stage records of the whole solve (default: they fit), of a few checkpoint segments (4 MB budget) or of one
    segment at a time (budget 0: re-integration from every checkpoint) give the same gradient to FP32 noise."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=22, save_stride=11, ckpt_stride=ckpt)
    th, x0, bcs, Q, tgt = _problem(d, 50)
    tot, comps, g = oracle_loss_grad(d, th, x0, bcs, tgt, W_GRAD)
    if aux_gb is not None:
        monkeypatch.setenv("CPZ_ADJ_AUX_GB", aux_gb)
    m = engine.Model(ctx, d, th)
    loss, grad = m.loss_grad(x0, bcs, tgt, W_GRAD)
    m.close()
    print(f"record budget {aux_gb} GB, ckpt_stride {ckpt}: loss {abs(loss[6] - tot) / abs(tot):.2e} grad {_rel(grad, g):.2e}")
    assert abs(loss[6] - tot) / abs(tot) <= TOL and _rel(grad, g) <= TOL


def test_wgrad_contraction_matches_plain_fp32(ctx, monkeypatch):
    """wgrad_tc_kernel (3xTF32 on tcgen05) against the plain FP32 contraction of the same records (CPZ_WGRAD_REF=1)."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4)
    th, x0, bcs, Q, tgt = _problem(d, 200)
    m = engine.Model(ctx, d, th)
    l1, g1 = m.loss_grad(x0, bcs, tgt, W_GRAD)
    monkeypatch.setenv("CPZ_WGRAD_REF", "1")
    l2, g2 = m.loss_grad(x0, bcs, tgt, W_GRAD)
    m.close()
    print(f"wgrad tcgen05 vs fp32 reference contraction: {_rel(g1, g2):.2e}")
    assert _rel(g1, g2) <= 5e-6 and l1[6] == l2[6]


def test_tc_adjoint_is_deterministic_and_shards_add_up(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=9, save_stride=3, ckpt_stride=3)
    th, x0, bcs, Q, tgt = _problem(d, 75)
    m = engine.Model(ctx, d, th)
    l_all, g_all = m.loss_grad(x0, bcs, tgt, W_GRAD)
    l_again, g_again = m.loss_grad(x0, bcs, tgt, W_GRAD)
    l_a, g_a = m.loss_grad(x0[:31], bcs[:31], tgt[:31], W_GRAD)
    l_b, g_b = m.loss_grad(x0[31:], bcs[31:], tgt[31:], W_GRAD)
    m.close()
    assert np.array_equal(g_all, g_again) and np.array_equal(l_all, l_again)   # fixed reduction order, no atomics
    assert _rel((31 * g_a + 44 * g_b) / 75, g_all) <= 1e-5
    assert np.abs((31 * l_a + 44 * l_b) / 75 - l_all).max() / abs(l_all[6]) <= 1e-5
