"""Block-wise parity (util.assert_blocks) on the cases where a whole-vector error cannot see a small block:

- gradients at the reference's initial weights (weights / 1e5), where the W blocks carry 1e-12 .. 1e-9 of the gradient's
  norm, on every adjoint path: the tensor-core adjoint (both CTA layouts), the FP32 adjoint, the single-column T-only
  kernel (fc1) and the T-only tile adjoint; cpz_solve_vjp's and cpz_rhs_vjp's pullbacks; wgrad_tc_kernel against the plain
  FP32 contraction;
- the tcgen05 forward RHS per field at the layouts it has: layer-1 rows past 128 (3 h1 > 128), 3 and 4 layer-3 K steps,
  28- and 32-column tiles, and each net alone in the N=48 chain (net q in lanes 32q.., accumulator columns 16q..), where a
  lane or column slip of the wT net moves only the T tendency, ~1 % of the RHS.

Every case asserts the path it takes. Tolerances are the suite's (1e-5 on RHS evaluations, 1e-4 on solves and gradients)
per block, or the FP32 oracle's error on that block times the factor the whole-vector test of the same path uses. The wT
net's gradient blocks are ill-conditioned in FP32 at these weights (see util.py): their floor is SPREAD_K times the largest
FP32-oracle error over the plain run and runs at x0 nudged by one ulp (1.4e-4 .. 7.2e-4 on the 18-step u/v/T case)."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import FLAG_CA, FLAG_MPP, RHS_INFER, RHS_TRAIN
from test_adjoint_gpu import W_GRAD, W_T, _targets
from test_batch_schedules_gpu import _env, cdiv, sm_count, tc_forward_seven
from test_rhs_vjp_gpu import _check as rhs_vjp_check
from test_solve_vjp_gpu import check_vjp_blocks, expected_path, oracle_solve_vjp, tbar_of
from test_tc_gpu import _desc
from util import (assert_block_errors, assert_blocks, field_blocks, fp32_spread, oracle_loss_grad, oracle_rhs, oracle_solve,
                  rel_inf, theta_blocks, ulp_nudge)

pytestmark = pytest.mark.gpu
TOL = 1e-4


# ---- 1. gradients at the initial weights on every adjoint path ------------------------------------------------------------
@pytest.fixture(scope="module")
def uvt_init():
    """test_adjoint_gpu.py::test_grad_reference_initial_weights' problem on 45 columns, with its FP64 and FP32 oracles."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=18, save_stride=9, ckpt_stride=9)
    th = syn.theta_init(d)
    x0, bcs = syn.columns(d, 45)
    tgt = _targets(d, syn.theta_random(d, scale=0.3), x0, bcs)
    return _oracles(d, th, x0, bcs, tgt, W_GRAD)


def _oracles(d, th, x0, bcs, tgt, w):
    tot, _, g = oracle_loss_grad(d, th, x0, bcs, tgt, w)
    tot32, _, g32 = oracle_loss_grad(d, th, x0, bcs, tgt, w, dtype=torch.float32)
    spread = fp32_spread(lambda s: oracle_loss_grad(d, th, ulp_nudge(x0, s), bcs, tgt, w, dtype=torch.float32)[2])
    return dict(d=d, th=th, x0=x0, bcs=bcs, tgt=tgt, tot=tot, g=g, g32=g32, f_l=abs(tot32 - tot) / abs(tot), spread=spread)


def _grad_blocks(ctx, c, env, kernels, label, k=1.0, w=W_GRAD):
    with _env(**env):
        m = engine.Model(ctx, c["d"], c["th"])
        assert kernels in m.describe(), m.describe()
        loss, grad = m.loss_grad(c["x0"], c["bcs"], c["tgt"], w)
        m.close()
    e_l = abs(loss[6] - c["tot"]) / abs(c["tot"])
    print(f"{label}: loss {e_l:.2e} (fp32-oracle {c['f_l']:.2e})")
    assert np.isfinite(grad).all() and e_l <= max(TOL, k * c["f_l"])
    worst = assert_blocks(label, grad, c["g"], c["g32"], theta_blocks(c["d"]), TOL, k=k, norm="l2", spread=c["spread"])
    print(f"{label}: worst block error / bound {worst:.2f}")
    return grad


@pytest.mark.parametrize("split", ["0", "1"])
def test_tc_adjoint_at_initial_weights(ctx, uvt_init, split):
    _grad_blocks(ctx, uvt_init, {"CPZ_TC_SPLIT": split, "CPZ_NO_TC_ADJ": None}, "adjoint kernels: tcgen05",
                 f"tc adjoint at theta_init, split={split}")


def test_fp32_adjoint_at_initial_weights(ctx, uvt_init):
    _grad_blocks(ctx, uvt_init, {"CPZ_NO_TC_ADJ": "1"}, "adjoint kernels: fp32-simt", "fp32 adjoint at theta_init")


@pytest.mark.parametrize("ncol,path", [(3, "fc1"), (40, "fp32")])
def test_t_only_adjoint_at_initial_weights(ctx, ncol, path):
    """T-only model with convective adjustment and the mPP base: fc1 (one CTA per column, <= 32 columns) and the FP32 tile
    adjoint. 3 x the floor, the rule of the T-only CA gradients elsewhere (the adjustment switch flips under rounding)."""
    d = syn.free_convection_desc(ca=True, mpp=True, n_steps=12, save_stride=4, ckpt_stride=4)
    th = syn.theta_init(d)
    x0, bcs = syn.columns(d, ncol)
    tgt = _targets(d, syn.theta_random(d, scale=0.3), x0, bcs)
    m = engine.Model(ctx, d, th)
    assert expected_path(m, ncol, False) == path, m.describe()
    m.close()
    c = _oracles(d, th, x0, bcs, tgt, W_T)
    _grad_blocks(ctx, c, {}, "", f"T-only {path} adjoint at theta_init, {ncol} columns", k=3.0, w=W_T)


@pytest.mark.parametrize("path", ["tc", "fp32"])
def test_solve_vjp_at_initial_weights(ctx, path):
    """cpz_solve_vjp at weights / 1e5 on the tensor-core adjoint and on the FP32 adjoint (with mpp_bar)."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4)
    th = syn.theta_init(d)
    ncol = 40
    x0, bcs = syn.columns(d, ncol)
    want_mpp = path == "fp32"
    m = engine.Model(ctx, d, th)
    assert expected_path(m, ncol, want_mpp) == path, m.describe()
    tb_in = tbar_of(d, ncol, m.n_saved)
    got = m.solve_vjp(x0, bcs, tb_in, want_mpp=want_mpp)
    m.close()
    ref = oracle_solve_vjp(d, th, x0, bcs, tb_in, want_mpp=want_mpp)
    ref32 = oracle_solve_vjp(d, th, x0, bcs, tb_in, dtype=torch.float32, want_mpp=want_mpp)
    print(f"solve_vjp at theta_init ({path}):")
    check_vjp_blocks(d, got, ref, ref32, path, fp32_spread(
        lambda s: oracle_solve_vjp(d, th, ulp_nudge(x0, s), bcs, tb_in, dtype=torch.float32, want_mpp=want_mpp)))


def test_rhs_vjp_at_initial_weights(ctx):
    """cpz_rhs_vjp at weights / 1e5 on the inference RHS with mPP and convective adjustment, 257 columns (9 tiles, the last
    ragged), every output held per block by test_rhs_vjp_gpu.py's checker (its own initial-weight case is the training RHS
    on 64 columns)."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA)
    rhs_vjp_check(ctx, d, syn.theta_init(d), 257, label="theta_init")


def test_wgrad_contraction_per_block_at_initial_weights(ctx, monkeypatch):
    """wgrad_tc_kernel (3xTF32) against the plain FP32 contraction of the same records (CPZ_WGRAD_REF=1), block by block,
    to test_adjoint_tc_gpu.py's whole-vector bound of 5e-6."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4)
    th = syn.theta_init(d)
    x0, bcs = syn.columns(d, 200)
    tgt = _targets(d, syn.theta_random(d, scale=0.3), x0, bcs)
    m = engine.Model(ctx, d, th)
    assert "adjoint kernels: tcgen05" in m.describe()
    l1, g1 = m.loss_grad(x0, bcs, tgt, W_GRAD)
    monkeypatch.setenv("CPZ_WGRAD_REF", "1")
    l2, g2 = m.loss_grad(x0, bcs, tgt, W_GRAD)
    m.close()
    assert l1[6] == l2[6]
    g1, g2 = g1.astype(np.float64), g2.astype(np.float64)
    rows = [(name, np.linalg.norm(g1[sl] - g2[sl]) / np.linalg.norm(g2[sl]), 0.0, np.linalg.norm(g2[sl]))
            for name, sl in theta_blocks(d)]
    assert_block_errors("wgrad tcgen05 vs fp32 contraction", rows, 5e-6)


# ---- 2. tcgen05 forward RHS per field -------------------------------------------------------------------------------------
def _rhs_fields(ctx, d, th, ncol, label, t=0.37):
    x, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    desc = m.describe()
    got = m.rhs(x, bcs, t=t)
    m.close()
    ref, ref32 = oracle_rhs(d, th, x, bcs, t), oracle_rhs(d, th, x, bcs, t, dtype=torch.float32)
    assert np.isfinite(got).all()
    assert rel_inf(got, ref) <= 1e-5
    worst = assert_blocks(label, got, ref, ref32, field_blocks(d), 1e-5)
    print(f"{label}: worst field error / bound {worst:.2f}")
    return desc


@pytest.mark.parametrize("h1,h2,act", [(53, 20, "mish"), (50, 24, "tanh"), (50, 25, "mish"), (53, 32, "relu")])
@pytest.mark.parametrize("variant", [RHS_TRAIN, RHS_INFER])
def test_tc_rhs_per_field_layouts(ctx, h1, h2, act, variant):
    """3 h1 > 128 runs the layer-1 rows past 128; h2 <= 24 gives 3 layer-3 K steps, h2 > 24 four."""
    d = _desc(h1, h2, act, variant=variant)
    n1b = max(0, 3 * h1 - 128)
    desc = _rhs_fields(ctx, d, syn.theta_random(d, scale=1.0), 70, f"tcgen05 rhs h1={h1} h2={h2} {act} variant={variant}")
    assert "forward kernel: tcgen05" in desc, desc
    assert f"layer-1 rows {3 * h1 - n1b}+{n1b}," in desc and f"layer-3 {3 if h2 <= 24 else 4} K steps" in desc, desc


def test_tc_rhs_per_field_28_and_32_column_tiles(ctx):
    sms = sm_count()
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=1.0)
    n = 28 * sms + 1
    x, bcs = syn.columns(d, n)
    ref, ref32 = oracle_rhs(d, th, x, bcs, 0.21), oracle_rhs(d, th, x, bcs, 0.21, dtype=torch.float32)
    m = engine.Model(ctx, d, th)
    assert "forward kernel: tcgen05" in m.describe()
    out = {}
    for ncol in (28 * sms, 28 * sms + 1):
        seven = tc_forward_seven(ncol, sms)
        assert seven == (ncol == 28 * sms)
        got = m.rhs(x[:ncol], bcs[:ncol], t=0.21)
        label = f"tcgen05 rhs {ncol} columns, {cdiv(ncol, 28 if seven else 32)} tiles of {28 if seven else 32}"
        assert rel_inf(got, ref[:ncol]) <= 1e-5
        assert_blocks(label, got, ref[:ncol], ref32[:ncol], field_blocks(d), 1e-5)
        out[ncol] = got
    m.close()
    np.testing.assert_array_equal(out[28 * sms], out[28 * sms + 1][:28 * sms])


# ---- 3. one net at a time ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", [RHS_TRAIN, RHS_INFER])
@pytest.mark.parametrize("net", [0, 1, 2])
def test_tc_one_net_at_a_time(ctx, net, variant):
    """theta non-zero in net `net` only: that net's flux must reach its own field and no other, in the RHS and in an
    8-step solve."""
    d = syn.wind_mixing_desc(variant=variant, n_steps=8, save_stride=4)
    full = syn.theta_random(d, scale=0.3)
    th = np.zeros_like(full)
    for name, sl in theta_blocks(d):
        if name.startswith(f"net{net}."):
            th[sl] = full[sl]
    desc = _rhs_fields(ctx, d, th, 70, f"tcgen05 rhs, net {net} alone, variant={variant}")
    assert "forward kernel: tcgen05" in desc
    x0, bcs = syn.columns(d, 45)
    m = engine.Model(ctx, d, th)
    assert "forward kernel: tcgen05" in m.describe(), m.describe()
    got = m.solve(x0, bcs)
    m.close()
    ref, ref32 = oracle_solve(d, th, x0, bcs), oracle_solve(d, th, x0, bcs, dtype=torch.float32)
    assert rel_inf(got, ref) <= TOL
    assert_blocks(f"tcgen05 8-step solve, net {net} alone", got, ref, ref32, field_blocks(d), TOL)
