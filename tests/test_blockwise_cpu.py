"""The block-wise rule of util.assert_blocks, pinned with oracle mutants (no GPU).

Each mutant is an FP64-oracle result with one plausible kernel fault built in, on the inputs of an existing GPU test. The
whole-vector rule that test applies accepts the mutant, because the faulty block is small next to the largest one; the
block-wise rule rejects it. The FP32 oracle gives the floors in both rules, as on the GPU."""
import numpy as np
import pytest
import torch

from cpz_b200 import synthetic as syn
from cpz_b200.desc import FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_TRAIN, NetDesc
from oracle import flux_nn, nde
from test_adjoint_gpu import W_GRAD, _targets
from test_mpp_gpu import _case
from util import (assert_blocks, field_blocks, fp32_spread, mpp_blocks, mpp_scale, oracle_loss_grad, oracle_rhs, rel_inf, t32,
                  t64, theta_blocks, ulp_nudge)


def test_theta_blocks_follow_destructure_order():
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    d.nets = [NetDesc([96, 50, 20, 31], ["mish", "mish", "identity"]), NetDesc([96, 40, 31], ["relu", "identity"]),
              NetDesc([96, 53, 24, 31], ["tanh", "tanh", "identity"])]
    th = np.arange(d.n_params, dtype=np.float64)
    blocks = dict(theta_blocks(d))
    assert len(blocks) == 2 * (3 + 2 + 3)
    for q, part in enumerate(nde.split_thetas(d, torch.tensor(th))):
        for l, (W, b) in enumerate(flux_nn.reconstruct(part.numpy(), d.nets[q].sizes)):
            np.testing.assert_array_equal(th[blocks[f"net{q}.W{l + 1}"]], W.flatten(order="F"))
            np.testing.assert_array_equal(th[blocks[f"net{q}.b{l + 1}"]], b)
    assert [n for n, _ in field_blocks(d)] == ["u", "v", "T"]
    assert [n for n, _ in field_blocks(syn.free_convection_desc())] == ["T"]


def test_exact_zero_blocks_take_an_absolute_bound():
    ref = np.array([1.0, 2.0, 0.0, 0.0])
    blocks = [("a", slice(0, 2)), ("z", slice(2, 4))]
    assert_blocks("zero block", ref + [0, 0, 1e-5, 0], ref, ref, blocks, 1e-4)
    with pytest.raises(AssertionError):
        assert_blocks("zero block", ref + [0, 0, 1e-3, 0], ref, ref, blocks, 1e-4)


def _tf32(t):
    """Round to the 10 explicit mantissa bits of TF32 (nearest, ties away from zero), as a 1xTF32 MMA reads its operands."""
    u = t.to(torch.float32).view(torch.int32)
    u = (u + 0x1000) & ~0x1FFF
    return u.view(torch.float32).to(t.dtype)


def _chain_tf32(theta, sizes, acts, x):
    h = x
    for (W, b), a in zip(flux_nn.reconstruct(theta, sizes), acts):
        h = flux_nn.act_torch(a, _tf32(h) @ _tf32(W).t() + b)
    return h


def test_wT_net_in_one_pass_tf32_passes_the_global_rule_and_fails_per_field(monkeypatch):
    """test_tc_gpu.py::test_tc_rhs_parity_net_shapes (50/20 mish, theta_random(1), 70 columns) with the wT net (net 2)
    evaluated in plain 1xTF32, the 3xTF32 correction dropped: the T tendency is ~1 % of the RHS's max."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small")
    th = syn.theta_random(d, scale=1.0)
    x, bcs = syn.columns(d, 70)
    ref = oracle_rhs(d, th, x, bcs, 0.37)
    ref32 = oracle_rhs(d, th, x, bcs, 0.37, dtype=torch.float32)
    calls = []

    def chain(theta, sizes, acts, xx):
        calls.append(None)
        return (_chain_tf32 if len(calls) % 3 == 0 else flux_nn.chain_torch)(theta, sizes, acts, xx)

    monkeypatch.setattr(nde, "chain_torch", chain)
    mutant = oracle_rhs(d, th, x, bcs, 0.37)
    monkeypatch.undo()
    assert len(calls) == 3
    e = rel_inf(mutant, ref)
    print(f"wT net in 1xTF32: global rel_inf {e:.2e} (rule 1e-5)")
    assert e <= 1e-5
    with pytest.raises(AssertionError, match="'T'"):
        assert_blocks("wT net in 1xTF32", mutant, ref, ref32, field_blocks(d), 1e-5)
    assert_blocks("fp32 oracle", ref32, ref, ref32, field_blocks(d), 1e-5)


def test_zero_weight_gradients_at_the_initial_weights_pass_the_global_rule_and_fail_per_block():
    """test_adjoint_gpu.py::test_grad_reference_initial_weights (weights / 1e5, 18 steps; 45 columns here) with every W
    gradient returned as zero: the b3 blocks carry almost all of the gradient's norm."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=18, save_stride=9, ckpt_stride=9)
    th = syn.theta_init(d)
    x0, bcs = syn.columns(d, 45)
    tgt = _targets(d, syn.theta_random(d, scale=0.3), x0, bcs)
    _, _, g = oracle_loss_grad(d, th, x0, bcs, tgt, W_GRAD)
    _, _, g32 = oracle_loss_grad(d, th, x0, bcs, tgt, W_GRAD, dtype=torch.float32)
    mutant = g.copy()
    for name, sl in theta_blocks(d):
        if ".W" in name:
            mutant[sl] = 0.0
    e, f = np.linalg.norm(mutant - g) / np.linalg.norm(g), np.linalg.norm(g32 - g) / np.linalg.norm(g)
    print(f"W gradients zeroed at theta_init: global L2 {e:.2e} (rule max(1e-4, {f:.2e}))")
    assert e <= max(1e-4, f)
    # the spread floor (FP32 oracle at ulp-nudged x0) used by the GPU gradient checks does not rescue it either
    spread = fp32_spread(lambda s: oracle_loss_grad(d, th, ulp_nudge(x0, s), bcs, tgt, W_GRAD, dtype=torch.float32)[2])
    with pytest.raises(AssertionError, match=r"net0\.W1"):
        assert_blocks("W gradients zeroed", mutant, g, g32, theta_blocks(d), 1e-4, norm="l2", spread=spread)
    assert spread()
    assert_blocks("fp32 oracle", g32, g, g32, theta_blocks(d), 1e-4, norm="l2")


def test_nu0_derivative_off_by_what_the_scaled_rule_allows_fails_per_parameter():
    """test_mpp_gpu.py::test_mpp_parameter_gradient_nn_free (training RHS, 9 columns) with d/d(nu0) scaled by 1 + delta,
    delta the largest relative error the scaled-space L2 rule max(1e-4, 3 x FP32 floor) still accepts."""
    d, th, x0, bcs, tgt = _case(RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS, None, 9)
    w = np.array([0.7, 0.7, 1.0, 3e-3, 3e-3, 5e-3], dtype=np.float32)
    _, g = nde.loss_grad_mpp(d, t64(th), t64(x0), t64(bcs), None, t64(tgt), w)
    _, g32 = nde.loss_grad_mpp(d, t32(th), t32(x0), t32(bcs), None, t32(tgt), w)
    p = mpp_scale(d)
    gs, gs32 = g.numpy() * p, g32.numpy().astype(np.float64) * p
    bound = max(1e-4, 3 * np.linalg.norm(gs32 - gs) / np.linalg.norm(gs))
    delta = 0.99 * bound * np.linalg.norm(gs) / abs(gs[0])
    mutant = gs.copy()
    mutant[0] *= 1 + delta
    e = np.linalg.norm(mutant - gs) / np.linalg.norm(gs)
    print(f"d/d(nu0) off by {delta:.2e} relative ({abs(gs[0]) / np.linalg.norm(gs):.2e} of the scaled norm): "
          f"scaled-space L2 {e:.2e} (rule {bound:.2e})")
    assert e <= bound
    with pytest.raises(AssertionError, match="nu0"):
        assert_blocks("d/d(nu0) off", mutant, gs, gs32, mpp_blocks(), 1e-4, k=3.0)
    assert_blocks("fp32 oracle", gs32, gs, gs32, mpp_blocks(), 1e-4, k=3.0)
