"""S1 parity: single RHS evaluation, CUDA (through the C ABI) vs the FP64 oracle.
Tolerance (BASELINE.json north_star): relative 1e-5 in the inf-norm."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import (FLAG_CA, FLAG_CA_LITERAL_U, FLAG_DIURNAL, FLAG_DIURNAL_UNSHIFTED, FLAG_MPP, FLAG_SMOOTH_NN,
                           FLAG_SMOOTH_RI, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN)
from util import assert_blocks, field_blocks, oracle_rhs, rel_inf

pytestmark = pytest.mark.gpu
TOL_RHS = 1e-5

UVT_CASES = [
    (RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS),
    (RHS_TRAIN, FLAG_MPP),
    (RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_SMOOTH_NN | FLAG_SMOOTH_RI),
    (RHS_TRAIN, FLAG_CA),
    (RHS_TRAIN, 0),
    (RHS_TRAIN, FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL),
    (RHS_INFER, FLAG_MPP | FLAG_ZERO_WEIGHTS),
    (RHS_INFER, FLAG_MPP | FLAG_CA),
    (RHS_INFER, FLAG_MPP | FLAG_CA | FLAG_CA_LITERAL_U),
    (RHS_INFER, FLAG_DIURNAL),
    (RHS_INFER, FLAG_DIURNAL | FLAG_DIURNAL_UNSHIFTED),
]


def _check(ctx, d, theta, ncol, t=0.37, use_q=False, seed=1000):
    x, bcs = syn.columns(d, ncol, seed=seed)
    Q = syn.diurnal_Q(ncol) if use_q else None
    m = engine.Model(ctx, d, theta)
    got = m.rhs(x, bcs, t=t, Q=Q)
    m.close()
    ref = oracle_rhs(d, theta, x, bcs, t, Q)
    ref32 = oracle_rhs(d, theta, x, bcs, t, Q, dtype=torch.float32)
    err, floor = rel_inf(got, ref), rel_inf(ref32, ref)
    print(f"rhs variant={d.variant} flags={d.flags} ncol={ncol}: cuda {err:.2e}  fp32-oracle {floor:.2e}")
    assert np.isfinite(got).all()
    assert err <= TOL_RHS, (err, floor)
    assert_blocks("rhs", got, ref, ref32, field_blocks(d), TOL_RHS)


@pytest.mark.parametrize("variant,flags", UVT_CASES)
def test_rhs_uvt_small_net(ctx, variant, flags):
    d = syn.wind_mixing_desc(variant=variant, flags=flags, net="uvT_small")
    _check(ctx, d, syn.theta_random(d, scale=1.0), 70, use_q=bool(flags & FLAG_DIURNAL))


def test_rhs_reference_initial_weights(ctx):
    """weights / 1e5 as the reference initialises them (train_NDE.jl:105-107): the NDE is the base closure."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN)
    _check(ctx, d, syn.theta_init(d), 64)


@pytest.mark.parametrize("ncol", [1, 3, 31, 32, 33, 257])
def test_rhs_ragged_column_counts(ctx, ncol):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    _check(ctx, d, syn.theta_random(d, scale=1.0), ncol)


@pytest.mark.parametrize("act", ["relu", "mish", "swish", "leakyrelu", "tanh"])
def test_rhs_uvt_test_net_activations(ctx, act):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    d.nets = [syn.NET_SHAPES["uvT_test"](32, act) for _ in range(3)]
    _check(ctx, d, syn.theta_random(d, scale=1.0), 40)


def test_rhs_uvt_large_net_streams_weights(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, net="uvT_large")
    _check(ctx, d, syn.theta_random(d, scale=1.0), 40)


def test_rhs_nn_free_DE(ctx):
    """diffusivity_parameter_optimisation.jl:1-33 — the mPP-only RHS."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    _check(ctx, d, np.zeros(0, dtype=np.float32), 48)


@pytest.mark.parametrize("ca", [False, True])
def test_rhs_free_convection(ctx, ca):
    d = syn.free_convection_desc(ca=ca)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 50)


def test_rhs_other_Nz(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, Nz=16)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 20)
    d = syn.free_convection_desc(ca=True, Nz=64)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 20)
