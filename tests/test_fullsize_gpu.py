"""Full-length parity cases (VERDICT r01 'untested configs'): slices of the BASELINE configs at their real horizon
(1 152 steps x 2 sub-steps x 6 stages = 13 824 right-hand-side evaluations per column), CUDA through the C ABI vs the
FP64 oracle on identical seeded inputs, with the FP32 restatement of the oracle printed beside every error as the
noise floor of the arithmetic type.

Tolerance: 1e-4 relative (north star). Where the FP32 oracle itself is further than 1e-4 from the FP64 oracle (the long
horizon amplifies rounding through the tanh step of the Richardson-number diffusivity), the CUDA result must be within
LONG_FLOOR_FACTOR x that floor: two FP32 evaluation orders of a sensitive map differ from the FP64 answer by amounts of
the same size, not by identical amounts. This is a stated relaxation of the north-star number, reported in DESIGN.md."""
import os
import sys

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
import make_fullsize  # noqa: E402


def golden(name):
    """FP64-oracle answers computed once by tests/golden/make_fullsize.py (minutes of CPU per case) and committed."""
    return make_fullsize.load(name)

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import ClosureDesc, RHS_INFER, RHS_TRAIN
from oracle import nde
from util import oracle_loss_grad, oracle_rhs, oracle_solve, rel_inf, t64

pytestmark = pytest.mark.gpu
TOL = 1e-4
LONG_FLOOR_FACTOR = 3.0
W3 = np.array([1, 1, 1, 5e-3, 5e-3, 5e-3], dtype=np.float32)  # bench.py config 3 weights


class _env:
    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        for k, v in self.kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# ---- (a) config 3 slice at full length: loss and gradient ---------------------------------------------------------------
@pytest.fixture(scope="module")
def config3_slice():
    """36 columns (one full 32-column tile + a ragged one) of BASELINE config 3 with un-divided weights (scale 0.1) so
    that the MLP contributes; targets = FP64 oracle solution of a perturbed theta (SURVEY 8d); FP64 loss / gradient and
    the FP32-oracle floors from tests/golden/fullsize_config3_slice*.npz."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=1152, save_stride=9, ckpt_stride=9)
    th = syn.theta_random(d, scale=0.1)
    x0, bcs = syn.columns(d, 36)
    G = golden("fullsize_config3_slice")
    return dict(d=d, th=th, x0=x0, bcs=bcs, tgt=G["targets"], tot=float(G["loss"][6]), comps=G["loss"][:6], g=G["grad"],
                floor_g=float(G["floor_grad"]), floor_l=float(G["floor_loss"]))


@pytest.mark.parametrize("ckpt,kstore", [(9, True), (9, False), (1, True), (1, False)])
def test_grad_config3_slice_full_length(ctx, config3_slice, ckpt, kstore):
    c = config3_slice
    d = c["d"]
    d.ckpt_stride = ckpt
    m = engine.Model(ctx, d, c["th"])
    with _env(CPZ_NO_KSTORE=None if kstore else "1"):
        loss, grad = m.loss_grad(c["x0"], c["bcs"], c["tgt"], W3)
    m.close()
    d.ckpt_stride = 9
    e_l = abs(loss[6] - c["tot"]) / abs(c["tot"])
    e_g = np.linalg.norm(grad - c["g"]) / np.linalg.norm(c["g"])
    print(f"config-3 slice, 1152 steps x 2 sub-steps, 129 saves, ckpt_stride {ckpt}, stored stage tendencies {kstore}: "
          f"loss {e_l:.2e} (fp32-oracle {c['floor_l']:.2e})  grad L2 {e_g:.2e} (fp32-oracle {c['floor_g']:.2e})  |g| {np.linalg.norm(c['g']):.3e}")
    assert np.isfinite(grad).all()
    assert e_l <= max(TOL, LONG_FLOOR_FACTOR * c["floor_l"]), (e_l, c["floor_l"])
    assert e_g <= max(TOL, LONG_FLOOR_FACTOR * c["floor_g"]), (e_g, c["floor_g"])


def test_grad_config3_bench_theta_full_length(ctx):
    """The exact model bench.py times as config 3 (theta = Glorot / 1e5, ckpt_stride 1 and 9) on a 32-column slice."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=1152, save_stride=9, ckpt_stride=1)
    th = syn.theta_init(d, seed=42, scale=1e-5)
    x0, bcs = syn.columns(d, 32, seed=1000)
    G = golden("fullsize_config3_bench_theta")
    tgt, tot, g, floor = make_fullsize.bench_targets(d, x0), float(G["loss"][6]), G["grad"], float(G["floor_grad"])
    for ckpt in (1, 9):
        d.ckpt_stride = ckpt
        m = engine.Model(ctx, d, th)
        loss, grad = m.loss_grad(x0, bcs, tgt, W3)
        m.close()
        e_l = abs(loss[6] - tot) / abs(tot)
        e_g = np.linalg.norm(grad - g) / np.linalg.norm(g)
        print(f"config-3 bench model (theta/1e5), ckpt_stride {ckpt}: loss {e_l:.2e}  grad L2 {e_g:.2e} (fp32-oracle {floor:.2e})")
        assert e_l <= TOL
        assert e_g <= max(TOL, LONG_FLOOR_FACTOR * floor), (e_g, floor)


# ---- (b) NN-free solve kernel ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nc", ["2", "4"])
@pytest.mark.parametrize("ncol", [1, 2, 3, 45, 131])
@pytest.mark.parametrize("variant", [RHS_TRAIN, RHS_INFER])
def test_nnfree_solve_parity(ctx, nc, ncol, variant):
    """`DE` (diffusivity_parameter_optimisation.jl:1-33) through solve_nnfree_kernel<NC>, ragged column counts."""
    d = syn.wind_mixing_desc(variant=variant, net=None, n_steps=48, save_stride=4)
    th = np.zeros(0, dtype=np.float32)
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    assert "nn-free" in m.describe(), m.describe()
    with _env(CPZ_NNFREE_NC=nc):
        got = m.solve(x0, bcs)
        dx = m.rhs(x0, bcs, t=0.1)
    with _env(CPZ_NO_TC="1"):
        simt = m.solve(x0, bcs)
    m.close()
    ref = oracle_solve(d, th, x0, bcs)
    floor = rel_inf(oracle_solve(d, th, x0, bcs, dtype=torch.float32), ref)
    e, e_s, e_r = rel_inf(got, ref), rel_inf(simt, ref), rel_inf(dx, oracle_rhs(d, th, x0, bcs, 0.1))
    print(f"nn-free NC={nc} ncol={ncol} variant={variant}: solve {e:.2e} (tiled simt {e_s:.2e}, fp32-oracle {floor:.2e})  rhs {e_r:.2e}")
    np.testing.assert_array_equal(got[:, 0], x0)
    assert got.shape == ref.shape and np.isfinite(got).all()
    assert e_r <= 1e-5 and e <= TOL


@pytest.mark.parametrize("flags_extra", ["ca", "diurnal"])
def test_nnfree_solve_flags(ctx, flags_extra):
    from cpz_b200.desc import FLAG_CA, FLAG_DIURNAL, FLAG_MPP, FLAG_ZERO_WEIGHTS
    if flags_extra == "ca":
        d = syn.wind_mixing_desc(variant=RHS_INFER, net=None, flags=FLAG_MPP | FLAG_CA, n_steps=36, save_stride=9)
    else:
        d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=36, save_stride=9)
    ncol = 77
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol) if flags_extra == "diurnal" else None
    th = np.zeros(0, dtype=np.float32)
    m = engine.Model(ctx, d, th)
    got = m.solve(x0, bcs, Q=Q)
    m.close()
    e = rel_inf(got, oracle_solve(d, th, x0, bcs, Q))
    print(f"nn-free {flags_extra}: {e:.2e}")
    assert e <= TOL


def test_nnfree_solve_full_length_bench_config(ctx):
    """The model of bench.py's nn_free line (config-2 shape, 1152 steps, all frames) on a 64-column slice."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, net=None, n_steps=1152, save_stride=1)
    th = np.zeros(0, dtype=np.float32)
    x0, bcs = syn.columns(d, 64)
    m = engine.Model(ctx, d, th)
    got = m.solve(x0, bcs)
    m.close()
    G = golden("fullsize_nnfree")
    e = np.abs(got[:, G["frames"]] - G["traj"]).max() / float(G["scale"])
    print(f"nn-free 1152 steps: {e:.2e} (fp32-oracle {float(G['floor']):.2e})")
    assert np.isfinite(got).all()
    assert e <= max(TOL, LONG_FLOOR_FACTOR * float(G["floor"]))


# ---- (c) long forward solve with weights that matter -----------------------------------------------------------------
def test_solve_full_length_undivided_weights(ctx):
    """1 152 steps, every frame saved, theta_random at scale 0.1 (the MLP fluxes are of the size of the diffusive ones)."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=1152, save_stride=1)
    th = syn.theta_random(d, scale=0.1)
    x0, bcs = syn.columns(d, 64)
    m = engine.Model(ctx, d, th)
    assert "tcgen05" in m.describe()
    got = m.solve(x0, bcs)
    with _env(CPZ_NO_TC="1"):
        simt = m.solve(x0, bcs)
    m.close()
    G = golden("fullsize_config2_undivided")
    fr, ref, floor, sc = G["frames"], G["traj"], float(G["floor"]), float(G["scale"])
    e, e_s = np.abs(got[:, fr] - ref).max() / sc, np.abs(simt[:, fr] - ref).max() / sc
    print(f"config-2 slice, un-divided weights (scale 0.1): tcgen05 {e:.2e}  simt {e_s:.2e}  fp32-oracle {floor:.2e}; "
          f"the nets move the final profiles by {float(G['nn_share']):.2e} relative")
    assert float(G["nn_share"]) > 1e-3  # the MLP matters in this case
    assert np.isfinite(got).all()
    assert e <= max(TOL, LONG_FLOOR_FACTOR * floor), (e, floor)
    assert e_s <= max(TOL, LONG_FLOOR_FACTOR * floor), (e_s, floor)


# ---- (d) the other bench.py workloads on slices with the descriptions bench.py builds -----------------------------------
@pytest.mark.parametrize("scale", [1e-5, 0.1])
def test_config4_slice_full_length(ctx, scale):
    """FreeConvectionNDE inference, 1152 steps, save every 9th frame (bench.py 'free_convection')."""
    d = syn.free_convection_desc(ca=False, n_steps=1152, save_stride=9)
    th = syn.theta_init(d, seed=42, scale=scale) if scale < 1e-3 else syn.theta_random(d, scale=scale)
    x0, bcs = syn.columns(d, 300, seed=1000)
    m = engine.Model(ctx, d, th)
    assert "tcgen05" in m.describe()
    got = m.solve(x0, bcs)
    m.close()
    G = golden("fullsize_config4_init" if scale < 1e-3 else "fullsize_config4_random")
    e = np.abs(got[:, G["frames"]] - G["traj"]).max() / float(G["scale"])
    print(f"config-4 slice (scale {scale}): {e:.2e} (fp32-oracle {float(G['floor']):.2e})")
    assert got.shape == (300, 129, 32)
    assert e <= max(TOL, LONG_FLOOR_FACTOR * float(G["floor"]))


def test_config5_slice_bench_description(ctx):
    """The closure call bench.py times (512-wide rows, Nz = 32, theta/1e5 and a theta that matters)."""
    for scale in (1e-5, 0.5):
        d = syn.free_convection_desc(ca=False)
        th = syn.theta_init(d, seed=42, scale=scale) if scale < 1e-3 else syn.theta_random(d, scale=scale)
        nx, ny = 512, 5
        T, y = syn.gyre_field(nx, ny, 32)
        cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
        m = engine.Model(ctx, d, th)
        forcing, T_out = m.closure_step(cd, T, y)
        m.close()
        f_ref, T_ref = nde.closure_step(d, t64(th), cd, t64(T), t64(y))
        e_f, e_T = rel_inf(forcing, f_ref.numpy()), rel_inf(T_out, T_ref.numpy())
        print(f"config-5 slice (scale {scale}): forcing {e_f:.2e}  T {e_T:.2e}")
        assert e_f <= 1e-5 and e_T <= 1e-5
