"""tcgen05 forward path (csrc/cpz_tc.cuh): the production u/v/T nets run their MLP on the 5th-generation tensor cores in
3xTF32. These tests pin (i) that the eligible models really take that kernel, (ii) parity of the tensor-core path with the
FP64 oracle at the north-star tolerances (RHS 1e-5, profiles 1e-4) for several net widths / activations / ragged sizes,
and (iii) agreement with the FP32 SIMT kernel (CPZ_NO_TC=1) on identical inputs."""
import os

import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import FLAG_CA, FLAG_DIURNAL, FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN, NetDesc
from util import assert_blocks, field_blocks, oracle_rhs, oracle_solve, rel_inf

pytestmark = pytest.mark.gpu


def _desc(h1=50, h2=20, act="mish", **kw):
    d = syn.wind_mixing_desc(net=None, **kw)
    d.nets = [NetDesc([96, h1, h2, 31], [act, act, "identity"]) for _ in range(3)]
    return d


class _simt:
    def __enter__(self):
        os.environ["CPZ_NO_TC"] = "1"

    def __exit__(self, *a):
        os.environ.pop("CPZ_NO_TC", None)


def test_production_nets_take_the_tcgen05_kernel(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    m = engine.Model(ctx, d, syn.theta_init(d))
    assert "forward kernel: tcgen05" in m.describe(), m.describe()
    with _simt():
        assert "forward kernel: fp32-simt" in m.describe()
    m.close()
    d = syn.wind_mixing_desc(variant=RHS_INFER, net="uvT_large")
    m = engine.Model(ctx, d, syn.theta_init(d))
    assert "forward kernel: fp32-simt" in m.describe()
    m.close()


@pytest.mark.parametrize("h1,h2,act", [(50, 20, "mish"), (50, 20, "relu"), (32, 16, "tanh"), (53, 32, "swish"),
                                       (42, 8, "leakyrelu"), (20, 28, "mish"), (8, 4, "relu")])
@pytest.mark.parametrize("variant", [RHS_TRAIN, RHS_INFER])
def test_tc_rhs_parity_net_shapes(ctx, h1, h2, act, variant):
    d = _desc(h1, h2, act, variant=variant)
    th = syn.theta_random(d, scale=1.0)
    x, bcs = syn.columns(d, 70)
    m = engine.Model(ctx, d, th)
    assert "forward kernel: tcgen05" in m.describe()
    got = m.rhs(x, bcs, t=0.37)
    with _simt():
        simt = m.rhs(x, bcs, t=0.37)
    m.close()
    ref = oracle_rhs(d, th, x, bcs, 0.37)
    e_tc, e_simt = rel_inf(got, ref), rel_inf(simt, ref)
    print(f"rhs h1={h1} h2={h2} {act} variant={variant}: tcgen05 {e_tc:.2e}  simt {e_simt:.2e}  tc-vs-simt {rel_inf(got, simt):.2e}")
    assert np.isfinite(got).all()
    assert e_tc <= 1e-5, (e_tc, e_simt)
    assert_blocks("tcgen05 rhs", got, ref, oracle_rhs(d, th, x, bcs, 0.37, dtype=torch.float32), field_blocks(d), 1e-5)


@pytest.mark.parametrize("flags,variant", [(FLAG_MPP | FLAG_ZERO_WEIGHTS, RHS_TRAIN), (FLAG_MPP, RHS_TRAIN), (FLAG_CA, RHS_TRAIN),
                                           (0, RHS_TRAIN), (FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, RHS_TRAIN),
                                           (FLAG_MPP | FLAG_CA, RHS_INFER), (FLAG_DIURNAL, RHS_INFER)])
def test_tc_rhs_flags(ctx, flags, variant):
    d = syn.wind_mixing_desc(variant=variant, flags=flags)
    th = syn.theta_random(d, scale=1.0)
    x, bcs = syn.columns(d, 45)
    Q = syn.diurnal_Q(45) if flags & FLAG_DIURNAL else None
    m = engine.Model(ctx, d, th)
    assert "forward kernel: tcgen05" in m.describe()
    got = m.rhs(x, bcs, t=0.21, Q=Q)
    m.close()
    ref = oracle_rhs(d, th, x, bcs, 0.21, Q)
    assert rel_inf(got, ref) <= 1e-5, rel_inf(got, ref)
    assert_blocks("tcgen05 rhs", got, ref, oracle_rhs(d, th, x, bcs, 0.21, Q, dtype=torch.float32), field_blocks(d), 1e-5)


@pytest.mark.parametrize("ncol", [1, 7, 16, 17, 32, 33, 100, 4096 + 5])
def test_tc_rhs_ragged_column_counts(ctx, ncol):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=1.0)
    x, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    got = m.rhs(x, bcs, t=0.0)
    m.close()
    ref = oracle_rhs(d, th, x, bcs, 0.0)
    assert got.shape == ref.shape and rel_inf(got, ref) <= 1e-5
    assert_blocks("tcgen05 rhs", got, ref, oracle_rhs(d, th, x, bcs, 0.0, dtype=torch.float32), field_blocks(d), 1e-5)


@pytest.mark.parametrize("integrator", ["euler", "rk4", "tsit5"])
def test_tc_solve_parity_and_agreement_with_simt(ctx, integrator):
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=48, save_stride=4, integrator=integrator)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, 45)
    m = engine.Model(ctx, d, th)
    got = m.solve(x0, bcs)
    with _simt():
        simt = m.solve(x0, bcs)
    m.close()
    ref = oracle_solve(d, th, x0, bcs)
    ref32 = oracle_solve(d, th, x0, bcs, dtype=torch.float32)
    e_tc, e_simt, floor = rel_inf(got, ref), rel_inf(simt, ref), rel_inf(ref32, ref)
    print(f"solve {integrator}: tcgen05 {e_tc:.2e}  simt {e_simt:.2e}  fp32-oracle {floor:.2e}")
    np.testing.assert_array_equal(got[:, 0], x0)
    assert e_tc <= 1e-4, (e_tc, e_simt, floor)
    assert_blocks("tcgen05 solve", got, ref, ref32, field_blocks(d), 1e-4)


def test_tc_solve_sharding_invariant_bitwise(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=16, save_stride=4)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, 96)
    m = engine.Model(ctx, d, th)
    full = m.solve(x0, bcs)
    a = m.solve(x0[:37], bcs[:37])
    b = m.solve(x0[37:], bcs[37:])
    m.close()
    np.testing.assert_array_equal(full, np.concatenate([a, b]))


@pytest.mark.parametrize("net", ["uvT_small", "uvT_test"])
def test_host_solve_chunked_pipeline_matches_single_launch(ctx, net):
    """cpz_solve cuts long solves into time chunks so the D2H of finished frames overlaps the next chunk's kernel
    (trajectories >= 64 MB); the chunked result must be bitwise the single-launch result (both forward kernels)."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, net=net, n_steps=96, save_stride=1)
    th = syn.theta_random(d, scale=0.3)
    ncol = 2048 + 7
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    pinned = torch.empty((ncol, d.n_saved, d.S), dtype=torch.float32).pin_memory()  # chunking needs a page-locked destination
    host = m.solve(x0, bcs, out=pinned.numpy())   # 2055 x 97 x 96 floats = 76.5 MB -> chunked
    pageable = m.solve(x0, bcs)                   # pageable destination: single launch + one copy
    np.testing.assert_array_equal(host, pageable)
    x0d, bcsd = torch.tensor(x0, device="cuda"), torch.tensor(bcs, device="cuda")
    traj = torch.empty((ncol, d.n_saved, d.S), device="cuda")
    m.solve_dev(x0d, bcsd, traj)
    ctx.synchronize()
    m.close()
    np.testing.assert_array_equal(host, traj.cpu().numpy())
    np.testing.assert_array_equal(host[:, 0], x0)


@pytest.mark.parametrize("ncol", [1, 127, 128, 129, 300])
@pytest.mark.parametrize("ca", [False, True])
def test_fc_tcgen05_solve_ragged_sizes_and_simt_agreement(ctx, ncol, ca):
    """T-only free-convection nets run on the tcgen05 kernel with the columns on the M side (128-column tiles)."""
    d = syn.free_convection_desc(ca=ca, n_steps=27, save_stride=9)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    assert "forward kernel: tcgen05" in m.describe(), m.describe()
    got = m.solve(x0, bcs)
    dx = m.rhs(x0, bcs, t=0.0)
    with _simt():
        simt = m.solve(x0, bcs)
    m.close()
    ref = oracle_solve(d, th, x0, bcs)
    e_tc, e_simt = rel_inf(got, ref), rel_inf(simt, ref)
    e_rhs = rel_inf(dx, oracle_rhs(d, th, x0, bcs, 0.0))
    print(f"fc ncol={ncol} ca={ca}: tcgen05 solve {e_tc:.2e} (simt {e_simt:.2e})  rhs {e_rhs:.2e}")
    np.testing.assert_array_equal(got[:, 0], x0)
    assert e_rhs <= 1e-5 and e_tc <= 1e-4


@pytest.mark.parametrize("h1,h2,act", [(128, 128, "mish"), (40, 72, "tanh"), (16, 16, "relu")])
def test_fc_tcgen05_net_shapes(ctx, h1, h2, act):
    d = syn.free_convection_desc(ca=True, n_steps=18, save_stride=9, net=None)
    d.nets = [NetDesc([32, h1, h2, 31], [act, act, "identity"])]
    th = syn.theta_random(d, scale=0.5)
    x0, bcs = syn.columns(d, 200)
    m = engine.Model(ctx, d, th)
    assert "forward kernel: tcgen05" in m.describe()
    got = m.solve(x0, bcs)
    m.close()
    assert rel_inf(got, oracle_solve(d, th, x0, bcs)) <= 1e-4


def test_fc_host_solve_chunked_pipeline_matches_single_launch(ctx):
    """The time-chunked host solve (>= 64 MB of trajectory) restarts the T-only tcgen05 kernel from trajectory frames."""
    d = syn.free_convection_desc(ca=True, n_steps=72, save_stride=1)
    th = syn.theta_random(d, scale=0.3)
    ncol = 8192 + 5
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    pinned = torch.empty((ncol, d.n_saved, d.S), dtype=torch.float32).pin_memory()
    host = m.solve(x0, bcs, out=pinned.numpy())   # 8197 x 73 x 32 floats = 76.6 MB -> chunked
    x0d, bcsd = torch.tensor(x0, device="cuda"), torch.tensor(bcs, device="cuda")
    traj = torch.empty((ncol, d.n_saved, d.S), device="cuda")
    m.solve_dev(x0d, bcsd, traj)
    ctx.synchronize()
    m.close()
    np.testing.assert_array_equal(host, traj.cpu().numpy())


def test_host_solve_chunked_diurnal_bitwise_and_validation(ctx):
    """The chunked host solve passes a step offset to the kernels (stage times are not re-rounded per chunk), so a
    time-dependent (diurnal) model gives bitwise the single-launch trajectory; a missing diurnal_Q is refused whatever
    the trajectory size (ADVICE r01)."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=96, save_stride=1)
    th = syn.theta_random(d, scale=0.3)
    ncol = 2048 + 3
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol)
    m = engine.Model(ctx, d, th)
    pinned = torch.empty((ncol, d.n_saved, d.S), dtype=torch.float32).pin_memory()
    host = m.solve(x0, bcs, Q=Q, out=pinned.numpy())
    x0d, bcsd, Qd = torch.tensor(x0, device="cuda"), torch.tensor(bcs, device="cuda"), torch.tensor(Q, device="cuda")
    traj = torch.empty((ncol, d.n_saved, d.S), device="cuda")
    m.solve_dev(x0d, bcsd, traj, Q=Qd)
    ctx.synchronize()
    np.testing.assert_array_equal(host, traj.cpu().numpy())
    with pytest.raises(engine.CpzError):
        m.solve(x0, bcs, out=pinned.numpy())   # large trajectory, no Q
    with pytest.raises(engine.CpzError):
        m.solve(x0[:4], bcs[:4])               # small trajectory, no Q
    m.close()
