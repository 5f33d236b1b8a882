"""S1 pushforward: cpz_rhs_jvp (dxdt_dot = J x_dot + (df/dtheta) theta_dot + (df/dp) mpp_dot for every column), CUDA through
the C ABI vs torch.func.jvp of the FP64 oracle (oracle/nde.py: rhs). The same jvp in FP32 gives the noise floor, printed next
to every error. Tolerance: relative inf-norm error <= max(1e-5, FP32-oracle error), on the case matrix of test_rhs_vjp_gpu.py."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import (FLAG_CA, FLAG_DIURNAL, FLAG_IMPLICIT_DIFFUSION as IMP, FLAG_MPP, FLAG_SMOOTH_NN, FLAG_SMOOTH_RI,
                           FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN)
from oracle import nde
from test_jvp_oracle_cpu import oracle_rhs_jvp, p_of, tangents_of
from test_rhs_gpu import UVT_CASES
from test_rhs_vjp_gpu import ybar_of
from util import assert_blocks, field_blocks, rel_inf

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _check(ctx, d, theta, ncol, t=0.37, use_q=False, seed=1000, label=""):
    """Runs the pushforward with x_dot only, theta_dot only, mpp_dot only and all of them; compares with the FP64 oracle. The
    primal dxdt is compared with cpz_rhs."""
    x, bcs = syn.columns(d, ncol, seed=seed)
    Q = syn.diurnal_Q(ncol) if use_q else None
    xd, thd, pd = tangents_of(d, ncol)
    m = engine.Model(ctx, d, theta)
    f_ref = m.rhs(x, bcs, t=t, Q=Q)
    msg = [f"rhs_jvp {label} variant={d.variant} flags={d.flags} ncol={ncol}:"]
    combos = [("x", (xd, None, None))]
    if thd is not None:
        combos.append(("theta", (None, thd, None)))
    if pd is not None:
        combos.append(("p", (None, None, pd)))
    if len(combos) > 1:
        combos.append(("all", (xd, thd, pd)))
    for name, tans in combos:
        f, fd = m.rhs_jvp(x, bcs, *tans, t=t, Q=Q)
        assert np.isfinite(fd).all(), name
        e_f = rel_inf(f, f_ref)
        assert e_f <= 1e-5, (name, e_f)
        _, r = oracle_rhs_jvp(d, theta, x, bcs, *tans, t=t, Q=Q)
        _, r32 = oracle_rhs_jvp(d, theta, x, bcs, *tans, t=t, Q=Q, dtype=torch.float32)
        err, floor = rel_inf(fd, r), rel_inf(r32, r)
        msg.append(f"{name} {err:.2e} (fp32-oracle {floor:.2e})")
        assert err <= max(TOL, floor), (name, err, floor)
        assert_blocks(f"{name} tangent", fd, r, r32, field_blocks(d), TOL)
    m.close()
    print("  ".join(msg))


@pytest.mark.parametrize("variant,flags", UVT_CASES)
def test_rhs_jvp_uvt_small_net(ctx, variant, flags):
    d = syn.wind_mixing_desc(variant=variant, flags=flags, net="uvT_small")
    th = syn.theta_random(d, scale=1.0)
    for t in ((0.37, 2.9) if flags & FLAG_DIURNAL else (0.37,)):
        _check(ctx, d, th, 70, t=t, use_q=bool(flags & FLAG_DIURNAL), label=f"t={t}")


def test_rhs_jvp_reference_initial_weights(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN)
    _check(ctx, d, syn.theta_init(d), 64)


@pytest.mark.parametrize("ncol", [1, 3, 31, 32, 33, 257, 5000])
def test_rhs_jvp_ragged_column_counts(ctx, ncol):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    _check(ctx, d, syn.theta_random(d, scale=1.0), ncol)


@pytest.mark.parametrize("act", ["relu", "mish", "swish", "leakyrelu", "tanh"])
def test_rhs_jvp_uvt_activations(ctx, act):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    d.nets = [syn.NetDesc([d.S, 40, d.Nz - 1], [act, "identity"]) for _ in range(3)]
    _check(ctx, d, syn.theta_random(d, scale=1.0), 40)


@pytest.mark.parametrize("variant", [RHS_TRAIN, RHS_INFER])
def test_rhs_jvp_uvt_streamed_weights(ctx, variant):
    d = syn.wind_mixing_desc(variant=variant, net=None)
    d.nets = [syn.NetDesc([d.S, 128, d.Nz - 1], ["relu", "identity"]) for _ in range(3)]
    th = syn.theta_random(d, scale=1.0)
    m = engine.Model(ctx, d, th)
    assert "weights streamed from global memory" in m.describe()
    m.close()
    _check(ctx, d, th, 40)


def test_rhs_jvp_nn_free_DE(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP, net=None)
    _check(ctx, d, np.zeros(0, dtype=np.float32), 48)


@pytest.mark.parametrize("ca,mpp", [(False, False), (True, False), (True, True)])
def test_rhs_jvp_free_convection(ctx, ca, mpp):
    d = syn.free_convection_desc(ca=ca, mpp=mpp)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 50)


def test_rhs_jvp_other_Nz(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, Nz=16)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 20)
    d = syn.free_convection_desc(ca=True, Nz=64)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 20)


@pytest.mark.parametrize("model", ["uvT", "T_only"])
def test_rhs_jvp_implicit_diffusion(ctx, model):
    """The tangent of the explicit part cpz_rhs returns; the mpp tangent contributes exactly 0."""
    if model == "uvT":
        d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA | IMP, n_substeps=1)
    else:
        d = syn.free_convection_desc(ca=True, mpp=True, n_substeps=1)
        d.flags |= IMP
    th = syn.theta_random(d, scale=1.0)
    _check(ctx, d, th, 70)
    if model == "uvT":
        x, bcs = syn.columns(d, 9)
        m = engine.Model(ctx, d, th)
        _, fd = m.rhs_jvp(x, bcs, mpp_dot=np.ones(5, dtype=np.float32), want_dxdt=False)
        m.close()
        assert not fd.any()


# ---- the dense per-column Jacobian from S replicated columns with unit tangents, against torch.func.jacfwd of the oracle
@pytest.mark.parametrize("model", ["uvT_mpp", "T_only_ca"])
def test_rhs_jvp_dense_jacobian(ctx, model):
    d = (syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA) if model == "uvT_mpp"
         else syn.free_convection_desc(ca=True, mpp=True))
    th = syn.theta_random(d, scale=1.0)
    x, bcs = syn.columns(d, 3)
    S = d.S
    m = engine.Model(ctx, d, th)
    xr, br = np.repeat(x, S, axis=0), np.repeat(bcs, S, axis=0)
    eye = np.tile(np.eye(S, dtype=np.float32), (3, 1))
    _, J = m.rhs_jvp(xr, br, x_dot=eye, want_dxdt=False)
    m.close()
    J = J.reshape(3, S, S).transpose(0, 2, 1)  # [column][output][input]
    for c in range(3):
        def f(xc, dtype):
            return nde.rhs(d, torch.tensor(th, dtype=dtype), xc[None], torch.tensor(bcs[c:c + 1], dtype=dtype), 0.0)[0]
        ref = torch.func.jacfwd(lambda v: f(v, torch.float64))(torch.tensor(x[c], dtype=torch.float64)).numpy()
        r32 = torch.func.jacfwd(lambda v: f(v, torch.float32))(torch.tensor(x[c], dtype=torch.float32)).numpy()
        err, floor = rel_inf(J[c], ref), rel_inf(r32, ref)
        print(f"rhs_jvp dense Jacobian {model} column {c}: {err:.2e} (fp32-oracle {floor:.2e})")
        assert err <= max(TOL, floor), (c, err, floor)


# ---- duality with the pullback: <J v, w> = <v, J^T w>
@pytest.mark.parametrize("model", ["uvT_mpp", "uvT_smooth", "T_only_ca"])
def test_rhs_jvp_dot_product_with_rhs_vjp(ctx, model):
    if model == "uvT_mpp":
        d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS)
    elif model == "uvT_smooth":
        d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_SMOOTH_RI | FLAG_SMOOTH_NN)
    else:
        d = syn.free_convection_desc(ca=True, mpp=True)
    th = syn.theta_random(d, scale=1.0)
    ncol = 100
    x, bcs = syn.columns(d, ncol)
    xd, thd, pd = tangents_of(d, ncol)
    m = engine.Model(ctx, d, th)
    _, fd = m.rhs_jvp(x, bcs, xd, thd, pd, want_dxdt=False)
    w = ybar_of(d, ncol)
    xb, tb, pb = m.rhs_vjp(x, bcs, w, want_mpp=pd is not None)
    m.close()
    lhs = float(np.sum(fd.astype(np.float64) * w))
    rhs = float(np.sum(xb.astype(np.float64) * xd) + np.sum(tb.astype(np.float64) * thd)
                + (np.sum(pb.astype(np.float64) * pd) if pd is not None else 0.0))
    e = abs(lhs - rhs) / (np.linalg.norm(fd) * np.linalg.norm(w))
    print(f"rhs_jvp duality {model}: {lhs:.6e} vs {rhs:.6e}, {e:.2e} of |Jv||w|")
    assert e <= 1e-5, e


# ---- batch invariance: a column's tangent is bitwise independent of the batch it is in
def test_rhs_jvp_batch_invariance(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA)
    th = syn.theta_random(d, scale=1.0)
    ncol = 300
    x, bcs = syn.columns(d, ncol)
    xd, thd, pd = tangents_of(d, ncol)
    m = engine.Model(ctx, d, th)
    f, fd = m.rhs_jvp(x, bcs, xd, thd, pd)
    cuts = [0, 1, 33, 64, 190, 300]
    parts = [m.rhs_jvp(x[a:b], bcs[a:b], xd[a:b], thd, pd) for a, b in zip(cuts[:-1], cuts[1:])]
    m.close()
    assert np.array_equal(np.concatenate([p[1] for p in parts]), fd)
    assert np.array_equal(np.concatenate([p[0] for p in parts]), f)


# ---- device flavour on torch CUDA tensors: bitwise the host flavour
def test_rhs_jvp_dev_matches_host(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL)
    th = syn.theta_random(d, scale=1.0)
    ncol = 45
    x, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol)
    xd, thd, pd = tangents_of(d, ncol)
    m = engine.Model(ctx, d, th)
    f, fd = m.rhs_jvp(x, bcs, xd, thd, pd, t=0.6, Q=Q)
    dev = torch.device("cuda:0")
    xt, bt, qt, xdt, tdt, pdt = (torch.from_numpy(a).to(dev) for a in (x, bcs, Q, xd, thd, pd))
    outs = [torch.full((ncol, d.S), float("nan"), device=dev) for _ in range(2)]
    torch.cuda.synchronize()
    m.rhs_jvp_dev(xt, bt, outs[1], x_dot=xdt, theta_dot=tdt, mpp_dot=pdt, dxdt=outs[0], t=0.6, Q=qt)
    ctx.synchronize()
    assert np.array_equal(outs[0].cpu().numpy(), f) and np.array_equal(outs[1].cpu().numpy(), fd)
    assert np.array_equal(m.get_theta(), th) and np.array_equal(m.mpp_params(), p_of(d, torch.float32).numpy())
    m.close()


# ---- argument validation
def test_rhs_jvp_argument_checks(ctx):
    L = engine.lib()
    P = engine._ptr
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_SMOOTH_RI | FLAG_DIURNAL)
    th = syn.theta_random(d, scale=1.0)
    ncol = 5
    x, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol)
    xd, thd, _ = tangents_of(d, ncol)
    pd = np.ones(5, dtype=np.float32)
    out = np.full_like(x, 7.0)
    m = engine.Model(ctx, d, th)

    def call(x_=x, Q_=Q, xd_=xd, td_=thd, pd_=None, y_=out, n=ncol, h=m._h):
        return L.cpz_rhs_jvp(h, P(x_), P(bcs), P(Q_), 0.0, P(xd_), P(td_), P(pd_), None, P(y_), n)

    def rejected(rc, words):
        msg = L.cpz_last_error().decode()
        assert rc == -1 and words in msg, (rc, msg)

    rejected(call(x_=None), "null array")
    rejected(call(y_=None), "null array")
    rejected(call(Q_=None), "diurnal_Q")
    rejected(call(xd_=None, td_=None), "no tangent")
    rejected(call(pd_=pd), "smooth_Ri")
    rejected(call(n=0), "ncol must be positive")
    rejected(call(n=2 ** 40), "ncol too large")
    assert (out == 7).all()
    assert call() == 0 and np.isfinite(out).all()
    m.close()
    d2 = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None, flags=FLAG_MPP)
    m2 = engine.Model(ctx, d2, np.zeros(0, dtype=np.float32))
    x2, b2 = syn.columns(d2, 3)
    rejected(L.cpz_rhs_jvp(m2._h, P(x2), P(b2), None, 0.0, None, P(np.ones(4, dtype=np.float32)), None, None, P(x2.copy()), 3),
             "no parameters")
    m2.close()
    for d3 in (syn.free_convection_desc(ca=True, mpp=True), syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_CA)):
        m3 = engine.Model(ctx, d3, syn.theta_random(d3, scale=1.0))
        x3, b3 = syn.columns(d3, 3)
        with pytest.raises(engine.CpzError) as ei:
            m3.rhs_jvp(x3, b3, mpp_dot=pd)
        assert ei.value.code == -1 and "mPP-parameter gradient" in str(ei.value)
        m3.close()


def test_rhs_jvp_needs_the_adjoint_plan(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, net="uvT_large")
    m = engine.Model(ctx, d, syn.theta_random(d, scale=0.1))
    x, bcs = syn.columns(d, 2)
    with pytest.raises(engine.CpzError) as ei:
        m.rhs_jvp(x, bcs, x_dot=x)
    assert ei.value.code == -1 and "adjoint plan unavailable" in str(ei.value)
    m.close()
