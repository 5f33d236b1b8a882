"""S1 pullback: cpz_rhs_vjp (x_bar, theta_bar, mpp_bar of one RHS evaluation over a batch of columns), CUDA through the
C ABI vs torch.autograd of the FP64 oracle (oracle/nde.py: rhs). The same autograd in FP32 gives the noise floor, printed
next to every error. Tolerance (gradient rule): relative inf-norm err <= max(1e-4, FP32-oracle error)."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import (FLAG_CA, FLAG_DIURNAL, FLAG_IMPLICIT_DIFFUSION as IMP, FLAG_MPP, FLAG_SMOOTH_RI,
                           FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN)
from oracle import nde
from test_rhs_gpu import UVT_CASES
from util import (assert_blocks, field_blocks, fp32_spread, mpp_blocks, mpp_scale, oracle_loss_grad, oracle_solve, rel_inf,
                  theta_blocks, ulp_nudge)

pytestmark = pytest.mark.gpu
TOL = 1e-4


def mpp_allowed(d):
    """Where cpz_loss_grad_mpp (and so cpz_rhs_vjp) accepts a gradient wrt the five mPP parameters."""
    return d.n_fields == 3 and (d.has(FLAG_MPP) or d.variant == RHS_INFER) and not d.has(FLAG_SMOOTH_RI)


def oracle_rhs_vjp(d, theta, x, bcs, ybar, t=0.0, Q=None, dtype=torch.float64, want_mpp=False):
    """(x_bar [ncol, S], theta_bar [P], mpp_bar [5] or None): torch.autograd.grad of nde.rhs with cotangent ybar. theta and
    p = (nu0, nu_m, dRi, Ric, Pr) are leaves; an input f does not depend on (implicit diffusion: p) gets a zero cotangent."""
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    xt = conv(x).requires_grad_(True)
    th = conv(theta).requires_grad_(True)
    p = None
    if want_mpp:
        p = torch.tensor([float(np.float32(v)) for v in (d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr)], dtype=dtype, requires_grad=True)
    f = nde.rhs(d, th, xt, conv(bcs), t, None if Q is None else conv(Q), p_mpp=p)
    leaves = [xt, th] + ([p] if p is not None else [])
    g = torch.autograd.grad(f, leaves, grad_outputs=conv(ybar), allow_unused=True)
    g = [torch.zeros_like(l) if gi is None else gi for gi, l in zip(g, leaves)]
    return g[0].detach().numpy(), g[1].detach().numpy(), (g[2].detach().numpy() if p is not None else None)


def ybar_of(d, ncol, seed=77):
    return np.random.default_rng(seed).standard_normal((ncol, d.S)).astype(np.float32)


def _check(ctx, d, theta, ncol, t=0.37, use_q=False, seed=1000, want_mpp=None, label=""):
    """Runs the pullback on the GPU and compares every requested output with the FP64 oracle; returns the outputs."""
    x, bcs = syn.columns(d, ncol, seed=seed)
    Q = syn.diurnal_Q(ncol) if use_q else None
    yb = ybar_of(d, ncol)
    want_mpp = mpp_allowed(d) if want_mpp is None else want_mpp
    want_theta = theta.size > 0
    m = engine.Model(ctx, d, theta)
    xb, tb, pb = m.rhs_vjp(x, bcs, yb, t=t, Q=Q, want_theta=want_theta, want_mpp=want_mpp)
    m.close()
    ref = oracle_rhs_vjp(d, theta, x, bcs, yb, t, Q, want_mpp=want_mpp)
    ref32 = oracle_rhs_vjp(d, theta, x, bcs, yb, t, Q, dtype=torch.float32, want_mpp=want_mpp)
    msg = [f"rhs_vjp {label} variant={d.variant} flags={d.flags} ncol={ncol}:"]
    for name, got, r, r32 in (("x_bar", xb, ref[0], ref32[0]), ("theta_bar", tb, ref[1], ref32[1]), ("mpp_bar", pb, ref[2], ref32[2])):
        if got is None:
            continue
        assert np.isfinite(got).all(), name
        err, floor = rel_inf(got, r), rel_inf(r32, r)
        msg.append(f"{name} {err:.2e} (fp32-oracle {floor:.2e})")
        assert err <= max(TOL, floor), (name, err, floor)
    print("  ".join(msg))
    spread = fp32_spread(lambda s: oracle_rhs_vjp(d, theta, ulp_nudge(x, s), bcs, yb, t, Q, dtype=torch.float32, want_mpp=want_mpp))
    assert_blocks("x_bar", xb, ref[0], ref32[0], field_blocks(d), TOL, spread=lambda: [r[0] for r in spread()])
    if tb is not None:
        assert_blocks("theta_bar", tb, ref[1], ref32[1], theta_blocks(d), TOL, norm="l2", spread=lambda: [r[1] for r in spread()])
    if pb is not None:
        p = mpp_scale(d)
        assert_blocks("mpp_bar", pb * p, ref[2] * p, ref32[2] * p, mpp_blocks(), TOL, spread=lambda: [r[2] * p for r in spread()])
    return xb, tb, pb


# ---- 1. every (variant, flags) pair of the RHS parity test, small nets, random theta; diurnal forcing at two times
@pytest.mark.parametrize("variant,flags", UVT_CASES)
def test_rhs_vjp_uvt_small_net(ctx, variant, flags):
    d = syn.wind_mixing_desc(variant=variant, flags=flags, net="uvT_small")
    th = syn.theta_random(d, scale=1.0)
    for t in ((0.37, 2.9) if flags & FLAG_DIURNAL else (0.37,)):
        _check(ctx, d, th, 70, t=t, use_q=bool(flags & FLAG_DIURNAL), label=f"t={t}")


# ---- 2. the reference initial weights
def test_rhs_vjp_reference_initial_weights(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN)
    _check(ctx, d, syn.theta_init(d), 64)


# ---- 3. ragged and large batches (5 000 columns: some persistent CTAs take two tiles)
@pytest.mark.parametrize("ncol", [1, 3, 31, 32, 33, 257, 5000])
def test_rhs_vjp_ragged_column_counts(ctx, ncol):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    _check(ctx, d, syn.theta_random(d, scale=1.0), ncol)


# ---- 4. every activation; weights streamed from global memory. The adjoint plan keeps a and z of every layer of the three
# nets for 32 columns in shared memory, so the u/v/T hidden width is bounded (about 170 with one hidden layer): the
# activation nets are the test nets' shape at width 40 (weights in shared memory), the streamed case is width 128.
@pytest.mark.parametrize("act", ["relu", "mish", "swish", "leakyrelu", "tanh"])
def test_rhs_vjp_uvt_activations(ctx, act):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    d.nets = [syn.NetDesc([d.S, 40, d.Nz - 1], [act, "identity"]) for _ in range(3)]
    _check(ctx, d, syn.theta_random(d, scale=1.0), 40)


@pytest.mark.parametrize("variant", [RHS_TRAIN, RHS_INFER])
def test_rhs_vjp_uvt_streamed_weights(ctx, variant):
    d = syn.wind_mixing_desc(variant=variant, net=None)
    d.nets = [syn.NetDesc([d.S, 128, d.Nz - 1], ["relu", "identity"]) for _ in range(3)]
    th = syn.theta_random(d, scale=1.0)
    m = engine.Model(ctx, d, th)
    assert "weights streamed from global memory" in m.describe()
    m.close()
    _check(ctx, d, th, 40)


# ---- 5. the NN-free `DE` model: x_bar and mpp_bar; theta_bar is refused
def test_rhs_vjp_nn_free_DE(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    th = np.zeros(0, dtype=np.float32)
    _check(ctx, d, th, 48, want_mpp=True)
    x, bcs = syn.columns(d, 8)
    m = engine.Model(ctx, d, th)
    with pytest.raises(engine.CpzError) as ei:
        m.rhs_vjp(x, bcs, ybar_of(d, 8), want_theta=True)
    assert ei.value.code == -1 and "no parameters" in str(ei.value)
    m.close()


# ---- 6. T-only models, other Nz
@pytest.mark.parametrize("ca,mpp", [(False, False), (True, False), (True, True)])
def test_rhs_vjp_free_convection(ctx, ca, mpp):
    d = syn.free_convection_desc(ca=ca, mpp=mpp)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 50)


def test_rhs_vjp_other_Nz(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, Nz=16)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 20)
    d = syn.free_convection_desc(ca=True, Nz=64)
    _check(ctx, d, syn.theta_random(d, scale=1.0), 20)


# ---- 7. implicit diffusion: the pullback of the explicit part cpz_rhs returns; mpp_bar is exactly 0
@pytest.mark.parametrize("model", ["uvT", "T_only"])
def test_rhs_vjp_implicit_diffusion(ctx, model):
    if model == "uvT":
        d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA | IMP, n_substeps=1)
    else:
        d = syn.free_convection_desc(ca=True, mpp=True, n_substeps=1)
        d.flags |= IMP
    _, _, pb = _check(ctx, d, syn.theta_random(d, scale=1.0), 70)
    if model == "uvT":
        assert pb is not None and (pb == 0).all(), pb


# ---- 8. batch invariance
def test_rhs_vjp_batch_invariance(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA)
    th = syn.theta_random(d, scale=1.0)
    ncol = 300
    x, bcs = syn.columns(d, ncol)
    yb = ybar_of(d, ncol)
    m = engine.Model(ctx, d, th)
    xb, tb, _ = m.rhs_vjp(x, bcs, yb)
    xb2, tb2, _ = m.rhs_vjp(x, bcs, yb)
    assert np.array_equal(tb, tb2)  # fixed-order reductions: bitwise reproducible
    assert np.array_equal(xb, xb2)
    cuts = [0, 1, 33, 64, 190, 300]
    parts = [m.rhs_vjp(x[a:b], bcs[a:b], yb[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
    m.close()
    assert np.array_equal(np.concatenate([p[0] for p in parts]), xb)
    tsum = np.sum([p[1].astype(np.float64) for p in parts], axis=0)
    e = rel_inf(tb, tsum)
    print(f"rhs_vjp batch invariance: theta_bar vs sum over {len(parts)} shards {e:.2e}")
    assert e <= 1e-6, e


# ---- 9. device flavour on torch CUDA tensors: bitwise the host flavour; every output subset
def test_rhs_vjp_dev_matches_host(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL)
    th = syn.theta_random(d, scale=1.0)
    ncol = 45
    x, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol)
    yb = ybar_of(d, ncol)
    m = engine.Model(ctx, d, th)
    xb, tb, pb = m.rhs_vjp(x, bcs, yb, t=0.6, Q=Q, want_mpp=True)
    dev = torch.device("cuda:0")
    xt, bt, qt, yt = (torch.from_numpy(a).to(dev) for a in (x, bcs, Q, yb))

    def run(want_x, want_theta, want_mpp):
        outs = [torch.full((ncol, d.S), float("nan"), device=dev) if want_x else None,
                torch.full((m.P,), float("nan"), device=dev) if want_theta else None,
                torch.full((5,), float("nan"), device=dev) if want_mpp else None]
        torch.cuda.synchronize()  # the fills run on torch's stream, the pullback on the context's
        m.rhs_vjp_dev(xt, bt, yt, *outs, t=0.6, Q=qt)
        ctx.synchronize()
        return [None if o is None else o.cpu().numpy() for o in outs]

    got = run(True, True, True)
    assert np.array_equal(got[0], xb) and np.array_equal(got[1], tb) and np.array_equal(got[2], pb)
    for want in ((True, False, False), (False, True, False), (False, False, True)):
        sub = run(*want)
        for w, g, h in zip(want, sub, (xb, tb, pb)):
            if w:
                assert np.array_equal(g, h), want
    # outputs are overwritten, not accumulated
    again = m.rhs_vjp(x, bcs, yb, t=0.6, Q=Q, want_mpp=True)
    assert all(np.array_equal(a, b) for a, b in zip(again, (xb, tb, pb)))
    m.close()


# ---- 10. consistency with the discrete adjoint of one explicit Euler step
def test_rhs_vjp_consistent_with_one_step_adjoint(ctx):
    """loss(x1), x1 = x0 + h f(x0): d loss/d theta = h (df/dtheta)^T ybar with ybar = d loss/d x1."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, integrator="euler", n_steps=1, n_substeps=1, save_stride=0, ckpt_stride=1)
    th = syn.theta_random(d, scale=0.3)
    ncol = 64
    x0, bcs = syn.columns(d, ncol)
    w = np.array([1, 1, 1, 0, 0, 0], dtype=np.float32)
    tgt = oracle_solve(d, th, x0, bcs)
    tgt = (tgt + 0.05 * np.random.default_rng(5).standard_normal(tgt.shape)).astype(np.float32)
    m = engine.Model(ctx, d, th)
    x1 = m.solve(x0, bcs)[:, -1].astype(np.float64)
    _, grad = m.loss_grad(x0, bcs, tgt, w)
    N = d.Nz
    ybar = (2.0 * (x1 - tgt[:, -1]) / (ncol * N)).astype(np.float32)  # each field's loss is a mean over ncol x Nz
    _, tb, _ = m.rhs_vjp(x0, bcs, ybar, t=0.0)
    m.close()
    h = np.float32(d.dt)
    e = rel_inf(h * tb, grad)
    _, _, g64 = oracle_loss_grad(d, th, x0, bcs, tgt, w)
    print(f"rhs_vjp vs one-step adjoint: {e:.2e} (adjoint vs FP64 oracle {rel_inf(grad, g64):.2e})")
    assert e <= 1e-4, e


# ---- 11. argument validation
def test_rhs_vjp_argument_checks(ctx):
    L = engine.lib()
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_SMOOTH_RI | FLAG_DIURNAL)
    th = syn.theta_random(d, scale=1.0)
    ncol = 5
    x, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol)
    yb = ybar_of(d, ncol)
    xb = np.full_like(x, 7.0)
    tb = np.full(th.size, 7.0, dtype=np.float32)
    pb = np.full(5, 7.0, dtype=np.float32)
    m = engine.Model(ctx, d, th)
    P = engine._ptr

    def call(x_=x, Q_=Q, y_=yb, xb_=xb, tb_=tb, pb_=pb, n=ncol):
        return L.cpz_rhs_vjp(m._h, P(x_), P(bcs), P(Q_), 0.0, P(y_), P(xb_), P(tb_), P(pb_), n)

    def rejected(rc, words):
        msg = L.cpz_last_error().decode()
        assert rc == -1 and words in msg, (rc, msg)

    rejected(call(y_=None, pb_=None), "null array")
    rejected(call(Q_=None, pb_=None), "diurnal_Q")
    rejected(call(xb_=None, tb_=None, pb_=None), "no output")
    rejected(call(), "smooth_Ri")  # mpp_bar where cpz_loss_grad_mpp refuses it
    assert call(n=0) == 0 and (xb == 7).all() and (tb == 7).all() and (pb == 7).all()  # ncol = 0: a no-op
    assert call(pb_=None) == 0 and np.isfinite(xb).all() and not (tb == 7).any()
    m.close()
    # mpp_bar: needs the u/v/T model and the mPP closure
    for d2 in (syn.free_convection_desc(ca=True, mpp=True), syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_CA)):
        th2 = syn.theta_random(d2, scale=1.0)
        x2, b2 = syn.columns(d2, 3)
        m2 = engine.Model(ctx, d2, th2)
        with pytest.raises(engine.CpzError) as ei:
            m2.rhs_vjp(x2, b2, ybar_of(d2, 3), want_mpp=True)
        assert ei.value.code == -1 and "mPP-parameter gradient" in str(ei.value)
        m2.close()


def test_rhs_vjp_needs_the_adjoint_plan(ctx):
    """The large u/v/T nets (construct_NN.jl:32-34) have cpz_rhs but no 32-column adjoint plan: the pullback is refused
    with the planner's reason."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, net="uvT_large")
    m = engine.Model(ctx, d, syn.theta_random(d, scale=0.1))
    assert "adjoint plan: unavailable" in m.describe()
    x, bcs = syn.columns(d, 2)
    assert np.isfinite(m.rhs(x, bcs)).all()
    with pytest.raises(engine.CpzError) as ei:
        m.rhs_vjp(x, bcs, ybar_of(d, 2))
    assert ei.value.code == -1 and "adjoint plan unavailable" in str(ei.value)
    m.close()
