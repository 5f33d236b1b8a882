"""S2 pushforward: cpz_solve_jvp (the tangent-linear model of the fixed-step solve), CUDA through the C ABI vs torch.func.jvp
of the FP64 oracle (oracle/nde.py: solve), with the FP32 jvp as the noise floor. Tolerance (the rule of test_solve_vjp_gpu.py):
relative L2 error <= max(1e-4, 3 x FP32-oracle error). The factor 3 is the one that file gives its T-only CA and tensor-core
cases, here for every case: the engine evaluates the activations and the Richardson-number step with MUFU intrinsics (about
1e-6 relative); its RHS tangent measured at up to 8.6x the FP32 oracle's error (2.6e-6, test_rhs_jvp_gpu.py), its solve
tangents at up to 1.5x. Each case also checks the dot-product identity
<traj_dot, tbar> = <x0_dot, x0_bar> + <theta_dot, theta_bar> + <mpp_dot, mpp_bar> against cpz_solve_vjp on the adjoint path
the case selects (asserted as in test_solve_vjp_gpu.py): an independent check of each adjoint path, with tbar = traj_dot + noise
so that the inner product is not small, to 1e-4 of |traj_dot| |tbar|. Where the tangent itself moves by more than that under
FP32 rounding of the trajectory (the pullback linearises about its own forward pass), the bound is that sensitivity: the FP32
oracle's tangent error, or at full length the change of the engine's tangent when theta and x0 move by 2 ulp."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn, wind_mixing as wm
from cpz_b200.desc import FLAG_CA, FLAG_DIURNAL, FLAG_MPP, FLAG_SMOOTH_RI, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN
from oracle import nde
from test_batch_schedules_gpu import _env
from test_jvp_oracle_cpu import oracle_solve_jvp, p_of, tangents_of
from test_solve_vjp_gpu import CASES, expected_path, rel_l2
from util import assert_blocks, field_blocks

pytestmark = pytest.mark.gpu
TOL = 1e-4
DUAL_TOL = 1e-4

JVP_CASES = dict(CASES)
JVP_CASES.update({
    "fp32_rk4": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP, n_steps=12, save_stride=4, ckpt_stride=4,
                                              integrator="rk4"), 40, "fp32", {}, True, False),
    "fp32_euler": (lambda: syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=12, save_stride=4, ckpt_stride=4,
                                                integrator="euler"), 40, "fp32", {}, True, False),
    "fc1_config1": (lambda: syn.free_convection_desc(ca=True, mpp=True, n_steps=36, save_stride=9, ckpt_stride=9), 1, "fc1", {}, False, False),
})


def _theta(d):
    return syn.theta_random(d, scale=0.1) if d.n_params > 0 else np.zeros(0, dtype=np.float32)


def _dual(m, x0, bcs, Q, tans, traj_dot, want_mpp, seed=17):
    """(|lhs - rhs| / (|traj_dot| |tbar|), lhs, rhs) of the dot-product identity against cpz_solve_vjp."""
    xd, thd, pd = tans
    tbar = (traj_dot + np.random.default_rng(seed).standard_normal(traj_dot.shape) * np.abs(traj_dot).mean()).astype(np.float32)
    xb, tb, pb = m.solve_vjp(x0, bcs, tbar, Q=Q, want_theta=m.P > 0, want_mpp=want_mpp)
    lhs = float(np.sum(traj_dot.astype(np.float64) * tbar))
    rhs = float(np.sum(xb.astype(np.float64) * xd))
    if tb is not None and thd is not None:
        rhs += float(np.sum(tb.astype(np.float64) * thd))
    if pb is not None and pd is not None:
        rhs += float(np.sum(pb.astype(np.float64) * pd))
    return abs(lhs - rhs) / (np.linalg.norm(traj_dot) * np.linalg.norm(tbar)), lhs, rhs


@pytest.mark.parametrize("case", list(JVP_CASES))
def test_solve_jvp_matches_the_oracle_and_each_adjoint_path(ctx, case):
    mk, ncol, path, env, want_mpp, diurnal = JVP_CASES[case]
    d = mk()
    th = _theta(d)
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol) if diurnal else None
    tans = tangents_of(d, ncol, with_p=want_mpp)
    with _env(**env):
        m = engine.Model(ctx, d, th)
        assert expected_path(m, ncol, want_mpp) == path, m.describe()
        traj, traj_dot = m.solve_jvp(x0, bcs, *tans, Q=Q)
        ref_traj = m.solve(x0, bcs, Q=Q)
        e_dual, lhs, rhs = _dual(m, x0, bcs, Q, tans, traj_dot, want_mpp)
        m.close()
    t64, r = oracle_solve_jvp(d, th, x0, bcs, *tans, Q=Q)
    t32, r32 = oracle_solve_jvp(d, th, x0, bcs, *tans, Q=Q, dtype=torch.float32)
    assert np.isfinite(traj_dot).all() and np.isfinite(traj).all()
    err, floor = rel_l2(traj_dot, r), rel_l2(r32, r)
    e_p, f_p = rel_l2(traj, ref_traj), rel_l2(t32, t64)
    print(f"solve_jvp {case} ({path}) ncol={ncol}: traj_dot {err:.2e} (fp32-oracle {floor:.2e}); traj vs cpz_solve {e_p:.2e} "
          f"(fp32-oracle {f_p:.2e}); duality {e_dual:.2e} ({lhs:.6e} vs {rhs:.6e})")
    assert err <= max(TOL, 3.0 * floor), (err, floor)
    assert_blocks("traj_dot", traj_dot, r, r32, field_blocks(d), TOL, k=3.0)
    assert e_p <= max(TOL, 3.0 * f_p), (e_p, f_p)
    assert e_dual <= max(DUAL_TOL, floor), (e_dual, floor)


@pytest.mark.parametrize("path", ["tc", "fp32"])
def test_solve_jvp_duality_full_length(ctx, path):
    """A config-3 slice (u/v/T nets of train_NDE.jl, training RHS with mPP, 1 152 steps x 2 sub-steps, 129 frames, 64
    columns): the tangent-linear solve against the adjoint of that path."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, save_stride=9, n_substeps=2)
    ncol = 64
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, ncol)
    want_mpp = path == "fp32"
    tans = tangents_of(d, ncol, with_p=want_mpp)
    env = {"CPZ_NO_TC_ADJ": "1"} if path == "fp32" else {}
    with _env(**env):
        m = engine.Model(ctx, d, th)
        assert m.n_saved == 129 and expected_path(m, ncol, want_mpp) == path
        _, traj_dot = m.solve_jvp(x0, bcs, *tans, want_traj=False)
        e, lhs, rhs = _dual(m, x0, bcs, None, tans, traj_dot, want_mpp)
        # sensitivity of the tangent to rounding-level changes of the trajectory: theta and x0 moved by 2 ulp
        rng = np.random.default_rng(9)
        nudge = (lambda a: (a.astype(np.float64) * (1.0 + 2.0 ** -22 * rng.choice([-1.0, 1.0], a.shape))).astype(np.float32))
        m.set_theta(nudge(th))
        _, traj_dot2 = m.solve_jvp(nudge(x0), bcs, *tans, want_traj=False)
        m.close()
    floor = rel_l2(traj_dot2, traj_dot)
    print(f"solve_jvp duality full length ({path}): {lhs:.6e} vs {rhs:.6e}, {e:.2e} of |traj_dot||tbar| (tangent moves by "
          f"{floor:.2e} under 2-ulp changes of theta and x0)")
    assert np.isfinite(traj_dot).all()
    assert e <= max(DUAL_TOL, floor), (e, floor)


def test_solve_jvp_batch_invariance(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=8, save_stride=4, ckpt_stride=4)
    ncol = 160
    th = _theta(d)
    x0, bcs = syn.columns(d, ncol)
    xd, thd, pd = tangents_of(d, ncol)
    m = engine.Model(ctx, d, th)
    traj, td = m.solve_jvp(x0, bcs, xd, thd, pd)
    cuts = [0, 1, 33, 96, 160]
    parts = [m.solve_jvp(x0[a:b], bcs[a:b], xd[a:b], thd, pd) for a, b in zip(cuts[:-1], cuts[1:])]
    m.close()
    assert np.array_equal(np.concatenate([p[1] for p in parts]), td)
    assert np.array_equal(np.concatenate([p[0] for p in parts]), traj)


def test_solve_jvp_dev_matches_host_and_leaves_the_model_alone(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=8, save_stride=4, ckpt_stride=4)
    ncol = 45
    th = _theta(d)
    x0, bcs = syn.columns(d, ncol)
    xd, thd, pd = tangents_of(d, ncol)
    m = engine.Model(ctx, d, th)
    tgt = m.solve(x0, bcs)
    m.train_step(x0, bcs, tgt + 0.01, np.ones(6, dtype=np.float32), 1e-3)  # a non-trivial ADAM state
    theta0, adam0, p0 = m.get_theta(), m.adam_state(), m.mpp_params()
    traj, traj_dot = m.solve_jvp(x0, bcs, xd, thd, pd)
    dev = torch.device("cuda:0")
    xt, bt, xdt, tdt, pdt = (torch.from_numpy(a).to(dev) for a in (x0, bcs, xd, thd, pd))
    outs = [torch.full((ncol, m.n_saved, d.S), float("nan"), device=dev) for _ in range(2)]
    torch.cuda.synchronize()
    m.solve_jvp_dev(xt, bt, outs[1], x0_dot=xdt, theta_dot=tdt, mpp_dot=pdt, traj=outs[0])
    ctx.synchronize()
    assert np.array_equal(outs[0].cpu().numpy(), traj) and np.array_equal(outs[1].cpu().numpy(), traj_dot)
    # outputs are overwritten, not accumulated; theta, the ADAM state and the mPP parameters are untouched
    again = m.solve_jvp(x0, bcs, xd, thd, pd)
    assert np.array_equal(again[0], traj) and np.array_equal(again[1], traj_dot)
    assert np.array_equal(m.get_theta(), theta0) and np.array_equal(m.mpp_params(), p0)
    assert all(np.array_equal(a, b) for a, b in zip(m.adam_state(), adam0))
    m.close()


def test_solve_jvp_argument_checks(ctx):
    L = engine.lib()
    P = engine._ptr
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_SMOOTH_RI, n_steps=4, save_stride=2, ckpt_stride=2)
    th = _theta(d)
    ncol = 5
    x0, bcs = syn.columns(d, ncol)
    xd, thd, _ = tangents_of(d, ncol)
    m = engine.Model(ctx, d, th)
    out = np.full((ncol, m.n_saved, d.S), 7.0, dtype=np.float32)

    def call(x_=x0, xd_=xd, td_=thd, pd_=None, y_=out, n=ncol, Q_=None, h=m._h):
        return L.cpz_solve_jvp(h, P(x_), P(bcs), P(Q_), P(xd_), P(td_), P(pd_), None, P(y_), n)

    def rejected(rc, words):
        msg = L.cpz_last_error().decode()
        assert rc == -1 and words in msg, (rc, msg)

    rejected(call(x_=None), "null array")
    rejected(call(y_=None), "null array")
    rejected(call(xd_=None, td_=None), "no tangent")
    rejected(call(pd_=np.ones(5, dtype=np.float32)), "smooth_Ri")
    rejected(call(n=0), "ncol must be positive")
    rejected(call(n=2 ** 40), "ncol too large")
    assert (out == 7).all()
    assert call() == 0 and np.isfinite(out).all()
    m.close()
    d2 = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=4, save_stride=2, ckpt_stride=2)
    m2 = engine.Model(ctx, d2, _theta(d2))
    x2, b2 = syn.columns(d2, 3)
    with pytest.raises(engine.CpzError) as ei:
        m2.solve_jvp(x2, b2, x0_dot=x2)
    assert "diurnal_Q" in str(ei.value)
    m2.close()
    for d3, tan, words in ((syn.free_convection_desc(ca=True, mpp=True, n_steps=4, save_stride=2, ckpt_stride=2), "p", "mPP-parameter gradient"),
                           (syn.wind_mixing_desc(variant=RHS_TRAIN, net=None, flags=FLAG_MPP, n_steps=4, save_stride=2, ckpt_stride=2), "theta",
                            "no parameters"),
                           (syn.wind_mixing_desc(variant=RHS_INFER, net="uvT_large", n_steps=4, save_stride=2, ckpt_stride=2), "x",
                            "adjoint plan unavailable")):
        m3 = engine.Model(ctx, d3, _theta(d3))
        x3, b3 = syn.columns(d3, 3)
        one = np.ones(5, dtype=np.float32)
        y3 = np.empty((3, m3.n_saved, d3.S), dtype=np.float32)
        rejected(L.cpz_solve_jvp(m3._h, P(x3), P(b3), None, P(x3) if tan == "x" else None, P(one) if tan == "theta" else None,
                                 P(one) if tan == "p" else None, None, P(y3), 3), words)
        m3.close()


# ---- solve_autograd: forward mode is cpz_solve_jvp, reverse mode cpz_solve_vjp
def test_solve_autograd_forward_and_reverse_mode(ctx):
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=8, save_stride=4, ckpt_stride=4)
    ncol = 40
    th = _theta(d)
    x0, bcs = syn.columns(d, ncol)
    xd, thd, pd = tangents_of(d, ncol)
    m = engine.Model(ctx, d, th)
    _, ref_dot = m.solve_jvp(x0, bcs, xd, thd, pd)
    tbar = np.random.default_rng(2).standard_normal(ref_dot.shape).astype(np.float32)
    ref_bar = m.solve_vjp(x0, bcs, tbar, want_mpp=True)
    dev = torch.device("cuda:0")
    T = (lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32)).to(dev))
    p0 = p_of(d, torch.float32).to(dev)

    def f(th_, x_, p_):
        return wm.solve_autograd(m, th_, x_, T(bcs), p=p_)

    _, tan = torch.func.jvp(f, (T(th), T(x0), p0), (T(thd), T(xd), T(pd)))
    assert np.array_equal(tan.cpu().numpy(), ref_dot)
    import torch.autograd.forward_ad as fwAD
    with fwAD.dual_level():
        out = f(fwAD.make_dual(T(th), T(thd)), fwAD.make_dual(T(x0), T(xd)), fwAD.make_dual(p0, T(pd)))
        assert np.array_equal(fwAD.unpack_dual(out).tangent.cpu().numpy(), ref_dot)
    th_t, x_t, p_t = (a.clone().requires_grad_(True) for a in (T(th), T(x0), p0))
    (f(th_t, x_t, p_t) * T(tbar)).sum().backward()
    for got, ref in zip((x_t.grad, th_t.grad, p_t.grad), ref_bar):
        assert np.array_equal(got.cpu().numpy(), ref)
    m.close()


def test_solve_autograd_mpp_jacobian_of_the_nn_free_model(ctx):
    """Five forward-mode calls with unit mpp tangents give the trajectory Jacobian wrt p = (nu0, nu_m, dRi, Ric, Pr) of the
    NN-free `DE` model: the forward sensitivities of optimise_modified_pacanowski_philander's parameters."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, n_steps=36, save_stride=9, ckpt_stride=9, net=None)
    ncol = 8
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, np.zeros(0, dtype=np.float32))
    dev = torch.device("cuda:0")
    th0 = torch.zeros(0, device=dev)
    xt, bt = torch.from_numpy(x0).to(dev), torch.from_numpy(bcs).to(dev)
    p0 = p_of(d, torch.float32).to(dev)
    cols = []
    for i in range(5):
        e = torch.zeros(5, device=dev)
        e[i] = 1.0
        _, tan = torch.func.jvp(lambda p_: wm.solve_autograd(m, th0, xt, bt, p=p_), (p0,), (e,))
        cols.append(tan.cpu().numpy())
    m.close()
    got = np.stack(cols, axis=-1)

    def jac(dtype):
        b = torch.tensor(bcs, dtype=dtype)
        x = torch.tensor(x0, dtype=dtype)
        return torch.func.jacfwd(lambda p_: nde.solve(d, torch.zeros(0, dtype=dtype), x, b, None, mpp=p_))(p_of(d, dtype)).numpy()

    ref, r32 = jac(torch.float64), jac(torch.float32)
    for i, name in enumerate(("nu0", "nu_m", "dRi", "Ric", "Pr")):
        err, floor = rel_l2(got[..., i], ref[..., i]), rel_l2(r32[..., i], ref[..., i])
        print(f"d traj / d {name}: {err:.2e} (fp32-oracle {floor:.2e})")
        assert err <= max(TOL, floor), (name, err, floor)
