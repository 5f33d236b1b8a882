"""S2 pullback: cpz_solve_vjp (x0_bar, theta_bar, mpp_bar of the batched solve for a cotangent of its trajectory), CUDA
through the C ABI vs torch.autograd of the FP64 oracle (oracle/nde.py: solve). The same autograd in FP32 gives the noise
floor, printed next to every error. Tolerance (the gradient rule of test_adjoint_tc_gpu.py): relative L2 error
<= max(1e-4, FP32-oracle error), 3x the floor for T-only models with convective adjustment and for x0_bar on the
tensor-core path: its Xbar chain (W1 delta1 on tcgen05) is 3xTF32, and on these sensitive random problems its x0_bar was
measured at 1.0-1.7x the FP32 floor while theta_bar stays within 1x. Every case asserts the adjoint path it takes,
mirroring loss_grad_core's selection (cpz_capi_train.inc) the way test_batch_schedules_gpu.py does."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn
from cpz_b200.desc import (FLAG_CA, FLAG_DIURNAL, FLAG_IMPLICIT_DIFFUSION as IMP, FLAG_MPP, FLAG_SMOOTH_RI,
                           FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN)
from oracle import nde
from test_batch_schedules_gpu import _env
from util import rel_inf

pytestmark = pytest.mark.gpu
TOL = 1e-4


def oracle_solve_vjp(d, theta, x0, bcs, tbar, Q=None, dtype=torch.float64, want_mpp=False):
    """(x0_bar, theta_bar, mpp_bar or None): torch.autograd.grad of nde.solve with cotangent tbar of the trajectory."""
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    xt = conv(x0).requires_grad_(True)
    th = conv(theta).requires_grad_(True)
    p = None
    if want_mpp:
        p = torch.tensor([float(np.float32(v)) for v in (d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr)], dtype=dtype, requires_grad=True)
    traj = nde.solve(d, th, xt, conv(bcs), None if Q is None else conv(Q), mpp=p)
    leaves = [xt, th] + ([p] if p is not None else [])
    g = torch.autograd.grad(traj, leaves, grad_outputs=conv(tbar), allow_unused=True)
    g = [torch.zeros_like(l) if gi is None else gi for gi, l in zip(g, leaves)]
    return g[0].detach().numpy(), g[1].detach().numpy(), (g[2].detach().numpy() if p is not None else None)


def rel_l2(a, ref):
    a, ref = np.asarray(a, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return float(np.linalg.norm(a - ref) / max(np.linalg.norm(ref), 1e-300))


def tbar_of(d, ncol, n_saved, seed=91):
    return np.random.default_rng(seed).standard_normal((ncol, n_saved, d.S)).astype(np.float32)


def expected_path(m, ncol, want_mpp):
    """loss_grad_core's choice: the tensor-core adjoint (P > 0, no mpp_bar), fc1 (T-only, <= 32 columns, no mpp_bar),
    otherwise the FP32 adjoint at train_tile's width."""
    desc = m.describe()
    if m.P > 0 and not want_mpp and "adjoint kernels: tcgen05" in desc:
        return "tc"
    if m.P > 0 and not want_mpp and "one CTA per column" in desc and ncol <= 32:
        return "fc1"
    return "fp32"


def uvt_relu():
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4, net=None)
    d.nets = [syn.NetDesc([d.S, 50, 20, d.Nz - 1], ["relu", "relu", "identity"]) for _ in range(3)]
    return d


def uvt_streamed():
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=8, save_stride=2, ckpt_stride=4, net=None)
    d.nets = [syn.NetDesc([d.S, 128, d.Nz - 1], ["relu", "identity"]) for _ in range(3)]
    return d


def fc_implicit():
    d = syn.free_convection_desc(ca=True, mpp=True, n_steps=12, save_stride=4, ckpt_stride=4, n_substeps=1)
    d.flags |= IMP
    return d


# name: (description, ncol, path, environment, want_mpp, diurnal). The ragged-batch cases leave the mPP closure out: some of the
# 257 columns sit on its Richardson-number step, where the FP32 oracle's theta_bar is 1e-2 from FP64 and says nothing about
# the column handling these cases are for.
CASES = {
    "tc_mish_split": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4), 40, "tc", {}, False, False),
    "tc_mish_two_groups": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4), 40, "tc",
                           {"CPZ_TC_SPLIT": "0"}, False, False),
    "tc_relu": (uvt_relu, 40, "tc", {}, False, False),
    "tc_implicit": (lambda: syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | IMP, n_steps=12, save_stride=3,
                                                 ckpt_stride=4, n_substeps=1), 40, "tc", {}, False, False),
    "tc_record_segments_ckpt1": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=22, save_stride=11, ckpt_stride=1), 50, "tc",
                                 {"CPZ_ADJ_AUX_GB": "0.004"}, False, False),
    "tc_record_segments_ckpt9": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=22, save_stride=11, ckpt_stride=9), 50, "tc",
                                 {"CPZ_ADJ_AUX_GB": "0"}, False, False),
    "tc_diurnal": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=12, save_stride=4,
                                                ckpt_stride=4), 40, "tc", {}, False, True),
    "tc_final_frame_only": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=10, save_stride=0, ckpt_stride=4), 40, "tc", {}, False, False),
    "tc_ncol1": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_ZERO_WEIGHTS, n_steps=6, save_stride=2, ckpt_stride=3), 1, "tc",
                 {}, False, False),
    "tc_ncol31": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_ZERO_WEIGHTS, n_steps=6, save_stride=2, ckpt_stride=3), 31, "tc",
                 {}, False, False),
    "tc_ncol257": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_ZERO_WEIGHTS, n_steps=6, save_stride=2, ckpt_stride=3), 257, "tc",
                 {}, False, False),
    "fp32_small_tiles_mpp": (lambda: syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=12, save_stride=1,
                                                          ckpt_stride=9), 33, "fp32", {}, True, False),
    "fp32_32col_tiles_streamed": (uvt_streamed, 70, "fp32", {"CPZ_SMALL_NCOL": "0"}, True, False),
    "fp32_no_tc_adj": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4), 40, "fp32",
                       {"CPZ_NO_TC_ADJ": "1"}, False, False),
    "fp32_implicit_mpp": (lambda: syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | IMP, n_steps=12, save_stride=3,
                                                       ckpt_stride=4, n_substeps=1), 31, "fp32", {}, True, False),
    "fp32_T_only_ncol33": (lambda: syn.free_convection_desc(ca=True, n_steps=12, save_stride=4, ckpt_stride=4), 33, "fp32", {}, False, False),
    "fc1_explicit": (lambda: syn.free_convection_desc(ca=True, mpp=True, n_steps=12, save_stride=4, ckpt_stride=4), 3, "fc1", {}, False, False),
    "fc1_implicit": (fc_implicit, 2, "fc1", {}, False, False),
    "nn_free": (lambda: syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, n_steps=12, save_stride=4, ckpt_stride=4,
                                             net=None), 37, "fp32", {}, True, False),
}


@pytest.mark.parametrize("case", list(CASES))
def test_solve_vjp_matches_the_oracle(ctx, case):
    mk, ncol, path, env, want_mpp, diurnal = CASES[case]
    d = mk()
    th = syn.theta_random(d, scale=0.1) if d.n_params > 0 else np.zeros(0, dtype=np.float32)
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol) if diurnal else None
    with _env(**env):
        m = engine.Model(ctx, d, th)
        assert expected_path(m, ncol, want_mpp) == path, m.describe()
        if path == "fp32" and "CPZ_SMALL_NCOL" in env:
            assert "weights streamed from global memory" in m.describe()
        tb_in = tbar_of(d, ncol, m.n_saved)
        got = m.solve_vjp(x0, bcs, tb_in, Q=Q, want_theta=m.P > 0, want_mpp=want_mpp)
        m.close()
    ref = oracle_solve_vjp(d, th, x0, bcs, tb_in, Q, want_mpp=want_mpp)
    ref32 = oracle_solve_vjp(d, th, x0, bcs, tb_in, Q, dtype=torch.float32, want_mpp=want_mpp)
    msg = [f"solve_vjp {case} ({path}) ncol={ncol}:"]
    for name, g, r, r32 in zip(("x0_bar", "theta_bar", "mpp_bar"), got, ref, ref32):
        if g is None:
            continue
        factor = 3.0 if (d.n_fields == 1 and d.has(FLAG_CA)) or (path == "tc" and name == "x0_bar") else 1.0
        assert np.isfinite(g).all(), name
        err, floor = rel_l2(g, r), rel_l2(r32, r)
        msg.append(f"{name} {err:.2e} (fp32-oracle {floor:.2e}; inf-norm {rel_inf(g, r):.2e})")
        assert err <= max(TOL, factor * floor), (name, err, floor)
    print("  ".join(msg))


# ---- consistency with the fused loss over a full-length solve: traj_bar = d loss/d traj of the oracle's loss functions
W_GRAD = np.array([0.7, 0.7, 1.0, 3e-3, 3e-3, 5e-3], dtype=np.float32)


def loss_cotangent(d, traj, tgt, w):
    t = torch.tensor(traj, dtype=torch.float64, requires_grad=True)
    comps = nde.loss_components(d, t, torch.tensor(tgt, dtype=torch.float64))
    total = sum(float(w[i]) * comps[i] for i in range(6))
    (g,) = torch.autograd.grad(total, t)
    return g.numpy().astype(np.float32)


@pytest.mark.parametrize("path", ["tc", "fp32"])
def test_solve_vjp_consistent_with_loss_grad_full_length(ctx, path):
    """A config-3 slice (u/v/T nets of train_NDE.jl, training RHS, 1 152 steps, 64 columns): solve_vjp's theta_bar for
    traj_bar = d loss/d traj equals cpz_loss_grad's gradient to 1e-5 relative, and its mpp_bar cpz_loss_grad_mpp's to 1e-4.
    mpp_bar is a sum of terms of both signs (FP64 partial sums in the kernel), so the rounding of the injected cotangent
    (computed in FP32 inside the kernel by cpz_loss_grad_mpp, rounded from FP64 here) shows at 7e-5 of the result."""
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS)
    ncol = 64
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, ncol)
    env = {"CPZ_NO_TC_ADJ": "1"} if path == "fp32" else {}
    with _env(**env):
        m = engine.Model(ctx, d, th)
        assert expected_path(m, ncol, False) == path
        traj = m.solve(x0, bcs)
        tgt = (traj + 0.05 * np.random.default_rng(4).standard_normal(traj.shape)).astype(np.float32)
        tbar = loss_cotangent(d, traj, tgt, W_GRAD)
        _, grad = m.loss_grad(x0, bcs, tgt, W_GRAD)
        _, tb, pb = m.solve_vjp(x0, bcs, tbar, want_x0=False, want_mpp=path == "fp32")
        e_t = float(np.linalg.norm(tb - grad) / np.linalg.norm(grad))
        msg = f"solve_vjp vs loss_grad ({path}, {d.n_steps} steps): theta {e_t:.2e}"
        if path == "fp32":
            _, gp, _ = m.loss_grad_mpp(x0, bcs, tgt, W_GRAD)
            e_p = float(np.linalg.norm(pb - gp) / np.linalg.norm(gp))
            msg += f", mpp {e_p:.2e}"
            assert e_p <= 1e-4, e_p
        m.close()
    print(msg)
    assert e_t <= 1e-5, e_t


# ---- exact identities
@pytest.mark.parametrize("path", ["tc", "fp32"])
def test_solve_vjp_exact_identities(ctx, path):
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_CA, n_steps=4, save_stride=2, ckpt_stride=2)
    ncol = 45
    th = syn.theta_random(d, scale=0.1)
    x0, bcs = syn.columns(d, ncol)
    want_mpp = path == "fp32"
    m = engine.Model(ctx, d, th)
    assert expected_path(m, ncol, want_mpp) == path
    a, b = tbar_of(d, ncol, m.n_saved, seed=1), tbar_of(d, ncol, m.n_saved, seed=2)
    f0 = np.zeros_like(a)
    f0[:, 0] = a[:, 0]
    xb, tb, pb = m.solve_vjp(x0, bcs, f0, want_mpp=want_mpp)
    assert np.array_equal(xb, a[:, 0])  # frame 0 is x0 itself
    assert not tb.any() and (pb is None or not pb.any())
    va, vb = m.solve_vjp(x0, bcs, a, want_mpp=want_mpp), m.solve_vjp(x0, bcs, b, want_mpp=want_mpp)
    vc = m.solve_vjp(x0, bcs, 2 * a - b, want_mpp=want_mpp)
    m.close()
    for name, ga, gb, gc in zip(("x0_bar", "theta_bar", "mpp_bar"), va, vb, vc):
        if ga is None:
            continue
        e = rel_l2(gc, 2 * ga.astype(np.float64) - gb)
        print(f"solve_vjp linearity ({path}) {name}: {e:.2e}")
        # FP32 rounding carried through the reverse sweep: 3.3e-6 .. 3.6e-6 measured on x0_bar, 4 steps
        assert e <= 1e-5, (name, e)


# ---- batch invariance
@pytest.mark.parametrize("path", ["tc", "fp32"])
def test_solve_vjp_batch_invariance(ctx, path):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=8, save_stride=4, ckpt_stride=4)
    ncol = 160
    th = syn.theta_random(d, scale=0.1)
    x0, bcs = syn.columns(d, ncol)
    env = {"CPZ_NO_TC_ADJ": "1", "CPZ_SMALL_NCOL": "0"} if path == "fp32" else {}  # 32-column tiles throughout
    with _env(**env):
        m = engine.Model(ctx, d, th)
        assert expected_path(m, ncol, False) == path
        tbar = tbar_of(d, ncol, m.n_saved)
        xb, tb, _ = m.solve_vjp(x0, bcs, tbar)
        cuts = [0, 32, 96, 160]  # whole 32-column tiles: every column keeps its place in its tile
        parts = [m.solve_vjp(x0[p:q], bcs[p:q], tbar[p:q]) for p, q in zip(cuts[:-1], cuts[1:])]
        m.close()
    assert np.array_equal(np.concatenate([p[0] for p in parts]), xb)
    tsum = np.sum([p[1].astype(np.float64) for p in parts], axis=0)
    e = rel_l2(tb, tsum)
    print(f"solve_vjp batch invariance ({path}): theta_bar vs sum over shards {e:.2e}")
    assert e <= 1e-6, e


# ---- flavours and side effects
def test_solve_vjp_dev_matches_host_and_leaves_training_alone(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_DIURNAL, n_steps=8, save_stride=4, ckpt_stride=4)
    ncol = 45
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, ncol)
    Q = syn.diurnal_Q(ncol)
    m = engine.Model(ctx, d, th)
    tbar = tbar_of(d, ncol, m.n_saved)
    host = m.solve_vjp(x0, bcs, tbar, Q=Q, want_mpp=True)
    dev = torch.device("cuda:0")
    xt, bt, qt, tt = (torch.from_numpy(a).to(dev) for a in (x0, bcs, Q, tbar))
    outs = [torch.full((ncol, d.S), float("nan"), device=dev), torch.full((m.P,), float("nan"), device=dev),
            torch.full((5,), float("nan"), device=dev)]
    torch.cuda.synchronize()  # the fills run on torch's stream, the pullback on the context's
    m.solve_vjp_dev(xt, bt, tt, *outs, Q=qt)
    ctx.synchronize()
    for g, h in zip(outs, host):
        assert np.array_equal(g.cpu().numpy(), h)
    # a train_step sequence interleaved with solve_vjp calls ends at the same theta, bitwise
    tgt = (tbar * 0.01 + m.solve(x0, bcs, Q=Q)).astype(np.float32)

    def train(with_vjp):
        mm = engine.Model(ctx, d, th)
        for _ in range(3):
            if with_vjp:
                mm.solve_vjp(x0, bcs, tbar, Q=Q, want_mpp=True)
            mm.train_step(x0, bcs, tgt, W_GRAD, 1e-3, Q=Q)
        loss, grad = mm.loss_grad(x0, bcs, tgt, W_GRAD, Q=Q)
        out = (mm.get_theta(), mm.adam_state(), loss, grad)
        mm.close()
        return out

    a, b = train(False), train(True)
    m.close()
    assert np.array_equal(a[0], b[0]) and all(np.array_equal(p, q) for p, q in zip(a[1], b[1]))
    assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])


# ---- a non-MSE loss end to end through a torch.autograd.Function (the INTEGRATION.md rrule, in torch)
class EngineSolve(torch.autograd.Function):
    """traj = solve(theta, x0): forward cpz_solve_dev, backward cpz_solve_vjp_dev. theta is the model's (set before)."""

    @staticmethod
    def forward(fctx, model, theta, x0, bcs):
        traj = torch.empty((x0.shape[0], model.n_saved, model.desc.S), device=x0.device)
        torch.cuda.synchronize()
        model.solve_dev(x0, bcs, traj)
        model.ctx.synchronize()
        fctx.model = model
        fctx.save_for_backward(x0, bcs)
        return traj

    @staticmethod
    def backward(fctx, traj_bar):
        x0, bcs = fctx.saved_tensors
        m = fctx.model
        xb, tb = torch.empty_like(x0), torch.empty(m.P, device=x0.device)
        tbar = traj_bar.contiguous()
        torch.cuda.synchronize()
        m.solve_vjp_dev(x0, bcs, tbar, x0_bar=xb, theta_bar=tb)
        m.ctx.synchronize()
        return None, tb, xb, None


def test_solve_vjp_non_mse_loss_through_autograd(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, n_steps=12, save_stride=4, ckpt_stride=4)
    ncol = 40
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, ncol)
    wcol = np.linspace(0.5, 2.0, ncol)

    def loss_of(traj, dt):  # per-column weights, a nonlinear loss on the last frame and a log-cosh misfit
        w = torch.tensor(wcol, dtype=dt, device=traj.device)
        return (w[:, None] * torch.log(torch.cosh(3.0 * (traj[:, -1] - 0.1)))).sum() + (traj[:, 1:] ** 3).mean()

    m = engine.Model(ctx, d, th)
    dev = torch.device("cuda:0")
    tht = torch.tensor(th, device=dev, requires_grad=True)
    xt = torch.tensor(x0, device=dev, requires_grad=True)
    traj = EngineSolve.apply(m, tht, xt, torch.from_numpy(bcs).to(dev))
    loss_of(traj, torch.float32).backward()
    m.close()
    th64 = torch.tensor(th, dtype=torch.float64, requires_grad=True)
    x64 = torch.tensor(x0, dtype=torch.float64, requires_grad=True)
    loss_of(nde.solve(d, th64, x64, torch.tensor(bcs, dtype=torch.float64)), torch.float64).backward()
    th32 = torch.tensor(th, dtype=torch.float32, requires_grad=True)
    x32 = torch.tensor(x0, dtype=torch.float32, requires_grad=True)
    loss_of(nde.solve(d, th32, x32, torch.tensor(bcs, dtype=torch.float32)), torch.float32).backward()
    for name, g, r, r32 in (("x0.grad", xt.grad, x64.grad, x32.grad), ("theta.grad", tht.grad, th64.grad, th32.grad)):
        err, floor = rel_l2(g.cpu().numpy(), r.numpy()), rel_l2(r32.numpy(), r.numpy())
        print(f"solve_vjp through autograd: {name} {err:.2e} (fp32-oracle {floor:.2e})")
        assert err <= max(TOL, floor), (name, err, floor)


# ---- argument checks
def test_solve_vjp_argument_checks(ctx):
    L = engine.lib()
    P = engine._ptr
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_SMOOTH_RI, n_steps=4, save_stride=2, ckpt_stride=2)
    th = syn.theta_random(d, scale=0.3)
    ncol = 5
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    tbar = tbar_of(d, ncol, m.n_saved)
    xb = np.full_like(x0, 7.0)
    tb = np.full(th.size, 7.0, dtype=np.float32)
    pb = np.full(5, 7.0, dtype=np.float32)

    def rejected(h, args, words):
        rc = L.cpz_solve_vjp(h, *args)
        msg = L.cpz_last_error().decode()
        assert rc == -1 and words in msg, (rc, msg)

    rejected(m._h, (P(x0), P(bcs), None, None, P(xb), P(tb), None, ncol), "null array")
    rejected(m._h, (P(x0), P(bcs), None, P(tbar), None, None, None, ncol), "no output")
    rejected(m._h, (P(x0), P(bcs), None, P(tbar), P(xb), P(tb), P(pb), ncol), "smooth_Ri")
    rejected(m._h, (P(x0), P(bcs), None, P(tbar), P(xb), P(tb), None, 0), "ncol must be positive")
    assert (xb == 7).all() and (tb == 7).all() and (pb == 7).all()
    m.close()
    for d2, words in ((syn.free_convection_desc(ca=True, mpp=True, n_steps=4, save_stride=2, ckpt_stride=2), "mPP-parameter gradient"),
                      (syn.wind_mixing_desc(variant=RHS_TRAIN, net=None, flags=FLAG_MPP, n_steps=4, save_stride=2, ckpt_stride=2), "no parameters")):
        th2 = syn.theta_random(d2, scale=0.3) if d2.n_params > 0 else np.zeros(0, dtype=np.float32)
        x2, b2 = syn.columns(d2, 3)
        m2 = engine.Model(ctx, d2, th2)
        with pytest.raises(engine.CpzError) as ei:
            m2.solve_vjp(x2, b2, tbar_of(d2, 3, m2.n_saved), want_theta=d2.n_params == 0, want_mpp=d2.n_params > 0)
        assert ei.value.code == -1 and words in str(ei.value), str(ei.value)
        m2.close()
