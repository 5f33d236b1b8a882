"""S7b pullback: cpz_closure_step_uvt_vjp (u_bar, v_bar, T_bar, theta_bar, mpp_bar of one embedded u/v/T closure step), CUDA
through the C ABI vs torch.autograd of the FP64 oracle step (oracle/nde.py: closure_step_uvt). The same autograd in FP32
gives the noise floor, printed next to every error. Tolerance: relative inf-norm err <= max(1e-4, FP32-oracle error)."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, synthetic as syn, wind_mixing as wm
from cpz_b200.desc import ClosureUvtDesc, FLAG_MPP, FLAG_SMOOTH_RI, RHS_INFER, RHS_TRAIN
from oracle import nde
from test_closure_uvt_vjp_oracle_cpu import mpp_of, oracle_closure_uvt, oracle_closure_uvt_vjp
from util import rel_inf, t64

pytestmark = pytest.mark.gpu
TOL = 1e-4


def cots(nx, ny, seed=77):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((3, 32, ny, nx)).astype(np.float32), rng.standard_normal((3, 32, ny, nx)).astype(np.float32))


def cdesc(nx, ny, ca=True, **kw):
    kw = dict(dict(dz=8.0, dt=60.0, uw_top=-1e-4, vw_top=2e-5, wT_top=3e-5), **kw)
    return ClosureUvtDesc(Nx=nx, Ny=ny, Nz=32, convective_adjustment=ca, **kw)


def _check(ctx, d, th, cd, u, v, T, fb, ob, label="", m=None):
    """Runs the host flavour with every output and compares them with the FP64 oracle; returns the outputs."""
    own = m is None
    m = engine.Model(ctx, d, th) if own else m
    xb, tb, pb = m.closure_step_uvt_vjp(cd, u, v, T, fb, ob, want_mpp=True)
    if own:
        m.close()
    ref = oracle_closure_uvt_vjp(d, th, cd, u, v, T, fb, ob)
    ref32 = oracle_closure_uvt_vjp(d, th, cd, u, v, T, fb, ob, dtype=torch.float32)
    msg = [f"closure_uvt_vjp {label} {cd.Nx}x{cd.Ny} ca={cd.convective_adjustment} "
           f"cot={'D' if fb is not None else ''}{'Y' if ob is not None else ''}:"]
    names = ("u_bar", "v_bar", "T_bar", "theta_bar", "mpp_bar")
    got = (xb[0], xb[1], xb[2], tb, pb)
    rr = (ref[0][0], ref[0][1], ref[0][2], ref[1], ref[2])
    r32 = (ref32[0][0], ref32[0][1], ref32[0][2], ref32[1], ref32[2])
    for name, g, r, f32 in zip(names, got, rr, r32):
        assert np.isfinite(g).all(), name
        if np.abs(r).max() == 0:  # a cotangent that does not reach this output
            assert np.abs(g).max() == 0, name
            msg.append(f"{name} 0")
            continue
        err, floor = rel_inf(g, r), rel_inf(f32, r)
        msg.append(f"{name} {err:.2e} (fp32-oracle {floor:.2e})")
        assert err <= max(TOL, floor), (name, err, floor)
    print("  ".join(msg))
    return xb, tb, pb


# ---- 1. production nets (the forward runs on the tcgen05 closure): convective adjustment off / on with unstable columns
@pytest.mark.parametrize("ca", [False, True])
def test_closure_uvt_vjp_production_nets(ctx, ca):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=0.5)
    nx, ny = 40, 3
    u, v, T = syn.uvt_fields(d, nx, ny, unstable_every=3 if ca else 0)
    cd = cdesc(nx, ny, ca=ca, dz=d.H / 32)
    m = engine.Model(ctx, d, th)
    desc = m.describe()
    assert "closure_uvt_vjp_kernel" in desc
    # the pullback linearises the step the deployed forward computes
    dzf, out = m.closure_step_uvt(cd, u, v, T)
    dzf_ref, out_ref = nde_step(d, th, cd, u, v, T)
    assert rel_inf(dzf, dzf_ref) <= 1e-5 and rel_inf(out, out_ref) <= 1e-5
    fb, ob = cots(nx, ny)
    _check(ctx, d, th, cd, u, v, T, fb, ob, label="production", m=m)
    m.close()
    if ca:
        assert (np.abs(out_ref[2] - T) > 1e-3).any()  # the kappa_ca branch acted


def nde_step(d, th, cd, u, v, T):
    with torch.no_grad():
        dzf, out = oracle_closure_uvt(d, t64(th), cd, t64(u), t64(v), t64(T), mpp_of(d))
    return dzf.numpy(), out.numpy()


# ---- 2. every activation (width-40 one-hidden-layer nets, weights in shared memory); width 128 streams the weights
@pytest.mark.parametrize("act", ["relu", "mish", "swish", "leakyrelu", "tanh"])
def test_closure_uvt_vjp_activations(ctx, act):
    d = syn.wind_mixing_desc(variant=RHS_INFER, net=None)
    d.nets = [syn.NetDesc([d.S, 40, d.Nz - 1], [act, "identity"]) for _ in range(3)]
    th = syn.theta_random(d, scale=1.0)
    u, v, T = syn.uvt_fields(d, 24, 2, unstable_every=5)
    fb, ob = cots(24, 2)
    _check(ctx, d, th, cdesc(24, 2), u, v, T, fb, ob, label=act)


def test_closure_uvt_vjp_streamed_weights(ctx):
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net=None)
    d.nets = [syn.NetDesc([d.S, 128, d.Nz - 1], ["relu", "identity"]) for _ in range(3)]
    th = syn.theta_random(d, scale=1.0)
    m = engine.Model(ctx, d, th)
    line = [s for s in m.describe().splitlines() if "closure_uvt_vjp_kernel" in s]
    assert len(line) == 1 and "weights streamed from global memory" in line[0]
    u, v, T = syn.uvt_fields(d, 40, 1, unstable_every=4)
    fb, ob = cots(40, 1)
    _check(ctx, d, th, cdesc(40, 1, wT_top=-4e-5, dz=5.0, dt=600.0, kappa_ca=0.3), u, v, T, fb, ob, label="width-128", m=m)
    m.close()


# ---- 3. field sizes: a single column, ragged last tiles, and more tiles than SMs (persistent CTAs take several)
@pytest.mark.parametrize("nx,ny", [(1, 1), (31, 1), (33, 1), (512, 64)])
def test_closure_uvt_vjp_field_sizes(ctx, nx, ny):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=0.5)
    u, v, T = syn.uvt_fields(d, nx, ny, unstable_every=3)
    fb, ob = cots(nx, ny)
    _check(ctx, d, th, cdesc(nx, ny), u, v, T, fb, ob, label="size")


# ---- 4. one cotangent or both
@pytest.mark.parametrize("which", ["uvT_bar", "dz_flux_bar", "both"])
def test_closure_uvt_vjp_cotangent_modes(ctx, which):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=0.5)
    u, v, T = syn.uvt_fields(d, 37, 2, unstable_every=3)
    fb, ob = cots(37, 2)
    fb = None if which == "uvT_bar" else fb
    ob = None if which == "dz_flux_bar" else ob
    xb, tb, pb = _check(ctx, d, th, cdesc(37, 2), u, v, T, fb, ob, label=which)
    if ob is None:
        assert np.all(pb == 0)  # the mPP parameters act on the state step only
    if fb is None:
        assert np.all(tb == 0)  # the nets act on dz_flux only


# ---- 5. exact properties
def _setup(nx=48, ny=4):
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=0.5)
    u, v, T = syn.uvt_fields(d, nx, ny, unstable_every=3)
    fb, ob = cots(nx, ny)
    return d, th, cdesc(nx, ny), u, v, T, fb, ob


def test_closure_uvt_vjp_is_linear_in_the_cotangents(ctx):
    d, th, cd, u, v, T, fb, ob = _setup()
    m = engine.Model(ctx, d, th)
    both = m.closure_step_uvt_vjp(cd, u, v, T, fb, ob, want_mpp=True)
    only_d = m.closure_step_uvt_vjp(cd, u, v, T, fb, None, want_mpp=True)
    only_y = m.closure_step_uvt_vjp(cd, u, v, T, None, ob, want_mpp=True)
    scaled = m.closure_step_uvt_vjp(cd, u, v, T, 2 * fb, -0.5 * ob, want_mpp=True)
    half = m.closure_step_uvt_vjp(cd, u, v, T, fb, -0.5 * ob, want_mpp=True)
    m.close()
    for i in range(3):
        assert rel_inf(both[i], only_d[i] + only_y[i]) <= 1e-6, i
    # scaling a cotangent by a power of two scales its part exactly
    assert np.array_equal(scaled[1], 2 * both[1]) and np.array_equal(half[2], -0.5 * both[2])


def test_closure_uvt_vjp_slab_decomposition(ctx):
    """theta_bar of a field is the sum of theta_bar over y-slab shards; a column's u_bar, v_bar, T_bar do not depend on the
    slab it is in (bitwise)."""
    d, th, cd, u, v, T, fb, ob = _setup(nx=48, ny=4)
    m = engine.Model(ctx, d, th)
    xb, tb, pb = m.closure_step_uvt_vjp(cd, u, v, T, fb, ob, want_mpp=True)
    tsum, psum = np.zeros_like(tb, dtype=np.float64), np.zeros(5)
    for j0, j1 in ((0, 1), (1, 3), (3, 4)):
        cds = cdesc(48, j1 - j0)
        sl = (slice(None), slice(j0, j1))
        xs, ts, ps = m.closure_step_uvt_vjp(cds, u[sl], v[sl], T[sl], fb[:, :, j0:j1], ob[:, :, j0:j1], want_mpp=True)
        assert np.array_equal(xs, xb[:, :, j0:j1])
        tsum += ts
        psum += ps
    m.close()
    assert rel_inf(tsum, tb) <= 1e-6 and rel_inf(psum, pb) <= 1e-6


def test_closure_uvt_vjp_host_equals_device_and_leaves_the_step_unchanged(ctx):
    d, th, cd, u, v, T, fb, ob = _setup(nx=40, ny=3)
    m = engine.Model(ctx, d, th)
    dzf0, out0 = m.closure_step_uvt(cd, u, v, T)
    xb, tb, pb = m.closure_step_uvt_vjp(cd, u, v, T, fb, ob, want_mpp=True)
    dev = torch.device("cuda:0")
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    ud, vd, Td, fbd, obd = (tt(a) for a in (u, v, T, fb, ob))
    xbd = torch.empty((3,) + u.shape, device=dev)
    tbd, pbd = torch.empty(m.P, device=dev), torch.empty(5, device=dev)
    torch.cuda.synchronize()
    m.closure_step_uvt_vjp_dev(cd, ud, vd, Td, fbd, obd, xbd[0], xbd[1], xbd[2], tbd, pbd)
    m.ctx.synchronize()
    assert np.array_equal(xbd.cpu().numpy(), xb) and np.array_equal(tbd.cpu().numpy(), tb) and np.array_equal(pbd.cpu().numpy(), pb)
    dzf1, out1 = m.closure_step_uvt(cd, u, v, T)
    m.close()
    assert np.array_equal(dzf0, dzf1) and np.array_equal(out0, out1)


# ---- 6. an a-posteriori gradient through a few host steps, with torch autograd around the device flavours
def test_closure_uvt_vjp_a_posteriori_gradient_through_autograd(ctx):
    """A loss on the state after three host steps (closure step, then the stand-in dynamics) differentiated in theta by torch
    autograd over wind_mixing.closure_step_uvt_autograd, against FP64 autograd of the same chain on the oracle. The oracle
    chain is evaluated along the engine's frames (value of the engine's state, derivative of the oracle's chain): a
    free-running chain is not comparable, because in the weakly stratified layer the Richardson number turns a 1e-7 rounding
    of T into an O(1e-3) change of the diffusivity at the next step."""
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=0.3)
    nx, ny, n_steps = 16, 2, 3
    u, v, T = syn.uvt_fields(d, nx, ny)
    cd = cdesc(nx, ny, ca=True, dz=d.H / 32)
    w = np.random.default_rng(3).standard_normal((3, 32, ny, nx))

    def chain(step, theta, x, frames=None):
        seen = []
        for k in range(n_steps):
            if frames is not None:
                x = [xi + (torch.as_tensor(f, dtype=xi.dtype) - xi).detach() for xi, f in zip(x, frames[k])]
            seen.append([xi.detach().cpu().numpy() for xi in x])
            dzf, out = step(theta, x)
            x = wm._standin_dynamics(out[0], out[1], out[2], dzf, cd.dt, d.f)
        loss = sum((x[q] * torch.as_tensor(w[q], dtype=x[q].dtype, device=x[q].device)).sum() for q in range(3))
        return loss, seen

    m = engine.Model(ctx, d, th)
    dev = torch.device("cuda:0")
    tht = torch.tensor(th, device=dev, requires_grad=True)
    x0 = [torch.from_numpy(a).to(dev) for a in (u, v, T)]
    loss, frames = chain(lambda theta, x: wm.closure_step_uvt_autograd(m, cd, theta, *x), tht, x0)
    loss.backward()
    g = tht.grad.cpu().numpy()
    m.close()

    def oracle_grad(dtype):
        t = torch.tensor(th, dtype=dtype, requires_grad=True)
        x = [torch.tensor(a, dtype=dtype) for a in (u, v, T)]
        L, _ = chain(lambda theta, xx: nde.closure_step_uvt(d, theta, cd, *xx), t, x, frames)
        return torch.autograd.grad(L, t)[0].numpy()

    ref, ref32 = oracle_grad(torch.float64), oracle_grad(torch.float32)
    err, floor = rel_inf(g, ref), rel_inf(ref32, ref)
    print(f"a-posteriori theta gradient through {n_steps} host steps: {err:.2e} (fp32-oracle {floor:.2e})")
    assert err <= max(TOL, floor)


# ---- 7. argument checks
def test_closure_uvt_vjp_refusals(ctx):
    z = np.zeros((32, 1, 4), dtype=np.float32)
    c3 = np.zeros((3, 32, 1, 4), dtype=np.float32)
    cd = cdesc(4, 1)

    def refused(d, th, words, **kw):
        m = engine.Model(ctx, d, th)
        args = dict(dz_flux_bar=c3, uvT_bar=c3)
        args.update(kw)
        with pytest.raises(engine.CpzError) as ei:
            m.closure_step_uvt_vjp(cd, z, z, z, **args)
        m.close()
        assert ei.value.code == engine.ERR_INVALID and words in str(ei.value), str(ei.value)

    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=0.5)
    # the 400-wide nets have no adjoint plan: refused with the planner's reason
    dl = syn.wind_mixing_desc(variant=RHS_INFER, net="uvT_large")
    ml = engine.Model(ctx, dl, syn.theta_random(dl, scale=0.1))
    reason = ml.describe().split("adjoint plan: unavailable (")[1].split("\n")[0][:-1]
    ml.close()
    refused(dl, syn.theta_random(dl, scale=0.1), "adjoint plan unavailable: " + reason)
    refused(d, th, "no output requested", want_uvT=False, want_theta=False, want_mpp=False)
    refused(d, th, "no cotangent given", dz_flux_bar=None, uvT_bar=None)
    dn = syn.wind_mixing_desc(variant=RHS_INFER, net=None)
    refused(dn, np.zeros(0, dtype=np.float32), "no parameters", want_theta=True)
    ds = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_SMOOTH_RI)
    refused(ds, syn.theta_random(ds, scale=0.5), "smooth_Ri", want_uvT=False, want_theta=False, want_mpp=True)
    df = syn.free_convection_desc(ca=False)
    refused(df, syn.theta_random(df), "u/v/T model")
