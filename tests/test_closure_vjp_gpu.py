"""S7 pullback: cpz_closure_step_vjp (T_bar, theta_bar of one gyre closure step), CUDA through the C ABI vs torch.autograd of
the FP64 oracle step (oracle/nde.py: closure_step). The same autograd in FP32 gives the noise floor, printed next to every
error. Tolerance: relative inf-norm err <= max(1e-4, FP32-oracle error).

The forcing is O(1e-6) of T, so with unit cotangents the forcing path's part of T_bar is invisible next to the T' path's.
Each case therefore runs forcing_bar alone (the whole of T_bar and theta_bar come from the net) and both cotangents with
forcing_bar scaled by 1 / max|forcing|, so that both paths show in T_bar."""
import numpy as np
import pytest
import torch

from cpz_b200 import engine, free_convection as fc, synthetic as syn
from cpz_b200.desc import ClosureDesc, NetDesc, RHS_INFER
from oracle import nde
from test_closure_vjp_oracle_cpu import gyre_inputs, oracle_closure_vjp
from util import assert_blocks, rel_inf, t64, theta_blocks

pytestmark = pytest.mark.gpu
TOL = 1e-4


def t_only(h1, h2, act):
    d = syn.free_convection_desc(ca=False, net=None)
    d.nets = [NetDesc([32, h1, h2, 31], [act, act, "identity"])]
    return d


def cots(d, th, cd, T, y, which, seed=77):
    """(forcing_bar, T_out_bar) for `which` in {"forcing_bar", "T_out_bar", "both"}; with both, forcing_bar is scaled by
    1 / max|forcing| of the oracle step."""
    rng = np.random.default_rng(seed)
    shp = (cd.Nz, cd.Ny, cd.Nx)
    fb, ob = rng.standard_normal(shp).astype(np.float32), rng.standard_normal(shp).astype(np.float32)
    if which == "both":
        with torch.no_grad():
            forcing, _ = nde.closure_step(d, t64(th), cd, t64(T), t64(y))
        fb = (fb / float(forcing.abs().max())).astype(np.float32)
    return (None if which == "T_out_bar" else fb), (None if which == "forcing_bar" else ob)


def branch_ties(d, th, cd, T, y):
    """[Ny, Nx] mask of the columns on a branch tie: those whose FP32-oracle T_bar is outside the tolerance of the FP64 one
    for a unit forcing_bar alone (the net's branches) or a unit T_out_bar alone (the adjustment's switch)."""
    ties = np.zeros((cd.Ny, cd.Nx), dtype=bool)
    for which in ("forcing_bar", "T_out_bar"):
        fb, ob = cots(d, th, cd, T, y, which)
        r = oracle_closure_vjp(d, th, cd, T, y, fb, ob)[0]
        r32 = oracle_closure_vjp(d, th, cd, T, y, fb, ob, dtype=torch.float32)[0]
        ties |= np.abs(r32 - r).max(axis=0) > TOL * max(np.abs(r).max(), 1e-30)
    return ties


def _check(ctx, d, th, cd, T, y, which, label="", m=None):
    """Runs the host flavour with both outputs for the cotangents of `which` and compares them with the FP64 oracle; returns
    (forcing_bar, T_out_bar, T_bar, theta_bar).

    A column whose FP32 oracle T_bar is itself outside the tolerance sits on a branch tie: a relu pre-activation or a
    centred gradient of the adjustment switch so close to 0 that FP64 and FP32 evaluate different branches (measured: a
    second-layer pre-activation of 1.8e-6 in FP64 and -2.3e-8 in FP32 on the 512 x 64 field). The pullback takes the branch
    its FP32 forward evaluated, so the FP64 derivative of the other branch is no reference there. Such columns are found
    from the two oracles alone, never from the engine's output; they must be rare, and they get zero cotangents (the
    pullback is linear in them, so this removes exactly their contribution) before the comparison is made."""
    own = m is None
    m = engine.Model(ctx, d, th) if own else m
    ties = branch_ties(d, th, cd, T, y)
    n_ties = int(ties.sum())
    assert n_ties <= max(1, ties.size // 1000), (n_ties, ties.size)
    fb, ob = cots(d, th, cd, T, y, which)
    if n_ties:
        fb = None if fb is None else np.where(ties[None], np.float32(0), fb).astype(np.float32)
        ob = None if ob is None else np.where(ties[None], np.float32(0), ob).astype(np.float32)
    ref = oracle_closure_vjp(d, th, cd, T, y, fb, ob)
    ref32 = oracle_closure_vjp(d, th, cd, T, y, fb, ob, dtype=torch.float32)
    Tb, tb = m.closure_step_vjp(cd, T, fb, ob)
    if own:
        m.close()
    msg = [f"closure_vjp {label} {cd.Nx}x{cd.Ny} cot={which}" + (f" ({n_ties} tie column(s) zeroed)" if n_ties else "") + ":"]
    for name, g, r, f32 in zip(("T_bar", "theta_bar"), (Tb, tb), ref, ref32):
        assert np.isfinite(g).all(), name
        if np.abs(r).max() == 0:  # a cotangent that does not reach this output
            assert np.abs(g).max() == 0, name
            msg.append(f"{name} 0")
            continue
        err, floor = rel_inf(g, r), rel_inf(f32, r)
        msg.append(f"{name} {err:.2e} (fp32-oracle {floor:.2e})")
        assert err <= max(TOL, floor), (name, err, floor)
    print("  ".join(msg))
    assert_blocks("theta_bar", tb, ref[1], ref32[1], theta_blocks(d), TOL, norm="l2")
    return fb, ob, Tb, tb


def _adjusted(d, th, cd, T, y):
    with torch.no_grad():
        _, T_out = nde.closure_step(d, t64(th), cd, t64(T), t64(y))
    return np.abs(T_out.numpy() - T).max() > 1e-3


# ---- 1. the production net (32 -> 128 -> 128 -> 31 relu; its forward runs on the tcgen05 closure)
@pytest.mark.parametrize("which", ["forcing_bar", "both"])
def test_closure_vjp_production_net(ctx, which):
    d = syn.free_convection_desc(ca=False)
    assert [n.sizes for n in d.nets] == [[32, 128, 128, 31]] and d.nets[0].acts == ["relu", "relu", "identity"]
    th = syn.theta_random(d, scale=1.0)
    nx, ny = 40, 3
    T, y = gyre_inputs(nx, ny)
    assert _adjusted(d, th, ClosureDesc(Nx=nx, Ny=ny, Nz=32), T, y)
    cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
    m = engine.Model(ctx, d, th)
    assert "closure_vjp_kernel" in m.describe()
    # the pullback linearises the step the deployed forward computes
    forcing, T_out = m.closure_step(cd, T, y)
    with torch.no_grad():
        f_ref, T_ref = nde.closure_step(d, t64(th), cd, t64(T), t64(y))
    assert rel_inf(forcing, f_ref.numpy()) <= 1e-5 and rel_inf(T_out, T_ref.numpy()) <= 1e-5
    _check(ctx, d, th, cd, T, y, which, label="production", m=m)
    m.close()


# ---- 2. the net shapes of the forward's tcgen05 test, and every activation
@pytest.mark.parametrize("h1,h2,act", [(128, 128, "relu"), (128, 128, "mish"), (64, 48, "tanh"), (20, 100, "swish"), (8, 8, "relu"),
                                       (40, 40, "leakyrelu")])
def test_closure_vjp_net_shapes(ctx, h1, h2, act):
    d = t_only(h1, h2, act)
    th = syn.theta_random(d, scale=1.0)
    T, y = gyre_inputs(50, 2)
    cd = ClosureDesc(Nx=50, Ny=2, Nz=32)
    for which in ("forcing_bar", "both"):
        _check(ctx, d, th, cd, T, y, which, label=f"{h1}x{h2} {act}")


def test_closure_vjp_streamed_weights(ctx):
    d = t_only(192, 192, "relu")
    th = syn.theta_random(d, scale=1.0)
    m = engine.Model(ctx, d, th)
    line = [s for s in m.describe().splitlines() if "closure_vjp_kernel" in s]
    assert len(line) == 1 and "weights streamed from global memory" in line[0]
    T, y = gyre_inputs(40, 1)
    cd = ClosureDesc(Nx=40, Ny=1, Nz=32, dz=40.0, dt=1800.0, K=5.0)
    for which in ("forcing_bar", "both"):
        _check(ctx, d, th, cd, T, y, which, label="width-192", m=m)
    m.close()


# ---- 3. field sizes: a single column, ragged last tiles, and more tiles than SMs (persistent CTAs take several)
@pytest.mark.parametrize("nx,ny", [(1, 1), (31, 1), (33, 1), (512, 64)])
def test_closure_vjp_field_sizes(ctx, nx, ny):
    d = syn.free_convection_desc(ca=False)
    th = syn.theta_random(d, scale=1.0)
    T, y = gyre_inputs(nx, ny)
    cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
    m = engine.Model(ctx, d, th)
    for which in ("forcing_bar", "both"):
        _check(ctx, d, th, cd, T, y, which, label="size", m=m)
    m.close()


# ---- 4. one cotangent or both
@pytest.mark.parametrize("which", ["forcing_bar", "T_out_bar", "both"])
def test_closure_vjp_cotangent_modes(ctx, which):
    d = syn.free_convection_desc(ca=False)
    th = syn.theta_random(d, scale=1.0)
    T, y = gyre_inputs(37, 2)
    cd = ClosureDesc(Nx=37, Ny=2, Nz=32)
    assert _adjusted(d, th, cd, T, y)
    _, _, Tb, tb = _check(ctx, d, th, cd, T, y, which, label=which)
    if which == "T_out_bar":
        assert np.all(tb == 0)  # the net acts on the forcing only
    assert np.abs(Tb).max() > 0


# ---- 5. exact properties
def _setup(nx=48, ny=4):
    d = syn.free_convection_desc(ca=False)
    th = syn.theta_random(d, scale=1.0)
    T, y = gyre_inputs(nx, ny)
    cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
    fb, ob = cots(d, th, cd, T, y, "both")
    return d, th, cd, T, y, fb, ob


def test_closure_vjp_is_linear_in_the_cotangents(ctx):
    d, th, cd, T, y, fb, ob = _setup()
    m = engine.Model(ctx, d, th)
    both = m.closure_step_vjp(cd, T, fb, ob)
    only_f = m.closure_step_vjp(cd, T, fb, None)
    only_y = m.closure_step_vjp(cd, T, None, ob)
    scaled = m.closure_step_vjp(cd, T, 2 * fb, 2 * ob)
    half = m.closure_step_vjp(cd, T, 0.5 * fb, None)
    m.close()
    assert rel_inf(both[0], only_f[0] + only_y[0]) <= 1e-5
    assert np.array_equal(both[1], only_f[1]) and np.all(only_y[1] == 0)  # theta_bar comes from forcing_bar alone
    # scaling the cotangents by a power of two scales the outputs exactly
    assert np.array_equal(scaled[0], 2 * both[0]) and np.array_equal(scaled[1], 2 * both[1])
    assert np.array_equal(half[0], 0.5 * only_f[0]) and np.array_equal(half[1], 0.5 * only_f[1])


def test_closure_vjp_slab_decomposition(ctx):
    """theta_bar of a field is the sum of theta_bar over y-slab shards; a column's T_bar does not depend on the slab it is in
    (bitwise)."""
    d, th, cd, T, y, fb, ob = _setup(nx=48, ny=4)
    m = engine.Model(ctx, d, th)
    Tb, tb = m.closure_step_vjp(cd, T, fb, ob)
    tsum = np.zeros_like(tb, dtype=np.float64)
    for j0, j1 in ((0, 1), (1, 3), (3, 4)):
        cds = ClosureDesc(Nx=48, Ny=j1 - j0, Nz=32)
        sl = (slice(None), slice(j0, j1))
        Ts, ts = m.closure_step_vjp(cds, T[sl], fb[sl], ob[sl])
        assert np.array_equal(Ts, Tb[sl])
        tsum += ts
    m.close()
    assert rel_inf(tsum, tb) <= 1e-6


def test_closure_vjp_host_equals_device_and_leaves_the_step_unchanged(ctx):
    d, th, cd, T, y, fb, ob = _setup(nx=40, ny=3)
    m = engine.Model(ctx, d, th)
    f0, o0 = m.closure_step(cd, T, y)
    Tb, tb = m.closure_step_vjp(cd, T, fb, ob)
    dev = torch.device("cuda:0")
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    Td, fbd, obd = (tt(a) for a in (T, fb, ob))
    Tbd, tbd = torch.empty_like(Td), torch.empty(m.P, device=dev)
    torch.cuda.synchronize()
    m.closure_step_vjp_dev(cd, Td, fbd, obd, Tbd, tbd)
    m.ctx.synchronize()
    assert np.array_equal(Tbd.cpu().numpy(), Tb) and np.array_equal(tbd.cpu().numpy(), tb)
    f1, o1 = m.closure_step(cd, T, y)
    m.close()
    assert np.array_equal(f0, f1) and np.array_equal(o0, o1)


# ---- 6. an a-posteriori gradient through a few host steps, with torch autograd around the device flavours
def test_closure_vjp_a_posteriori_gradient_through_autograd(ctx):
    """A loss on T after three host steps (closure step, then bench.py's stand-in dynamics T <- T' + dt forcing)
    differentiated in theta by torch autograd over free_convection.closure_step_autograd, against FP64 autograd of the same
    chain on the oracle. The oracle chain is evaluated along the engine's frames (value of the engine's T, derivative of the
    oracle's chain), so that a rounding-level difference cannot flip the convective-adjustment switch between the two."""
    d = syn.free_convection_desc(ca=False)
    th = syn.theta_random(d, scale=1.0)
    nx, ny, n_steps = 16, 2, 3
    T, y = gyre_inputs(nx, ny)
    cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
    w = np.random.default_rng(3).standard_normal((32, ny, nx))

    def chain(step, theta, x, frames=None):
        seen = []
        for k in range(n_steps):
            if frames is not None:
                x = x + (torch.as_tensor(frames[k], dtype=x.dtype) - x).detach()
            seen.append(x.detach().cpu().numpy())
            forcing, T_out = step(theta, x)
            x = T_out + cd.dt * forcing
        return (x * torch.as_tensor(w, dtype=x.dtype, device=x.device)).sum(), seen

    m = engine.Model(ctx, d, th)
    dev = torch.device("cuda:0")
    tht = torch.tensor(th, device=dev, requires_grad=True)
    yd = torch.from_numpy(y).to(dev)
    loss, frames = chain(lambda theta, x: fc.closure_step_autograd(m, cd, theta, x, yd), tht, torch.from_numpy(T).to(dev))
    loss.backward()
    g = tht.grad.cpu().numpy()
    m.close()
    assert np.abs(frames[-1] - frames[0]).max() > 1e-2  # the steps move T

    def oracle_grad(dtype):
        t = torch.tensor(th, dtype=dtype, requires_grad=True)
        yy = torch.tensor(y, dtype=dtype)
        L, _ = chain(lambda theta, x: nde.closure_step(d, theta, cd, x, yy), t, torch.tensor(T, dtype=dtype), frames)
        return torch.autograd.grad(L, t)[0].numpy()

    ref, ref32 = oracle_grad(torch.float64), oracle_grad(torch.float32)
    err, floor = rel_inf(g, ref), rel_inf(ref32, ref)
    print(f"a-posteriori theta gradient through {n_steps} gyre steps: {err:.2e} (fp32-oracle {floor:.2e})")
    assert err <= max(TOL, floor)


# ---- 7. argument checks
def test_closure_vjp_refusals(ctx):
    z = np.zeros((32, 1, 4), dtype=np.float32)
    cd = ClosureDesc(Nx=4, Ny=1, Nz=32)

    def refused(d, th, words, **kw):
        m = engine.Model(ctx, d, th)
        args = dict(forcing_bar=z, T_out_bar=z)
        args.update(kw)
        with pytest.raises(engine.CpzError) as ei:
            m.closure_step_vjp(cd, z, **args)
        m.close()
        assert ei.value.code == engine.ERR_INVALID and words in str(ei.value), str(ei.value)

    d = syn.free_convection_desc(ca=False)
    th = syn.theta_random(d)
    # 400-wide layers: the T-only net has no adjoint plan, refused with the planner's reason
    dl = t_only(400, 400, "relu")
    thl = syn.theta_random(dl, scale=0.1)
    ml = engine.Model(ctx, dl, thl)
    desc = ml.describe()
    ml.close()
    assert "adjoint plan: unavailable (" in desc and "closure_vjp_kernel" not in desc
    reason = desc.split("adjoint plan: unavailable (")[1].split("\n")[0][:-1]
    refused(dl, thl, "adjoint plan unavailable: " + reason)
    refused(d, th, "no output requested", want_T=False, want_theta=False)
    refused(d, th, "no cotangent given", forcing_bar=None, T_out_bar=None)
    du = syn.wind_mixing_desc(variant=RHS_INFER)
    refused(du, syn.theta_random(du, scale=0.5), "T-only model with one net")
