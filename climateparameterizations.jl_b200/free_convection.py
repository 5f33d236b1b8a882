"""Host-side mirror of the FreeConvection NDE interface (free_convection/src/FreeConvection.jl:3-23), backed by libcpz.so.

FreeConvectionNDE / ConvectiveAdjustmentNDE build the T-only problem (free_convection_nde.jl:1-47,
convective_adjustment_nde.jl:1-57); FreeConvectionNDEParameters packs [bottom_flux, top_flux, σ_T, σ_wT, H, τ]
(:49-62); solve_nde integrates (solve.jl:1-51); train_neural_differential_equation is training.jl:44-74.
Batched over simulations; fixed-step explicit time stepping (see wind_mixing.py header).
"""
from __future__ import annotations

import logging
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import engine
from .desc import FLAG_CA, RHS_FREE_CONVECTION, ModelDesc
from .flux import ADAM, Chain, destructure
from .ocean_parameterizations import ZeroMeanUnitVarianceScaling
from .wind_mixing import _integrator

log = logging.getLogger("FreeConvection")


@dataclass
class FreeConvectionDataset:
    """One simulation's inputs as the NDE constructors read them from `ds` (free_convection_nde.jl:4-14,49-62):
    T [Nt, Nz] (deg C), wT bottom value and the imposed surface temperature flux, zf[0] (= -H), times [Nt] seconds."""
    T: np.ndarray
    wT_bottom: float
    temperature_flux: float
    H: float
    times: np.ndarray


@dataclass
class NDEProblem:
    """The ODEProblem returned by FreeConvectionNDE / ConvectiveAdjustmentNDE, reduced to what the engine needs."""
    nn: Chain
    convective_adjustment: bool
    Nz: int
    Nt: int
    H: float
    tau: float
    iterations: np.ndarray  # 0-based frame indices to save


def _problem(NN: Chain, ds: FreeConvectionDataset, iterations, ca: bool) -> NDEProblem:
    Nt, Nz = ds.T.shape
    its = np.arange(Nt) if iterations is None else np.asarray(iterations, dtype=np.int64)
    return NDEProblem(NN, ca, Nz, Nt, float(ds.H), float(ds.times[-1]), its)


def FreeConvectionNDE(NN: Chain, ds: FreeConvectionDataset, iterations=None) -> NDEProblem:
    return _problem(NN, ds, iterations, False)


def ConvectiveAdjustmentNDE(NN: Chain, ds: FreeConvectionDataset, iterations=None) -> NDEProblem:
    return _problem(NN, ds, iterations, True)


def FreeConvectionNDEParameters(ds: FreeConvectionDataset, T_scaling, wT_scaling) -> np.ndarray:
    """[bottom_flux, top_flux, σ_T, σ_wT, H, τ] (free_convection_nde.jl:49-62)"""
    return np.array([wT_scaling(ds.wT_bottom), wT_scaling(ds.temperature_flux), T_scaling.sigma, wT_scaling.sigma, ds.H,
                     ds.times[-1]], dtype=np.float32)


def _desc(nde: NDEProblem, T_scaling, wT_scaling, integrator: str, n_substeps: Optional[int], K: float = 10.0) -> ModelDesc:
    its = nde.iterations
    stride = int(its[1] - its[0]) if len(its) > 1 else 1
    if len(its) > 1 and np.any(np.diff(its) != stride):
        raise ValueError("the fixed-step engine needs uniformly strided iterations")
    n_steps = int(its[-1] - its[0]) if len(its) > 1 else 1
    mu = [0, 0, T_scaling.mu, 0, 0, wT_scaling.mu]
    sg = [1, 1, T_scaling.sigma, 1, 1, wT_scaling.sigma]
    d = ModelDesc(Nz=nde.Nz, n_fields=1, variant=RHS_FREE_CONVECTION, flags=(FLAG_CA if nde.convective_adjustment else 0),
                  nets=[nde.nn.net_desc()], H=nde.H, tau=nde.tau, mu=mu, sigma=sg, K_ca=K, integrator=integrator,
                  dt=1.0 / nde.Nt, t0=float(its[0]) / nde.Nt,  # tspan = (0, max(iterations)/Nt), free_convection_nde.jl:40
                  n_steps=n_steps, save_stride=stride, ckpt_stride=stride)
    if n_substeps is None:
        from .synthetic import n_substeps_for
        n_substeps = n_substeps_for(d)
    d.n_substeps = n_substeps
    return d


def solve_nde(ndes: Sequence[NDEProblem], NN: Chain, T0: np.ndarray, alg, nde_params: np.ndarray, T_scaling, wT_scaling,
              ctx: Optional[engine.Context] = None, n_substeps: Optional[int] = None) -> np.ndarray:
    """solve.jl:1-6 for a batch: T0 [n_sim, Nz] scaled, nde_params [n_sim, 6] -> scaled T [n_sim, n_saved, Nz]."""
    own = ctx is None
    ctx = ctx or engine.Context(0)
    d = _desc(ndes[0], T_scaling, wT_scaling, _integrator(alg), n_substeps)
    m = engine.Model(ctx, d, destructure(NN)[0])
    try:
        return m.solve(np.atleast_2d(T0), np.ascontiguousarray(np.atleast_2d(nde_params)[:, :2], dtype=np.float32))
    finally:
        m.close()
        if own:
            ctx.close()


def solve_nde_dataset(ds: FreeConvectionDataset, NN: Chain, NDEType, algorithm, T_scaling, wT_scaling, T0: Optional[np.ndarray] = None,
                      ctx: Optional[engine.Context] = None, n_substeps: Optional[int] = None) -> Dict[str, np.ndarray]:
    """The six-argument solve_nde (free_convection/src/solve.jl:8-51): integrate one dataset's NDE, reconstruct the total
    temperature flux wT = [bottom; NN(T_n); top] (minus min(0, 10 dT/dz) for ConvectiveAdjustmentNDE) at every saved frame
    and unscale both. Returns {"T": [Nt, Nz] deg C, "wT": [Nt, Nz+1]}. The per-frame NN evaluations run on the device in
    one batched cpz_predict_flux call over all frames."""
    own = ctx is None
    ctx = ctx or engine.Context(0)
    nde = NDEType(NN, ds)
    params = FreeConvectionNDEParameters(ds, T_scaling, wT_scaling)
    if T0 is None:
        T0 = T_scaling(ds.T[0])  # :28-30
    d = _desc(nde, T_scaling, wT_scaling, _integrator(algorithm), n_substeps)
    m = engine.Model(ctx, d, destructure(NN)[0])
    try:
        bcs = np.ascontiguousarray(params[None, :2], dtype=np.float32)
        T = m.solve(np.atleast_2d(np.asarray(T0, dtype=np.float32)), bcs)[0]          # [Nt, Nz] scaled
        wT = m.predict_flux(T, np.repeat(bcs, T.shape[0], axis=0))[:, 0, :]            # [Nt, Nz+1] scaled
        return {"T": T_scaling.unscale(T), "wT": wT_scaling.unscale(wT)}  # inv(T_scaling).(T), :50
    finally:
        m.close()
        if own:
            ctx.close()


def masked_weight_penalty(NN: Chain, layer: int, mask: np.ndarray):
    """causal_penalty() = sum(abs2, NN[layer].W[mask]) of train_free_convection_nde.jl:190-195 with its gradient, as a
    function of the destructured parameter vector."""
    off = 0
    for i, l in enumerate(NN.layers):
        if i == layer:
            break
        off += l.n_in * l.n_out + l.n_out
    L = NN.layers[layer]
    mflat = np.asarray(mask, dtype=bool).reshape(L.n_out, L.n_in).flatten(order="F")  # vec(W) is column-major (out x in)
    idx = off + np.nonzero(mflat)[0]

    def penalty(theta):
        g = np.zeros_like(theta, dtype=np.float64)
        g[idx] = 2.0 * theta[idx]
        return float(np.sum(theta[idx].astype(np.float64) ** 2)), g

    return penalty


def train_neural_differential_equation(NN: Chain, NDEType, algorithm, datasets: Dict[int, FreeConvectionDataset], T_scaling,
                                       wT_scaling, iterations, opt: ADAM, epochs: int, history: Optional[List[float]] = None,
                                       ctx: Optional[engine.Context] = None, n_substeps: Optional[int] = None,
                                       causal_penalty=None) -> Chain:
    """training.jl:44-74: loss = Flux.mse over all simulations' saved frames (+ causal_penalty(NN) when given, :57-58);
    one ADAM step per epoch (Flux.train! over Iterators.repeated((), epochs)). Returns the trained Chain (the reference
    mutates NN in place).
    causal_penalty: callable(theta) -> (value, d value / d theta) on the destructured parameter vector — the reference
    passes a closure over NN and lets Zygote differentiate it (train_free_convection_nde.jl:195:
    `sum(abs2, NN[i].W[mask])`); without an AD system the caller supplies the gradient, see `masked_weight_penalty`."""
    own = ctx is None
    ctx = ctx or engine.Context(0)
    ids = sorted(datasets.keys())
    ndes = [NDEType(NN, datasets[i], iterations) for i in ids]
    params = np.stack([FreeConvectionNDEParameters(datasets[i], T_scaling, wT_scaling) for i in ids])
    its = ndes[0].iterations
    T0 = np.stack([T_scaling(datasets[i].T[its[0]]) for i in ids]).astype(np.float32)
    true_sols = np.stack([T_scaling(datasets[i].T[its]) for i in ids]).astype(np.float32)
    d = _desc(ndes[0], T_scaling, wT_scaling, _integrator(algorithm), n_substeps)
    theta, re = destructure(NN)
    m = engine.Model(ctx, d, theta)
    w = np.array([0, 0, 1, 0, 0, 0], dtype=np.float32)
    bcs = np.ascontiguousarray(params[:, :2], dtype=np.float32)
    try:
        if opt.state:
            m.set_adam_state(opt.state["m"], opt.state["v"], opt.state["beta_pow"])
        for e in range(epochs):
            if causal_penalty is None:
                l = m.train_step(T0, bcs, true_sols, w, opt.eta, opt.beta[0], opt.beta[1], opt.eps)
                total = float(l[6])
            else:
                # gradient of the data term from the device, penalty term and its gradient from the caller, then the same
                # Flux-0.11 ADAM arithmetic as cpz_train_step on the combined gradient (a P-vector update per epoch)
                th = m.get_theta()
                l, g = m.loss_grad(T0, bcs, true_sols, w)
                pv, pg = causal_penalty(th)
                total = float(l[6]) + float(pv)
                mt, vt, bp = m.adam_state()
                if bp[0] == 0 and bp[1] == 0:
                    bp = np.array(opt.beta, dtype=np.float32)
                gg = g.astype(np.float64) + np.asarray(pg, dtype=np.float64)
                mt = opt.beta[0] * mt + (1 - opt.beta[0]) * gg
                vt = opt.beta[1] * vt + (1 - opt.beta[1]) * gg * gg
                th = th - mt / (1 - bp[0]) / (np.sqrt(vt / (1 - bp[1])) + opt.eps) * opt.eta
                m.set_theta(th.astype(np.float32))
                m.set_adam_state(mt.astype(np.float32), vt.astype(np.float32), np.array([bp[0] * opt.beta[0], bp[1] * opt.beta[1]], dtype=np.float32))
            log.info("Training free convection NDE... MSE loss: %.12e", total)
            if history is not None:
                history.append(total)
        mm, vv, bp = m.adam_state()
        opt.state = {"m": mm, "v": vv, "beta_pow": bp}
        return re(m.get_theta())
    finally:
        m.close()
        if own:
            ctx.close()


def closure_step_autograd(model: engine.Model, cdesc, theta, T, y):
    """One gyre closure step (cpz_closure_step_dev) as a torch autograd node whose backward is cpz_closure_step_vjp_dev:
    (forcing [Nz,Ny,Nx], T' [Nz,Ny,Nx]) of a CUDA float32 field T [Nz,Ny,Nx] and y [Ny] on the model's device. `theta` ([P]
    tensor) is copied into the model first and receives theta_bar; T receives T_bar, y no cotangent (it enters the forcing
    additively). A host model written in torch can chain through several closure steps and train the T-only net
    "a posteriori" on the discretisation it is deployed in."""
    global _CLOSURE_STEP
    if _CLOSURE_STEP is None:  # built on first use: importing this module does not import torch
        _CLOSURE_STEP = _closure_autograd_function()
    return _CLOSURE_STEP.apply(model, cdesc, theta, T, y)


_CLOSURE_STEP = None


def _closure_autograd_function():
    import torch

    class ClosureStep(torch.autograd.Function):
        @staticmethod
        def forward(fctx, model, cdesc, theta, T, y):
            model.set_theta(theta.detach().float().cpu().numpy())
            T = T.detach().float().contiguous()
            y = y.detach().float().contiguous()
            forcing = torch.empty_like(T)
            T_out = torch.empty_like(T)
            torch.cuda.synchronize(T.device)
            model.closure_step_dev(cdesc, T, y, forcing, T_out)
            model.ctx.synchronize()
            fctx.model, fctx.cdesc, fctx.theta_meta = model, cdesc, (theta.dtype, theta.device)
            fctx.save_for_backward(T)
            return forcing, T_out

        @staticmethod
        def backward(fctx, forcing_bar, T_out_bar):
            (T,) = fctx.saved_tensors
            m = fctx.model
            fb = None if forcing_bar is None else forcing_bar.float().contiguous()
            ob = None if T_out_bar is None else T_out_bar.float().contiguous()
            if fb is None and ob is None:
                return None, None, None, None, None
            Tb = torch.empty_like(T)
            tb = torch.empty(m.P, device=T.device)
            torch.cuda.synchronize(T.device)
            m.closure_step_vjp_dev(fctx.cdesc, T, fb, ob, Tb, tb)
            m.ctx.synchronize()
            dtype, device = fctx.theta_meta
            return None, None, tb.to(dtype=dtype, device=device), Tb, None

    return ClosureStep
