"""Host-side mirror of the WindMixing NDE interface (wind_mixing/src/WindMixing.jl:3-23), backed by libcpz.so.

Same names, argument meaning and error behaviour as the reference functions, with two declared differences:
  * simulations are batched — every function takes/returns arrays with a leading column (simulation) axis and the
    engine integrates all of them at once, where the reference loops `for i in 1:n_simulations`
    (wind_mixing/src/NDE_training.jl:291);
  * time stepping is fixed-step explicit (Tsit5 / RK4 / Euler tableau, optional sub-steps) with the exact discrete
    adjoint, where the reference passes an adaptive OrdinaryDiffEq solver and a continuous adjoint.
Julia's 1-based, column-major (3Nz × Nt) matrices become (…, Nt, 3Nz) row-major arrays; `tsteps` are 0-based.
"""
from __future__ import annotations

import logging
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import engine
from .desc import (FLAG_CA, FLAG_DIURNAL, FLAG_MPP, FLAG_SMOOTH_NN, FLAG_SMOOTH_RI, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN,
                   ModelDesc)
from .flux import ADAM, Chain, destructure
from .ocean_parameterizations import Dc, Df, ZeroMeanUnitVarianceScaling

log = logging.getLogger("WindMixing")

LOSS_KEYS = ("u", "v", "T", "∂u∂z", "∂v∂z", "∂T∂z")
_INTEGRATORS = {"tsit5": "tsit5", "rk4": "rk4", "euler": "euler"}


def _integrator(timestepper) -> str:
    name = (timestepper if isinstance(timestepper, str) else type(timestepper).__name__).lower().replace("()", "")
    if name not in _INTEGRATORS:
        raise ValueError(f"timestepper {timestepper!r} is not available in the fixed-step engine; use Tsit5, RK4 or Euler "
                         "(adaptive/implicit OrdinaryDiffEq solvers such as ROCK4 are out of scope, see DESIGN.md)")
    return _INTEGRATORS[name]


@dataclass
class ProfileData:
    """What the NDE path reads from `WindMixing.data(...)` (wind_mixing/src/data_containers.jl:260-427), batched:
    uvT_scaled [n_sim, Nt, 3Nz], t [Nt] seconds, boundary fluxes scaled [n_sim, 6] = (uw_b, uw_t, vw_b, vw_t, wT_b, wT_t)
    taken at the first frame (NDE_training.jl:238-243), scalings name -> ZeroMeanUnitVarianceScaling, zF [Nz+1]."""
    uvT_scaled: np.ndarray
    t: np.ndarray
    bcs_scaled: np.ndarray
    scalings: Dict[str, ZeroMeanUnitVarianceScaling]
    zF: np.ndarray
    diurnal_Q: Optional[np.ndarray] = None

    @property
    def Nz(self) -> int:
        return self.uvT_scaled.shape[-1] // 3


# ---- loss.jl -------------------------------------------------------------------------------------------------------------
def loss(a, b) -> float:
    """Flux.mse (wind_mixing/src/loss.jl:1-3)"""
    return float(np.mean((np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64)) ** 2))


def calculate_loss_scalings(losses: Dict[str, float], fractions: Dict[str, float], train_gradient: bool) -> Dict[str, float]:
    """wind_mixing/src/loss.jl:11-31; fractions keys: T, ∂T∂z, profile."""
    velocity_scaling = (1 - fractions["T"]) / fractions["T"] * losses["T"] / (losses["u"] + losses["v"])
    profile_loss = velocity_scaling * (losses["u"] + losses["v"]) + losses["T"]
    if train_gradient:
        vgs = (1 - fractions["∂T∂z"]) / fractions["∂T∂z"] * losses["∂T∂z"] / (losses["∂u∂z"] + losses["∂v∂z"])
        gradient_loss = vgs * (losses["∂u∂z"] + losses["∂v∂z"]) + losses["∂T∂z"]
        tgs = (1 - fractions["profile"]) / fractions["profile"] * profile_loss / gradient_loss
    else:
        vgs = tgs = 0.0
    return {"u": velocity_scaling, "v": velocity_scaling, "T": 1.0, "∂u∂z": tgs * vgs, "∂v∂z": tgs * vgs, "∂T∂z": tgs}


def apply_loss_scalings(losses: Dict[str, float], scalings: Dict[str, float]) -> Dict[str, float]:
    """wind_mixing/src/loss.jl:33-42"""
    return {k: scalings[k] * losses[k] for k in LOSS_KEYS}


# ---- NDE_training.jl -----------------------------------------------------------------------------------------------------
def prepare_parameters_NDE_training(data: ProfileData, uw_NN: Chain, vw_NN: Chain, wT_NN: Chain, f, Nz, g, alpha, nu0, nu_m,
                                    Ric, dRi, Pr, kappa, conditions: dict):
    """wind_mixing/src/NDE_training.jl:1-44 — returns (constants, scalings, derivatives, NN_constructions, weights,
    NN_sizes, NN_ranges)."""
    H = abs(float(data.zF[-1] - data.zF[0]))
    tau = abs(float(data.t[-1] - data.t[0]))
    uw_w, re_uw = destructure(uw_NN)
    vw_w, re_vw = destructure(vw_NN)
    wT_w, re_wT = destructure(wT_NN)
    constants = dict(H=H, tau=tau, f=f, Nz=Nz, g=g, alpha=alpha)
    if conditions.get("modified_pacanowski_philander"):
        constants.update(nu0=nu0, nu_m=nu_m, Ric=Ric, dRi=dRi, Pr=Pr)
    if conditions.get("convective_adjustment"):
        constants.update(kappa=kappa)
    scalings = {k: data.scalings[k] for k in ("u", "v", "T", "uw", "vw", "wT")}
    derivatives = dict(cell=np.float32(Dc(Nz, 1 / Nz)), face=np.float32(Df(Nz, 1 / Nz)))
    NN_constructions = dict(uw=re_uw, vw=re_vw, wT=re_wT)
    weights = np.concatenate([uw_w, vw_w, wT_w]).astype(np.float32)
    sizes = dict(uw=len(uw_w), vw=len(vw_w), wT=len(wT_w))
    ranges = dict(uw=slice(0, sizes["uw"]), vw=slice(sizes["uw"], sizes["uw"] + sizes["vw"]),
                  wT=slice(sizes["uw"] + sizes["vw"], sizes["uw"] + sizes["vw"] + sizes["wT"]))
    return constants, scalings, derivatives, NN_constructions, weights, sizes, ranges


def _model_desc(nets: Sequence[Chain], constants: dict, scalings: dict, conditions: dict, variant: int, Nz: int,
                integrator: str, dt: float, t0: float, n_steps: int, n_substeps: int, save_stride: int,
                ckpt_stride: int) -> ModelDesc:
    flags = 0
    if conditions.get("modified_pacanowski_philander"): flags |= FLAG_MPP
    if conditions.get("convective_adjustment"): flags |= FLAG_CA
    if conditions.get("zero_weights"): flags |= FLAG_ZERO_WEIGHTS
    if conditions.get("smooth_NN"): flags |= FLAG_SMOOTH_NN
    if conditions.get("smooth_Ri"): flags |= FLAG_SMOOTH_RI
    if conditions.get("diurnal"): flags |= FLAG_DIURNAL
    names = ("u", "v", "T", "uw", "vw", "wT")
    return ModelDesc(Nz=Nz, n_fields=3, variant=variant, flags=flags, nets=[n.net_desc() for n in nets],
                     H=constants["H"], tau=constants["tau"], f=constants["f"], g=constants["g"], alpha=constants["alpha"],
                     nu0=constants.get("nu0", 1e-4), nu_m=constants.get("nu_m", 0.1), Ric=constants.get("Ric", 0.25),
                     dRi=constants.get("dRi", 0.1), Pr=constants.get("Pr", 1.0), kappa=constants.get("kappa", 10.0),
                     mu=[scalings[k].mu for k in names], sigma=[scalings[k].sigma for k in names], integrator=integrator,
                     dt=dt, t0=t0, n_steps=n_steps, n_substeps=n_substeps, save_stride=save_stride, ckpt_stride=ckpt_stride)


def NDE(x, p, t, NN_sizes, nets: Sequence[Chain], conditions, scalings, constants, ctx: engine.Context, diurnal_Q=None):
    """RHS seam f(x, p, t) -> dx (wind_mixing/src/NDE_training.jl:56-81): p = [theta_uw; theta_vw; theta_wT; 6 BCs]
    per column. x [ncol, 3Nz], p [ncol, P+6] (theta taken from the first row) -> [ncol, 3Nz]."""
    x = np.atleast_2d(np.asarray(x, dtype=np.float32))
    p = np.atleast_2d(np.asarray(p, dtype=np.float32))
    P = sum(NN_sizes.values())
    d = _model_desc(nets, constants, scalings, conditions, RHS_TRAIN, constants["Nz"], "tsit5", 1.0, 0.0, 1, 1, 1, 1)
    m = engine.Model(ctx, d, p[0, :P])
    try:
        return m.rhs(x, p[:, P:P + 6], t=float(t), Q=diurnal_Q)
    finally:
        m.close()


def predict_NDE(uw_NN, vw_NN, wT_NN, x, BCs, conditions, scalings, constants, ctx: engine.Context, t: float = 0.0):
    """wind_mixing/src/NDE_training.jl:149-165 for a batch: x [ncol, 3Nz], BCs [ncol, 6] -> d(uvT)/dt [ncol, 3Nz]."""
    nets = (uw_NN, vw_NN, wT_NN)
    theta = np.concatenate([destructure(n)[0] for n in nets])
    d = _model_desc(nets, constants, scalings, conditions, RHS_TRAIN, constants["Nz"], "tsit5", 1.0, 0.0, 1, 1, 1, 1)
    m = engine.Model(ctx, d, theta)
    try:
        return m.rhs(np.atleast_2d(x), np.atleast_2d(BCs), t=t)
    finally:
        m.close()


def _time_grid(t: np.ndarray, tsteps: Sequence[int], tau: float) -> Tuple[float, float, int, int]:
    tsteps = np.asarray(tsteps, dtype=np.int64)
    assert tsteps.ndim == 1 and len(tsteps) >= 2, "tsteps needs at least two frames"
    stride = int(tsteps[1] - tsteps[0])
    if stride <= 0 or np.any(np.diff(tsteps) != stride):
        raise ValueError("the fixed-step engine needs uniformly strided tsteps (e.g. range(0, 1153, 9))")
    dts = np.diff(np.asarray(t, dtype=np.float64))
    if np.abs(dts - dts[0]).max() > 1e-6 * abs(dts[0]):
        raise ValueError("frame times must be uniformly spaced")
    return float(dts[0] / tau), float((t[tsteps[0]] - 0.0) / tau), int(tsteps[-1] - tsteps[0]), stride


def default_substeps(constants: dict, conditions: dict, dt_hat: float, Nz: int, integrator: str) -> int:
    """Sub-steps keeping nu_max*dt/dz^2 inside the explicit stability interval (SURVEY 7 'Stiffness')."""
    lim = {"tsit5": 0.8, "rk4": 0.65, "euler": 0.45}[integrator]
    nu = 0.0
    if conditions.get("modified_pacanowski_philander"):
        nu = constants.get("nu0", 0.0) + constants.get("nu_m", 0.0)
    if conditions.get("convective_adjustment"):
        nu = max(nu, constants.get("kappa", 0.0))
    dz = constants["H"] / Nz
    return max(1, int(np.ceil(nu * dt_hat * constants["tau"] / dz ** 2 / lim)))


@dataclass
class TrainingRecord:
    """What write_data_NDE_training appends per iteration (wind_mixing/src/data_writing.jl:28-78)."""
    losses: List[Dict[str, float]] = field(default_factory=list)
    totals: List[float] = field(default_factory=list)
    loss_scalings: Optional[Dict[str, float]] = None
    adam_state: Optional[dict] = None


def train_NDE(uw_NN: Chain, vw_NN: Chain, wT_NN: Chain, data: ProfileData, tsteps, timestepper, optimizers: Sequence[ADAM],
              epochs: int, FILE_PATH=None, stage=1, *, maxiters=500, nu0=1e-4, nu_m=1e-1, dRi=1.0, Ric=0.25, Pr=1.0,
              kappa=10.0, f=1e-4, alpha=2e-4, g=9.80665, modified_pacanowski_philander=False, convective_adjustment=False,
              smooth_profile=False, smooth_NN=False, smooth_Ri=False, train_gradient=False, zero_weights=False,
              gradient_scaling=5e-3, training_fractions=None, diurnal=False, ctx: Optional[engine.Context] = None,
              n_substeps: Optional[int] = None, ckpt_stride: Optional[int] = None,
              callback: Optional[Callable] = None, record: Optional[TrainingRecord] = None):
    """wind_mixing/src/NDE_training.jl:167-374. Returns the three trained Chains (rebuilt from the best-loss theta,
    as GalacticOptim's `res.minimizer` is, :371-373)."""
    # :171, :192-194
    assert not modified_pacanowski_philander or not convective_adjustment
    if zero_weights:
        assert modified_pacanowski_philander
    own_ctx = ctx is None
    ctx = ctx or engine.Context(0)
    Nz = data.Nz
    conditions = dict(modified_pacanowski_philander=modified_pacanowski_philander, convective_adjustment=convective_adjustment,
                      smooth_profile=smooth_profile, smooth_NN=smooth_NN, smooth_Ri=smooth_Ri, train_gradient=train_gradient,
                      zero_weights=zero_weights, diurnal=diurnal)
    constants, scalings, derivatives, NN_constructions, weights, NN_sizes, NN_ranges = prepare_parameters_NDE_training(
        data, uw_NN, vw_NN, wT_NN, f, Nz, g, alpha, nu0, nu_m, Ric, dRi, Pr, kappa, conditions)
    integrator = _integrator(timestepper)
    dt_hat, t0, n_steps, stride = _time_grid(data.t, tsteps, constants["tau"])
    nsub = n_substeps or default_substeps(constants, conditions, dt_hat, Nz, integrator)
    tsteps = np.asarray(tsteps)
    uvT0 = np.ascontiguousarray(data.uvT_scaled[:, tsteps[0]], dtype=np.float32)           # :220
    targets = np.ascontiguousarray(data.uvT_scaled[:, tsteps], dtype=np.float32)           # :222
    BCs = np.ascontiguousarray(data.bcs_scaled, dtype=np.float32)                           # :238-243
    Q = data.diurnal_Q if diurnal else None
    d = _model_desc((uw_NN, vw_NN, wT_NN), constants, scalings, conditions, RHS_TRAIN, Nz, integrator, dt_hat, t0, n_steps,
                    nsub, stride, ckpt_stride or stride)
    model = engine.Model(ctx, d, weights)

    def unit_losses(want: bool = True) -> Dict[str, float]:
        w = np.array([1, 1, 1, 1, 1, 1] if train_gradient else [1, 1, 1, 0, 0, 0], dtype=np.float32)
        l, _ = model.loss_grad(uvT0, BCs, targets, w, Q=Q, want_grad=False)
        return dict(zip(LOSS_KEYS, map(float, l[:6])))

    # determine_loss_scalings :256-288
    if training_fractions is None:
        gs = gradient_scaling if train_gradient else 0.0
        loss_scalings = {"u": 1.0, "v": 1.0, "T": 1.0, "∂u∂z": gs, "∂v∂z": gs, "∂T∂z": gs}
    else:
        loss_scalings = calculate_loss_scalings(unit_losses(), training_fractions, train_gradient)
        if not train_gradient:
            loss_scalings.update({"∂u∂z": 0.0, "∂v∂z": 0.0, "∂T∂z": 0.0})
    w = np.array([loss_scalings[k] for k in LOSS_KEYS], dtype=np.float32)
    record = record if record is not None else TrainingRecord()
    record.loss_scalings = loss_scalings

    best_theta, best_loss = weights.copy(), np.inf
    try:
        for i, opt in enumerate(optimizers):
            resume = opt.state  # a state the CALLER attached (checkpoint/resume); consumed by this optimizer's first epoch
            for epoch in range(1, epochs + 1):
                # Every `solve(prob, opt, ...)` of the reference copies theta (GalacticOptim 1.2.0), and Flux keys the ADAM
                # moments by array identity, so each epoch of each optimizer starts from zero moments and full bias
                # correction (NDE_training.jl:370); the device state is therefore reset here, never carried over from the
                # previous optimizer or epoch.
                if resume:
                    model.set_adam_state(resume["m"], resume["v"], resume["beta_pow"])
                    resume = None
                else:
                    model.reset_adam_state()
                for it in range(1, maxiters + 1):
                    theta_before = model.get_theta()
                    try:
                        l = model.train_step(uvT0, BCs, targets, w, opt.eta, opt.beta[0], opt.beta[1], opt.eps, Q=Q)
                    except engine.CpzError as e:
                        if e.code != engine.ERR_NONFINITE:
                            raise
                        raise FloatingPointError(f"non-finite loss at iteration {it}: reduce dt (n_substeps={nsub}) or the learning rate") from e
                    total = float(l[6])
                    losses = dict(zip(LOSS_KEYS, map(float, l[:6])))
                    if not np.isfinite(total):
                        raise FloatingPointError(f"non-finite loss at iteration {it}: reduce dt (n_substeps={nsub}) or the learning rate")
                    if total < best_loss:  # GalacticOptim keeps the best-seen parameters (loss is at theta BEFORE the update)
                        best_loss = total
                        best_theta = theta_before
                    # cb :343-369
                    prof = losses["u"] + losses["v"] + losses["T"]
                    grad = losses["∂u∂z"] + losses["∂v∂z"] + losses["∂T∂z"]
                    log.info("loss = %s: uvT%.3g%% grad%.3g%% %s opt%d/%d epoch%d/%d iter%d/%d", total, 100 * prof / total,
                             100 * grad / total, stage, i + 1, len(optimizers), epoch, epochs, it, maxiters)
                    record.losses.append(losses)
                    record.totals.append(total)
                    if FILE_PATH is not None:  # write_data_NDE_training inside cb (:364-366): the networks at the evaluated theta
                        from . import data_writing
                        data_writing.write_data_NDE_training(
                            FILE_PATH, losses, loss_scalings, NN_constructions["uw"](theta_before[NN_ranges["uw"]]),
                            NN_constructions["vw"](theta_before[NN_ranges["vw"]]), NN_constructions["wT"](theta_before[NN_ranges["wT"]]),
                            stage, opt, flush_every=25)
                    if callback is not None:
                        callback(theta_before, total, losses, loss_scalings)
                m_, v_, bp_ = model.adam_state()
                record.adam_state = {"m": m_, "v": v_, "beta_pow": bp_}  # what write_data_NDE_training checkpoints
                # weights .= res.minimizer  (:371): continue the next epoch from the best-seen theta
                final_theta = model.get_theta()
                l_final, _ = model.loss_grad(uvT0, BCs, targets, w, Q=Q, want_grad=False)
                if float(l_final[6]) < best_loss:
                    best_loss, best_theta = float(l_final[6]), final_theta
                model.set_theta(best_theta)
        weights = best_theta
    finally:
        model.close()
        if own_ctx:
            ctx.close()
        if FILE_PATH is not None:
            from . import data_writing
            data_writing.flush(FILE_PATH)
    return (NN_constructions["uw"](weights[NN_ranges["uw"]]), NN_constructions["vw"](weights[NN_ranges["vw"]]),
            NN_constructions["wT"](weights[NN_ranges["wT"]]))


# ---- training_postprocessing.jl --------------------------------------------------------------------------------------------
def prepare_BCs(data: ProfileData) -> np.ndarray:
    """wind_mixing/src/training_postprocessing.jl:35-53 — scaled boundary fluxes of the first frame, [n_sim, 6]."""
    return np.ascontiguousarray(data.bcs_scaled, dtype=np.float32)


def solve_NDE_mutating(uw_NN: Chain, vw_NN: Chain, wT_NN: Chain, scalings, constants, BCs, derivatives, uvT0, ts,
                       timestepper, conditions, ctx: Optional[engine.Context] = None, n_substeps: Optional[int] = None,
                       diurnal_Q=None) -> np.ndarray:
    """wind_mixing/src/training_postprocessing.jl:55-159 (inference RHS) for a batch of columns.
    uvT0 [ncol, 3Nz], BCs [ncol, 6], ts: uniformly spaced non-dimensional save times -> [ncol, len(ts), 3Nz].
    `derivatives` is accepted for signature compatibility; the engine applies Dᶜ/Dᶠ as stencils."""
    own_ctx = ctx is None
    ctx = ctx or engine.Context(0)
    ts = np.asarray(ts, dtype=np.float64)
    assert len(ts) >= 2
    dt = float(ts[1] - ts[0])
    if np.abs(np.diff(ts) - dt).max() > 1e-6 * abs(dt):
        raise ValueError("ts must be uniformly spaced")
    integrator = _integrator(timestepper)
    cond = dict(conditions)
    cond["modified_pacanowski_philander"] = True  # the mutating inference RHS always applies mPP (:114-128)
    nsub = n_substeps or default_substeps(constants, cond, dt, constants["Nz"], integrator)
    nets = (uw_NN, vw_NN, wT_NN)
    theta = np.concatenate([destructure(n)[0] for n in nets])
    d = _model_desc(nets, constants, scalings, cond, RHS_INFER, constants["Nz"], integrator, dt, float(ts[0]), len(ts) - 1, nsub, 1, 1)
    m = engine.Model(ctx, d, theta)
    try:
        return m.solve(np.atleast_2d(uvT0), np.atleast_2d(BCs), Q=diurnal_Q)
    finally:
        m.close()
        if own_ctx:
            ctx.close()


# ---- diffusivity_parameter_optimisation.jl ----------------------------------------------------------------------------------
MPP_KEYS = ("nu0", "nu_m", "dRi", "Ric", "Pr")


def DE(x, p, t, scalings, constants, BCs, ctx: engine.Context, conditions: Optional[dict] = None):
    """RHS of the NN-free base closure, p = (nu0, nu_m, dRi, Ric, Pr) (wind_mixing/src/diffusivity_parameter_optimisation.jl:1-33),
    batched: x [ncol, 3Nz], BCs [ncol, 6] -> [ncol, 3Nz]."""
    cond = dict(modified_pacanowski_philander=True, zero_weights=True)
    cond.update(conditions or {})
    c = dict(constants)
    c.update(dict(zip(MPP_KEYS, map(float, p))))
    d = _model_desc((), c, scalings, cond, RHS_TRAIN, constants["Nz"], "tsit5", 1.0, 0.0, 1, 1, 1, 1)
    m = engine.Model(ctx, d, np.zeros(0, dtype=np.float32))
    try:
        return m.rhs(np.atleast_2d(x), np.atleast_2d(BCs), t=float(t))
    finally:
        m.close()


def optimise_modified_pacanowski_philander(data: ProfileData, tsteps, timestepper, maxiters: int, *, nu0=1e-4, nu_m=1e-1, dRi=0.1,
                                           Ric=0.25, Pr=1.0, f=1e-4, alpha=2e-4, g=9.80665, train_gradient=True,
                                           gradient_scaling=5e-3, training_fractions=None, ctx: Optional[engine.Context] = None,
                                           n_substeps: Optional[int] = None, callback: Optional[Callable] = None,
                                           record: Optional[TrainingRecord] = None):
    """wind_mixing/src/diffusivity_parameter_optimisation.jl:35-235: fit the five mPP parameters of the NN-free column model
    to the profiles. As in the reference the optimiser works on p .* (1 ./ p_initial) inside the box [0, 10]^5
    (`OptimizationProblem(..., lb=0, ub=10)` with `LBFGS()`, optimise_modified_pacanowski_philander.jl:40); the box-constrained
    quasi-Newton iteration itself stays on the host (scipy L-BFGS-B), loss and gradient come from cpz_loss_grad_mpp.
    Returns (dict of fitted parameters, TrainingRecord). dRi and Pr are kept >= 1e-6 (they divide)."""
    from scipy.optimize import minimize

    own_ctx = ctx is None
    ctx = ctx or engine.Context(0)
    Nz = data.Nz
    H = abs(float(data.zF[-1] - data.zF[0]))
    tau = abs(float(data.t[-1] - data.t[0]))
    constants = dict(H=H, tau=tau, f=f, Nz=Nz, g=g, alpha=alpha, nu0=nu0, nu_m=nu_m, dRi=dRi, Ric=Ric, Pr=Pr)
    scalings = {k: data.scalings[k] for k in ("u", "v", "T", "uw", "vw", "wT")}
    conditions = dict(modified_pacanowski_philander=True, zero_weights=True)
    integrator = _integrator(timestepper)
    dt_hat, t0, n_steps, stride = _time_grid(data.t, tsteps, tau)
    p_init = np.array([nu0, nu_m, dRi, Ric, Pr], dtype=np.float64)
    if n_substeps is None:  # stable for diffusivities up to twice the initial nu0 + nu_m
        c2 = dict(constants); c2["nu_m"] = 2 * nu_m; c2["nu0"] = 2 * nu0
        n_substeps = default_substeps(c2, conditions, dt_hat, Nz, integrator)
    tsteps = np.asarray(tsteps)
    uvT0 = np.ascontiguousarray(data.uvT_scaled[:, tsteps[0]], dtype=np.float32)
    targets = np.ascontiguousarray(data.uvT_scaled[:, tsteps], dtype=np.float32)
    BCs = np.ascontiguousarray(data.bcs_scaled, dtype=np.float32)
    d = _model_desc((), constants, scalings, conditions, RHS_TRAIN, Nz, integrator, dt_hat, t0, n_steps, n_substeps, stride, stride)
    model = engine.Model(ctx, d, np.zeros(0, dtype=np.float32))
    record = record if record is not None else TrainingRecord()
    try:
        if training_fractions is None:
            gs = gradient_scaling if train_gradient else 0.0
            loss_scalings = {"u": 1.0, "v": 1.0, "T": 1.0, "∂u∂z": gs, "∂v∂z": gs, "∂T∂z": gs}
        else:
            wu = np.array([1, 1, 1, 1, 1, 1] if train_gradient else [1, 1, 1, 0, 0, 0], dtype=np.float32)
            l, _ = model.loss_grad(uvT0, BCs, targets, wu, want_grad=False)
            loss_scalings = calculate_loss_scalings(dict(zip(LOSS_KEYS, map(float, l[:6]))), training_fractions, train_gradient)
            if not train_gradient:
                loss_scalings.update({"∂u∂z": 0.0, "∂v∂z": 0.0, "∂T∂z": 0.0})
        record.loss_scalings = loss_scalings
        w = np.array([loss_scalings[k] for k in LOSS_KEYS], dtype=np.float32)
        best = {"loss": np.inf, "p": p_init.copy()}

        def fun(scaled):
            p = np.asarray(scaled, dtype=np.float64) * p_init  # unscale_parameter (:50-52)
            p[2] = max(p[2], 1e-6); p[4] = max(p[4], 1e-6)
            model.set_mpp_params(*p)
            l, gp, _ = model.loss_grad_mpp(uvT0, BCs, targets, w)
            total = float(l[6])
            losses = dict(zip(LOSS_KEYS, map(float, l[:6])))
            record.losses.append(losses); record.totals.append(total)
            if total < best["loss"]:
                best["loss"], best["p"] = total, p.copy()
            log.info("nu0 = %g, nu_m = %g, dRi = %g, Ric = %g, Pr = %g, loss = %g", *p, total)
            if callback is not None:
                callback(p, total, losses, loss_scalings)
            return total, gp.astype(np.float64) * p_init  # chain rule to the scaled parameters

        minimize(fun, np.ones(5), jac=True, method="L-BFGS-B", bounds=[(0.0, 10.0)] * 5, options={"maxiter": int(maxiters)})
        return dict(zip(MPP_KEYS, map(float, best["p"]))), record
    finally:
        model.close()
        if own_ctx:
            ctx.close()


# ---- the trained NDE embedded in a host ocean model (SURVEY 8f-2) -----------------------------------------------------

def _standin_dynamics(u, v, T, dz_flux, dt, f):
    """Stand-in for the host model's own time step between two callbacks (Oceananigans' IncompressibleModel is third-party
    and out of scope): forward Euler with the three NN forcings -dz_flux (NDE_oceananigans.jl:346-359) and the f-plane
    Coriolis terms (:366). Works on numpy arrays and torch tensors alike."""
    return (u + dt * (-dz_flux[0] + f * v), v + dt * (-dz_flux[1] - f * u), T + dt * (-dz_flux[2]))


def oceananigans_modified_pacanowski_philander_nn(model: engine.Model, cdesc, u, v, T, n_iterations: int, output_every: int = 10,
                                                  f: float = 1e-4, wT_flux: Optional[Callable[[float], float]] = None,
                                                  dynamics: Optional[Callable] = None) -> List[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
    """Mirror of the neural-network simulation of oceananigans_modified_pacanowski_philander_nn
    (wind_mixing/src/NDE_oceananigans.jl:103-475): every iteration the callback progress_neural_network (:380-405) — the
    three NN forcing chains on the current state, then the backward-Euler modified Pacanowski–Philander step — runs on the
    GPU through cpz_closure_step_uvt for every column of the (Nz, Ny, Nx) fields, and the host model advances the state with
    those forcings (`dynamics(u, v, T, dz_flux, dt, f)`; default: the forward-Euler stand-in above). A time-dependent top
    temperature flux is `wT_flux(t)` (:129,332). Returns the frames saved every `output_every` iterations (the reference
    writes every 600 s at dt = 60 s, :407-440), frame 0 = initial state."""
    import copy
    dyn = dynamics or _standin_dynamics
    cd = copy.copy(cdesc)
    u, v, T = (np.ascontiguousarray(a, dtype=np.float32) for a in (u, v, T))
    frames = [(u.copy(), v.copy(), T.copy())]
    for it in range(n_iterations):
        if wT_flux is not None:
            cd.wT_top = float(wT_flux(it * cd.dt))
        dz_flux, out = model.closure_step_uvt(cd, u, v, T)
        u, v, T = (np.ascontiguousarray(a, dtype=np.float32) for a in dyn(out[0], out[1], out[2], dz_flux, cd.dt, f))
        if (it + 1) % output_every == 0:
            frames.append((u.copy(), v.copy(), T.copy()))
    return frames


def closure_step_uvt_autograd(model: engine.Model, cdesc, theta, u, v, T):
    """One embedded closure step (cpz_closure_step_uvt_dev) as a torch autograd node whose backward is
    cpz_closure_step_uvt_vjp_dev: (dz_flux [3,Nz,Ny,Nx], uvT' [3,Nz,Ny,Nx]) of CUDA float32 fields [Nz,Ny,Nx] on the model's
    device. `theta` ([P] tensor) is copied into the model first and receives theta_bar; u, v, T receive their cotangents. A host
    model written in torch can chain through several closure steps and train the nets "a posteriori" on the discretisation
    they are deployed in."""
    global _CLOSURE_STEP_UVT
    if _CLOSURE_STEP_UVT is None:  # built on first use: importing this module does not import torch
        _CLOSURE_STEP_UVT = _closure_autograd_function()
    return _CLOSURE_STEP_UVT.apply(model, cdesc, theta, u, v, T)


_CLOSURE_STEP_UVT = None


def _closure_autograd_function():
    import torch

    class ClosureStepUvt(torch.autograd.Function):
        @staticmethod
        def forward(fctx, model, cdesc, theta, u, v, T):
            model.set_theta(theta.detach().float().cpu().numpy())
            u, v, T = (a.detach().float().contiguous() for a in (u, v, T))
            dzf = torch.empty((3,) + tuple(u.shape), device=u.device)
            out = torch.empty_like(dzf)
            torch.cuda.synchronize(u.device)
            model.closure_step_uvt_dev(cdesc, u, v, T, dzf, out)
            model.ctx.synchronize()
            fctx.model, fctx.cdesc, fctx.theta_meta = model, cdesc, (theta.dtype, theta.device)
            fctx.save_for_backward(u, v, T)
            return dzf, out

        @staticmethod
        def backward(fctx, dzf_bar, out_bar):
            u, v, T = fctx.saved_tensors
            m = fctx.model
            fb = None if dzf_bar is None else dzf_bar.float().contiguous()
            ob = None if out_bar is None else out_bar.float().contiguous()
            if fb is None and ob is None:
                return None, None, None, None, None, None
            xb = torch.empty((3,) + tuple(u.shape), device=u.device)
            tb = torch.empty(m.P, device=u.device)
            torch.cuda.synchronize(u.device)
            m.closure_step_uvt_vjp_dev(fctx.cdesc, u, v, T, fb, ob, xb[0], xb[1], xb[2], tb)
            m.ctx.synchronize()
            dtype, device = fctx.theta_meta
            return None, None, tb.to(dtype=dtype, device=device), xb[0], xb[1], xb[2]

    return ClosureStepUvt



def solve_autograd(model: engine.Model, theta, x0, bcs, Q=None, p=None):
    """The batched solve (cpz_solve_dev) as a torch autograd node for any model, u/v/T or T-only: traj [ncol, n_saved, S] of
    CUDA float32 x0 [ncol, S] and bcs [ncol, n_bc] (and diurnal amplitudes Q [ncol]) on the model's device. `theta` ([P]
    tensor) is copied into the model first; `p` (optional [5] tensor (nu0, nu_m, dRi, Ric, Pr)) sets the mPP parameters.
    Reverse mode runs cpz_solve_vjp_dev (theta, x0 and p receive their cotangents), forward mode (torch.autograd.forward_ad,
    torch.func.jvp) cpz_solve_jvp_dev with the tangents of theta, x0 and p. bcs and Q are data: they get no derivative."""
    global _SOLVE
    if _SOLVE is None:  # built on first use: importing this module does not import torch
        _SOLVE = _solve_autograd_function()
    return _SOLVE.apply(model, theta, x0, bcs, Q, p)


_SOLVE = None


def _solve_autograd_function():
    import torch
    from torch._C import _functorch
    from torch._functorch.pyfunctorch import temporarily_clear_interpreter_stack

    # Under torch.func transforms the tensors a Function sees (and the ones it allocates) are functorch wrappers without
    # storage; the engine needs raw device pointers, so every engine call runs on the unwrapped tensors with the transform
    # stack cleared (torch's own private hooks for this: there is no public one in this torch version).
    def raw(a):
        while a is not None and _functorch.is_functorch_wrapped_tensor(a):
            a = _functorch.get_unwrapped(a)
        return None if a is None else a.detach().float().contiguous()

    class Solve(torch.autograd.Function):
        @staticmethod
        def forward(model, theta, x0, bcs, Q, p):
            with temporarily_clear_interpreter_stack():
                if model.P > 0:
                    model.set_theta(raw(theta).cpu().numpy())
                if p is not None:
                    model.set_mpp_params(*(float(v) for v in raw(p).cpu()))
                x0, bcs, Q = raw(x0), raw(bcs), raw(Q)
                traj = torch.empty((x0.shape[0], model.n_saved, model.desc.S), device=x0.device)
                torch.cuda.synchronize(x0.device)
                model.solve_dev(x0, bcs, traj, Q=Q)
                model.ctx.synchronize()
            return traj

        @staticmethod
        def setup_context(fctx, inputs, output):
            model, theta, x0, bcs, Q, p = inputs
            fctx.model, fctx.has_p = model, p is not None
            fctx.meta = [(a.dtype, a.device) if a is not None else None for a in (theta, x0, p)]
            fctx.data = (x0, bcs, Q)

        @staticmethod
        def backward(fctx, traj_bar):
            m = fctx.model
            want = fctx.needs_input_grad
            with temporarily_clear_interpreter_stack():
                x0, bcs, Q = (raw(a) for a in fctx.data)
                xb = torch.empty_like(x0) if want[2] else None
                tb = torch.empty(m.P, device=x0.device) if want[1] and m.P > 0 else None
                pb = torch.empty(5, device=x0.device) if want[5] and fctx.has_p else None
                if xb is None and tb is None and pb is None:
                    return None, None, None, None, None, None
                torch.cuda.synchronize(x0.device)
                m.solve_vjp_dev(x0, bcs, raw(traj_bar), x0_bar=xb, theta_bar=tb, mpp_bar=pb, Q=Q)
                m.ctx.synchronize()
            out = [tb, xb, pb]
            for i, meta in enumerate(fctx.meta):
                if out[i] is not None:
                    out[i] = out[i].to(dtype=meta[0], device=meta[1])
            return None, out[0], out[1], None, None, out[2]

        @staticmethod
        def jvp(fctx, model_t, theta_t, x0_t, bcs_t, Q_t, p_t):
            m = fctx.model
            with temporarily_clear_interpreter_stack():
                x0, bcs, Q = (raw(a) for a in fctx.data)
                dev = x0.device
                td = raw(theta_t).to(dev) if (theta_t is not None and m.P > 0) else None
                xd = None if x0_t is None else raw(x0_t).to(dev)
                pd = raw(p_t).to(dev) if (p_t is not None and fctx.has_p) else None
                traj_dot = torch.zeros((x0.shape[0], m.n_saved, m.desc.S), device=dev)
                if xd is not None or td is not None or pd is not None:
                    torch.cuda.synchronize(dev)
                    m.solve_jvp_dev(x0, bcs, traj_dot, x0_dot=xd, theta_dot=td, mpp_dot=pd, Q=Q)
                    m.ctx.synchronize()
            return traj_dot

    return Solve
