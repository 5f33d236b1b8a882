"""Shared helpers for the parity tests (oracle = checker only)."""
import numpy as np
import torch

from oracle import nde


def t64(a):
    return torch.tensor(np.asarray(a), dtype=torch.float64)


def t32(a):
    return torch.tensor(np.asarray(a), dtype=torch.float32)


def rel_inf(a, ref):
    a = np.asarray(a, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    return float(np.abs(a - ref).max() / max(np.abs(ref).max(), 1e-300))


# ---- block-wise comparison ----------------------------------------------------------------------------------------------
# A whole-vector error is dominated by its largest block: the T tendency is ~1 % of the u/v/T RHS, and at the reference's
# initial weights (weights / 1e5) the W blocks carry 1e-12 .. 1e-9 of the gradient's norm. Each block is therefore also held
# to the rule on its own: err_b <= max(tol, k floor_b), both relative to the block's own FP64 norm. A block whose FP64 value
# is exactly zero must be within tol of the whole vector's norm.
#
# floor_b is the FP32 oracle's error on the block. Some gradient blocks are ill-conditioned in FP32, so that one FP32
# evaluation is a poor estimate of it: at weights / 1e5 (test_adjoint_gpu.py's 18-step problem) the wT net's blocks of the
# FP32-oracle gradient are 1.4e-4 .. 7.2e-4 from FP64 when x0 is moved by one FP32 ulp per element, while the FP64 gradient
# itself moves by 7e-6 .. 2e-5; the engine, an equally valid FP32 evaluation, lands at 3e-4. On the 64-column case of
# test_grad_reference_initial_weights, 13 such FP32-oracle runs put net 2's b3 block at 0.9e-4 .. 5.6e-4 (median 1.6e-4)
# and the engine at 7.7e-4: it rounds every intermediate of the solve and evaluates the Richardson-number step with MUFU
# exp (~1e-6 relative, against ~6e-8), a larger perturbation than one ulp of x0. Where a gradient check passes `spread`,
# floor_b is therefore SPREAD_K times the largest error of the FP32 oracle over its plain run and runs at ulp-nudged inputs
# (ulp_nudge, SPREAD_SEEDS), all against the FP64 oracle at the unchanged inputs. The nudged runs are evaluated only when
# the plain floor does not already hold every block: the floor can only grow with them, so the verdict is the same.
MPP_NAMES = ("nu0", "nu_m", "dRi", "Ric", "Pr")
SPREAD_SEEDS = (1, 2, 3, 4)
SPREAD_K = 2.0


def ulp_nudge(a, seed):
    """a as float32 with every element moved by one ulp, up or down at random."""
    a = np.asarray(a, dtype=np.float32)
    to = np.where(np.random.default_rng(seed).random(a.shape) < 0.5, -np.inf, np.inf).astype(np.float32)
    return np.nextafter(a, to)


def fp32_spread(fn):
    """A callable returning [fn(seed) for seed in SPREAD_SEEDS], computed on the first call and kept (fn(seed) runs the FP32
    oracle at inputs nudged by ulp_nudge(., seed))."""
    cache = []

    def get():
        if not cache:
            cache.extend(fn(s) for s in SPREAD_SEEDS)
        return cache
    return get


def theta_blocks(desc):
    """[(name, slice)] of every W and b of every net, in Flux.destructure order (oracle.flux_nn.reconstruct's offsets)."""
    out, off = [], 0
    for q, n in enumerate(desc.nets):
        for l in range(len(n.sizes) - 1):
            for kind, size in (("W", n.sizes[l] * n.sizes[l + 1]), ("b", n.sizes[l + 1])):
                out.append((f"net{q}.{kind}{l + 1}", slice(off, off + size)))
                off += size
    assert off == desc.n_params
    return out


def field_blocks(desc):
    """[(name, slice)] of the fields along the last axis of states, tendencies, trajectories and their cotangents."""
    N = desc.Nz
    if desc.n_fields == 1:
        return [("T", slice(0, N))]
    return [(f, slice(i * N, (i + 1) * N)) for i, f in enumerate("uvT")]


def mpp_blocks():
    return [(n, slice(i, i + 1)) for i, n in enumerate(MPP_NAMES)]


def mpp_scale(desc):
    """p = (nu0, nu_m, dRi, Ric, Pr) as float32 values: g * p is the gradient in the optimiser's scaled space."""
    return np.array([np.float32(getattr(desc, n)) for n in MPP_NAMES], dtype=np.float64)


def _norm(a, norm):
    return float(np.abs(a).max()) if norm == "inf" else float(np.linalg.norm(a))


def block_errors(got, ref, ref32, blocks, norm="inf"):
    """[(name, err, floor, |ref_b|)] over the last axis; err and floor relative to |ref_b|, absolute where ref_b == 0.
    ref32 is one FP32-oracle result or a list of them (floor: the largest error among them)."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    samples = [np.asarray(r, dtype=np.float64) for r in (ref32 if isinstance(ref32, (list, tuple)) else [ref32])]
    out = []
    for name, sl in blocks:
        r = ref[..., sl]
        scale = _norm(r, norm)
        den = scale if scale > 0 else 1.0
        floor = max(_norm(s[..., sl] - r, norm) for s in samples) / den
        out.append((name, _norm(got[..., sl] - r, norm) / den, floor, scale))
    return out


def assert_blocks(label, got, ref, ref32, blocks, tol, k=1.0, norm="inf", spread=None):
    """Prints one line per block and asserts err_b <= max(tol, k floor_b) on every block; a block whose FP64 value is exactly
    zero is held to tol times the whole vector's norm. spread: optional callable giving more FP32-oracle results (at
    ulp-nudged inputs) for the floor. Returns the worst err_b / max(tol, k floor_b)."""
    whole = _norm(np.asarray(ref, dtype=np.float64), norm)
    rows = block_errors(got, ref, ref32, blocks, norm)
    if spread is not None and any(scale > 0 and err > max(tol, k * floor) for _, err, floor, scale in rows):
        rows = [(n, e, SPREAD_K * f, s) for n, e, f, s in block_errors(got, ref, [ref32] + list(spread()), blocks, norm)]
        label += f" (floor: {SPREAD_K:g} x max over ulp-nudged fp32-oracle runs)"
    return assert_block_errors(label, rows, tol, k, whole)


def assert_block_errors(label, rows, tol, k=1.0, whole=0.0):
    """assert_blocks' rule on precomputed [(name, err, floor, |ref_b|)] rows."""
    worst, bad = 0.0, []
    for name, err, floor, scale in rows:
        if scale == 0:
            bound = tol * whole
            print(f"    {label} {name}: exact zero, |got| {err:.2e} (bound {bound:.2e})")
            if err > bound:
                bad.append((name, err, bound))
            continue
        bound = max(tol, k * floor)
        worst = max(worst, err / bound)
        print(f"    {label} {name}: {err:.2e} (fp32-oracle {floor:.2e}, |ref| {scale:.2e}; {err / bound:.2f} of the bound)")
        if not err <= bound:
            bad.append((name, err, floor))
    assert not bad, (label, bad)
    return worst


def oracle_rhs(desc, theta, x, bcs, t=0.0, Q=None, dtype=torch.float64):
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    q = None if Q is None else conv(Q)
    return nde.rhs(desc, conv(theta), conv(x), conv(bcs), t, q).numpy()


def oracle_solve(desc, theta, x0, bcs, Q=None, dtype=torch.float64):
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    q = None if Q is None else conv(Q)
    with torch.no_grad():
        return nde.solve(desc, conv(theta), conv(x0), conv(bcs), q).numpy()


def oracle_loss_grad(desc, theta, x0, bcs, targets, w, Q=None, dtype=torch.float64):
    conv = (lambda a: torch.tensor(np.asarray(a), dtype=dtype))
    q = None if Q is None else conv(Q)
    total, scaled, g = nde.loss_grad(desc, conv(theta), conv(x0), conv(bcs), q, conv(targets), w)
    return float(total), np.array([float(s) for s in scaled]), g.numpy()
