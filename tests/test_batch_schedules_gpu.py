"""Launch schedules that only large and mid-size batches take, against the FP64 oracle.

The launchers pick different code once a batch outgrows one wave of the device: several reverse launches per record
segment and re-integrated segments in the tensor-core adjoint, 8- / 16-column and multi-tile CTAs in the FP32 adjoint,
two-tile CTAs in solve_fc_tc_kernel, the persistent loops of the closure kernels, the 28-/32-column tile choice of the
tcgen05 forward solve and the NN-free kernel's 4-column warps. Each case derives its sizes from the SM count, mirrors the
launcher arithmetic that selects the path (helpers below, each citing its C++ source) and asserts that the path it exists
for is the one taken, so that a change of a threshold fails the test instead of silently dropping its coverage.

Tolerances are the suite's: 1e-4 on solves, losses and gradients, where a result may also be as far from the FP64 oracle
as the FP32 restatement of the oracle is (the floor printed beside each error); 1e-5 on RHS evaluations and on the gyre
closure; the u/v/T closure rules of test_closure_uvt_gpu.py. Two kinds of case need the floor:
- Gradients of the T-only model with convective adjustment: the switch on dT/dz < 0 flips under rounding in the
  well-mixed layers, and the FP32 oracle itself misses the FP64 gradient by 1e-3 at these batch sizes. There the CUDA
  gradient must be within 3 x that floor (the suite's rule for sensitive maps, test_adjoint_gpu.py smoothing filters,
  test_fullsize_gpu.py), and the same batch without the adjustment, where the floor is far below 1e-4, is held to 1e-4.
- Trajectories of thousands of u/v/T columns: a few columns of the batch sit on the tanh step of the Richardson number,
  and the FP32 oracle's worst column is 5e-4 .. 1e-3 from FP64 after a few steps (the FP32 SIMT kernel misses those
  columns by the same amount as the tcgen05 one). The worst column must be within 3 x the FP32 oracle's worst, and
  the batch as a whole (Frobenius norm) within 1e-4, which a single wrong tile of 28 or 32 columns exceeds by orders
  of magnitude. Where two launch schedules compute the same columns, they must agree bitwise."""
import os
import sys

import numpy as np
import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
import make_batch_schedules as mbs  # noqa: E402

from cpz_b200 import engine, synthetic as syn  # noqa: E402
from cpz_b200.desc import (FLAG_IMPLICIT_DIFFUSION, FLAG_MPP, FLAG_SMOOTH_NN, FLAG_ZERO_WEIGHTS, RHS_INFER,  # noqa: E402
                           RHS_TRAIN, ClosureDesc, ClosureUvtDesc, NetDesc, RHS_EVALS)
from oracle import nde  # noqa: E402
from util import oracle_loss_grad, oracle_rhs, oracle_solve, rel_inf, t32, t64  # noqa: E402

pytestmark = pytest.mark.gpu
TOL = 1e-4
W3 = mbs.W3
W_T = np.array([0, 0, 1.0, 0, 0, 0], dtype=np.float32)
W_GRAD = np.array([0.7, 0.7, 1.0, 3e-3, 3e-3, 5e-3], dtype=np.float32)


class _env:
    def __init__(self, **kv):
        self.kv = kv

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        for k, v in self.kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# ---- mirrors of the launchers' path selection --------------------------------------------------------------------------
def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def cdiv(a, b):
    return (a + b - 1) // b


def train_tile(ncol, sms):
    """train_tile (cpz_k_solve.cu): the smallest of 4 / 8 / 16 columns whose tiles fit one wave, else 32."""
    for ct in (4, 8, 16):
        if cdiv(ncol, ct) <= sms:
            return ct
    return 32


def tc_forward_seven(ncol, sms):
    """`seven` of launch_tc_t (cpz_k_tc.cu) for a solve without checkpoints, records or implicit step: 28-column tiles when
    that does not add a wave and gives more tiles."""
    t32, t28 = cdiv(ncol, 32), cdiv(ncol, 28)
    return cdiv(t28, sms) <= cdiv(t32, sms) and t28 > t32


def fc_tc_ctas(ncol, sms):
    """(n_pair, n_single) of launch_fc_tc_t (cpz_k_closure.cu): full waves of two-tile CTAs, a remainder of at most one
    wave as single-tile CTAs, otherwise pairs throughout (the last one with a phantom second tile when the count is odd)."""
    n_tiles = cdiv(ncol, 128)
    n_pair, n_single = (n_tiles + 1) // 2, 0
    full = n_tiles // (2 * sms)
    rem = n_tiles - full * 2 * sms
    if 0 < rem <= sms:
        n_pair, n_single = full * sms, rem
    return n_pair, n_single


def tiles_per_cta(n_tiles, grid):
    """Tiles of the persistent loops `for (tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)` per CTA."""
    return [len(range(b, n_tiles, grid)) for b in range(grid)]


def tc_adjoint_schedule(ncol, d, sms, budget_floats, h1=50, h2=20):
    """The tensor-core adjoint's schedule (loss_grad_tc, cpz_k_adjoint_tc.cu; record rows from tc_aux_rows,
    cpz_adjoint_tc.cuh): split mode, steps per reverse launch `rs`, record-segment length and boundaries, and the reverse
    launches (segment, n0, n1, ev0, first) in the order they run."""
    n_tiles = cdiv(ncol, 32)
    epst = d.n_substeps * RHS_EVALS[d.integrator]
    rx, r1, r2, r3 = 104, (3 * h1 + 1 + 7) & ~7, (3 * h2 + 1 + 7) & ~7, 96
    xp = n_tiles * d.n_substeps * rx * 32 if d.flags & FLAG_IMPLICIT_DIFFUSION else 0
    xz_step = n_tiles * epst * (rx + r1 + r2) * 32 + xp
    d_step = n_tiles * epst * (r1 + r2 + r3) * 32
    n_steps, cs = d.n_steps, d.ckpt_stride
    split = 2 * n_tiles <= sms
    rs = max(1, min(n_steps, (1 << 30) // d_step))
    seg_len = min(n_steps, budget_floats // xz_step)
    if seg_len < n_steps:
        seg_len = max(cs, seg_len // cs * cs)
    s_last = 0 if seg_len >= n_steps else cdiv(n_steps - seg_len, cs) * cs
    bnd = list(range(0, s_last, seg_len)) + [s_last, n_steps]
    launches = []
    for seg in range(len(bnd) - 2, -1, -1):
        a0, a1 = bnd[seg], bnd[seg + 1]
        n1 = a1
        while n1 > a0:
            n0 = n1 - min(rs, n1 - a0)
            launches.append(dict(seg=seg, n0=n0, n1=n1, ev0=(n0 - a0) * epst, first=n1 == n_steps))
            n1 = n0
    return dict(n_tiles=n_tiles, split=split, rs=rs, seg_len=seg_len, bnd=bnd, launches=launches, xz_step=xz_step,
                d_step=d_step, n_reint=len(bnd) - 2)


def aux_gb(xz_step, steps):
    """CPZ_ADJ_AUX_GB for records of `steps` steps (half a step of slack, so the float parse cannot round below)."""
    return f"{(steps * xz_step + xz_step // 2) * 4 / 1e9:.9f}"


def aux_budget_floats(gb):
    return int(float(gb) * 1e9 / 4)  # loss_grad_tc: (size_t)(atof(gb) * 1e9 / sizeof(float))


def drift_targets(d, x0):
    return mbs.bench_targets(d, x0)


def assert_trajectories(got, ref, ref32, label):
    """Worst column within max(1e-4, 3 x the FP32 oracle's worst column); Frobenius-norm error of the batch within 1e-4."""
    n, sc = ref.shape[0], np.abs(ref).max()
    e = np.abs(got.astype(np.float64) - ref).reshape(n, -1).max(1) / sc
    f = np.abs(ref32.astype(np.float64) - ref).reshape(n, -1).max(1) / sc
    e_fro = np.linalg.norm(got.astype(np.float64) - ref) / np.linalg.norm(ref)
    f_fro = np.linalg.norm(ref32.astype(np.float64) - ref) / np.linalg.norm(ref)
    print(f"  {label}: worst column {e.max():.2e} (fp32-oracle {f.max():.2e}; columns above 1e-4: {int((e > TOL).sum())}, fp32-oracle "
          f"{int((f > TOL).sum())} of {n})  batch norm {e_fro:.2e} (fp32-oracle {f_fro:.2e})")
    assert np.isfinite(got).all()
    assert e.max() <= max(TOL, 3 * f.max()), (e.max(), f.max())
    assert e_fro <= TOL, e_fro


# ---- 1. tensor-core adjoint: reverse launches and record segments (FP64 golden) -----------------------------------------
@pytest.fixture(scope="module")
def adj_case():
    cache = {}

    def get(name):
        if name not in cache:
            d, th, x0, bcs, tgt = mbs.case_inputs(name)
            G = mbs.load(name)
            cache[name] = dict(d=d, th=th, x0=x0, bcs=bcs, tgt=tgt, tot=float(G["loss"][6]), g=G["grad"],
                               floor_g=float(G["floor_grad"]), floor_l=float(G["floor_loss"]))
        return cache[name]
    return get


def _adj_err(c, loss, grad):
    e_l = abs(float(loss[6]) - c["tot"]) / abs(c["tot"])
    e_g = np.linalg.norm(grad - c["g"]) / np.linalg.norm(c["g"])
    return e_l, e_g


def _adj_assert(c, loss, grad, what):
    e_l, e_g = _adj_err(c, loss, grad)
    print(f"  {what}: loss {e_l:.2e} (fp32-oracle {c['floor_l']:.2e})  grad L2 {e_g:.2e} (fp32-oracle {c['floor_g']:.2e})")
    assert np.isfinite(grad).all()
    assert e_l <= max(TOL, c["floor_l"]), (what, e_l, c["floor_l"])
    assert e_g <= max(TOL, c["floor_g"]), (what, e_g, c["floor_g"])


def test_adjoint_tc_several_reverse_launches_two_groups_per_cta(ctx, adj_case):
    """A1: 300 tiles (two column groups per CTA), 72 steps. With records for all 72 steps: one record segment, reverse
    launches of 29 / 29 / 14 steps. With records for 36 steps: two segments, the first re-integrated from its checkpoint,
    each with launches of 29 and 7 steps (the second of each starts at ev0 = 0 of its segment, the first at ev0 != 0)."""
    sms = sm_count()
    c = adj_case("batch_adjoint_tc_a1")
    d, ncol = c["d"], c["x0"].shape[0]
    assert cdiv(ncol, 32) > sms // 2
    m = engine.Model(ctx, d, c["th"])
    assert "adjoint kernels: tcgen05" in m.describe(), m.describe()
    xz = tc_adjoint_schedule(ncol, d, sms, 0)["xz_step"]
    counts = {}
    for steps in (72, 36):
        gb = aux_gb(xz, steps)
        S = tc_adjoint_schedule(ncol, d, sms, aux_budget_floats(gb))
        L = S["launches"]
        assert not S["split"] and S["rs"] < d.n_steps
        if steps == 72:
            assert S["n_reint"] == 0 and len(L) >= 3 and sum(not l["first"] for l in L) >= 2
        else:
            assert S["n_reint"] >= 1 and any(l["seg"] < len(S["bnd"]) - 2 and l["ev0"] != 0 for l in L)
            assert all(sum(l["seg"] == s for l in L) >= 2 for s in range(len(S["bnd"]) - 1))
        with _env(CPZ_ADJ_AUX_GB=gb, CPZ_NO_TC_ADJ=None):
            l1, g1 = m.loss_grad(c["x0"], c["bcs"], c["tgt"], W3)
            n0 = ctx.launch_count
            l2, g2 = m.loss_grad(c["x0"], c["bcs"], c["tgt"], W3)
            counts[steps] = (ctx.launch_count - n0, S)
        what = (f"A1 {ncol} columns, {d.n_steps} steps, records for {S['seg_len']} steps: rs={S['rs']}, segments {S['bnd']}, "
                f"{len(L)} reverse launches {[(l['n0'], l['n1'], l['ev0']) for l in L]}, {S['n_reint']} re-integrated")
        _adj_assert(c, l1, g1, what)
        np.testing.assert_array_equal(l1, l2)
        np.testing.assert_array_equal(g1, g2)
    # the library ran the schedule above: every reverse launch is an adjoint + weight-gradient pair of kernels, every
    # earlier record segment one re-integration
    (n72, S72), (n36, S36) = counts[72], counts[36]
    assert n36 - n72 == 2 * (len(S36["launches"]) - len(S72["launches"])) + S36["n_reint"] - S72["n_reint"], (n36, n72)
    with _env(CPZ_NO_TC_ADJ="1"):
        assert "adjoint kernels: fp32-simt" in m.describe()
        l3, g3 = m.loss_grad(c["x0"], c["bcs"], c["tgt"], W3)
    m.close()
    assert train_tile(ncol, sms) == 32 and cdiv(ncol, 32) > sms
    _adj_assert(c, l3, g3, f"A1 on the FP32 adjoint: 32-column tiles, {cdiv(ncol, 32)} tiles on {sms} CTAs, stored tendencies")


def test_adjoint_tc_split_mode_two_reverse_launches_and_halves(ctx, adj_case):
    """A2: 72 tiles (one column group per CTA, two CTAs per tile), 144 steps: reverse launches of 124 + 20 steps. The same
    golden from the FP32 adjoint (16-column tiles) and from the two halves combined by column count, each half on the FP32
    adjoint (8-column tiles) and on the tensor-core adjoint. (theta_random at scale 0.1: see make_batch_schedules.py.)
    This case found the weight-gradient contraction losing accuracy with the number of records one accumulator sums
    (1.5e-4 from FP64, against an FP32-oracle floor of 9e-6), fixed by the blocked accumulation of wgrad_tc_kernel."""
    sms = sm_count()
    c = adj_case("batch_adjoint_tc_a2")
    d, ncol = c["d"], c["x0"].shape[0]
    x0, bcs, tgt = c["x0"], c["bcs"], c["tgt"]
    S0 = tc_adjoint_schedule(ncol, d, sms, 0)
    gb = aux_gb(S0["xz_step"], d.n_steps)
    S = tc_adjoint_schedule(ncol, d, sms, aux_budget_floats(gb))
    assert S["split"] and S["n_reint"] == 0 and len(S["launches"]) >= 2 and S["launches"][-1]["n0"] == 0
    assert not S["launches"][-1]["first"]
    m = engine.Model(ctx, d, c["th"])
    assert "adjoint kernels: tcgen05" in m.describe()
    with _env(CPZ_ADJ_AUX_GB=gb, CPZ_NO_TC_ADJ=None):
        l1, g1 = m.loss_grad(x0, bcs, tgt, W3)
        l2, g2 = m.loss_grad(x0, bcs, tgt, W3)
    _adj_assert(c, l1, g1, f"A2 {ncol} columns, {d.n_steps} steps: split mode, rs={S['rs']}, "
                           f"{len(S['launches'])} reverse launches {[(l['n0'], l['n1']) for l in S['launches']]}")
    np.testing.assert_array_equal(l1, l2)
    np.testing.assert_array_equal(g1, g2)
    with _env(CPZ_NO_TC_ADJ="1"):
        l3, g3 = m.loss_grad(x0, bcs, tgt, W3)
    assert train_tile(ncol, sms) == 16
    _adj_assert(c, l3, g3, "A2 on the FP32 adjoint, 16-column tiles")
    h = ncol // 2
    assert train_tile(h, sms) == 8
    for kind in ("fp32-simt", "tcgen05"):
        parts = []
        for sl in (slice(0, h), slice(h, ncol)):
            n = sl.stop - sl.start
            Sh = tc_adjoint_schedule(n, d, sms, 0)
            with _env(CPZ_NO_TC_ADJ="1" if kind == "fp32-simt" else None, CPZ_ADJ_AUX_GB=aux_gb(Sh["xz_step"], d.n_steps)):
                parts.append((n,) + m.loss_grad(x0[sl], bcs[sl], tgt[sl], W3))
        lm = sum(n * l.astype(np.float64) for n, l, _ in parts) / ncol
        gm = sum(n * g.astype(np.float64) for n, _, g in parts) / ncol
        _adj_assert(c, lm, gm, f"A2 as two halves of {h} columns on the {kind} adjoint"
                               + (" (8-column tiles)" if kind == "fp32-simt" else f" (rs={Sh['rs']})"))
    m.close()


# ---- 2. FP32 adjoint tile widths and multi-tile CTAs (inline oracle) ----------------------------------------------------
SIZES = {"tile8": lambda s: 4 * s + 1, "tile16": lambda s: 8 * s + 1, "tile32": lambda s: 16 * s + 1,
         "tile32x2": lambda s: 32 * s + 5}
TILE_OF = {"tile8": 8, "tile16": 16, "tile32": 32, "tile32x2": 32}


def _grad_check(ctx, d, th, ncol, w, label, floor_factor=1.0, env=None):
    x0, bcs = syn.columns(d, ncol)
    tgt = drift_targets(d, x0)
    m = engine.Model(ctx, d, th)
    with _env(**(env or {})):
        loss, grad = m.loss_grad(x0, bcs, tgt, w)
    desc = m.describe()
    m.close()
    tot, _, g = oracle_loss_grad(d, th, x0, bcs, tgt, w)
    tot32, _, g32 = oracle_loss_grad(d, th, x0, bcs, tgt, w, dtype=torch.float32)
    f_l, f_g = abs(tot32 - tot) / abs(tot), np.linalg.norm(g32 - g) / np.linalg.norm(g)
    e_l, e_g = abs(loss[6] - tot) / abs(tot), np.linalg.norm(grad - g) / np.linalg.norm(g)
    print(f"  {label}: loss {e_l:.2e} (fp32-oracle {f_l:.2e})  grad L2 {e_g:.2e} (fp32-oracle {f_g:.2e})")
    assert np.isfinite(grad).all() and np.linalg.norm(g) > 0
    assert e_l <= max(TOL, floor_factor * f_l), (e_l, f_l)
    assert e_g <= max(TOL, floor_factor * f_g), (e_g, f_g)
    return desc


def _fp32_adjoint_path(ncol, sms, size):
    ct = train_tile(ncol, sms)
    assert ct == TILE_OF[size], (ncol, ct)
    n_tiles = cdiv(ncol, ct)
    per = tiles_per_cta(n_tiles, min(n_tiles, sms))
    assert ncol % ct != 0  # a ragged last tile
    assert cdiv(ncol, 4) > sms  # past the 4-column tiles every earlier test runs on
    if size == "tile32x2":
        assert per[0] >= 2
    else:
        assert max(per) == 1
    return f"{ct}-column tiles, {n_tiles} tiles on {min(n_tiles, sms)} CTAs (up to {max(per)} per CTA)"


@pytest.mark.parametrize("ca", [True, False])
@pytest.mark.parametrize("size", list(SIZES))
def test_fp32_adjoint_tile_widths_t_only(ctx, size, ca):
    """The T-only model with and without convective adjustment: forward with checkpoints on solve_fc_tc_kernel, reverse
    sweep on the FP32 adjoint at the tile width the batch selects."""
    sms = sm_count()
    ncol = SIZES[size](sms)
    d = syn.free_convection_desc(ca=ca, n_steps=6, save_stride=2, ckpt_stride=3)
    th = syn.theta_random(d, scale=0.3)
    path = _fp32_adjoint_path(ncol, sms, size)
    desc = _grad_check(ctx, d, th, ncol, W_T, f"T-only{' CA' if ca else ''}, {ncol} columns: {path}", floor_factor=3.0 if ca else 1.0)
    assert "adjoint kernels: fp32-simt" in desc and "tcgen05 3xTF32, columns on the M side" in desc
    assert "small-batch training pass" in desc  # the 8- / 16-column plans exist, so train_tile's mirror holds


@pytest.mark.parametrize("size", ["tile8", "tile16"])
def test_fp32_adjoint_tile_widths_t_only_ca_mpp(ctx, size):
    sms = sm_count()
    ncol = SIZES[size](sms)
    d = syn.free_convection_desc(ca=True, mpp=True, n_steps=4, save_stride=2, ckpt_stride=2)
    th = syn.theta_random(d, scale=0.3)
    path = _fp32_adjoint_path(ncol, sms, size)
    _grad_check(ctx, d, th, ncol, W_T, f"T-only CA + mPP, {ncol} columns: {path}", floor_factor=3.0)


@pytest.mark.parametrize("size", ["tile8", "tile16", "tile32"])
def test_fp32_adjoint_tile_widths_smoothing_filter(ctx, size):
    """u/v/T with smooth_NN (not tensor-core eligible): the FP32 forward and adjoint at every tile width. nu_m = 0.01 and
    the 3 x floor rule as in test_adjoint_gpu.py::test_grad_smoothing_filters."""
    sms = sm_count()
    ncol = SIZES[size](sms)
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_SMOOTH_NN, n_steps=4, save_stride=2,
                             ckpt_stride=2, nu_m=0.01)
    th = syn.theta_random(d, scale=0.3)
    path = _fp32_adjoint_path(ncol, sms, size)
    desc = _grad_check(ctx, d, th, ncol, W_GRAD, f"u/v/T smooth_NN, {ncol} columns: {path}", floor_factor=3.0)
    assert "adjoint kernels: fp32-simt" in desc and "small-batch training pass" in desc


@pytest.mark.parametrize("size", ["tile8", "tile16"])
def test_fp32_adjoint_tile_widths_mpp_parameter_gradient(ctx, size):
    """loss_grad_mpp (always the FP32 adjoint): NN-free model, targets from other mPP parameters."""
    sms = sm_count()
    ncol = SIZES[size](sms)
    kw = dict(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, net=None, n_steps=6, save_stride=3, ckpt_stride=3)
    d = syn.wind_mixing_desc(**kw)
    d_true = syn.wind_mixing_desc(**kw, n_substeps=d.n_substeps, nu_m=0.07, Ric=0.3, Pr=1.3, dRi=0.15, nu0=2e-4)
    th = np.zeros(0, dtype=np.float32)
    x0, bcs = syn.columns(d, ncol)
    tgt = oracle_solve(d_true, th, x0, bcs).astype(np.float32)
    path = _fp32_adjoint_path(ncol, sms, size)
    m = engine.Model(ctx, d, th)
    loss, gp, _ = m.loss_grad_mpp(x0, bcs, tgt, W_GRAD)
    m.close()
    tot, g = nde.loss_grad_mpp(d, t64(th), t64(x0), t64(bcs), None, t64(tgt), W_GRAD)
    _, g32 = nde.loss_grad_mpp(d, t32(th), t32(x0), t32(bcs), None, t32(tgt), W_GRAD)
    g, g32 = g.numpy(), g32.numpy().astype(np.float64)
    p = np.array([np.float32(v) for v in (d.nu0, d.nu_m, d.dRi, d.Ric, d.Pr)], dtype=np.float64)
    e_s, f_s = np.linalg.norm((gp - g) * p) / np.linalg.norm(g * p), np.linalg.norm((g32 - g) * p) / np.linalg.norm(g * p)
    e_l = abs(loss[6] - float(tot)) / abs(float(tot))
    print(f"  mPP-parameter gradient, {ncol} columns: {path}: loss {e_l:.2e}  scaled-space L2 {e_s:.2e} (fp32-oracle {f_s:.2e})")
    assert e_l <= TOL
    assert e_s <= max(TOL, 3 * f_s), (e_s, f_s)  # test_mpp_gpu.py's rule


@pytest.mark.parametrize("ca", [True, False])
def test_fp32_adjoint_many_tiles_per_cta_after_pair_forward(ctx, ca):
    """T-only model, small nets (32 x 32, still on tcgen05) at (sms + 2) * 128 + 77 columns: checkpoints from two-tile
    solve_fc_tc_kernel CTAs (odd tile count, phantom tile), FP32 adjoint with 4-5 32-column tiles per CTA."""
    sms = sm_count()
    ncol = (sms + 2) * 128 + 77
    d = syn.free_convection_desc(ca=ca, net=None, n_steps=4, save_stride=2, ckpt_stride=2)
    d.nets = [NetDesc([32, 32, 32, 31], ["relu", "relu", "identity"])]
    th = syn.theta_random(d, scale=0.5)
    n_pair, n_single = fc_tc_ctas(ncol, sms)
    assert n_single == 0 and 2 * n_pair > cdiv(ncol, 128)  # pairs only, the last one with a phantom tile
    assert train_tile(ncol, sms) == 32
    per = tiles_per_cta(cdiv(ncol, 32), sms)
    assert min(per) >= 4
    desc = _grad_check(ctx, d, th, ncol, W_T, f"T-only{' CA' if ca else ''} 32x32 nets, {ncol} columns: forward {n_pair} pair CTAs; "
                                              f"adjoint {cdiv(ncol, 32)} 32-column tiles, {min(per)}-{max(per)} per CTA",
                       floor_factor=3.0 if ca else 1.0)
    assert "tcgen05 3xTF32, columns on the M side" in desc


# ---- 3. solve_fc_tc_kernel pair mode (inline oracle) --------------------------------------------------------------------
FC_TILES = {"odd_pairs": lambda s: (s + 2) * 128 + 77, "exact_pairs": lambda s: 2 * s * 128,
            "pairs_and_singles": lambda s: (2 * s + 3) * 128 + 100}


def _fc_desc(act, ca, mpp):
    d = syn.free_convection_desc(ca=ca, mpp=mpp, net=None, n_steps=9, save_stride=3)
    d.nets = [NetDesc([32, 128, 128, 31], [act, act, "identity"])]
    return d


@pytest.mark.parametrize("tiles,act,ca,mpp", [
    ("odd_pairs", "relu", True, False), ("odd_pairs", "mish", False, False), ("odd_pairs", "tanh", True, True),
    ("exact_pairs", "tanh", False, False), ("exact_pairs", "relu", True, True),
    ("pairs_and_singles", "mish", True, False), ("pairs_and_singles", "relu", False, False)])
def test_fc_tc_pair_ctas(ctx, tiles, act, ca, mpp):
    sms = sm_count()
    ncol = FC_TILES[tiles](sms)
    n_tiles = cdiv(ncol, 128)
    n_pair, n_single = fc_tc_ctas(ncol, sms)
    if tiles == "odd_pairs":
        assert n_tiles % 2 == 1 and n_single == 0 and 2 * n_pair == n_tiles + 1 and ncol % 128 != 0
    elif tiles == "exact_pairs":
        assert n_single == 0 and 2 * n_pair == n_tiles
    else:
        assert n_pair == sms and n_single == n_tiles - 2 * sms > 0
    d = _fc_desc(act, ca, mpp)
    th = syn.theta_random(d, scale=0.5)
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    assert "tcgen05 3xTF32, columns on the M side" in m.describe()
    got = m.solve(x0, bcs)
    dx = m.rhs(x0, bcs, t=0.1)
    # the same columns in shards of at most `sms` tiles run as single-tile CTAs only
    step = sms * 128
    assert fc_tc_ctas(min(step, ncol), sms) == (0, cdiv(min(step, ncol), 128))
    shards = [m.solve(x0[a:a + step], bcs[a:a + step]) for a in range(0, ncol, step)]
    m.close()
    ref = oracle_solve(d, th, x0, bcs)
    floor = rel_inf(oracle_solve(d, th, x0, bcs, dtype=torch.float32), ref)
    e, e_r = rel_inf(got, ref), rel_inf(dx, oracle_rhs(d, th, x0, bcs, 0.1))
    print(f"  fc_tc {ncol} columns ({n_pair} pair CTAs + {n_single} single) {act} ca={ca} mpp={mpp}: solve {e:.2e} "
          f"(fp32-oracle {floor:.2e})  rhs {e_r:.2e}")
    assert np.isfinite(got).all()
    assert e <= TOL and e_r <= 1e-5
    # a tile's arithmetic does not depend on whether its CTA owns one tile or two
    np.testing.assert_array_equal(got, np.concatenate(shards))


# ---- 4. closures with many tiles per CTA (inline oracle) ----------------------------------------------------------------
def _gyre(nx, ny):
    T, y = syn.gyre_field(nx, ny, 32)
    T[:, :, ::3] = T[::-1, :, ::3] * 1.0  # every third column statically unstable
    return T, y


@pytest.mark.parametrize("nx,ny", [(512, 64), (509, 131)])
@pytest.mark.parametrize("act", ["relu", "mish", "tanh"])
def test_gyre_closure_persistent_tiles(ctx, nx, ny, act):
    sms = sm_count()
    n_tiles = cdiv(nx * ny, 128)
    per = tiles_per_cta(n_tiles, min(n_tiles, sms))
    assert n_tiles > sms and max(per) >= 2
    if (nx, ny) == (509, 131):
        assert (nx * ny) % 128 != 0 and len(set(per)) == 2 and {p % 2 for p in per} == {0, 1}
    d = syn.free_convection_desc(ca=False, net=None)
    d.nets = [NetDesc([32, 128, 128, 31], [act, act, "identity"])]
    th = syn.theta_random(d, scale=1.0)
    T, y = _gyre(nx, ny)
    cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
    m = engine.Model(ctx, d, th)
    forcing, T_out = m.closure_step(cd, T, y)
    with _env(CPZ_NO_TC="1"):
        f_simt, T_simt = m.closure_step(cd, T, y)
    m.close()
    f_ref, T_ref = nde.closure_step(d, t64(th), cd, t64(T), t64(y))
    f_ref, T_ref = f_ref.numpy(), T_ref.numpy()
    e_f, e_T, e_fs, e_Ts = rel_inf(forcing, f_ref), rel_inf(T_out, T_ref), rel_inf(f_simt, f_ref), rel_inf(T_simt, T_ref)
    n32 = cdiv(nx * ny, 32)
    print(f"  gyre closure {nx}x{ny} {act}: tcgen05 {n_tiles} tiles, {min(per)}-{max(per)} per CTA: forcing {e_f:.2e} T {e_T:.2e}; "
          f"fp32 {n32} tiles, {max(tiles_per_cta(n32, sms))} per CTA: forcing {e_fs:.2e} T {e_Ts:.2e}")
    assert e_f <= 1e-5 and e_T <= 1e-5
    assert e_fs <= 1e-5 and e_Ts <= 1e-5
    assert np.abs(T_out - T).max() > 1e-3


@pytest.mark.parametrize("kernel", ["tcgen05", "fp32-simt"])
@pytest.mark.parametrize("ca", [False, True])
@pytest.mark.parametrize("nx,ny", [(512, 64), (509, 13)])
def test_uvt_closure_persistent_tiles(ctx, nx, ny, ca, kernel):
    """The CLOSURE instantiation of solve_tc_kernel (32-column tiles; persistent loop with the next tile's prefetch) and the
    FP32 closure_uvt_kernel, both with several tiles per CTA. 509 x 13 is ragged and not a multiple of 4 (scalar I/O)."""
    sms = sm_count()
    n_tiles = cdiv(nx * ny, 32)
    per = tiles_per_cta(n_tiles, min(n_tiles, sms))
    assert n_tiles > sms and max(per) >= 2
    if ny == 13:
        assert (nx * ny) % 32 != 0 and (nx * ny) % 4 != 0
    d = syn.wind_mixing_desc(variant=RHS_INFER)
    th = syn.theta_random(d, scale=0.5)
    u, v, T = syn.uvt_fields(d, nx, ny, unstable_every=3 if ca else 0)
    cd = ClosureUvtDesc(Nx=nx, Ny=ny, Nz=32, dz=d.H / 32, dt=60.0, uw_top=-1e-4, vw_top=2e-5, wT_top=3e-5, convective_adjustment=ca)
    m = engine.Model(ctx, d, th)
    with _env(CPZ_NO_TC="1" if kernel == "fp32-simt" else None):
        dzf, out = m.closure_step_uvt(cd, u, v, T)
    m.close()
    dzf_ref, out_ref = nde.closure_step_uvt(d, t64(th), cd, t64(u), t64(v), t64(T))
    dzf_ref, out_ref = dzf_ref.numpy(), out_ref.numpy()
    x = np.stack([u, v, T])
    inc, inc_ref = out.astype(np.float64) - x, out_ref - x.astype(np.float64)
    e = [rel_inf(dzf[q], dzf_ref[q]) for q in range(3)] + [rel_inf(out[q], out_ref[q]) for q in range(3)]
    e_inc = [float(np.abs(inc[q] - inc_ref[q]).max() / max(np.abs(inc_ref[q]).max(), 1e-30)) for q in range(3)]
    print(f"  u/v/T closure [{kernel}] {nx}x{ny} ca={ca}: {n_tiles} tiles, {min(per)}-{max(per)} per CTA: dz_flux {max(e[:3]):.1e} "
          f"state {max(e[3:]):.1e} increments {max(e_inc):.1e}")
    assert max(e) <= 1e-5
    rel = 1e-5 if kernel == "fp32-simt" else 1e-4  # test_closure_uvt_gpu.py's increment rule
    for q in range(3):
        assert np.abs(inc[q] - inc_ref[q]).max() <= 4e-7 * np.abs(x[q]).max() + rel * np.abs(inc_ref[q]).max()
    if ca:
        assert np.abs(inc_ref[2]).max() > 1e-3


# ---- 5. tcgen05 forward tile-width boundary and the NN-free default -------------------------------------------------------
@pytest.fixture(scope="module")
def boundary_columns():
    """One u/v/T column set of 28 * sms + 1 columns with its FP64 (and FP32) oracle trajectory, 24 steps, all frames."""
    sms = sm_count()
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=24, save_stride=1)
    th = syn.theta_random(d, scale=0.3)
    n = max(28 * sms + 1, 4096)
    x0, bcs = syn.columns(d, n)
    return dict(d=d, th=th, x0=x0, bcs=bcs, ref=oracle_solve(d, th, x0, bcs), ref32=oracle_solve(d, th, x0, bcs, dtype=torch.float32))


def test_tc_forward_tile_width_boundary(ctx, boundary_columns):
    sms = sm_count()
    c = boundary_columns
    sizes = {"28*sms (28-column tiles)": 28 * sms, "28*sms+1 (32-column tiles)": 28 * sms + 1, "4096 (bench config 2)": 4096}
    assert tc_forward_seven(28 * sms, sms) and not tc_forward_seven(28 * sms + 1, sms) and tc_forward_seven(4096, sms) == (sms >= 147)
    m = engine.Model(ctx, c["d"], c["th"])
    assert "forward kernel: tcgen05" in m.describe()
    out = {}
    for label, n in sizes.items():
        got = m.solve(c["x0"][:n], c["bcs"][:n])
        assert_trajectories(got, c["ref"][:n], c["ref32"][:n], f"tcgen05 solve {label}: {cdiv(n, 28 if tc_forward_seven(n, sms) else 32)} tiles")
        out[n] = got
    m.close()
    # a column's arithmetic does not depend on the tile width it ran in
    k = min(sizes.values())
    np.testing.assert_array_equal(out[28 * sms][:k], out[28 * sms + 1][:k])
    np.testing.assert_array_equal(out[4096][:k], out[28 * sms + 1][:k])


def test_tc_forward_implicit_diffusion_bench_config(ctx):
    """4 096 columns with the implicit-diffusion step and one sub-step (32-column tiles: `seven` is off for it)."""
    d = syn.wind_mixing_desc(variant=RHS_INFER, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS | FLAG_IMPLICIT_DIFFUSION, n_substeps=1,
                             n_steps=24, save_stride=1)
    th = syn.theta_random(d, scale=0.3)
    x0, bcs = syn.columns(d, 4096)
    m = engine.Model(ctx, d, th)
    assert "forward kernel: tcgen05" in m.describe()
    got = m.solve(x0, bcs)
    m.close()
    assert_trajectories(got, oracle_solve(d, th, x0, bcs), oracle_solve(d, th, x0, bcs, dtype=torch.float32),
                   "tcgen05 implicit-diffusion solve, 4096 columns")


def test_nnfree_default_four_columns_per_warp(ctx):
    """32 768 + 5 columns with no override: solve_nnfree_kernel<4> (launch_solve_nnfree, cpz_k_tc.cu: NC = 4 from 32 768
    columns)."""
    assert os.environ.get("CPZ_NNFREE_NC") is None
    ncol = 32768 + 5
    d = syn.wind_mixing_desc(variant=RHS_INFER, net=None, n_steps=12, save_stride=3)
    th = np.zeros(0, dtype=np.float32)
    x0, bcs = syn.columns(d, ncol)
    m = engine.Model(ctx, d, th)
    assert "nn-free" in m.describe()
    got = m.solve(x0, bcs)
    with _env(CPZ_NNFREE_NC="2"):
        got2 = m.solve(x0, bcs)
    m.close()
    ref, ref32 = oracle_solve(d, th, x0, bcs), oracle_solve(d, th, x0, bcs, dtype=torch.float32)
    assert_trajectories(got, ref, ref32, f"nn-free {ncol} columns, 4 columns per warp")
    # a column's arithmetic does not depend on how many columns its warp carries
    np.testing.assert_array_equal(got, got2)
