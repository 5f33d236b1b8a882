"""Generates tests/golden/batch_*.npz: FP64-oracle losses and gradients (and FP32-oracle noise floors) for the tensor-core
adjoint cases of tests/test_batch_schedules_gpu.py. Those cases need thousands of columns (a second reverse launch per
record segment only happens past ~3.4 M column-evaluations), so their FP64 autograd gradient takes minutes of CPU and is
computed here once and committed. Inputs and targets are regenerated from seeds by the test; save() / load() are
make_fullsize.py's.

The oracle runs in chunks of at most CHUNK columns, each weighted n_c / N: every loss term is a mean over columns and
columns are independent, so the weighted sum is the loss (and gradient) of the whole batch.

    python tests/golden/make_batch_schedules.py [case ...]
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import make_fullsize  # noqa: E402  (puts the repository and tests/ on sys.path, loads the package)
from make_fullsize import W3, bench_targets, load, save  # noqa: E402,F401
from cpz_b200 import synthetic as syn  # noqa: E402
from cpz_b200.desc import RHS_TRAIN  # noqa: E402
from util import SPREAD_SEEDS, oracle_loss_grad, theta_blocks, ulp_nudge  # noqa: E402

CHUNK = 300

# (columns, steps, theta scale): A1 = 300 tiles of 32 (two column groups per CTA), A2 = 72 tiles (one column group per
# CTA). Over A2's 144 steps the nets of theta_random(scale=0.3) make the FP32 oracle's gradient 13 % off the FP64 one (a
# floor that would hide any kernel error); at scale 0.1, the scale of the config-3 full-length slice, it is well-conditioned.
SHAPES = {"batch_adjoint_tc_a1": (9600, 72, 0.3), "batch_adjoint_tc_a2": (2304, 144, 0.1)}


def case_inputs(name):
    """Description, theta, x0, bcs and targets of a case (shared with the test)."""
    ncol, n_steps, scale = SHAPES[name]
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=n_steps, save_stride=9, ckpt_stride=9)
    th = syn.theta_random(d, scale=scale)
    x0, bcs = syn.columns(d, ncol)
    return d, th, x0, bcs, bench_targets(d, x0)


def chunked_loss_grad(d, th, x0, bcs, tgt, w, dtype):
    n = x0.shape[0]
    tot, comps, g = 0.0, np.zeros(6), 0.0
    for c0 in range(0, n, CHUNK):
        c1 = min(n, c0 + CHUNK)
        t_c, comps_c, g_c = oracle_loss_grad(d, th, x0[c0:c1], bcs[c0:c1], tgt[c0:c1], w, dtype=dtype)
        wt = (c1 - c0) / n
        tot, comps, g = tot + wt * t_c, comps + wt * comps_c, g + wt * g_c.astype(np.float64)
    return tot, comps, g


def block_floors(d, th, x0, bcs, tgt, g, g32):
    """Per (net, layer, W/b) block of theta (util.theta_blocks order): the largest relative L2 error of the FP32-oracle gradient
    over its plain run and runs at x0 nudged by one ulp (util.assert_blocks' spread floor; the first two SPREAD_SEEDS, as each
    run takes minutes here)."""
    runs = [g32] + [chunked_loss_grad(d, th, ulp_nudge(x0, s), bcs, tgt, W3, torch.float32)[2] for s in SPREAD_SEEDS[:2]]
    return np.array([max(np.linalg.norm(r[sl] - g[sl]) for r in runs) / np.linalg.norm(g[sl]) for _, sl in theta_blocks(d)])


def adjoint_case(name):
    d, th, x0, bcs, tgt = case_inputs(name)
    tot, comps, g = chunked_loss_grad(d, th, x0, bcs, tgt, W3, torch.float64)
    tot32, _, g32 = chunked_loss_grad(d, th, x0, bcs, tgt, W3, torch.float32)
    return dict(loss=np.concatenate([comps, [tot]]), grad=g, floor_grad=np.linalg.norm(g32 - g) / np.linalg.norm(g),
                floor_loss=abs(tot32 - tot) / abs(tot), floor_grad_blocks=block_floors(d, th, x0, bcs, tgt, g, g32))


CASES = {name: (lambda name=name: adjoint_case(name)) for name in SHAPES}

if __name__ == "__main__":
    for name in (sys.argv[1:] or CASES):
        save(name, CASES[name]())
        print("wrote", name, flush=True)
