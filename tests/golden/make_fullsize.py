"""Generates tests/golden/fullsize_*.npz: FP64-oracle answers (and FP32-oracle noise floors) for the full-length
parity cases of tests/test_fullsize_gpu.py (1 152 steps x 2 sub-steps x Tsit5 = 13 824 right-hand-side evaluations per
column). The FP64 autograd gradient of one case takes minutes of CPU, so it is computed here once and committed; the
inputs themselves are regenerated from seeds by the test. Like make_golden.py these are outputs of THIS repo's oracle,
not of the (un-runnable) Julia reference: parity unpinned.

    python tests/golden/make_fullsize.py [case ...]
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cpzload  # noqa: E402

cpzload.load()
from cpz_b200 import synthetic as syn  # noqa: E402
from cpz_b200.desc import RHS_INFER, RHS_TRAIN  # noqa: E402
from util import oracle_loss_grad, oracle_solve, rel_inf  # noqa: E402

W3 = np.array([1, 1, 1, 5e-3, 5e-3, 5e-3], dtype=np.float32)
FRAMES = lambda n: np.unique(np.concatenate([np.arange(0, n, 64), [n - 1]]))  # frames kept of an all-frames trajectory


def grad_case(d, th, x0, bcs, tgt, w):
    tot, comps, g = oracle_loss_grad(d, th, x0, bcs, tgt, w)
    tot32, comps32, g32 = oracle_loss_grad(d, th, x0, bcs, tgt, w, dtype=torch.float32)
    return dict(targets=tgt, loss=np.concatenate([comps, [tot]]), grad=g, floor_grad=np.linalg.norm(g32 - g) / np.linalg.norm(g),
                floor_loss=abs(tot32 - tot) / abs(tot))


def config3_slice():
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=1152, save_stride=9, ckpt_stride=9)
    th = syn.theta_random(d, scale=0.1)
    x0, bcs = syn.columns(d, 36)
    th2 = (th * (1 + 0.3 * np.random.default_rng(0).standard_normal(th.shape))).astype(np.float32)
    tgt = oracle_solve(d, th2, x0, bcs).astype(np.float32)
    return grad_case(d, th, x0, bcs, tgt, W3)


def bench_targets(d, x0):
    """bench.py's config-3 targets: a smooth drift of the initial profiles (cheap to rebuild, so not stored)."""
    tgt = np.ascontiguousarray(np.repeat(x0[:, None, :], d.n_saved, axis=1))
    return (tgt + 0.05 * np.linspace(0, 1, d.n_saved, dtype=np.float32)[None, :, None]).astype(np.float32)


def config3_bench_theta():
    d = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=1152, save_stride=9, ckpt_stride=1)
    th = syn.theta_init(d, seed=42, scale=1e-5)
    x0, bcs = syn.columns(d, 32, seed=1000)
    out = grad_case(d, th, x0, bcs, bench_targets(d, x0), W3)
    del out["targets"]
    return out


def forward_case(d, th, ncol, seed=1000, frames=None):
    x0, bcs = syn.columns(d, ncol, seed=seed)
    ref = oracle_solve(d, th, x0, bcs)
    floor = rel_inf(oracle_solve(d, th, x0, bcs, dtype=torch.float32), ref)
    fr = np.arange(ref.shape[1]) if frames is None else frames(ref.shape[1])
    return dict(frames=fr, traj=ref[:, fr].astype(np.float32), floor=floor, scale=np.abs(ref).max())  # float32 storage: 6e-8


def config2_undivided():
    d = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=1152, save_stride=1)
    th = syn.theta_random(d, scale=0.1)
    out = forward_case(d, th, 64, frames=FRAMES)
    x0, bcs = syn.columns(d, 64)
    base = oracle_solve(d, 0 * th, x0, bcs)[:, -1]
    out["nn_share"] = np.abs(out["traj"][:, -1] - base).max() / np.abs(out["traj"][:, -1]).max()
    return out


def nnfree_full():
    d = syn.wind_mixing_desc(variant=RHS_INFER, net=None, n_steps=1152, save_stride=1)
    return forward_case(d, np.zeros(0, dtype=np.float32), 64, frames=FRAMES)


def config4_slice(scale):
    d = syn.free_convection_desc(ca=False, n_steps=1152, save_stride=9)
    th = syn.theta_init(d, seed=42, scale=scale) if scale < 1e-3 else syn.theta_random(d, scale=scale)
    return forward_case(d, th, 300, frames=lambda n: np.unique(np.concatenate([np.arange(0, n, 4), [n - 1]])))


W_T = np.array([0, 0, 1, 0, 0, 0], dtype=np.float32)


def config1(scale):
    """BASELINE config 1: ONE column of the T-only NDE with convective adjustment + mPP base, forward solve + loss gradient."""
    d = syn.free_convection_desc(ca=True, mpp=True, n_steps=1152, save_stride=9, ckpt_stride=9)
    th = syn.theta_init(d, seed=42, scale=scale) if scale < 1e-3 else syn.theta_random(d, scale=scale)
    x0, bcs = syn.columns(d, 1)
    th2 = (syn.theta_random(d, seed=8, scale=0.1)).astype(np.float32)
    tgt = oracle_solve(d, th2, x0, bcs).astype(np.float32)
    out = grad_case(d, th, x0, bcs, tgt, W_T)
    out["traj"] = oracle_solve(d, th, x0, bcs)
    out["floor_traj"] = rel_inf(oracle_solve(d, th, x0, bcs, dtype=torch.float32), out["traj"])
    return out


CASES = {"fullsize_config1_random": lambda: config1(0.1), "fullsize_config1_init": lambda: config1(1e-5),"fullsize_config3_slice": config3_slice, "fullsize_config3_bench_theta": config3_bench_theta,
         "fullsize_config2_undivided": config2_undivided, "fullsize_nnfree": nnfree_full,
         "fullsize_config4_init": lambda: config4_slice(1e-5), "fullsize_config4_random": lambda: config4_slice(0.1)}

# arrays that do not compress below 1 MB: written in this many parts along the column axis, the first part in <name>.npz
# with the other arrays, part i in <name>.<i>.npz
SPLIT = {"fullsize_config3_slice": ("targets", 2), "fullsize_config4_random": ("traj", 2)}


def save(name, out):
    if name not in SPLIT:
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        return
    key, n = SPLIT[name]
    parts = np.array_split(out[key], n)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **{**out, key: parts[0]})
    for i, part in enumerate(parts[1:], 1):
        np.savez_compressed(os.path.join(HERE, f"{name}.{i}.npz"), **{key: part})


def load(name):
    """The arrays save() wrote for `name`, split arrays joined again."""
    out = dict(np.load(os.path.join(HERE, name + ".npz")))
    if name in SPLIT:
        key, n = SPLIT[name]
        out[key] = np.concatenate([out[key]] + [np.load(os.path.join(HERE, f"{name}.{i}.npz"))[key] for i in range(1, n)])
    return out


if __name__ == "__main__":
    for name in (sys.argv[1:] or CASES):
        save(name, CASES[name]())
        print("wrote", name, flush=True)
