"""CUDA-event timing of the pushforwards next to the primal and the pullback on the same inputs, alternating in windows in
one process after a warm-up:
  (a) 4 096 u/v/T columns x 1 152 steps, Tsit5 x 2 sub-steps (the config-2 size; inference RHS, 3 x 96->50->20->31 mish, every
      9th step saved): cpz_solve_dev, cpz_solve_jvp_dev with an x0 tangent, with x0 + theta tangents, and cpz_solve_vjp_dev;
  (b) the NN-free `DE` model at the same size: cpz_solve_dev and cpz_solve_jvp_dev with an mPP-parameter tangent;
  (c) BASELINE config 1 (one T-only column, 32->128->128->31 relu, CA + mPP base): solve, jvp (x0 + theta), vjp;
  (d) cpz_rhs_jvp_dev (x tangent) next to cpz_rhs_dev and cpz_rhs_vjp_dev on the three cases of time_rhs_vjp.py.
A separate torch.profiler pass splits one call of each entry point into its kernels. The algorithmic MLP FLOPs (2 K N per
layer, column and evaluation; the tangent adds one such product for x_dot and one for theta_dot) are computed from the shapes.
Prints one JSON line with the GPU name and power limit (read with nvidia-smi --query-gpu; nothing is changed).
    python tools/time_solve_jvp.py [--windows 5] [--per 1] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import cpzload  # noqa: E402

cpzload.load()
from cpz_b200 import engine, synthetic as syn  # noqa: E402
from cpz_b200.desc import FLAG_MPP, FLAG_ZERO_WEIGHTS, RHS_INFER, RHS_TRAIN  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def mlp_flops(d):
    """FLOPs of the nets' dense products for one column and one RHS evaluation."""
    return sum(2 * a * b for n in d.nets for a, b in zip(n.sizes[:-1], n.sizes[1:]))


def timed(fns, windows, per, scale):
    """Median and range (in ms * scale) of each callable, alternating in `windows` windows of `per` calls; then the kernels
    time of one call of each callable, summed per kernel name (us), from a separate profiler pass."""
    names = list(fns)
    for _ in range(2):  # warm-up: module load, shared-memory attributes, scratch allocation
        for n in names:
            fns[n]()
    torch.cuda.synchronize()
    k = len(names)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range((k + 1) * windows)]
    for r in range(windows):
        ev[(k + 1) * r].record()
        for i, n in enumerate(names):
            for _ in range(per):
                fns[n]()
            ev[(k + 1) * r + i + 1].record()
    torch.cuda.synchronize()
    out = {}
    for i, n in enumerate(names):
        t = sorted(ev[(k + 1) * r + i].elapsed_time(ev[(k + 1) * r + i + 1]) * scale / per for r in range(windows))
        out[n] = {"median": round(t[len(t) // 2], 3), "min_max": [round(t[0], 3), round(t[-1], 3)]}
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:  # one pass, every entry point twice
        for _ in range(2):
            for n in names:
                fns[n]()
        torch.cuda.synchronize()
    kernels = {e.key[:60]: round(e.device_time_total / 2, 1) for e in prof.key_averages()  # us per call
               if e.device_type.name == "CUDA" and e.count > 0}
    return out, kernels


def solve_case(ctx, d, ncol, windows, per, want_theta=True, want_p=False):
    P = d.n_params
    m = engine.Model(ctx, d, syn.theta_random(d, scale=0.3) if P > 0 else None)
    x0, bcs = syn.columns(d, ncol)
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(3)
    xd, bd = torch.tensor(x0, device=dev), torch.tensor(bcs, device=dev)
    x0d = torch.randn(x0.shape, generator=g).to(dev)
    thd = torch.randn(P, generator=g).to(dev) if P > 0 else None
    pd = torch.tensor([1e-5, 1e-3, 1e-3, 1e-3, 1e-2], device=dev)
    shape = (ncol, m.n_saved, d.S)
    traj, traj_dot = torch.empty(shape, device=dev), torch.empty(shape, device=dev)
    tbar = torch.randn(shape, generator=g).to(dev) * 1e-4
    xb, tb = torch.empty_like(xd), torch.empty(max(P, 1), device=dev)
    fns = {"solve_ms": lambda: m.solve_dev(xd, bd, traj)}
    if not want_p:
        fns["jvp_x0_ms"] = lambda: m.solve_jvp_dev(xd, bd, traj_dot, x0_dot=x0d)
    if want_theta and P > 0:
        fns["jvp_x0_theta_ms"] = lambda: m.solve_jvp_dev(xd, bd, traj_dot, x0_dot=x0d, theta_dot=thd)
    if want_p:
        fns["jvp_p_ms"] = lambda: m.solve_jvp_dev(xd, bd, traj_dot, mpp_dot=pd)
    if P > 0:
        fns["vjp_ms"] = lambda: m.solve_vjp_dev(xd, bd, tbar, x0_bar=xb, theta_bar=tb)
    times, kernels = timed(fns, windows, per, 1.0)
    evals = d.n_steps * d.n_substeps * {"tsit5": 6, "rk4": 4, "euler": 1}[d.integrator]  # RHS evaluations per column
    f = mlp_flops(d) * evals * ncol
    out = {"ncol": ncol, "n_steps": d.n_steps, "n_substeps": d.n_substeps, "n_saved": m.n_saved, "P": P, "times": times,
           "kernels_us_per_call": kernels, "mlp_gflop_primal": round(f / 1e9, 2)}
    if "jvp_x0_ms" in times:  # primal + the x tangent: 2 products per layer
        out["jvp_x0_tflops_mlp"] = round(2 * f / (times["jvp_x0_ms"]["median"] * 1e-3) / 1e12, 2)
    if "jvp_x0_theta_ms" in times:  # + Wdot a: 3 products per layer
        out["jvp_x0_theta_tflops_mlp"] = round(3 * f / (times["jvp_x0_theta_ms"]["median"] * 1e-3) / 1e12, 2)
    out["describe"] = [l for l in m.describe().splitlines() if "tangents" in l or "forward kernel" in l.lower()][:2]
    m.close()
    return out


def rhs_case(ctx, d, ncol, windows, per):
    m = engine.Model(ctx, d, syn.theta_random(d, scale=0.3))
    x, bcs = syn.columns(d, ncol)
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(3)
    xd, bd = torch.tensor(x, device=dev), torch.tensor(bcs, device=dev)
    v = torch.randn(x.shape, generator=g).to(dev)
    f, fd, xb, tb = torch.empty_like(xd), torch.empty_like(xd), torch.empty_like(xd), torch.empty(m.P, device=dev)
    fns = {"rhs_us": lambda: m.rhs_dev(xd, bd, f), "jvp_x_us": lambda: m.rhs_jvp_dev(xd, bd, fd, x_dot=v),
           "vjp_us": lambda: m.rhs_vjp_dev(xd, bd, v, x_bar=xb, theta_bar=tb)}
    times, kernels = timed(fns, windows, per, 1e3)
    out = {"ncol": ncol, "n_fields": d.n_fields, "nets": [n.sizes for n in d.nets][:1], "P": m.P, "times": times,
           "kernels_us_per_call": kernels}
    out["jvp_x_tflops_mlp"] = round(2 * mlp_flops(d) * ncol / (times["jvp_x_us"]["median"] * 1e-6) / 1e12, 2)
    m.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=5, help="alternating windows per case")
    ap.add_argument("--per", type=int, default=1, help="calls of each entry point per window (the RHS cases take 50x this)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    # the library enqueues on a torch stream of its own so that the events below time its work
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = engine.Context(0, stream=stream.cuda_stream)
    w = args.windows
    d2 = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=1152, save_stride=9, ckpt_stride=9, n_substeps=2)
    dde = syn.wind_mixing_desc(variant=RHS_TRAIN, flags=FLAG_MPP | FLAG_ZERO_WEIGHTS, net=None, n_steps=1152, save_stride=9,
                               ckpt_stride=9, n_substeps=2)
    d1 = syn.free_convection_desc(ca=True, mpp=True, n_steps=1152, save_stride=9, ckpt_stride=9)
    res = {"metric": "solve_jvp_and_rhs_jvp", "unit": "ms per solve call, us per rhs call (median of the windows)", "gpu": gpu_info(),
           "cases": {}}
    res["cases"]["a_uvT_4096_solve"] = solve_case(ctx, d2, 4096, w, args.per)
    res["cases"]["b_DE_4096_solve"] = solve_case(ctx, dde, 4096, w, args.per, want_p=True)
    res["cases"]["c_config1_solve"] = solve_case(ctx, d1, 1, w, args.per)
    uvt = syn.wind_mixing_desc(variant=RHS_INFER)
    fc = syn.free_convection_desc(ca=False)
    for name, d, n in (("d_rhs_uvT_4096", uvt, 4096), ("d_rhs_uvT_9", uvt, 9), ("d_rhs_T_only_131072", fc, 131072)):
        res["cases"][name] = rhs_case(ctx, d, n, w, 50 * args.per)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
