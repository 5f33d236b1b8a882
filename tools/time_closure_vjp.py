"""CUDA-event timing of the gyre closure-step pullback (cpz_closure_step_vjp_dev: T_bar and theta_bar for both cotangents)
next to the closure step itself (cpz_closure_step_dev), the two alternating in one process, on the 512 x 64 x 32 BASELINE
config-5 slab (32 768 columns, every seventh column statically unstable so that the adjustment acts) with
  (a) the production net (32->128->128->31 relu; the forward runs on the tcgen05 closure, the pullback on FP32 SIMT),
  (b) a 32->192->192->31 relu net (weights streamed from global memory by the pullback).
A separate torch.profiler pass splits one call of each into its kernels. Algorithmic FLOPs per column are counted from the
net shapes (multiply-add = 2): the forward evaluates every layer; the pullback evaluates every layer but the last, then
backward-data and weight gradient of every layer. Prints one JSON line with the GPU name and power limit (read with
nvidia-smi --query-gpu; nothing is changed).
    python tools/time_closure_vjp.py [--calls 100] [--out FILE]"""
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
from cpz_b200.desc import ClosureDesc, NetDesc  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def mlp_flops(d):
    fwd = bwd = 0
    for n in d.nets:
        kn = [n.sizes[i] * n.sizes[i + 1] for i in range(len(n.sizes) - 1)]
        fwd += 2 * sum(kn)
        bwd += 2 * sum(kn[:-1]) + 4 * sum(kn)  # forward without the last layer; backward-data + weight gradient
    return fwd, bwd


def case(ctx, d, nx, ny, calls, reps=10):
    m = engine.Model(ctx, d, syn.theta_random(d, scale=1.0))
    T, y = syn.gyre_field(nx, ny, 32)
    T[:, :, ::7] = T[::-1, :, ::7]
    cd = ClosureDesc(Nx=nx, Ny=ny, Nz=32)
    dev = torch.device("cuda:0")
    Td, yd = torch.tensor(T, device=dev), torch.tensor(y, device=dev)
    g = torch.Generator().manual_seed(3)
    fb = (torch.randn(T.shape, generator=g) * 1e5).to(dev)  # ~ 1 / max|forcing|: both paths matter
    ob = torch.randn(T.shape, generator=g).to(dev)
    forcing, T_out, Tb = (torch.empty_like(Td) for _ in range(3))
    tb = torch.empty(m.P, device=dev)
    fwd = lambda: m.closure_step_dev(cd, Td, yd, forcing, T_out)
    vjp = lambda: m.closure_step_vjp_dev(cd, Td, fb, ob, Tb, tb)
    for _ in range(20):  # warm-up: module load, shared-memory attributes, weight images, scratch allocation
        fwd(); vjp()
    torch.cuda.synchronize()
    per = max(1, calls // reps)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * reps)]
    for r in range(reps):  # alternate: `per` closure steps, then `per` pullbacks
        ev[3 * r].record()
        for _ in range(per):
            fwd()
        ev[3 * r + 1].record()
        for _ in range(per):
            vjp()
        ev[3 * r + 2].record()
    torch.cuda.synchronize()
    t_fwd = [ev[3 * r].elapsed_time(ev[3 * r + 1]) * 1e3 / per for r in range(reps)]
    t_vjp = [ev[3 * r + 1].elapsed_time(ev[3 * r + 2]) * 1e3 / per for r in range(reps)]
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            fwd(); vjp()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count > 0:
            kernels[e.key[:60]] = round(e.device_time_total / 5, 2)  # us per call
    ff, fb_ = mlp_flops(d)
    ncol = nx * ny
    res = {"field": [32, ny, nx], "ncol": ncol, "nets": [n.sizes for n in d.nets], "P": m.P, "calls_each": per * reps,
           "closure_us": round(sorted(t_fwd)[reps // 2], 2), "vjp_us": round(sorted(t_vjp)[reps // 2], 2),
           "closure_us_min_max": [round(min(t_fwd), 2), round(max(t_fwd), 2)],
           "vjp_us_min_max": [round(min(t_vjp), 2), round(max(t_vjp), 2)],
           "mlp_flops_per_column": {"closure": ff, "vjp": fb_},
           "kernels_us_per_call": kernels,
           "describe": [l for l in m.describe().splitlines() if "closure-step pullback" in l or "forward kernel" in l.lower()]}
    res["vjp_over_closure"] = round(res["vjp_us"] / res["closure_us"], 2)
    res["vjp_tflops"] = round(fb_ * ncol / (res["vjp_us"] * 1e-6) / 1e12, 2)
    m.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=100, help="timed calls of each entry point per case (after warm-up)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    stream = torch.cuda.Stream()  # the library enqueues on this torch stream, so that the events below time its work
    torch.cuda.set_stream(stream)
    ctx = engine.Context(0, stream=stream.cuda_stream)
    prod = syn.free_convection_desc(ca=False)
    w192 = syn.free_convection_desc(ca=False, net=None)
    w192.nets = [NetDesc([32, 192, 192, 31], ["relu", "relu", "identity"])]
    res = {"metric": "closure_vjp_vs_closure", "unit": "us per call (median of 10 windows)", "gpu": gpu_info(),
           "cases": {"a_production_512x64": case(ctx, prod, 512, 64, args.calls),
                     "b_width192_512x64": case(ctx, w192, 512, 64, args.calls)}}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
