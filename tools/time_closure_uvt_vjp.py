"""CUDA-event timing of the u/v/T closure-step pullback (cpz_closure_step_uvt_vjp_dev: u_bar, v_bar, T_bar and theta_bar for
both cotangents) next to the closure step itself (cpz_closure_step_uvt_dev), the two alternating in one process, on the
512 x 64 x 32 bench slab (32 768 columns) with
  (a) the production nets (3 x 96->50->20->31 mish; the forward runs on the tcgen05 closure),
  (b) width-128 one-hidden-layer relu nets (weights streamed from global memory by the pullback).
A separate torch.profiler pass splits one call of each into its kernels. Algorithmic FLOPs per column are counted from the
net shapes (multiply-add = 2): the forward evaluates every layer; the pullback evaluates every layer but the last, then
backward-data and weight gradient of every layer. Prints one JSON line with the GPU name and power limit (read with
nvidia-smi --query-gpu; nothing is changed).
    python tools/time_closure_uvt_vjp.py [--calls 100] [--out FILE]"""
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
from cpz_b200.desc import ClosureUvtDesc, RHS_INFER  # noqa: E402


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
    m = engine.Model(ctx, d, syn.theta_random(d, scale=0.3))
    u, v, T = syn.uvt_fields(d, nx, ny, unstable_every=7)
    cd = ClosureUvtDesc(Nx=nx, Ny=ny, Nz=32, dz=d.H / 32, dt=60.0, uw_top=-1e-4, vw_top=2e-5, wT_top=3e-5, convective_adjustment=True)
    dev = torch.device("cuda:0")
    ud, vd, Td = (torch.tensor(a, device=dev) for a in (u, v, T))
    g = torch.Generator().manual_seed(3)
    fb = torch.randn((3,) + u.shape, generator=g).to(dev)
    ob = torch.randn((3,) + u.shape, generator=g).to(dev)
    dzf, out, xb = (torch.empty((3,) + u.shape, device=dev) for _ in range(3))
    tb = torch.empty(m.P, device=dev)
    fwd = lambda: m.closure_step_uvt_dev(cd, ud, vd, Td, dzf, out)
    vjp = lambda: m.closure_step_uvt_vjp_dev(cd, ud, vd, Td, fb, ob, xb[0], xb[1], xb[2], tb)
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
    res = {"field": [32, ny, nx], "ncol": ncol, "nets": [n.sizes for n in d.nets][:1], "P": m.P, "calls_each": per * reps,
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
    prod = syn.wind_mixing_desc(variant=RHS_INFER)
    w128 = syn.wind_mixing_desc(variant=RHS_INFER, net=None)
    w128.nets = [syn.NetDesc([w128.S, 128, w128.Nz - 1], ["relu", "identity"]) for _ in range(3)]
    res = {"metric": "closure_uvt_vjp_vs_closure_uvt", "unit": "us per call (median of 10 windows)", "gpu": gpu_info(),
           "cases": {"a_production_512x64": case(ctx, prod, 512, 64, args.calls),
                     "b_width128_512x64": case(ctx, w128, 512, 64, args.calls)}}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
