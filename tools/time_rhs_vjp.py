"""CUDA-event timing of the RHS pullback (cpz_rhs_vjp_dev: x_bar and theta_bar) next to the RHS itself (cpz_rhs_dev), the
two alternating in one process, on
  (a) 4 096 u/v/T columns with the production nets (3 x 96->50->20->31 mish, inference RHS; the config-2 size),
  (b) 9 u/v/T columns (the reference's batch of simulations),
  (c) 131 072 T-only columns (32->128->128->31 relu; the config-4 size).
A separate torch.profiler pass splits one call of each into its kernels. Prints one JSON line with the GPU name and power
limit (read with nvidia-smi --query-gpu; nothing is changed).
    python tools/time_rhs_vjp.py [--calls 200] [--out FILE]"""
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
from cpz_b200.desc import RHS_INFER  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def case(ctx, d, ncol, calls, reps=10):
    m = engine.Model(ctx, d, syn.theta_random(d, scale=0.3))
    x, bcs = syn.columns(d, ncol)
    dev = torch.device("cuda:0")
    xd, bd = torch.tensor(x, device=dev), torch.tensor(bcs, device=dev)
    yb = torch.randn(x.shape, generator=torch.Generator().manual_seed(3)).to(dev)
    f, xb, tb = torch.empty_like(xd), torch.empty_like(xd), torch.empty(m.P, device=dev)
    rhs = lambda: m.rhs_dev(xd, bd, f)
    vjp = lambda: m.rhs_vjp_dev(xd, bd, yb, x_bar=xb, theta_bar=tb)
    for _ in range(20):  # warm-up: module load, shared-memory attributes, scratch allocation
        rhs(); vjp()
    torch.cuda.synchronize()
    per = max(1, calls // reps)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * reps)]
    for r in range(reps):  # alternate: `per` RHS calls, then `per` pullback calls
        ev[3 * r].record()
        for _ in range(per):
            rhs()
        ev[3 * r + 1].record()
        for _ in range(per):
            vjp()
        ev[3 * r + 2].record()
    torch.cuda.synchronize()
    t_rhs = [ev[3 * r].elapsed_time(ev[3 * r + 1]) * 1e3 / per for r in range(reps)]
    t_vjp = [ev[3 * r + 1].elapsed_time(ev[3 * r + 2]) * 1e3 / per for r in range(reps)]
    # kernel split of one call each (profiler in its own pass, outside the timed window)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            rhs(); vjp()
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count > 0:
            kernels[e.key[:60]] = round(e.device_time_total / 5, 2)  # us per call
    out = {"ncol": ncol, "n_fields": d.n_fields, "nets": [n.sizes for n in d.nets][:1], "P": m.P, "calls_each": per * reps,
           "rhs_us": round(sorted(t_rhs)[reps // 2], 2), "vjp_us": round(sorted(t_vjp)[reps // 2], 2),
           "rhs_us_min_max": [round(min(t_rhs), 2), round(max(t_rhs), 2)], "vjp_us_min_max": [round(min(t_vjp), 2), round(max(t_vjp), 2)],
           "kernels_us_per_call": kernels, "describe": [l for l in m.describe().splitlines() if "rhs pullback" in l]}
    out["vjp_over_rhs"] = round(out["vjp_us"] / out["rhs_us"], 2)
    m.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200, help="timed calls of each entry point per case (after warm-up)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    # the library enqueues on a torch stream of its own (the legacy default stream has handle 0, which would mean "create
    # a private stream"), so that the events below time its work
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = engine.Context(0, stream=stream.cuda_stream)
    uvt = syn.wind_mixing_desc(variant=RHS_INFER)
    fc = syn.free_convection_desc(ca=False)
    res = {"metric": "rhs_vjp_vs_rhs", "unit": "us per call (median of 10 windows)", "gpu": gpu_info(),
           "cases": {"a_uvT_4096": case(ctx, uvt, 4096, args.calls), "b_uvT_9": case(ctx, uvt, 9, args.calls),
                     "c_T_only_131072": case(ctx, fc, 131072, args.calls)}}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
