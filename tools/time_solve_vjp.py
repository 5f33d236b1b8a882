"""CUDA-event timing of the solve pullback (cpz_solve_vjp_dev: x0_bar and theta_bar) next to the fused loss gradient
(cpz_loss_grad_dev) on the same inputs, the two alternating in windows in one process after a warm-up, on
  (a) BASELINE config 3: 9 216 u/v/T columns x 1 152 steps (training RHS, 3 x 96->50->20->31 mish, save every 9th step,
      ckpt_stride 9), on the tensor-core adjoint;
  (b) the same model with CPZ_NO_TC_ADJ=1 (FP32 SIMT adjoint) on 1 152 columns, which keeps the run short;
  (c) BASELINE config 1: one T-only column (32->128->128->31 relu, CA + mPP base), on the single-column kernel fc1.
Both entry points run the same checkpointing forward and reverse sweep, so parity is expected. Prints one JSON line with
the GPU name and power limit (read with nvidia-smi --query-gpu; nothing is changed).
    python tools/time_solve_vjp.py [--windows 5] [--per 2] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import cpzload  # noqa: E402

cpzload.load()
from cpz_b200 import engine, synthetic as syn  # noqa: E402
from cpz_b200.desc import RHS_TRAIN  # noqa: E402

W = np.array([1, 1, 1, 5e-3, 5e-3, 5e-3], dtype=np.float32)


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         check=True).stdout.strip()
    return dict(zip(q.split(","), (s.strip() for s in out.split(","))))


def case(ctx, d, ncol, windows, per, path_words):
    m = engine.Model(ctx, d, syn.theta_random(d, scale=0.3))
    desc = m.describe()
    assert path_words in desc, desc
    x0, bcs = syn.columns(d, ncol)
    dev = torch.device("cuda:0")
    xd, bd = torch.tensor(x0, device=dev), torch.tensor(bcs, device=dev)
    shape = (ncol, m.n_saved, d.S)
    tgt = torch.randn(shape, generator=torch.Generator().manual_seed(3)).to(dev) * 0.1 + xd[:, None, :]
    tbar = torch.randn(shape, generator=torch.Generator().manual_seed(4)).to(dev) * 1e-4
    loss, grad = torch.empty(7, device=dev), torch.empty(m.P, device=dev)
    xb, tb = torch.empty_like(xd), torch.empty(m.P, device=dev)
    lg = lambda: m.loss_grad_dev(xd, bd, tgt, W, loss, grad)
    vjp = lambda: m.solve_vjp_dev(xd, bd, tbar, x0_bar=xb, theta_bar=tb)
    for _ in range(2):  # warm-up: module load, shared-memory attributes, scratch and record allocation
        lg(); vjp()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * windows)]
    for r in range(windows):  # alternate: `per` loss-gradient calls, then `per` pullback calls
        ev[3 * r].record()
        for _ in range(per):
            lg()
        ev[3 * r + 1].record()
        for _ in range(per):
            vjp()
        ev[3 * r + 2].record()
    torch.cuda.synchronize()
    t_lg = [ev[3 * r].elapsed_time(ev[3 * r + 1]) / per for r in range(windows)]
    t_vjp = [ev[3 * r + 1].elapsed_time(ev[3 * r + 2]) / per for r in range(windows)]
    med = lambda t: round(sorted(t)[len(t) // 2], 3)
    out = {"ncol": ncol, "n_steps": d.n_steps, "P": m.P, "calls_each": per * windows,
           "loss_grad_ms": med(t_lg), "solve_vjp_ms": med(t_vjp),
           "loss_grad_ms_min_max": [round(min(t_lg), 3), round(max(t_lg), 3)],
           "solve_vjp_ms_min_max": [round(min(t_vjp), 3), round(max(t_vjp), 3)],
           "path": [l for l in desc.splitlines() if path_words in l][0][:120]}
    out["vjp_over_loss_grad"] = round(out["solve_vjp_ms"] / out["loss_grad_ms"], 3)
    m.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=5, help="alternating windows per case")
    ap.add_argument("--per", type=int, default=2, help="calls of each entry point per window")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    # the library enqueues on a torch stream of its own so that the events below time its work
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = engine.Context(0, stream=stream.cuda_stream)
    d3 = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=1152, save_stride=9, ckpt_stride=9)
    d1 = syn.free_convection_desc(ca=True, mpp=True, n_steps=1152, save_stride=9, ckpt_stride=9)
    res = {"metric": "solve_vjp_vs_loss_grad", "unit": "ms per call (median of the windows)", "gpu": gpu_info(), "cases": {}}
    res["cases"]["a_config3_tc_9216"] = case(ctx, d3, 9216, args.windows, args.per, "adjoint kernels: tcgen05")
    os.environ["CPZ_NO_TC_ADJ"] = "1"
    res["cases"]["b_config3_fp32_1152"] = case(ctx, d3, 1152, args.windows, args.per, "adjoint kernels: fp32-simt")
    del os.environ["CPZ_NO_TC_ADJ"]
    res["cases"]["c_config1_fc1"] = case(ctx, d1, 1, args.windows, args.per, "one CTA per column")
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
