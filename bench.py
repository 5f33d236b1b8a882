#!/usr/bin/env python
"""bench.py — headline benchmark of the NDE column engine (BASELINE.json: column-steps/s at Nz=32).

Workload at every N: BASELINE config 2 per GPU — wind_mixing u/v/T NDE forward solve (inference RHS, mPP base,
3 x (96->50 mish->20 mish->31) nets, Tsit5 fixed step with the sub-steps explicit diffusion needs), 4,096 synthetic
columns x 1,152 steps, every frame saved (1.81 GB of trajectory per solve, larger than L2) — weak scaling: columns
shard across ranks with no data-path collective. One bench "step" = one full solve of the rank's column batch.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Prints ONE JSON line (rank 0). `value` = device-resident throughput, `e2e` = through the host-pointer C ABI call
(pinned host buffers, H2D + D2H inside the timed region). Extra objects: roofline (tensor pipe of the tcgen05 kernel:
ALGORITHMIC FP32-equivalent flops = 2 x MACs of SURVEY 8d over the measured bf16 peak; the 3xTF32-issued rate and the
TF32 peak measured in this run are separate keys), roofline_hbm / roofline_compute (HBM and FP32-SIMT views of the same
run), adjoint (forward + discrete adjoint + ADAM, BASELINE config 3: the tensor-core adjoint with its stage records kept in HBM,
the same with a per-checkpoint-segment record budget = ckpt_stride 9 recompute, and the FP32 SIMT adjoint for A/B), config1 (one T-only column, CA + mPP base, forward + gradient, beside the oracle's single-column
CPU time), nn_free (the HBM-fair mPP-only variant), free_convection (config 4 slice), closure (config 5 slice, also as a
10^4-call CUDA-graph replay with a stand-in dynamics kernel between calls), cpu_baseline (the oracle on host cores:
batched on all cores, and one column at a time on one thread as the reference executes).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

NCOL = 4096
NSTEPS = 1152
DUMP_COLUMNS = 64
FP32_LANES_PER_SM = 128
# ncu --set full summaries of the dominant kernel at the bench configuration (newest round first); `traffic` and the
# tensor-pipe activity are READ from the committed file, not typed into this source
NCU_SUMMARIES = ("profiles/r02_tc_solve_ncu_summary.txt", "profiles/r01_tc_solve_ncu_summary.txt")


def ncu_summary():
    """dram bytes per launch and tensor-pipe activity of solve_tc_kernel from the committed ncu summary."""
    import re
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for rel in NCU_SUMMARIES:
        path = os.path.join(ROOT, rel)
        if not os.path.exists(path):
            continue
        txt = open(path).read()
        out = {"source": rel}
        tot = 0.0
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            mt = re.search(re.escape(key) + r"\s+([0-9.]+)\s+(\w+)", txt)
            if mt:
                tot += float(mt.group(1)) * unit.get(mt.group(2), 1.0)
        out["traffic"] = tot if tot > 0 else None
        mt = re.search(r"sm__pipe_tensor_cycles_active\.avg\.pct_of_peak_sustained_active\s+([0-9.]+)", txt)
        out["pipe_tensor_active_pct"] = float(mt.group(1)) if mt else None
        mt = re.search(r"gpu__time_duration\.sum\s+([0-9.]+)\s+ms", txt)
        out["ncu_kernel_ms"] = float(mt.group(1)) if mt else None
        return out
    return {"source": None, "traffic": None, "pipe_tensor_active_pct": None, "ncu_kernel_ms": None}


def measure_tf32_peak(torch):
    """Dense TF32 tensor-core throughput of this device, measured the MEASURED_PEAKS way (torch.matmul 8192^3, best of 5)."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device="cuda"); b = torch.randn(n, n, device="cuda")
        for _ in range(2):
            a @ b
        best = 1e30
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); a @ b; e1.record(); e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("sm_max_mhz", 1965.0), "measured", d.get("bf16_tflops_sustained", 1400.0)
    return 6650.0, 1965.0, "fallback", 1400.0


def bind_to_gpu_numa_node(local_rank, world):
    """Multi-rank runs: pin this process to the CPUs of its GPU's NUMA node BEFORE any pinned host allocation, so that the
    first-touch policy places the rank's staging buffers next to the GPU's PCIe root (the N = 8 end-to-end rate is bound by the
    host side of eight concurrent 1.81 GB D2H streams). No-op at N = 1, on single-node hosts, and when sysfs has no answer."""
    info = {"bound": False}
    if world <= 1:
        return info
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bus = bus[4:] if len(bus) > 12 else bus  # 00000000:1b:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        nodes = [n for n in os.listdir("/sys/devices/system/node") if n.startswith("node") and n[4:].isdigit()]
        info.update({"gpu_pci": bus, "node": node, "nodes": len(nodes)})
        if node < 0 or len(nodes) < 2:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info.update({"bound": True, "cpus": len(cpus)})
    except Exception as e:  # noqa: BLE001
        info["error"] = repr(e)
    return info


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        """number of samples taken so far (the timed region is rows[mark_begin:mark_end])"""
        return len(self.rows)

    def stop(self, lo=0, hi=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if hi is not None and hi - lo < 2:  # a timed region shorter than two sampling periods: wait for one more sample
            t_end = time.time() + 0.5
            while len(self.rows) <= hi and time.time() < t_end:
                time.sleep(0.02)
            hi = len(self.rows)
            lo = max(0, min(lo, hi - 2))
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[lo:hi]:
            try:
                sm.append(float(r[1])); smax.append(float(r[2]))
                for i, nm in enumerate(names):
                    if r[5 + i].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_workload(syn, RHS_INFER, n_steps):
    d = syn.wind_mixing_desc(variant=RHS_INFER, net="uvT_small", n_steps=n_steps, save_stride=1)
    theta = syn.theta_init(d, seed=42, scale=1e-5)
    return d, theta


def dump_outputs(out_dir, traj_d):
    """The trajectory [columns, frames, S] of the last timed solve, as float32 .npy: the final frame of every column and
    every frame of a fixed, seeded sample of DUMP_COLUMNS columns (about 30 MB; the whole trajectory is 1.81 GB)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cols = np.sort(np.random.default_rng(0).choice(traj_d.shape[0], DUMP_COLUMNS, replace=False))
    np.save(os.path.join(out_dir, "final_state.npy"), traj_d[:, -1].cpu().numpy())
    np.save(os.path.join(out_dir, "trajectory_sample.npy"), traj_d[torch.from_numpy(cols).to(traj_d.device)].cpu().numpy())


def flops_per_colstep(d):
    mlp = 2 * sum(n.macs for n in d.nets)
    return (mlp + 1200) * d.rhs_evals_per_step


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path. The Julia reference cannot run here (no julia
    binary, no LES data), so this times the oracle port (restated-reference CPU) with all host threads on a bounded
    sample of the same workload."""
    if rank != 0:
        return
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cpzload
    cpzload.load()
    from cpz_b200 import synthetic as syn
    from cpz_b200.desc import RHS_INFER
    from oracle import nde
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ncol_s, nsteps_s = 512, 12
    d, theta = build_workload(syn, RHS_INFER, nsteps_s)
    x0, bcs = syn.columns(d, ncol_s)
    th, x, b = torch.tensor(theta), torch.tensor(x0), torch.tensor(bcs)
    times = []
    with torch.no_grad():
        for it in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            nde.solve(d, th, x, b, None)
            dt = time.perf_counter() - t0
            if it >= args.warmup:
                times.append(dt)
    tot = sum(times)
    val = ncol_s * nsteps_s * len(times) / tot
    sample = f"{ncol_s} columns x {nsteps_s} steps (x{d.n_substeps} sub-steps, Tsit5) per step, FP32 torch-CPU oracle batched over columns"
    line = {
        "impl": "reference", "metric": "column-steps/sec (forward)", "value": val, "unit": "column-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE config 2 (wind_mixing u/v/T forward, Nz=32, small nets, Tsit5) — bounded sample",
                   "sample": sample},
        "cpu_baseline": {"value": val, "unit": "column-steps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "column-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference Julia path cannot run in this image (no julia, no LES data); restated-reference CPU oracle timed instead",
    }
    emit(line)


def cpu_baseline(syn, RHS_INFER):
    """Bounded oracle run on the host cores (about 10-30 s)."""
    import torch
    from oracle import nde
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ncol_s, nsteps_s = 512, 12
    d, theta = build_workload(syn, RHS_INFER, nsteps_s)
    x0, bcs = syn.columns(d, ncol_s)
    th, x, b = torch.tensor(theta), torch.tensor(x0), torch.tensor(bcs)
    with torch.no_grad():
        nde.solve(d, th, x, b, None)  # warm-up
        reps, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < 10.0 and reps < 20:
            nde.solve(d, th, x, b, None)
            reps += 1
        el = time.perf_counter() - t0
    out = {"value": ncol_s * nsteps_s * reps / el, "unit": "column-steps/s", "cores": cores, "kind": "port",
           "sample": f"{reps} x ({ncol_s} columns x {nsteps_s} steps x {d.n_substeps} sub-steps), FP32 torch-CPU oracle batched over columns"}
    # BASELINE.md section 3 leg: ONE thread, ONE column at a time — how the reference executes (`for i in 1:n_simulations`,
    # NDE_training.jl:291, with BLAS.set_num_threads(1), train_NDE.jl:11)
    torch.set_num_threads(1)
    try:
        with torch.no_grad():
            nde.solve(d, th, x[:1], b[:1], None)
            cols, t0 = 0, time.perf_counter()
            while time.perf_counter() - t0 < 8.0 and cols < ncol_s:
                nde.solve(d, th, x[cols:cols + 1], b[cols:cols + 1], None)
                cols += 1
            el1 = time.perf_counter() - t0
        out["serial_one_column_at_a_time"] = {
            "value": cols * nsteps_s / el1, "unit": "column-steps/s", "cores": 1,
            "sample": f"{cols} columns x {nsteps_s} steps, one column per solve call, torch.set_num_threads(1)"}
    finally:
        torch.set_num_threads(cores)
    return out


_REAL_STDOUT = None


def quiet_stdout():
    """Everything a library prints to fd 1 (e.g. NCCL's version banner) goes to stderr; the one JSON line is written to
    the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip adjoint / nn_free / cpu_baseline side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (rank 0's "
                    "columns) to DIR/*.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    numa = bind_to_gpu_numa_node(local_rank, world)
    import torch
    import cpzload
    cpzload.load()
    from cpz_b200 import engine, synthetic as syn
    from cpz_b200.desc import RHS_INFER, RHS_TRAIN

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # kernels are launched on a torch-owned stream so that torch.cuda.Event brackets them
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    ctx = engine.Context(local_rank, tstream.cuda_stream)
    d, theta = build_workload(syn, RHS_INFER, NSTEPS)
    model = engine.Model(ctx, d, theta)
    S, n_saved = d.S, d.n_saved
    x0, bcs = syn.columns(d, NCOL, seed=1000 + rank)
    x0_d, bcs_d = torch.tensor(x0, device="cuda"), torch.tensor(bcs, device="cuda")
    traj_d = torch.empty((NCOL, n_saved, S), dtype=torch.float32, device="cuda")

    # ---- device-resident timing (value) ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # started before the warm-up so that nvidia-smi is already streaming when the timed region begins
    for _ in range(args.warmup):
        model.solve_dev(x0_d, bcs_d, traj_d)
    barrier()
    mark0 = sampler.mark()
    l0 = ctx.launch_count
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_all0 = torch.cuda.Event(enable_timing=True); t_all1 = torch.cuda.Event(enable_timing=True)
    t_all0.record()
    for e0, e1 in evs:
        e0.record()
        model.solve_dev(x0_d, bcs_d, traj_d)
        e1.record()
    t_all1.record()
    barrier()
    launches = ctx.launch_count - l0
    clocks = sampler.stop(mark0, sampler.mark()) if rank == 0 else None
    ms_total = t_all0.elapsed_time(t_all1)
    kern_ms = float(np.mean([e0.elapsed_time(e1) for e0, e1 in evs]))
    t = torch.tensor([ms_total], device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    colsteps_per_step = NCOL * NSTEPS * world
    value = colsteps_per_step * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, traj_d)

    # ---- end-to-end through the host-pointer C ABI (pinned host buffers; H2D + D2H inside the timed region) ----
    x0_h = torch.tensor(x0).pin_memory(); bcs_h = torch.tensor(bcs).pin_memory()
    traj_h = torch.empty((NCOL, n_saved, S), dtype=torch.float32).pin_memory()
    e2e_steps = max(1, min(args.steps, 3))
    model.solve(x0_h.numpy(), bcs_h.numpy(), out=traj_h.numpy())
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        model.solve(x0_h.numpy(), bcs_h.numpy(), out=traj_h.numpy())  # synchronous on return
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_val = colsteps_per_step * e2e_steps / float(t.item())
    checksum = float(traj_h[:, -1].double().abs().mean())

    hbm_peak, sm_max_mhz, peak_src, bf16_peak = peaks()
    bytes_per_colstep = 4 * S * (n_saved / NSTEPS) + (4 * S + 4 * d.n_bc) / NSTEPS
    ach_gbs = bytes_per_colstep * NCOL * NSTEPS / (kern_ms * 1e-3) / 1e9
    fl = flops_per_colstep(d)
    ach_tf = fl * NCOL * NSTEPS / (kern_ms * 1e-3) / 1e12
    n_sm = torch.cuda.get_device_properties(local_rank).multi_processor_count
    sm_mhz = (clocks or {}).get("sm_mhz") or sm_max_mhz
    peak_tf_max = n_sm * FP32_LANES_PER_SM * 2 * sm_max_mhz * 1e6 / 1e12
    peak_tf_obs = n_sm * FP32_LANES_PER_SM * 2 * sm_mhz * 1e6 / 1e12

    tc = "forward kernel: tcgen05" in model.describe()
    if tc:
        # dominant kernel: solve_tc_kernel (tcgen05 kind::tf32, 3xTF32). `achieved` = ALGORITHMIC FP32-equivalent flops of
        # SURVEY 8d (2 x MACs of the three MLPs per RHS evaluation x the launch's column-steps) / the kernel's mean launch
        # time; `peak` = measured dense bf16 (sustained: the kernel runs for tens of ms). Every algorithmic MAC is issued as
        # three TF32 MACs (hi*lo + lo*hi + hi*hi) and the 150/60/93 output rows are padded to 128-row MMA blocks: those
        # rates are reported as separate keys, against the TF32 peak measured in this run.
        mlp_macs = sum(n.macs for n in d.nets)
        alg_flops = 2 * mlp_macs * d.rhs_evals_per_step * NCOL * NSTEPS
        h1 = d.nets[0].sizes[1]; h2 = d.nets[0].sizes[2]
        mma_per_rhs_group = (72 if 3 * h1 > 128 else 36) + 9 * 7 + 9 * (3 if h2 <= 24 else 4)
        issued_flops = mma_per_rhs_group * (2 * 128 * 16 * 8) * (NCOL / 16) * d.rhs_evals_per_step * NSTEPS
        ach = alg_flops / (kern_ms * 1e-3) / 1e12
        tf32_peak = measure_tf32_peak(torch)
        ncu = ncu_summary()
        roofline = {"bound": "tensor", "achieved": ach, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach / bf16_peak,
                    "traffic": ncu["traffic"], "traffic_source": ncu["source"], "peak_source": peak_src + " (bf16_tflops_sustained)",
                    "kernel": "solve_tc_kernel<ACT_MISH,3>", "kernel_ms": kern_ms,
                    "algorithmic_flop_per_colstep": 2 * mlp_macs * d.rhs_evals_per_step,
                    "tf32_peak_measured_tflops": tf32_peak,
                    "tf32_3x_algorithmic_tflops": 3 * ach, "frac_3xtf32_of_measured_tf32_peak": 3 * ach / tf32_peak,
                    "tf32_issued_tflops_incl_padding": issued_flops / (kern_ms * 1e-3) / 1e12,
                    "issued_over_algorithmic": issued_flops / (3 * alg_flops),
                    "pipe_tensor_active_pct_ncu": ncu["pipe_tensor_active_pct"], "ncu_kernel_ms": ncu["ncu_kernel_ms"],
                    "note": "3xTF32 on tcgen05 with M=128 x N=16 x K=8 MMAs; frac counts each MAC once (FP32-equivalent), the "
                            "three TF32 passes and the row padding are the separate keys; the kernel is latency-bound (two "
                            "dependent MLP chains per SM), see the ncu summary named in traffic_source"}
    else:
        roofline = {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak, "traffic": None,
                    "peak_source": peak_src, "kernel": "solve_kernel<32,256,true>", "kernel_ms": kern_ms,
                    "algorithmic_bytes_per_colstep": bytes_per_colstep}
    line = {
        "metric": "column-steps/sec (forward)", "value": value, "unit": "column-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE config 2: wind_mixing u/v/T NDE forward solve, 4096 synthetic columns x 1152 steps per GPU, all frames saved",
                   "Nz": 32, "columns_per_gpu": NCOL, "n_steps": NSTEPS, "n_substeps": d.n_substeps, "integrator": d.integrator,
                   "rhs_evals_per_step": d.rhs_evals_per_step, "nets": "3 x (96->50 mish->20 mish->31), P=19563",
                   "rhs": "inference (solve_NDE_mutating), mPP base, zero_weights BCs",
                   "arithmetic": "FP32 state/stencil/Runge-Kutta; MLP as 3xTF32 on tcgen05 (hi/lo operand split, FP32 accumulate in TMEM), RHS within 6e-7 of the FP64 oracle",
                   "l2": "no explicit flush: each solve writes a 1.81 GB trajectory (> 126 MB L2)", "parallelism": f"columns x{world}"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": "column-steps/s", "h2d_bytes_per_step": int(x0_h.numel() * 4 + bcs_h.numel() * 4),
                "d2h_bytes_per_step": int(traj_h.numel() * 4), "steps": e2e_steps, "final_state_checksum": checksum,
                "d2h_gbs_per_rank": traj_h.numel() * 4 * e2e_val / (NCOL * NSTEPS * world) / 1e9,
                "numa": numa},
        "roofline": roofline,
        "roofline_hbm": {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
                         "peak_source": peak_src, "algorithmic_bytes_per_colstep": bytes_per_colstep,
                         "note": "not the binding roof: arithmetic intensity ~ 1200 flop/B"},
        "roofline_compute": {"bound": "fp32_simt", "achieved": ach_tf, "unit": "TFLOP/s", "peak_at_max_clock": peak_tf_max,
                             "peak_at_observed_clock": peak_tf_obs, "frac": ach_tf / peak_tf_obs, "flop_per_colstep": fl,
                             "stage_evals_per_s": value * d.rhs_evals_per_step,
                             "note": "FP32-equivalent algorithmic flops against the FP32 SIMT peak (the roof of the non-tensor-core kernel)"},
    }
    if not args.no_extras:
        # ---- config 2 with the diffusive flux treated implicitly (SURVEY 8f-1): one Tsit5 step per saved frame, no sub-steps ----
        try:
            from cpz_b200.desc import FLAG_IMPLICIT_DIFFUSION as FLAG_IMPLICIT
            di = syn.wind_mixing_desc(variant=RHS_INFER, n_steps=NSTEPS, save_stride=1, n_substeps=1)
            di.flags |= FLAG_IMPLICIT
            mi = engine.Model(ctx, di, theta)
            mi.solve_dev(x0_d, bcs_d, traj_d)
            barrier()
            i0 = torch.cuda.Event(enable_timing=True); i1 = torch.cuda.Event(enable_timing=True)
            i0.record()
            for _ in range(3):
                mi.solve_dev(x0_d, bcs_d, traj_d)
            i1.record()
            barrier()
            ti = torch.tensor([i0.elapsed_time(i1)], device="cuda")
            if dist is not None:
                dist.all_reduce(ti, op=dist.ReduceOp.MAX)
            msi = float(ti.item()) / 3
            line["implicit_diffusion"] = {
                "metric": "column-steps/sec (forward, backward-Euler vertical diffusion + explicit NN flux)", "value": NCOL * NSTEPS * world / (msi * 1e-3),
                "ms_per_step": msi, "scaling": "weak",
                "config": {"workload": "BASELINE config 2 with CPZ_FLAG_IMPLICIT_DIFFUSION: the tridiagonal mPP solve of NDE_oceananigans.jl:61-101 at the "
                                       "start of every step (parallel cyclic reduction across the warp), then ONE Tsit5 step of the NN / boundary / Coriolis part",
                           "n_substeps": 1, "rhs_evals_per_step": di.rhs_evals_per_step, "kernel": mi.describe().splitlines()[0]},
                "note": "a different discretisation of the same model (Lie splitting, first order in the diffusion), not a faster path to the same numbers: "
                        "parity is against the oracle's implicit_diffusion restatement (tests/test_implicit_gpu.py)"}
            mi.close()
        except Exception as e:  # noqa: BLE001
            line["implicit_diffusion"] = {"error": repr(e)}
        # the headline model's device buffers are done with: the adjoint's stage records want the HBM
        model.close()
        del traj_d
        torch.cuda.empty_cache()
        # ---- fwd + discrete adjoint + ADAM (BASELINE config 3: 9 forcing cases x 1024 columns, sharded over ranks) ----
        # Three policies of the same training iteration (same loss, same gradient to FP32 noise):
        #   tc_records_in_hbm   tensor-core adjoint; the per-stage records (X_i, z1, z2) of as many steps as the free HBM holds are
        #                       written by the checkpointing forward pass itself (all 1 152 steps when they fit: no re-integration)
        #   tc_ckpt_stride_9    the same kernels with a 2 GB record budget: every 9-step checkpoint segment is re-integrated
        #                       (SURVEY config 3 as written: ckpt_stride 9, recompute)
        #   fp32_simt           the round-1 FP32 SIMT adjoint kernel (CPZ_NO_TC_ADJ=1), for A/B
        try:
            from cpz_b200 import parallel
            if dist is not None:
                parallel.attach_torch_allreduce(ctx)
            NC3 = 9216
            lo, hi = parallel.shard_columns(NC3, rank, world)
            x3 = b3 = None
            w3 = np.array([1, 1, 1, 5e-3, 5e-3, 5e-3], dtype=np.float32)
            adj = {}
            policies = (("tc_records_in_hbm", {}, 3), ("tc_ckpt_stride_9", {"CPZ_ADJ_AUX_GB": "2"}, 3), ("fp32_simt", {"CPZ_NO_TC_ADJ": "1"}, 1),
                        ("tc_implicit_diffusion", {"IMPLICIT": "1"}, 3))
            for name, env, n3 in policies:
                for k in ("CPZ_ADJ_AUX_GB", "CPZ_NO_TC_ADJ"):
                    os.environ.pop(k, None)
                os.environ.update({k: v for k, v in env.items() if k.startswith("CPZ_")})
                os.environ["CPZ_VERBOSE"] = "1"  # the library reports its record-segment policy (columns, GB, segments) on stderr
                d3 = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=NSTEPS, save_stride=9, ckpt_stride=9)
                if env.get("IMPLICIT"):  # the same training iteration with the diffusive flux implicit: one sub-step per step
                    from cpz_b200.desc import FLAG_IMPLICIT_DIFFUSION
                    d3 = syn.wind_mixing_desc(variant=RHS_TRAIN, net="uvT_small", n_steps=NSTEPS, save_stride=9, ckpt_stride=9, n_substeps=1)
                    d3.flags |= FLAG_IMPLICIT_DIFFUSION
                m3 = engine.Model(ctx, d3, syn.theta_init(d3, seed=42, scale=1e-5))
                adj_desc = [ln for ln in m3.describe().splitlines() if ln.startswith("adjoint kernels")]
                if x3 is None:
                    x3, b3 = syn.columns(d3, NC3, seed=1000)
                    x3_d, b3_d = torch.tensor(x3[lo:hi], device="cuda"), torch.tensor(b3[lo:hi], device="cuda")
                    # targets: a smooth drift of the initial profiles (any target gives the same cost)
                    tg = torch.tensor(x3[lo:hi], device="cuda")[:, None, :].repeat(1, d3.n_saved, 1).contiguous()
                    tg += 0.05 * torch.linspace(0, 1, d3.n_saved, device="cuda")[None, :, None]
                m3.train_step_dev(x3_d, b3_d, tg, w3, 3e-4)  # warm-up (allocates scratch)
                barrier()
                l0 = ctx.launch_count
                # every iteration is timed on its own (max over ranks each) and the MEDIAN is reported: with 86-163 GB of records
                # streaming through HBM single iterations run 5-10 % (once 85 %) slow on some boards; all samples are in the line
                ev3 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n3)]
                for e0_, e1_ in ev3:
                    e0_.record()
                    loss3 = m3.train_step_dev(x3_d, b3_d, tg, w3, 3e-4)
                    e1_.record()
                barrier()
                t3 = torch.tensor([e0_.elapsed_time(e1_) for e0_, e1_ in ev3], device="cuda")
                if dist is not None:
                    dist.all_reduce(t3, op=dist.ReduceOp.MAX)
                ms3_all = [float(v) for v in t3.tolist()]
                ms3 = float(np.median(ms3_all))
                # algorithmic FP32-equivalent flops: forward MLP + delta propagation + weight gradient = 3 x the forward MLP flops
                # (re-integration not counted); algorithmic HBM bytes per column-step: 129 (SURVEY 8d). The tensor-core policies
                # really move the per-stage records: per stage evaluation and column 1 224 B written + read twice (x, z1, z2)
                # and 1 212 B written + read (d1, d2, d3).
                mlp3 = 2 * sum(n.macs for n in d3.nets) * d3.rhs_evals_per_step
                tf3 = 3 * mlp3 * (hi - lo) * NSTEPS / (ms3 * 1e-3) / 1e12
                rec_bytes = d3.rhs_evals_per_step * (3 * 1224 + 2 * 1212) if name.startswith("tc") else None
                adj[name] = {
                    "value": NC3 * NSTEPS / (ms3 * 1e-3), "ms_per_step": ms3, "ms_each_iteration": ms3_all, "n_substeps": d3.n_substeps, "kernels": adj_desc[0] if adj_desc else None,
                    "gpu_launches_per_step": int((ctx.launch_count - l0) / n3), "loss": float(loss3[6]),
                    "roofline": {"fp32_equiv_tflops_algorithmic": tf3, "frac_of_fp32_simt_peak": tf3 / peak_tf_max, "frac_of_bf16_tensor_peak": tf3 / bf16_peak,
                                 "hbm_frac_algorithmic_129B": 129.0 * (hi - lo) * NSTEPS / (ms3 * 1e-3) / 1e9 / hbm_peak,
                                 "record_traffic_bytes_per_colstep": rec_bytes,
                                 "hbm_frac_record_traffic": (rec_bytes * (hi - lo) * NSTEPS / (ms3 * 1e-3) / 1e9 / hbm_peak) if rec_bytes else None}}
                m3.close()
            for k in ("CPZ_ADJ_AUX_GB", "CPZ_NO_TC_ADJ", "CPZ_VERBOSE"):
                os.environ.pop(k, None)
            best = adj["tc_records_in_hbm"]
            line["adjoint"] = {
                "metric": "column-steps/sec (forward + discrete adjoint + ADAM)", "value": best["value"],
                "unit": "column-steps/s", "ms_per_step": best["ms_per_step"], "scaling": "strong",
                "config": {"workload": "BASELINE config 3: 9 forcing cases x 1024 columns, training RHS, 1152 steps, 129 saved frames, Tsit5 x2 sub-steps, ADAM(3e-4), one allreduce of P+16 floats",
                           "columns_total": NC3, "columns_this_rank": hi - lo, "tiles": "32-column tiles (two 16-column MMA groups per CTA)"},
                **adj,
                "note": "value = tc_records_in_hbm. The tensor-core adjoint is three tcgen05 kernels (segment forward pass with stage records, "
                        "reverse sweep with transposed weights in tensor memory, weight-gradient contraction); they exchange ~73 KB of records "
                        "per column-step through HBM because forward weights, transposed weights and gradient accumulators do not fit 512 TMEM "
                        "columns together, so the real DRAM traffic (hbm_frac_record_traffic) is far above the algorithmic 129 B",
            }
        except Exception as e:  # noqa: BLE001
            line["adjoint"] = {"error": repr(e)}
        # ---- BASELINE config 1: ONE T-only column, convective adjustment + mPP base, forward solve + loss gradient ----
        try:
            d1 = syn.free_convection_desc(ca=True, mpp=True, n_steps=NSTEPS, save_stride=9, ckpt_stride=9)
            m1 = engine.Model(ctx, d1, syn.theta_init(d1, seed=42, scale=1e-5))
            x1, b1_ = syn.columns(d1, 1)
            x1_d, b1_d = torch.tensor(x1, device="cuda"), torch.tensor(b1_, device="cuda")
            tg1 = torch.tensor(x1, device="cuda")[:, None, :].repeat(1, d1.n_saved, 1).contiguous() + 0.05
            w1 = np.array([0, 0, 1, 0, 0, 0], dtype=np.float32)
            l1_d = torch.zeros(8, device="cuda"); g1_d = torch.zeros(m1.P, device="cuda")
            m1.loss_grad_dev(x1_d, b1_d, tg1, w1, l1_d, g1_d)
            barrier()
            c0 = torch.cuda.Event(enable_timing=True); c1 = torch.cuda.Event(enable_timing=True)
            c0.record()
            for _ in range(2):
                m1.loss_grad_dev(x1_d, b1_d, tg1, w1, l1_d, g1_d)
            c1.record()
            barrier()
            ms1 = c0.elapsed_time(c1) / 2
            line["config1"] = {
                "metric": "seconds per forward solve + loss gradient of ONE column", "value": ms1 * 1e-3, "unit": "s", "higher_is_better": False,
                "column_steps_per_s": NSTEPS / (ms1 * 1e-3),
                "config": {"workload": f"BASELINE config 1: single-column T-only NDE (32->128->128->31 relu), convective adjustment + mPP base, 1152 steps x {d1.n_substeps} sub-steps (Tsit5), save every 9th, MSE loss gradient wrt 24735 parameters",
                           "kernel": "fc1_train_kernel: one CTA per column (512 threads), weights in shared memory, weight gradients in registers, "
                                     "stage records streamed through HBM (cp.async double buffer), nothing recomputed; latency-bound on ONE SM by construction"},
                "loss": float(l1_d[6].item())}
            m1.close()
            try:  # the same column with the diffusive / convective-adjustment flux implicit: 1 sub-step instead of 15
                from cpz_b200.desc import FLAG_IMPLICIT_DIFFUSION as FLAG_IMPLICIT
                d1i = syn.free_convection_desc(ca=True, mpp=True, n_steps=NSTEPS, save_stride=9, ckpt_stride=9, n_substeps=1)
                d1i.flags |= FLAG_IMPLICIT
                m1i = engine.Model(ctx, d1i, syn.theta_init(d1i, seed=42, scale=1e-5))
                m1i.loss_grad_dev(x1_d, b1_d, tg1, w1, l1_d, g1_d)
                barrier()
                c0 = torch.cuda.Event(enable_timing=True); c1 = torch.cuda.Event(enable_timing=True)
                c0.record()
                for _ in range(2):
                    m1i.loss_grad_dev(x1_d, b1_d, tg1, w1, l1_d, g1_d)
                c1.record()
                barrier()
                line["config1"]["implicit_diffusion"] = {"value": c0.elapsed_time(c1) / 2 * 1e-3, "unit": "s", "n_substeps": 1,
                                                         "kernel": "fc1_train_kernel with the implicit step and its VJP on warp 0 (cyclic reduction across the lanes)",
                                                         "loss": float(l1_d[6].item())}
                m1i.close()
            except Exception as e:  # noqa: BLE001
                line["config1"]["implicit_diffusion"] = {"error": repr(e)}
            if rank == 0 and world == 1:
                # the same job on the CPU oracle (FP32 torch, 1 thread, the way the reference runs one simulation): bounded
                # sample of 36 steps, scaled to 1152
                from oracle import nde as _nde
                torch.set_num_threads(1)
                d1s = syn.free_convection_desc(ca=True, mpp=True, n_steps=36, save_stride=9, ckpt_stride=9)
                th1 = torch.tensor(syn.theta_init(d1s, seed=42, scale=1e-5))
                tgs = torch.tensor(x1)[:, None, :].repeat(1, d1s.n_saved, 1) + 0.05
                t0 = time.perf_counter()
                _nde.loss_grad(d1s, th1, torch.tensor(x1), torch.tensor(b1_), None, tgs, w1)
                cpu1 = (time.perf_counter() - t0) * NSTEPS / 36
                torch.set_num_threads(os.cpu_count() or 1)
                line["config1"]["cpu_oracle_seconds_scaled"] = cpu1
                line["config1"]["cpu_sample"] = "36 of 1152 steps (same sub-steps), FP32 torch oracle with autograd, 1 thread, scaled x32"
        except Exception as e:  # noqa: BLE001
            line["config1"] = {"error": repr(e)}
        # ---- NN-free mPP-only forward (SURVEY 8d '2-base', the HBM-fair variant) ----
        try:
            d0 = syn.wind_mixing_desc(variant=RHS_INFER, net=None, n_steps=NSTEPS, save_stride=1)
            m0 = engine.Model(ctx, d0, np.zeros(0, dtype=np.float32))
            traj_d = torch.empty((NCOL, n_saved, S), dtype=torch.float32, device="cuda")
            m0.solve_dev(x0_d, bcs_d, traj_d)
            barrier()
            b0 = torch.cuda.Event(enable_timing=True); b1 = torch.cuda.Event(enable_timing=True)
            b0.record()
            for _ in range(3):
                m0.solve_dev(x0_d, bcs_d, traj_d)
            b1.record()
            barrier()
            ms0 = b0.elapsed_time(b1) / 3
            gb0 = bytes_per_colstep * NCOL * NSTEPS / (ms0 * 1e-3) / 1e9
            line["nn_free"] = {"metric": "column-steps/sec (forward, mPP only)", "value": NCOL * NSTEPS * world / (ms0 * 1e-3),
                               "ms_per_step": ms0, "roofline": {"bound": "hbm", "achieved": gb0, "peak": hbm_peak, "unit": "GB/s", "frac": gb0 / hbm_peak}}
            m0.close()
        except Exception as e:  # noqa: BLE001
            line["nn_free"] = {"error": repr(e)}
        # ---- BASELINE config 4 slice: FreeConvectionNDE inference, 131072 columns per GPU (tcgen05, columns on the M side) ----
        try:
            NC4 = 131072
            d4 = syn.free_convection_desc(ca=False, n_steps=NSTEPS, save_stride=9)
            m4 = engine.Model(ctx, d4, syn.theta_init(d4, seed=42, scale=1e-5))
            x4, b4 = syn.columns(d4, NC4, seed=1000 + rank)
            x4_d, b4_d = torch.tensor(x4, device="cuda"), torch.tensor(b4, device="cuda")
            t4_d = torch.empty((NC4, d4.n_saved, d4.S), dtype=torch.float32, device="cuda")
            m4.solve_dev(x4_d, b4_d, t4_d)
            barrier()
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(2):
                m4.solve_dev(x4_d, b4_d, t4_d)
            a1.record()
            barrier()
            t4 = torch.tensor([a0.elapsed_time(a1)], device="cuda")
            if dist is not None:
                dist.all_reduce(t4, op=dist.ReduceOp.MAX)
            ms4 = float(t4.item()) / 2
            macs4 = sum(n.macs for n in d4.nets)
            line["free_convection"] = {
                "metric": "column-steps/sec (forward, T-only FreeConvectionNDE)", "value": NC4 * NSTEPS * world / (ms4 * 1e-3),
                "ms_per_step": ms4, "scaling": "weak",
                "config": {"workload": "BASELINE config 4 slice: 131072 columns per GPU x 1152 steps, 32->128->128->31 relu, Tsit5, save every 9th frame",
                           "kernel": m4.describe().splitlines()[0]},
                "tensor_tflops_tf32_algorithmic": 3 * 2 * macs4 * d4.rhs_evals_per_step * NC4 * NSTEPS / (ms4 * 1e-3) / 1e12}
            m4.close()
        except Exception as e:  # noqa: BLE001
            line["free_convection"] = {"error": repr(e)}
        # ---- BASELINE config 5 slice: per-step closure on a 512 x 64 x 32 y-slab (one call per host-model step) ----
        try:
            from cpz_b200.desc import ClosureDesc
            d5 = syn.free_convection_desc(ca=False)
            m5 = engine.Model(ctx, d5, syn.theta_init(d5, seed=42, scale=1e-5))
            nx5, ny5 = 512, 64
            T5, y5 = syn.gyre_field(nx5, ny5, 32)
            cd5 = ClosureDesc(Nx=nx5, Ny=ny5, Nz=32)
            T5_d, y5_d = torch.tensor(T5, device="cuda"), torch.tensor(y5, device="cuda")
            f5_d, o5_d = torch.empty_like(T5_d), torch.empty_like(T5_d)
            for _ in range(20):
                m5.closure_step_dev(cd5, T5_d, y5_d, f5_d, o5_d)
            barrier()
            n5 = 500
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(n5):
                m5.closure_step_dev(cd5, T5_d, y5_d, f5_d, o5_d)
            a1.record()
            barrier()
            t5 = torch.tensor([a0.elapsed_time(a1)], device="cuda")
            if dist is not None:
                dist.all_reduce(t5, op=dist.ReduceOp.MAX)
            us5 = float(t5.item()) / n5 * 1e3
            gb5 = 3 * nx5 * ny5 * 128 / (us5 * 1e-6) / 1e9
            line["closure"] = {
                "metric": "column-steps/sec (NN closure applied every host-model step)", "value": nx5 * ny5 * world / (us5 * 1e-6),
                "us_per_call": us5, "scaling": "weak",
                "config": {"workload": "BASELINE config 5 slice: 512 x 64 x 32 y-slab per GPU, implicit convective adjustment + NN forcing, T read / T' + forcing written every call"},
                "roofline": {"bound": "hbm", "achieved": gb5, "peak": hbm_peak, "unit": "GB/s", "frac": gb5 / hbm_peak,
                             "algorithmic_bytes_per_colstep": 384}}
            # SURVEY config 5 as specified: 10^4 host-model steps replayed from a CUDA graph, each step = the closure call
            # followed by a stand-in "dynamics" kernel of the host model (T <- T' + dt * forcing; a torch kernel, not ours)
            try:
                n_inner, n_replay = 100, 100
                Tg = T5_d.clone()
                cur = torch.cuda.current_stream()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=cur):
                    for _ in range(n_inner):
                        m5.closure_step_dev(cd5, Tg, y5_d, f5_d, o5_d)
                        torch.add(o5_d, f5_d, alpha=1e-3, out=Tg)
                graph.replay()
                barrier()
                a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
                a0.record()
                for _ in range(n_replay):
                    graph.replay()
                a1.record()
                barrier()
                tg5 = torch.tensor([a0.elapsed_time(a1)], device="cuda")
                if dist is not None:
                    dist.all_reduce(tg5, op=dist.ReduceOp.MAX)
                usg = float(tg5.item()) / (n_inner * n_replay) * 1e3
                line["closure"]["graph_replay"] = {
                    "host_model_steps": n_inner * n_replay, "us_per_step": usg, "value": nx5 * ny5 * world / (usg * 1e-6),
                    "finite": bool(torch.isfinite(Tg).all().item()),
                    "note": "CUDA graph of 100 x (cpz_closure_step_dev + stand-in dynamics kernel), replayed 100 times"}
            except Exception as e:  # noqa: BLE001
                line["closure"]["graph_replay"] = {"error": repr(e)}
            m5.close()
        except Exception as e:  # noqa: BLE001
            line["closure"] = {"error": repr(e)}
        # ---- SURVEY 8f-2: the embedded u/v/T NDE's per-step closure on a 512 x 64 x 32 slab ----
        try:
            from cpz_b200.desc import ClosureUvtDesc
            d6, th6 = build_workload(syn, RHS_INFER, NSTEPS)
            m6 = engine.Model(ctx, d6, th6)
            nx6, ny6 = 512, 64
            u6, v6, T6 = syn.uvt_fields(d6, nx6, ny6, unstable_every=3)
            cd6 = ClosureUvtDesc(Nx=nx6, Ny=ny6, Nz=32, dz=d6.H / 32, dt=60.0, uw_top=-1e-4, wT_top=2e-5, convective_adjustment=True)
            u6_d, v6_d, T6_d = (torch.tensor(a_, device="cuda") for a_ in (u6, v6, T6))
            f6_d = torch.empty((3,) + tuple(T6_d.shape), device="cuda"); o6_d = torch.empty_like(f6_d)
            for _ in range(5):
                m6.closure_step_uvt_dev(cd6, u6_d, v6_d, T6_d, f6_d, o6_d)
            barrier()
            n6 = 50
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(n6):
                m6.closure_step_uvt_dev(cd6, u6_d, v6_d, T6_d, f6_d, o6_d)
            a1.record()
            barrier()
            t6 = torch.tensor([a0.elapsed_time(a1)], device="cuda")
            if dist is not None:
                dist.all_reduce(t6, op=dist.ReduceOp.MAX)
            us6 = float(t6.item()) / n6 * 1e3
            gb6 = 9 * nx6 * ny6 * 128 / (us6 * 1e-6) / 1e9
            line["closure_uvt"] = {
                "metric": "column-steps/sec (u/v/T NN forcing chains + implicit mPP step applied every host-model step)",
                "value": nx6 * ny6 * world / (us6 * 1e-6), "us_per_call": us6, "scaling": "weak",
                "config": {"workload": "512 x 64 x 32 slab per GPU, three 96->50->20->31 mish nets, convective adjustment on; u, v, T read, "
                                       "three dz-flux fields and u', v', T' written every call (NDE_oceananigans.jl:380-405)",
                           "kernel": "solve_tc_kernel<CLOSURE>: one tcgen05 MLP evaluation + cyclic-reduction mPP step per 32-column tile, persistent CTAs (FP32 SIMT closure_uvt_kernel for other net shapes)"},
                "roofline": {"bound": "hbm", "achieved": gb6, "peak": hbm_peak, "unit": "GB/s", "frac": gb6 / hbm_peak,
                             "algorithmic_bytes_per_colstep": 1152}}
            m6.close()
        except Exception as e:  # noqa: BLE001
            line["closure_uvt"] = {"error": repr(e)}
    if rank == 0 and world == 1 and not args.no_extras:  # the CPU baseline is reported at N = 1 only
        try:
            line["cpu_baseline"] = cpu_baseline(syn, RHS_INFER)
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": repr(e)}
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
