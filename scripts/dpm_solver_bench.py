"""DPM-Solver++(2M) against DDIM on the CIFAR-10 conditional network (bench.py's flagship workload: v-prediction, CFG w = 1,
seeded random weights).  Prints a report and writes it to --out.

  1. per-step time of the fused sampler, 2M against DDIM, at batch --batch (alternating, one process), and the time of
     sampler_step_kernel for both from torch.profiler (eager steps, no graph);
  2. wall-clock images/s through p_sample: 2M at T in {10, 15, 20, 25} against DDIM at 100, at batch --wall-batch;
  3. distance of final samples from a T = 1000 DDIM trajectory with the same x_T, both solvers at T in {10, 15, 20, 25, 50,
     100}, at batch --conv-batch.  Random weights: this says how far each solver's trajectory is from the converged one,
     not anything about sample quality.

    python scripts/dpm_solver_bench.py --out profiles/r5_dpm_solver_bench.txt
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import build_model                                         # noqa: E402
from v_diffusion_b200 import _lib                                      # noqa: E402

SOLVER = "dpmpp_2m"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


def inputs(B, seed=1234):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, 3, 32, 32, generator=g), torch.randint(10, (B,), generator=g) + 1


def per_step(net, diff, B, steps, reps, log):
    """K steps from the start of the trajectory in one range call, timed with CUDA events; the solvers alternate."""
    noise, label = inputs(B)
    dev = torch.device("cuda", 0)
    plan = net.plan_for(32, dev)
    y = label.cuda()
    L = _lib.lib()
    T = diff.sample_timesteps
    scs = {name: diff.sampler_config(True, solver=s) for name, s in (("ddim", None), ("2m", SOLVER))}
    x, pred = noise.cuda(), torch.empty(B, 3, 32, 32, device="cuda")

    def run(sc, n):
        xx = x.clone()
        _lib.check(L.vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(xx), _lib.ptr(y), None, B, T - 1, n, _lib.ptr(pred),
                                        _lib.current_stream_ptr()))
    for sc in scs.values():                                             # graph capture and workspace outside the clock
        run(sc, 2)
    torch.cuda.synchronize()
    times = {k: [] for k in scs}
    for _ in range(reps):
        for name, sc in scs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(sc, steps)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    for name, ts in times.items():
        ts = sorted(ts)
        log(f"  {name:5s} per step: median {ts[len(ts) // 2]:.2f} ms  min {ts[0]:.2f}  max {ts[-1]:.2f}  ({reps} x {steps} steps)")
    # sampler_step_kernel from torch.profiler, eager steps (per-launch profiling mode runs the steps outside the graph)
    from torch.profiler import profile, ProfilerActivity
    L.vdt_profile_enable(1)
    kern = {}
    try:
        for name, sc in scs.items():
            run(sc, 2)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run(sc, steps)
                torch.cuda.synchronize()
            evs = [e for e in prof.events() if "sampler_step_kernel" in e.name]
            # one launch per chunk and step, in launch order; the first (chunk 0, step T-1) is a DDIM row for both solvers
            us = [e.device_time for e in evs] if hasattr(evs[0], "device_time") else [e.cuda_time for e in evs]
            kern[name] = us
    finally:
        L.vdt_profile_enable(0)
    for name, us in kern.items():
        later = sorted(us[1:])
        log(f"  {name:5s} sampler_step_kernel: launch 1 {us[0]:.1f} us, launches 2..{len(us)} median {later[len(later) // 2]:.1f} us "
            f"(min {later[0]:.1f}, max {later[-1]:.1f})")
    return times, kern


def wall_clock(net, diff_factory, B, log):
    noise, label = inputs(B, 99)
    rows = []
    for solver, T in [(None, 100), (SOLVER, 10), (SOLVER, 15), (SOLVER, 20), (SOLVER, 25)]:
        diff = diff_factory(T)
        diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=True, solver=solver)   # warm
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=True, solver=solver)
        torch.cuda.synchronize()
        s = time.perf_counter() - t0
        log(f"  {solver or 'ddim':9s} T={T:3d}: {s:7.3f} s  {B / s:8.1f} images/s")
        rows.append((solver, T, s))
    return rows


def convergence(net, diff_factory, B, log):
    noise, label = inputs(B, 7)
    ref = diff_factory(1000).p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=True)
    log(f"  reference: DDIM T=1000, |x| max {ref.abs().max().item():.3f}")
    for T in (10, 15, 20, 25, 50, 100):
        cells = []
        for solver in (None, SOLVER):
            out = diff_factory(T).p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=True,
                                           solver=solver)
            d = (out - ref).abs()
            cells.append(f"{solver or 'ddim'} max {d.max().item():.4f} mean {d.mean().item():.5f}")
        log(f"  T={T:3d}: " + "   ".join(cells))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--wall-batch", type=int, default=1024)
    ap.add_argument("--conv-batch", type=int, default=256)
    ap.add_argument("--conv-operand", default="fp16x3")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    torch.cuda.set_device(0)
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log(f"card: {card()}  (name, power limit, max SM clock; read in this run)")
    net, diff = build_model(torch.device("cuda", 0), 0)
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule

    def diff_factory(T):
        return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, diff.model_out_type, diff.model_var_type,
                                 "snr_trunc", "mse", intp_frac=diff.intp_frac, w_guide=diff.w_guide)
    log(f"\n[1] per-step time, cifar10_cond CFG w={diff.w_guide}, batch {args.batch} ({2 * args.batch} UNet rows), T=100, "
        f"fp16 operands")
    per_step(net, diff, args.batch, args.steps, args.reps, log)
    log(f"\n[2] wall clock through p_sample, batch {args.wall_batch}, fp16 operands (one warm call, then one timed call each)")
    wall_clock(net, diff_factory, args.wall_batch, log)
    net.operand_dtype = args.conv_operand
    log(f"\n[3] distance from a T=1000 DDIM trajectory, same x_T and labels, batch {args.conv_batch}, {args.conv_operand} operands; "
        "seeded random weights (no quality claim)")
    convergence(net, diff_factory, args.conv_batch, log)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
