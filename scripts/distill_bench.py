"""Cost of progressive distillation on the CIFAR-10 conditional network (bench.py's flagship network and weights, v-prediction).
Prints a report and writes it to --out.

  1. one DistillationStep iteration at --batch (128) with an unguided teacher (w = 0) and a guided one (w = 1): wall time per
     iteration, split into the teacher's two forwards, the two distillation kernels, the student's forward + backward and the
     optimizer (each phase ends in a device synchronise; phases are timed in separate iterations from the totals);
  2. distill_step_kernel and distill_target_kernel: CUDA-event time per launch and achieved GB/s against the bytes they must move,
     at --batch (whose tensors sit in L2) and at 4096 images (larger than L2);
  3. p_sample images/s at batch 4096: the teacher at 2N = --teacher-steps DDIM steps with CFG (w = 1) against a student at N
     steps without CFG (the same network; throughput does not depend on the weights);
  4. the card's name, power limit and max SM clock, read in the same run.

    python scripts/distill_bench.py --out profiles/r11_distill_bench.txt
"""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import build_model                                         # noqa: E402
from v_diffusion_b200 import _lib                                      # noqa: E402
from v_diffusion_b200.training import DistillationStep                # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


class Phases:
    """Accumulates synchronised wall time per phase by wrapping the callables a DistillationStep iteration goes through."""

    def __init__(self):
        self.t = {}
        self.on = False

    def wrap(self, name, fn):
        def timed(*a, **kw):
            if not self.on:
                return fn(*a, **kw)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn(*a, **kw)
            torch.cuda.synchronize()
            self.t[name] = self.t.get(name, 0.0) + time.perf_counter() - t0
            return out
        return timed


def iteration_split(w, B, iters, warmup):
    dev = torch.device("cuda", 0)
    teacher, diff = build_model(dev, 0)
    student, _ = build_model(dev, 0)
    student.train()
    diff.sample_timesteps = 64                                  # the student's N (the cost per iteration does not depend on it)
    ds = DistillationStep(student, teacher, diff, w_guide=w, lr=1e-4)
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(B, 3, 32, 32, generator=g) * 2 - 1).to(dev)
    y = (torch.randint(10, (B,), generator=g) + 1).to(dev)
    ph = Phases()
    L = _lib.lib()
    ds.teacher = ph.wrap("teacher forwards", teacher)
    L.vdt_op_distill_step = ph.wrap("distill kernels", L.vdt_op_distill_step)
    L.vdt_op_distill_target = ph.wrap("distill kernels", L.vdt_op_distill_target)
    ds.graph.forward = ph.wrap("student forward + loss", ds.graph.forward)
    L.vdt_train_loss = ph.wrap("student forward + loss", L.vdt_train_loss)
    ds.graph.backward = ph.wrap("student backward", ds.graph.backward)
    ds.optimizer.step = ph.wrap("optimizer", ds.optimizer.step)
    for _ in range(warmup):
        ds.step(x, y)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        ds.step(x, y)
    torch.cuda.synchronize()
    total = (time.perf_counter() - t0) / iters
    ph.on = True
    for _ in range(iters):
        ds.step(x, y)
    ph.on = False
    return total, {k: v / iters for k, v in ph.t.items()}


def kernel_rates(B, w, reps=50):
    """Per-launch time (CUDA events over reps launches) and achieved GB/s of both kernels at batch B."""
    L = _lib.lib()
    dev = torch.device("cuda", 0)
    _, diff = build_model(dev, 0)
    cfg = int(w > 0)
    chw = 3 * 32 * 32
    tab = diff.distill_coefficients(torch.randint(diff.sample_timesteps, (B,))).to(dev).contiguous()
    out = torch.randn(B * (1 + cfg), 3, 32, 32, device=dev)
    z, zm, x1, xt, et = (torch.randn(B, 3, 32, 32, device=dev) for _ in range(5))
    st = _lib.current_stream_ptr()
    calls = {
        "distill_step_kernel": (lambda: L.vdt_op_distill_step(_lib.ptr(out), _lib.ptr(z), _lib.ptr(zm), _lib.ptr(x1), _lib.ptr(tab),
                                                              B, 3, 1024, cfg, 3, float(w), st), (1 + cfg + 1 + 2) * B * chw * 4),
        "distill_target_kernel": (lambda: L.vdt_op_distill_target(_lib.ptr(out), _lib.ptr(zm), _lib.ptr(x1), _lib.ptr(z), _lib.ptr(xt),
                                                                  _lib.ptr(et), _lib.ptr(tab), B, 3, 1024, cfg, 3, float(w), st),
                                  (1 + cfg + 3 + 2) * B * chw * 4),
    }
    res = {}
    for name, (fn, nbytes) in calls.items():
        for _ in range(5):
            _lib.check(fn())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            _lib.check(fn())
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / reps
        res[name] = (us, nbytes, nbytes / (us * 1e-6) / 1e9)
    return res


def sample_rate(T, w, B=4096, reps=1):
    dev = torch.device("cuda", 0)
    net, diff = build_model(dev, 0)
    diff.sample_timesteps, diff.w_guide = T, w
    g = torch.Generator().manual_seed(1)
    noise = torch.randn(B, 3, 32, 32, generator=g)
    y = torch.randint(10, (B,), generator=g) + 1
    diff.p_sample(net, tuple(noise.shape), noise=noise, label=y, device=dev, use_ddim=True)       # graph capture, workspace
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        diff.p_sample(net, tuple(noise.shape), noise=noise, label=y, device=dev, use_ddim=True)
    torch.cuda.synchronize()
    return B * reps / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--teacher-steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    lines = [f"card: {card()}", ""]
    for w in (0.0, 1.0):
        total, split = iteration_split(w, args.batch, args.iters, args.warmup)
        lines.append(f"DistillationStep iteration, cifar10_cond network, batch {args.batch}, teacher w = {w:g} "
                     f"({'2B' if w > 0 else 'B'} teacher rows): {total * 1e3:.1f} ms (mean of {args.iters}, unsynchronised phases)")
        for k, v in split.items():
            lines.append(f"  {k:<24s} {v * 1e3:8.2f} ms")
        lines.append(f"  {'sum of phases':<24s} {sum(split.values()) * 1e3:8.2f} ms (synchronised after every phase)")
    lines.append("")
    for B in (args.batch, 4096):
        for w in (0.0, 1.0):
            for name, (us, nbytes, gbs) in kernel_rates(B, w).items():
                where = "L2-resident" if nbytes < 100e6 else "larger than L2"
                lines.append(f"{name:<22s} batch {B:5d} cfg {int(w > 0)}: {us:8.2f} us/launch, {nbytes / 1e6:7.2f} MB moved "
                             f"({where}), {gbs:7.1f} GB/s")
    lines.append("")
    N = args.teacher_steps // 2
    teacher_ips = sample_rate(2 * N, 1.0)
    student_ips = sample_rate(N, 0.0)
    lines.append(f"p_sample batch 4096 DDIM: teacher {2 * N} steps with CFG (w = 1): {teacher_ips:.1f} images/s; "
                 f"student {N} steps without CFG: {student_ips:.1f} images/s ({student_ips / teacher_ips:.2f}x)")
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
