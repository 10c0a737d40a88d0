"""Cost of DDIM inversion on the CIFAR-10 conditional network (bench.py's flagship workload: v-prediction, CFG w = 1, seeded
random weights, T = 100).  Prints a report and writes it to --out.

  1. per-step time of the fused inversion step (vdt_ddim_invert_range from step 0) and of the fused DDIM sampling step
     (vdt_p_sample_range from step T-1) at batch --batch, alternating in one process, CUDA events;
  2. invert_step_kernel and sampler_step_kernel time per launch (one 512-image chunk) under torch.profiler (eager steps);
  3. with --parent-tree (a built copy of the previous commit: `git archive HEAD~1 | tar -x -C DIR`, then its build()): each
     tree's own `bench.py --dump-outputs` must write byte-identical samples.npy.

    python scripts/inversion_bench.py --parent-tree build/parent --out profiles/r8_inversion_bench.txt
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import build_model                                         # noqa: E402
from v_diffusion_b200 import _lib                                      # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


class Runner:
    """K inversion steps from t = 0, or K sampling steps from t = 1, in one range call on the same plan."""

    def __init__(self, B):
        self.net, self.diff = build_model(torch.device("cuda", 0), 0)
        g = torch.Generator().manual_seed(1234)
        self.B = B
        self.x = (torch.rand(B, 3, 32, 32, generator=g) * 2 - 1).cuda()
        self.y = (torch.randint(10, (B,), generator=g) + 1).cuda()
        self.plan = self.net.plan_for(32, torch.device("cuda", 0))
        self.sc = self.diff.sampler_config(True)

    def run(self, n, invert):
        L, xx, T = _lib.lib(), self.x.clone(), self.diff.sample_timesteps
        if invert:
            _lib.check(L.vdt_ddim_invert_range(self.plan, C.byref(self.sc), _lib.ptr(xx), _lib.ptr(self.y), self.B, 0, n,
                                               _lib.current_stream_ptr()))
        else:
            _lib.check(L.vdt_p_sample_range(self.plan, C.byref(self.sc), _lib.ptr(xx), _lib.ptr(self.y), None, self.B, T - 1, n,
                                            None, _lib.current_stream_ptr()))

    def kernel_us(self, steps, invert, name):
        """Device times (us) of the named kernel, one per chunk and step, from torch.profiler over eager steps."""
        from torch.profiler import profile, ProfilerActivity
        L = _lib.lib()
        L.vdt_profile_enable(1)
        try:
            self.run(2, invert)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                self.run(steps, invert)
                torch.cuda.synchronize()
        finally:
            L.vdt_profile_enable(0)
        evs = [e for e in prof.events() if name in e.name and "begin" not in e.name]
        return [e.device_time for e in evs] if hasattr(evs[0], "device_time") else [e.cuda_time for e in evs]


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def per_step(r, steps, reps, log):
    modes = {"invert": True, "ddim": False}
    for inv in modes.values():                                          # graph capture and workspace outside the clock
        r.run(2, inv)
    torch.cuda.synchronize()
    times = {k: [] for k in modes}
    for _ in range(reps):
        for name, inv in modes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r.run(steps, inv)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    for name, ts in times.items():
        ts = sorted(ts)
        log(f"  {name:6s} per step: median {median(ts):.2f} ms  min {ts[0]:.2f}  max {ts[-1]:.2f}  ({reps} x {steps} steps)")
    for name, inv, kern in (("invert", True, "invert_step_kernel"), ("ddim", False, "sampler_step_kernel")):
        us = r.kernel_us(steps, inv, kern)
        log(f"  {name:6s} {kern}: median {median(us):.2f} us  min {min(us):.2f}  max {max(us):.2f}  "
            f"({len(us)} launches of one 512-image chunk)")


def ab(args, log):
    trees = {"parent": os.path.abspath(args.parent_tree), "this": ROOT}
    tmp = tempfile.mkdtemp(prefix="inversion_ab_")
    samples = {}
    for name in ("parent", "this", "parent", "this"):
        out = os.path.join(tmp, name)
        r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                            "--no-train-step", "--dump-outputs", out], cwd=trees[name], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        log(f"  bench.py {name}: {line['value']:.1f} {line['unit']}")
        samples[name] = open(os.path.join(out, "samples.npy"), "rb").read()
    log(f"  bench.py --dump-outputs samples.npy byte-identical: {samples['parent'] == samples['this']} "
        f"({len(samples['this'])} bytes)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    torch.cuda.set_device(0)
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log(f"card: {card()}  (name, power limit, max SM clock; read in this run)")
    r = Runner(args.batch)
    log(f"\n[1, 2] cifar10_cond CFG w={r.diff.w_guide}, batch {args.batch} ({2 * args.batch} UNet rows), T=100, fp16 operands: "
        "inversion steps from t = 0 against DDIM sampling steps from t = 1")
    per_step(r, args.steps, args.reps, log)
    del r
    if args.parent_tree:
        log("\n[3] bench.py of this build against the parent build (separate processes, alternating)")
        ab(args, log)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
