"""Cost of inpainting on the CIFAR-10 conditional network (bench.py's flagship workload: v-prediction, CFG w = 1, seeded random
weights, T = 100 DDIM).  Prints a report and writes it to --out.

  1. per-step time of the fused sampler with and without inpainting (left-half box mask, z' from the library's stream) at
     batch --batch, alternating in one process, CUDA events;
  2. sampler_step_kernel time per launch (one 512-image chunk) under torch.profiler, with and without inpainting (eager steps);
  3. with --parent-tree (a built copy of the previous commit: `git archive HEAD~1 | tar -x -C DIR`, then its build()): this
     build without inpainting against it.  Each tree's own `bench.py --dump-outputs` must write byte-identical samples.npy,
     and the kernel-time medians of (2) without inpainting are compared with the spread of the parent tree against itself
     (separate processes, alternating).

    python scripts/inpaint_bench.py --parent-tree build/parent --out profiles/r6_inpaint_bench.txt
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROOT = os.environ.get("INPAINT_BENCH_TREE", HERE)          # the tree whose package and library a --kernel-child run imports
sys.path.insert(0, ROOT)

from bench import build_model                                         # noqa: E402
from v_diffusion_b200 import _lib                                      # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


class Sampler:
    """K steps from the start of the trajectory in one range call, with or without inpainting."""

    def __init__(self, B):
        self.net, self.diff = build_model(torch.device("cuda", 0), 0)
        g = torch.Generator().manual_seed(1234)
        self.B = B
        self.x = torch.randn(B, 3, 32, 32, generator=g).cuda()
        self.y = (torch.randint(10, (B,), generator=g) + 1).cuda()
        self.known = (torch.rand(B, 3, 32, 32, generator=g) * 2 - 1).cuda()
        self.mask = torch.zeros(B, 3, 32, 32, device="cuda")
        self.mask[..., :16] = 1.0
        self.pred = torch.empty_like(self.x)
        self.plan = self.net.plan_for(32, torch.device("cuda", 0))
        self.sc = self.diff.sampler_config(True, seed=5)
        self.has_inpaint = hasattr(_lib.lib(), "vdt_p_sample_range_inpaint")
        if self.has_inpaint:
            self.ip = _lib.Inpaint(_lib.ptr(self.known), _lib.ptr(self.mask), None)

    def run(self, n, inpaint):
        L, xx, T = _lib.lib(), self.x.clone(), self.diff.sample_timesteps
        if inpaint:
            _lib.check(L.vdt_p_sample_range_inpaint(self.plan, C.byref(self.sc), C.byref(self.ip), _lib.ptr(xx), _lib.ptr(self.y),
                                                    None, self.B, T - 1, n, _lib.ptr(self.pred), _lib.current_stream_ptr()))
        else:
            _lib.check(L.vdt_p_sample_range(self.plan, C.byref(self.sc), _lib.ptr(xx), _lib.ptr(self.y), None, self.B, T - 1, n,
                                            _lib.ptr(self.pred), _lib.current_stream_ptr()))

    def kernel_us(self, steps, inpaint):
        """sampler_step_kernel device times (us), one per chunk and step, from torch.profiler over eager steps."""
        from torch.profiler import profile, ProfilerActivity
        L = _lib.lib()
        L.vdt_profile_enable(1)
        try:
            self.run(2, inpaint)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                self.run(steps, inpaint)
                torch.cuda.synchronize()
        finally:
            L.vdt_profile_enable(0)
        evs = [e for e in prof.events() if "sampler_step_kernel" in e.name]
        return [e.device_time for e in evs] if hasattr(evs[0], "device_time") else [e.cuda_time for e in evs]


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def per_step(s, steps, reps, log):
    modes = {"plain": False, "inpaint": True}
    for inp in modes.values():                                          # graph capture and workspace outside the clock
        s.run(2, inp)
    torch.cuda.synchronize()
    times = {k: [] for k in modes}
    for _ in range(reps):
        for name, inp in modes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            s.run(steps, inp)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    for name, ts in times.items():
        ts = sorted(ts)
        log(f"  {name:8s} per step: median {median(ts):.2f} ms  min {ts[0]:.2f}  max {ts[-1]:.2f}  ({reps} x {steps} steps)")
    for name, inp in modes.items():
        us = s.kernel_us(steps, inp)
        log(f"  {name:8s} sampler_step_kernel: median {median(us):.2f} us  min {min(us):.2f}  max {max(us):.2f}  "
            f"({len(us)} launches of one 512-image chunk)")


def kernel_child(args):
    """Runs on the tree INPAINT_BENCH_TREE names: sampler_step_kernel medians without inpainting, one JSON line."""
    s = Sampler(args.batch)
    s.run(2, False)
    print("KERNEL " + json.dumps([median(s.kernel_us(args.steps, False)) for _ in range(args.reps)]), flush=True)


def ab(args, log):
    trees = {"parent": os.path.abspath(args.parent_tree), "this": HERE}
    tmp = tempfile.mkdtemp(prefix="inpaint_ab_")
    samples = {}
    for name, tree in trees.items():
        out = os.path.join(tmp, name)
        r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                            "--no-train-step", "--dump-outputs", out], cwd=tree, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        log(f"  bench.py {name}: {line['value']:.1f} {line['unit']}")
        samples[name] = open(os.path.join(out, "samples.npy"), "rb").read()
    log(f"  bench.py --dump-outputs samples.npy byte-identical: {samples['parent'] == samples['this']} "
        f"({len(samples['this'])} bytes)")
    runs = {"parent": [], "this": []}
    for name in ("parent", "this", "parent", "this", "parent"):
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--kernel-child", "--batch", str(args.batch), "--steps",
                            str(args.steps), "--reps", "3"], cwd=HERE, env=dict(os.environ, INPAINT_BENCH_TREE=trees[name]),
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-3000:]
        runs[name] += json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("KERNEL ")][-1][len("KERNEL "):])
    for name, v in runs.items():
        log(f"  {name:6s} sampler_step_kernel medians without inpainting (us): {', '.join(f'{x:.2f}' for x in v)}")
    p, t = runs["parent"], runs["this"]
    log(f"  parent against itself: {min(p):.2f} .. {max(p):.2f} us; this build {min(t):.2f} .. {max(t):.2f} us; "
        f"this build within the parent's spread: {min(p) <= min(t) and max(t) <= max(p)}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--out", default=None)
    ap.add_argument("--kernel-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    torch.cuda.set_device(0)
    if args.kernel_child:
        return kernel_child(args)
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    log(f"card: {card()}  (name, power limit, max SM clock; read in this run)")
    s = Sampler(args.batch)
    log(f"\n[1, 2] cifar10_cond CFG w={s.diff.w_guide}, batch {args.batch} ({2 * args.batch} UNet rows), T=100 DDIM, fp16 operands; "
        "inpainting: left-half mask, known image, z' from the library's stream")
    per_step(s, args.steps, args.reps, log)
    del s
    if args.parent_tree:
        log("\n[3] this build without inpainting against the parent build (separate processes, alternating)")
        ab(args, log)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
