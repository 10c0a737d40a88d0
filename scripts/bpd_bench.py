"""Cost of the likelihood bound (calc_all_bpd) on the CIFAR-10 conditional network (bench.py's seeded, de-zeroed weights, v-prediction,
fixed_medium, T = 100) at batch 4096, unguided.  Prints a report and writes it to --out.

  1. per-step time of the fused bound step (vdt_calc_bpd_range) and of an unguided fused DDIM sampling step
     (vdt_p_sample_range, w = 0) at batch --batch, alternating in one process, CUDA events; the images/s of a full T = 1000
     evaluation derived from the bound's step time;
  2. bpd_qsample_kernel, bpd_term_kernel and bpd_finalize_kernel time per launch (one chunk) under torch.profiler (eager
     steps);
  3. with --parent-tree (a built copy of the previous commit: `git archive HEAD~1 | tar -x -C DIR`, then its build()): each
     tree's own `bench.py --dump-outputs` must write byte-identical samples.npy, and the two throughputs alternate.

    python scripts/bpd_bench.py --parent-tree build/parent --out profiles/r9_bpd_bench.txt
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

KERNELS = ("bpd_qsample_kernel", "bpd_term_kernel", "bpd_finalize_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


class Runner:
    """K bound steps, or K unguided DDIM sampling steps from t = 1, in one range call on the same plan."""

    def __init__(self, B):
        self.net, self.diff = build_model(torch.device("cuda", 0), 0)
        g = torch.Generator().manual_seed(1234)
        self.B = B
        self.x = (torch.randint(0, 256, (B, 3, 32, 32), generator=g).float() / 127.5 - 1).cuda()
        self.y = (torch.randint(10, (B,), generator=g) + 1).cuda()
        self.plan = self.net.plan_for(32, torch.device("cuda", 0))
        self.T = self.diff.sample_timesteps
        self.sc_bpd = self.diff.sampler_config(False, seed=3)
        self.sc_ddim = self.diff.sampler_config(True)
        self.sc_ddim.w_guide = 0.0                                      # unguided: one UNet row per image, like the bound
        self.terms = torch.empty((B, self.T), dtype=torch.float64, device="cuda")
        self.mse = torch.empty_like(self.terms)

    def run(self, n, bpd):
        L = _lib.lib()
        if bpd:
            _lib.check(L.vdt_calc_bpd_range(self.plan, C.byref(self.sc_bpd), _lib.ptr(self.x), _lib.ptr(self.y), None, 1, self.B,
                                            self.T - n, n, _lib.ptr(self.terms), _lib.ptr(self.mse), _lib.current_stream_ptr()))
        else:
            xx = self.x.clone()
            _lib.check(L.vdt_p_sample_range(self.plan, C.byref(self.sc_ddim), _lib.ptr(xx), _lib.ptr(self.y), None, self.B,
                                            self.T - 1, n, None, _lib.current_stream_ptr()))

    def kernel_us(self, steps):
        """Device times (us) of each named kernel, one per chunk and step, from torch.profiler over eager steps."""
        from torch.profiler import profile, ProfilerActivity
        L = _lib.lib()
        L.vdt_profile_enable(1)
        try:
            self.run(2, True)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                self.run(steps, True)
                torch.cuda.synchronize()
        finally:
            L.vdt_profile_enable(0)
        out = {}
        for name in KERNELS:
            evs = [e for e in prof.events() if name in e.name]
            out[name] = [e.device_time for e in evs] if evs and hasattr(evs[0], "device_time") else [e.cuda_time for e in evs]
        return out


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def per_step(r, steps, reps, log):
    modes = {"bpd": True, "ddim": False}
    for b in modes.values():                                            # graph capture and workspace outside the clock
        r.run(2, b)
    torch.cuda.synchronize()
    times = {k: [] for k in modes}
    for _ in range(reps):
        for name, b in modes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r.run(steps, b)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    for name, ts in times.items():
        ts = sorted(ts)
        log(f"  {name:4s} per step: median {median(ts):.2f} ms  min {ts[0]:.2f}  max {ts[-1]:.2f}  ({reps} x {steps} steps)")
    step_ms = median(times["bpd"])
    log(f"  derived from the bound's step time (not measured end to end): a T = 1000 evaluation of {r.B} images takes "
        f"{1000 * step_ms / 1e3:.0f} s, {r.B / (1000 * step_ms / 1e3):.2f} images/s on one GPU")
    us = r.kernel_us(steps)
    added = 0.0
    for name in KERNELS:
        v = us[name]
        chunks = max(1, len(v) // steps)
        added += median(v) * chunks
        log(f"  {name}: median {median(v):.2f} us  min {min(v):.2f}  max {max(v):.2f}  ({len(v)} launches, {chunks} chunks per step)")
    log(f"  the three kernels per step: {added:.1f} us = {100 * added / (1e3 * step_ms):.3f} % of the bound's step")


def ab(args, log):
    trees = {"parent": os.path.abspath(args.parent_tree), "this": ROOT}
    tmp = tempfile.mkdtemp(prefix="bpd_ab_")
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
    log(f"\n[1, 2] cifar10_cond unguided, batch {args.batch} ({args.batch} UNet rows), T={r.T}, fp16 operands: bound steps "
        "against DDIM sampling steps with w = 0")
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
