#!/usr/bin/env python
"""Rates of the backward kernels at the CelebA widths, one CelebA training step, and an A/B of the existing widths against
another build of the library.  Everything runs in one process on cuda:0; the card's name and power limit are printed first.

    scripts/build_variant.sh HEAD~1 parent && scripts/build_variant.sh WORKTREE pr      # here, before the run
    python scripts/backward_widths_bench.py --ab parent pr

Kernel times come from torch.profiler CUDA activity (kernel time only: the C-ABI hooks allocate scratch and synchronise per
call, which the rates leave out).  Bytes and FLOPs are computed from shapes: GroupNorm backward moves x and dA twice and
writes dx once (20 B per element); wgrad counts 2 * pixels * cout * cin * taps useful FLOPs.
"""
import ctypes as C
import math
import os
import subprocess
import sys
import time

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from v_diffusion_b200 import _lib  # noqa: E402

dev = "cuda"
p = lambda t: None if t is None else C.c_void_p(t.data_ptr())      # noqa: E731
GN_KERNELS = ("gn_stats_kernel", "gn_bwd_")
WGRAD_KERNELS = ("wgrad_kernel",)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def kernel_us(fn, names, reps=10):
    """Mean CUDA time per call (us) of the kernels whose names contain one of `names`, over `reps` calls after a warm-up."""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    tot = 0.0
    for e in prof.key_averages():
        if any(n in e.key for n in names):
            tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
    return tot / reps


def bind(L):
    vp, i32 = C.c_void_p, C.c_int32
    L.vdt_last_error.restype = C.c_char_p
    L.vdt_op_groupnorm_backward.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, i32, C.c_float, C.c_uint64, i32, vp, vp, vp, vp, vp]
    L.vdt_op_conv_wgrad.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, i32, vp]
    return L


def ok(L, rc):
    if rc != 0:
        raise RuntimeError(L.vdt_last_error().decode())


def gn_inputs(B, H, Cc, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed + Cc)
    x = torch.randn(B, H, H, Cc, device=dev, generator=g)
    go = torch.randn(B, H, H, Cc, device=dev, generator=g)
    gamma = torch.rand(Cc, device=dev, generator=g) + 0.5
    beta = torch.randn(Cc, device=dev, generator=g) * 0.2
    film = torch.randn(B, 2 * Cc, device=dev, generator=g) * 0.3
    return x, go, gamma, beta, film


def gn_call(L, B, H, Cc, ins, drop=0.1):
    x, go, gamma, beta, film = ins
    out = [torch.empty_like(x), torch.empty(Cc, device=dev), torch.empty(Cc, device=dev), torch.empty_like(film)]
    fn = lambda: ok(L, L.vdt_op_groupnorm_backward(p(x), p(go), Cc, B, H, H, p(gamma), p(beta), p(film), 1, C.c_float(drop), 7, 3,  # noqa: E731
                                                   *map(p, out), None))
    return fn, out


def wgrad_inputs(B, H, cin, cout, k, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed + cin + cout + k)
    x = torch.randn(B, H, H, cin, device=dev, generator=g).half()
    dy = torch.randn(B, H, H, cout, device=dev, generator=g).half()
    return x, dy


def wgrad_call(L, B, H, cin, cout, k, ins):
    x, dy = ins
    out = [torch.empty(cout, cin, k, k, device=dev), torch.empty(cout, device=dev)]
    fn = lambda: ok(L, L.vdt_op_conv_wgrad(p(x), p(dy), B, H, H, cin, cout, k, p(out[0]), p(out[1]), 1, None))  # noqa: E731
    return fn, out


def gn_rates(L):
    print("\n## GroupNorm backward (FiLM + SiLU + dropout 0.1), ~2^24 elements per tensor (x and dA 2 x 67 MB: above L2)")
    print(f"{'C':>6} {'HxW':>7} {'B':>4} {'vec':>4} {'MB moved':>9} {'kernel us':>10} {'GB/s':>7}")
    for Cc, H in [(256, 32), (192, 64), (384, 32), (576, 16), (768, 8), (960, 32), (1152, 16), (1344, 16), (1536, 8), (64, 64)]:
        B = max(1, round(2 ** 24 / (H * H * Cc)))
        fn, _ = gn_call(L, B, H, Cc, gn_inputs(B, H, Cc))
        us = kernel_us(fn, GN_KERNELS)
        mb = 20.0 * B * H * H * Cc / 1e6
        tag = "  (existing width)" if Cc in (128, 256, 512, 1024) else ""
        print(f"{Cc:>6} {H:>3}x{H:<3} {B:>4} {4 if (Cc // 32) % 4 == 0 else 2:>4} {mb:>9.1f} {us:>10.1f} {mb * 1e3 / us:>7.0f}{tag}")


def wgrad_rates(L):
    print("\n## wgrad (fp16 operands), useful FLOPs 2 * pixels * cout * cin * taps; wgrad_kernel time only (without the split")
    print("## reduction and the bias kernel).  cout % 128 == 64: the last 128-row MMA block has 64 zero rows -- half of that block's")
    print("## tensor work is spent on zeros; 'issued' counts them")
    print(f"{'cin->cout':>11} {'k':>2} {'HxW':>6} {'B':>4} {'GFLOP':>8} {'kernel us':>10} {'TFLOP/s':>8} {'issued TFLOP/s':>15}")
    for (cin, cout, k, H, B) in [(192, 192, 3, 32, 64), (384, 384, 3, 32, 64), (576, 576, 3, 32, 64), (768, 768, 3, 32, 64),
                                 (192, 192, 3, 64, 16), (384, 384, 3, 64, 16), (576, 576, 3, 16, 16), (768, 768, 3, 16, 16)]:
        fn, _ = wgrad_call(L, B, H, cin, cout, k, wgrad_inputs(B, H, cin, cout, k))
        us = kernel_us(fn, WGRAD_KERNELS)
        fl = 2.0 * B * H * H * cout * cin * k * k
        issued = fl * (128 * math.ceil(cout / 128)) / cout
        print(f"{cin:>5}->{cout:<5} {k:>2} {H:>2}x{H:<3} {B:>4} {fl / 1e9:>8.1f} {us:>10.1f} {fl / us / 1e6:>8.0f} {issued / us / 1e6:>15.0f}")


def celeba_step(B=16, steps=3):
    from tests.cases import CELEBA
    from tests.train_step_worker import build
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    from v_diffusion_b200.training import TrainingStep
    print(f"\n## one CelebA TrainingStep.step at batch {B} (celeba.json: hid 192, 64x64, drop_rate 0.1, 'both', fixed_large, snr_trunc)")
    print("## the untuned composition: per-call scratch allocation and synchronisation inside the C-ABI hooks, fp32 attention")
    print("## backward -- a statement of what runs today, not a throughput claim")
    _, net = build(CELEBA, 5, "fp16", drop_rate=0.1)
    net.train()
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 256, "both", "fixed_large", "snr_trunc", "mse", intp_frac=0.0,
                             p_uncond=0.1)
    ts = TrainingStep(net, diff, timesteps=0, lr=2e-4, weight_decay=0.0, grad_norm=1.0, use_ema=True, ema_decay=0.9999)
    x = (torch.rand(B, 3, 64, 64, generator=torch.Generator().manual_seed(3)) * 2 - 1).to(dev)
    ts.step(x, None)                                               # warm-up: module loads, first allocations
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        loss = ts.step(x, None)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    print(f"step wall time (s, each with a device synchronise): {', '.join(f'{t:.3f}' for t in times)}; loss {float(loss):.4f}")
    print(f"peak memory allocated by torch: {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB "
          "(the hooks' own cudaMalloc scratch is not counted by torch)")


def ab(names, rounds=5):
    libs = {n: bind(C.CDLL(os.path.join(_lib.LIB_DIR, f"libvdt_b200_{n}.so"))) for n in names}
    print(f"\n## A/B at the existing widths: {' vs '.join(names)} (libvdt_b200_<name>.so), {rounds} alternating rounds, kernel us per call")
    gn_shapes = [(128, 32, 256), (64, 16, 512), (128, 16, 128), (32, 8, 1024)]          # (B, H, C)
    wg_shapes = [(128, 32, 256, 256, 3), (128, 16, 256, 256, 3), (128, 32, 512, 256, 3), (64, 16, 128, 128, 3),
                 (64, 32, 512, 256, 1), (16, 64, 192, 384, 3)]                           # (B, H, cin, cout, k)
    for (B, H, Cc) in gn_shapes:
        ins = gn_inputs(B, H, Cc)
        runs = {n: gn_call(L, B, H, Cc, ins) for n, L in libs.items()}
        t = {n: [] for n in names}
        for _ in range(rounds):
            for n in names:
                t[n].append(kernel_us(runs[n][0], GN_KERNELS, reps=5))
        for n in names:
            runs[n][0]()
        torch.cuda.synchronize()
        same = all(torch.equal(a, b) for a, b in zip(runs[names[0]][1], runs[names[1]][1]))
        print(f"groupnorm backward B={B} {H}x{H} C={Cc}: " + "; ".join(f"{n} {min(v):.1f}-{max(v):.1f}" for n, v in t.items())
              + f"; outputs (dx, dgamma, dbeta, dfilm) bit-identical: {same}")
    for (B, H, cin, cout, k) in wg_shapes:
        ins = wgrad_inputs(B, H, cin, cout, k)
        runs = {n: wgrad_call(L, B, H, cin, cout, k, ins) for n, L in libs.items()}
        t = {n: [] for n in names}
        for _ in range(rounds):
            for n in names:
                t[n].append(kernel_us(runs[n][0], WGRAD_KERNELS + ("wgrad_reduce", "bias_grad"), reps=5))
        for n in names:
            runs[n][0]()
        torch.cuda.synchronize()
        same = all(torch.equal(a, b) for a, b in zip(runs[names[0]][1], runs[names[1]][1]))
        print(f"wgrad + reduce + dbias {cin}->{cout} k{k} B={B} {H}x{H}: " + "; ".join(f"{n} {min(v):.1f}-{max(v):.1f}" for n, v in t.items())
              + f"; outputs (dW, db) bit-identical: {same}")


if __name__ == "__main__":
    assert torch.cuda.is_available(), "this script measures on the GPU; there is no CPU path"
    torch.cuda.set_device(0)
    print("card (name, power limit, max SM clock):", card())
    L = bind(_lib.lib())
    gn_rates(L)
    wgrad_rates(L)
    if "--ab" in sys.argv:
        i = sys.argv.index("--ab")
        ab(sys.argv[i + 1:i + 3])
    if "--no-step" not in sys.argv:
        celeba_step()
