#!/usr/bin/env python
"""wgrad on ragged tiles (28², 14², 7²: 112 / 98 / 98 pixels per 128-row tile) next to the full-tile sizes 32², 16², 8² at the
same channels and pixel count, one TrainingStep.step of BASELINE configs[3]'s network, and an A/B of the existing full-tile
geometries against another build of the library.  Everything runs in one process on cuda:0; the card's name and power limit are
printed first.

    scripts/build_variant.sh <parent commit> parent && scripts/build_variant.sh WORKTREE pr      # before the run
    python scripts/ragged_wgrad_bench.py --ab parent pr
    cp v-diffusion-torch_b200/lib/libvdt_b200_parent.so v-diffusion-torch_b200/lib/libvdt_b200_parent2.so
    python scripts/ragged_wgrad_bench.py --ab parent parent2 --no-step      # the same build twice: the A/B's own noise

Kernel times come from torch.profiler CUDA activity (wgrad_kernel only, as in scripts/backward_widths_bench.py, whose helpers this
script uses).  Useful FLOPs are 2 * pixels * cout * cin * taps; executed FLOPs count the MMAs issued: per tile ceil(pixels / 16)
MMAs of 16 pixel rows on 128-row output-channel blocks.
"""
import math
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import backward_widths_bench as bw                 # noqa: E402
from v_diffusion_b200 import _lib                  # noqa: E402


def tile_rows(B, H):
    """(pixels per tile, tiles) of the forward conv's tiling (plan.cu conv_geom) for a square H x H map; only the executed-FLOP
    column uses it, and the checks keep it from counting fewer or wider tiles than the kernel can run."""
    if 2 * H * H > 128:
        bh = max(d for d in range(1, H + 1) if H % d == 0 and d * H <= 128)
        rows, tiles = bh * H, B * (H // bh)
    else:
        bn = 128 // (H * H)
        rows, tiles = bn * H * H, (B + bn - 1) // bn
    assert rows <= 128 and rows * tiles >= B * H * H, (B, H, rows, tiles)
    return rows, tiles


def wgrad_rates(L):
    print("\n## wgrad (fp16 operands, 256 -> 256, 3x3), 100352 pixels per call (activations 2 x 51 MB); wgrad_kernel time only")
    print("## useful = 2 * pixels * cout * cin * taps; executed = 2 * tiles * 16 * ceil(rows / 16) * cout * cin * taps")
    print(f"{'HxW':>6} {'B':>5} {'rows/tile':>9} {'MMA rows':>8} {'GFLOP':>7} {'kernel us':>10} {'useful TFLOP/s':>15} "
          f"{'executed TFLOP/s':>17}")
    cin = cout = 256
    k = 3
    for H, B in [(28, 128), (32, 98), (14, 512), (16, 392), (7, 2048), (8, 1568)]:
        rows, tiles = tile_rows(B, H)
        mma_rows = 16 * math.ceil(rows / 16)
        fn, _ = bw.wgrad_call(L, B, H, cin, cout, k, bw.wgrad_inputs(B, H, cin, cout, k))
        us = bw.kernel_us(fn, bw.WGRAD_KERNELS)
        fl = 2.0 * B * H * H * cout * cin * k * k
        ex = 2.0 * tiles * mma_rows * cout * cin * k * k
        print(f"{H:>2}x{H:<3} {B:>5} {rows:>9} {mma_rows:>8} {fl / 1e9:>7.1f} {us:>10.1f} {fl / us / 1e6:>15.0f} {ex / us / 1e6:>17.0f}")


def cfg3_step(B=128, steps=3):
    from tests.mnist28_train_worker import CASES
    from tests.train_step_worker import build
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    from v_diffusion_b200.training import TrainingStep
    print(f"\n## one TrainingStep.step of BASELINE configs[3]'s network at batch {B} (1 channel 28x28, hid 256, mult 1-1-1, 3 residual")
    print("## blocks, attention at 14x14 / 7x7, 10 classes; drop_rate 0.2; v, fixed_medium, snr_trunc, p_uncond 0.1).  The untuned")
    print("## composition: per-call scratch allocation and synchronisation inside the C-ABI hooks, fp32 attention backward --")
    print("## a statement of what runs today, not a throughput claim")
    cfg = CASES["mnist_cfg3"]["cfg"]                              # the network tests/test_train_mnist28_gpu.py checks
    _, net = build(cfg, 5, "fp16", drop_rate=0.2)
    net.train()
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 1000, "v", "fixed_medium", "snr_trunc", "mse", intp_frac=0.3,
                             w_guide=3.0, p_uncond=0.1)
    ts = TrainingStep(net, diff, timesteps=0, lr=2e-4, weight_decay=0.0, grad_norm=1.0, use_ema=True, ema_decay=0.9999)
    g = torch.Generator().manual_seed(3)
    x = (torch.rand(B, 1, 28, 28, generator=g) * 2 - 1).to(bw.dev)
    y = torch.randint(1, 11, (B,), generator=g).to(bw.dev)
    ts.step(x, y)                                                  # warm-up: module loads, first allocations
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        loss = ts.step(x, y)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    print(f"step wall time (s, each with a device synchronise): {', '.join(f'{t:.3f}' for t in times)}; loss {float(loss):.4f}")
    print(f"peak memory allocated by torch: {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB "
          "(the hooks' own cudaMalloc scratch is not counted by torch)")


def ab(names, rounds=8):
    import ctypes as C
    libs = {n: bw.bind(C.CDLL(os.path.join(_lib.LIB_DIR, f"libvdt_b200_{n}.so"))) for n in names}
    print(f"\n## A/B at the existing 128-row geometries: {' vs '.join(names)} (libvdt_b200_<name>.so), {rounds} rounds, the order")
    print("## of the two builds swapped every round,")
    print("## wgrad + split reduction + bias kernel us per call (min-max over the rounds)")
    shapes = [(128, 32, 256, 256, 3), (128, 16, 256, 256, 3), (128, 8, 256, 256, 3), (128, 32, 512, 256, 3), (64, 16, 128, 128, 3),
              (64, 32, 512, 256, 1), (16, 64, 192, 384, 3), (64, 32, 192, 192, 3)]       # (B, H, cin, cout, k)
    for (B, H, cin, cout, k) in shapes:
        ins = bw.wgrad_inputs(B, H, cin, cout, k)
        runs = {n: bw.wgrad_call(L, B, H, cin, cout, k, ins) for n, L in libs.items()}
        t = {n: [] for n in names}
        for r in range(rounds):
            for n in (names if r % 2 == 0 else names[::-1]):      # alternate which build goes first
                t[n].append(bw.kernel_us(runs[n][0], bw.WGRAD_KERNELS + ("wgrad_reduce", "bias_grad"), reps=5))
        for n in names:
            runs[n][0]()
        torch.cuda.synchronize()
        same = all(torch.equal(a, b) for a, b in zip(runs[names[0]][1], runs[names[1]][1]))
        med = {n: sorted(v)[len(v) // 2] for n, v in t.items()}
        print(f"wgrad {cin}->{cout} k{k} B={B} {H}x{H}: " + "; ".join(f"{n} {min(v):.1f}-{max(v):.1f}" for n, v in t.items())
              + f"; median {names[1]} / {names[0]} {med[names[1]] / med[names[0]] - 1:+.2%} (spread over the rounds: "
              + ", ".join(f"{n} {(max(v) - min(v)) / med[n]:.2%}" for n, v in t.items()) + f"); outputs (dW, db) bit-identical: {same}")


if __name__ == "__main__":
    assert torch.cuda.is_available(), "this script measures on the GPU; there is no CPU path"
    torch.cuda.set_device(0)
    print("card (name, power limit, max SM clock):", bw.card())
    L = bw.bind(_lib.lib())
    wgrad_rates(L)
    if "--ab" in sys.argv:
        i = sys.argv.index("--ab")
        ab(sys.argv[i + 1:i + 3])
    if "--no-step" not in sys.argv:
        cfg3_step()
