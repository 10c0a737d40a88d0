#!/usr/bin/env python
"""Headline benchmark: DDIM images/sec, CIFAR-10 class-conditional UNet, CFG w=1 (cond/uncond batched as 2B
rows in one UNet call), 100-step DDIM, batch 4096 per GPU (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A "step" is one denoising step of the real sampling loop over the whole per-GPU batch: one UNet forward on
2*B rows plus the fused sampler update (diffusion.py:360-392).  100 such steps make B images, so
images/s = N_gpus * B * K / (100 * t_K).  Inputs are synthetic (seeded normal noise, random labels, random
non-zero weights of the reference architecture); every tensor a step touches is far larger than L2.
One process per GPU; multi-GPU is weak scaling with no collective in the loop (SURVEY §8e).

The N=1 line also carries, outside every timed region: `cpu_baseline` (the unmodified reference on the host cores),
`reference_gpu_eager` (the unmodified reference in stock PyTorch eager on the same GPU) and `train_step` (BASELINE configs[4]:
one cifar10_cond training step at batch 128 through v_diffusion_b200.training.TrainingStep beside the reference's own step under
autograd, measured in a child process; the composition is parity-green but untuned, see DESIGN.md section 7).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_STEPS = 100
W_GUIDE = 1.0
METRIC = "ddim_images_per_sec_cifar10_cfg_100step"
# extra workloads (parity-test configs of BASELINE.json, measurable with --workload; the headline stays cifar10_cond)
CELEBA_MODEL = dict(in_channels=3, hid_channels=192, ch_multipliers=[1, 2, 3, 4], num_res_blocks=3,
                    apply_attn=[False, True, True, True], embedding_dim=768, drop_rate=0.1, head_dim=64, num_heads=1)
WORKLOADS = {
    # name: (model kwargs, out_channels, num_classes, resolution, model_out_type, var_type, cfg, default batch, text)
    "cifar10_cond": None,
    "celeba": (CELEBA_MODEL, 6, 0, 64, "both", "fixed_large", False, 1024,
               "CelebA 64x64 UNet (celeba.json), unconditional, 100-step DDIM"),
    "cifar10_uncond": (dict(in_channels=3, hid_channels=256, ch_multipliers=[1, 1, 1], num_res_blocks=3,
                            apply_attn=[False, True, True], drop_rate=0.2, num_heads=1), 3, 0, 32, "x0", "fixed_large",
                       False, 4096, "CIFAR-10 unconditional UNet (cifar10_uncond.json), 100-step DDIM"),
    # BASELINE configs[3]: defaults.json model block with in_channels=1, 10 classes, 28x28 (28 -> 14 -> 7), CFG w=3,
    # 1000-step ancestral sampling with on-device noise: small images, launch-bound, one CUDA graph per step
    "mnist28": (dict(in_channels=1, hid_channels=256, ch_multipliers=[1, 1, 1], num_res_blocks=3,
                     apply_attn=[False, True, True], drop_rate=0.2, num_heads=1), 1, 10, 28, "v", "fixed_medium",
                True, 256, "MNIST 28x28 conditional UNet (defaults.json model, 1 channel), CFG w=3, 1000-step ancestral sampling",
                1000, 3.0, False),
}


def workload_params(name):
    """(T, w_guide, use_ddim, in_channels) of a workload; the 100-step DDIM workloads use w = 1."""
    wl = WORKLOADS[name]
    if wl is None or len(wl) < 12:
        return T_STEPS, W_GUIDE, True, 3
    return wl[9], wl[10], wl[11], wl[0]["in_channels"]


# cifar10_cond.json merged with defaults.json (tests/golden/merged_configs.json pins this in the CPU tests)
CIFAR_COND_MODEL = dict(in_channels=3, hid_channels=256, ch_multipliers=[1, 1, 1], num_res_blocks=3,
                        apply_attn=[False, True, True], drop_rate=0.2, num_heads=1)
FLOP_PER_ROW = 37.644423168e9          # conv 35.965 + attention 1.648 + linear 0.031 GF (vdt_plan_flops, SURVEY §6)


def read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(tflops=p["bf16_tflops_sustained"], tflops_burst=p["bf16_tflops"], hbm=p["hbm_gbs"], source="measured")
    except Exception:
        return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        busy = sorted(sm)[len(sm) // 4:]                     # drop idle samples at the edges
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in self.rows if len(r) >= 7)}


def build_model(device, seed, workload="cifar10_cond"):
    import torch
    from v_diffusion_b200 import UNet, GaussianDiffusion, get_logsnr_schedule
    torch.manual_seed(seed)
    wl = WORKLOADS[workload]
    if wl is None:
        net = UNet(out_channels=3, num_classes=10, multitags=False, **CIFAR_COND_MODEL)
        out_type, var_type = "v", "fixed_medium"
    else:
        net = UNet(out_channels=wl[1], num_classes=wl[2], multitags=False, **wl[0])
        out_type, var_type = wl[4], wl[5]
    g = torch.Generator().manual_seed(seed + 7)
    with torch.no_grad():
        for name, p in net.named_parameters():
            # the reference zero-initialises conv2 / proj_out / out_conv (SURVEY §9.1): a zero network would
            # exercise nothing, so every all-zero matrix gets N(0, 1/fan_in) and biases / norms get jitter
            if p.ndim >= 2 and not bool(p.any()):
                fan_in = p[0].numel()
                p.copy_(torch.randn(p.shape, generator=g) / fan_in ** 0.5)
            elif p.ndim == 1:
                p.add_(0.05 * torch.randn(p.shape, generator=g))
    net = net.to(device).eval()
    T, w, _, _ = workload_params(workload)
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, out_type, var_type, "snr_trunc",
                             "mse", intp_frac=0.3, w_guide=w)
    return net, diff


def reference_staged():
    from oracle import stage_ref
    return stage_ref.staged()


def reference_objects(state_dict, device):
    """The UNMODIFIED reference (oracle/_ref, staged by oracle/stage_ref.py) built the way generate.py:48-98 builds it
    for cifar10_cond.json, with this bench's weights and w_guide = 1, 100 steps.  Returns (model, diffusion)."""
    import torch
    from oracle import stage_ref
    ref = stage_ref.load()
    cfg = stage_ref.config("cifar10_cond")
    d = dict(cfg["diffusion"])
    logsnr_fn = ref.get_logsnr_schedule(d.pop("logsnr_schedule"), logsnr_min=d.pop("logsnr_min"),
                                        logsnr_max=d.pop("logsnr_max"), rescale=d.pop("allow_rescale"))
    d.pop("train_timesteps")
    d["sample_timesteps"] = T_STEPS
    diffusion = ref.GaussianDiffusion(logsnr_fn=logsnr_fn, w_guide=W_GUIDE, **d)
    model = ref.UNet(out_channels=3, num_classes=10, multitags=False, **cfg["model"])
    model.load_state_dict({k: v.detach().float().cpu() for k, v in state_dict.items()}, strict=True)
    return model.to(device).eval(), diffusion


def reference_steps(diffusion, model, x_t, label, first_ti, n_steps, sync=None):
    """n_steps iterations of the body of the reference's own p_sample loop (diffusion.py:410-413) from step index
    first_ti downwards (a run longer than the trajectory keeps repeating step 1).  Returns x after the last step."""
    import torch
    t = torch.empty((x_t.shape[0],), device=x_t.device, dtype=torch.float64)
    ti = first_ti
    with torch.inference_mode():
        for _ in range(n_steps):
            t.fill_(ti)
            x_t = diffusion.p_sample_step(model, x_t, step=t, y=label, generator=None, use_ddim=True)
            ti = max(ti - 1, 1)
    if sync:
        sync()
    return x_t


def oracle_trajectory(sd, cfg, x_t, label, n_warm, n_steps, budget_s=None):
    """Fallback when oracle/_ref is not staged: the same steps with the oracle port (test infrastructure, pinned to
    the reference by tests/golden).  Returns (x after the last step, seconds per timed step, timed steps)."""
    import torch
    from oracle import unet_forward
    from oracle.diffusion_ref import step_coefficients, _pred_x0
    co = step_coefficients(T_STEPS, use_ddim=True)
    B = x_t.shape[0]

    def step(x_t, ti):
        xin = x_t.repeat_interleave(2, dim=0)
        yin = label.repeat_interleave(2).clone(); yin[1::2] = 0
        t = torch.full((2 * B,), co["t_model"][ti], dtype=torch.float64)
        out = unet_forward(sd, cfg, xin, t, yin)
        x0 = _pred_x0(xin, out, torch.tensor(co["logsnr_t"][ti]), "v").clamp(-1, 1)
        mean = float(co["c1"][ti]) * xin + float(co["c2"][ti]) * x0
        return mean[0::2] + W_GUIDE * (mean[0::2] - mean[1::2])
    ti = T_STEPS - 1
    for _ in range(n_warm):
        x_t = step(x_t, ti); ti = max(ti - 1, 1)       # (a run longer than the trajectory keeps timing step 1)
    n, t0 = 0, time.perf_counter()
    while n < n_steps and (budget_s is None or n < 2 or time.perf_counter() - t0 < budget_s):
        x_t = step(x_t, ti); ti = max(ti - 1, 1); n += 1
    return x_t, (time.perf_counter() - t0) / max(n, 1), n


def cpu_reference_trajectory(state_dict, x_t, label, n_warm, n_steps, budget_s=None):
    """First n_warm + n_steps denoising steps of the CIFAR-10 cond CFG DDIM trajectory on the host CPU: the unmodified
    reference when it is staged (kind "reference"), else the oracle port (kind "port").
    Returns (kind, x after the last step, seconds per timed step, timed steps)."""
    import torch
    torch.set_num_threads(os.cpu_count())
    if reference_staged():
        model, diffusion = reference_objects(state_dict, "cpu")
        x = reference_steps(diffusion, model, x_t, label, T_STEPS - 1, n_warm)
        ti = max(T_STEPS - 1 - n_warm, 1)
        n, t0 = 0, time.perf_counter()
        while n < n_steps and (budget_s is None or n < 2 or time.perf_counter() - t0 < budget_s):
            x = reference_steps(diffusion, model, x, label, ti, 1); ti = max(ti - 1, 1); n += 1
        return "reference", x, (time.perf_counter() - t0) / max(n, 1), n
    from oracle.unet_ref import unet_config_from_json
    cfg = unet_config_from_json(CIFAR_COND_MODEL, 3, 3, num_classes=10)
    sd = {k: v.detach().cpu().float() for k, v in state_dict.items()}
    x, dt, n = oracle_trajectory(sd, cfg, x_t, label, n_warm, n_steps, budget_s)
    return "port", x, dt, n


def cpu_baseline(net, diff, noise2, label2, device, seconds_budget=20.0):
    """The reference's CPU implementation on the host cores on a bounded sample of the same workload: the FIRST
    denoising steps of the bench's own trajectory for its first two images (4 UNet rows per step), on the bench's own
    weights, scaled by 100 steps / image.  The same steps are then run through the CUDA path and compared (`parity`)."""
    import ctypes as C
    import torch
    from v_diffusion_b200 import _lib
    B = noise2.shape[0]
    kind, x_cpu, dt, n = cpu_reference_trajectory(net.state_dict(), noise2.clone(), label2, 1, 16, seconds_budget)
    steps = n + 1
    x = noise2.to(device).contiguous().clone()
    y = label2.to(device).contiguous()
    sc = diff.sampler_config(use_ddim=True)
    plan = net.plan_for(noise2.shape[2], device)
    _lib.check(_lib.lib().vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(y), None, B, T_STEPS - 1, steps,
                                             None, _lib.current_stream_ptr()))
    torch.cuda.synchronize()
    err = (x.cpu() - x_cpu).abs().max().item()
    return {"value": B / (dt * T_STEPS), "unit": "images/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"first {steps} denoising steps of the bench trajectory for its first {B} images "
                      f"({2 * B} UNet rows per step, CFG pair), {n} timed at {dt:.3f} s/step, scaled by {T_STEPS} steps per image",
            "parity": {"steps": steps, "images": B, "max_abs_vs_cuda_path": err}}


def reference_gpu_eager(net, diff, noise, label, device, batch=256, parity_batch=32, steps=4):
    """The untouched reference on this same GPU in stock PyTorch eager (what a user of the reference gets on a B200):
    throughput of its own p_sample loop body at `batch` images per step -- once with PyTorch's default flags (cuDNN
    convolutions in TF32, generate.py:115-116 sets cudnn.benchmark) and once in strict fp32 -- and, outside any timed
    region, all 100 steps of `parity_batch` images in strict fp32 against the CUDA path on the same noise / labels."""
    import torch
    if not reference_staged():
        return {"unavailable": "oracle/_ref not staged (build() stages it where /root/reference exists)"}
    model, rdiff = reference_objects(net.state_dict(), device)
    out = {"batch": batch, "rows_per_unet_call": 2 * batch, "steps_timed": steps,
           "note": "unmodified reference (oracle/_ref) in torch eager on this GPU, its own p_sample_step loop"}
    saved = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        torch.backends.cudnn.benchmark = True                           # generate.py:115-116
        x0, y0 = noise[:batch].clone(), label[:batch].clone()
        for mode, tf32 in (("stock_flags_tf32_convs", True), ("strict_fp32", False)):
            torch.backends.cudnn.allow_tf32 = tf32
            reference_steps(rdiff, model, x0, y0, T_STEPS - 1, 2, torch.cuda.synchronize)       # warm-up / autotune
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            reference_steps(rdiff, model, x0, y0, T_STEPS - 3, steps)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"ms_per_step": ms, "images_per_s": batch / (ms * 1e-3 * T_STEPS)}
        torch.backends.cudnn.allow_tf32 = False
        xn, yn = noise[:parity_batch].clone(), label[:parity_batch].clone()
        with torch.inference_mode():
            ref_imgs = rdiff.p_sample(model, tuple(xn.shape), noise=xn, label=yn, device=device, use_ddim=True)
        ours = diff.p_sample(net, tuple(xn.shape), noise=xn.cpu(), label=yn.cpu(), device=device, use_ddim=True)
        out["parity_full_100_steps"] = {"images": parity_batch, "reference": "strict fp32 eager on this GPU",
                                        "max_abs": (ours - ref_imgs).abs().max().item(),
                                        "mean_abs": (ours - ref_imgs).abs().mean().item()}
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
        del model
        torch.cuda.empty_cache()
    return out


def train_step_child(batch=128, steps=2, device=None):
    """BASELINE configs[4], run in a child process of the N=1 bench (never inside its timed region): one training step of the
    CIFAR-10 conditional v-objective network (cifar10_cond.json: drop_rate 0.2, snr_trunc re-weighting, p_uncond 0.1, AdamW
    2e-4 / wd 1e-3, clip 1.0, EMA) on a synthetic batch of 128 images on one GPU -- through v_diffusion_b200.training.
    TrainingStep (UNet forward + backward composed from this library's kernels, DESIGN.md section 7: a parity-green
    composition, NOT tuned -- the kernel-level hooks allocate, pack weights and synchronise per call) and, beside it, the
    unmodified reference (oracle/_ref) doing the same step under autograd in stock PyTorch eager on the same GPU.
    Prints one line: TRAIN_STEP {json}."""
    import torch
    from v_diffusion_b200 import _lib
    from v_diffusion_b200.training import TrainingStep
    if device is None:
        device = torch.device("cuda", 0)
        torch.cuda.set_device(device)
    net, diff = build_model(device, seed=0)
    sd0 = {k: v.detach().clone() for k, v in net.state_dict().items()}
    lr, wd, gn, decay = 2e-4, 0.001, 1.0, 0.9999                        # cifar10_cond.json "train"
    g = torch.Generator().manual_seed(4321)
    x = (torch.rand(batch, 3, 32, 32, generator=g) * 2 - 1).to(device)      # SURVEY 8(d) cfg 5: x0 ~ U[-1, 1], t ~ U[0, 1) fp64
    y = (torch.randint(10, (batch,), generator=g) + 1).to(device)
    gf_per_sample = 112.92                                                # fwd + bwd of the cifar10_cond UNet (SURVEY 8(d))
    peak = read_peaks()["tflops"]

    def rate(ms):
        tf = gf_per_sample * batch / (ms * 1e-3) / 1e3
        return {"ms_per_step": ms, "images_per_s": batch / (ms * 1e-3), "unet_tflops": tf, "frac_of_sustained_bf16_peak": tf / peak}
    out = {"workload": "BASELINE configs[4]: cifar10_cond.json training step (v objective, continuous time, snr_trunc, "
                       f"p_uncond 0.1, drop_rate 0.2, clip 1.0 + AdamW + EMA), synthetic batch {batch} on one GPU",
           "batch": batch, "steps_timed": steps, "unit": "images/s"}

    def timed(fn, warm):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps, float(last)

    try:
        net.train()
        ts = TrainingStep(net, diff, timesteps=0, lr=lr, weight_decay=wd, grad_norm=gn, use_ema=True, ema_decay=decay)
        n0 = _lib.lib().vdt_kernel_launches()
        ms, loss = timed(lambda: ts.step(x, y.clone()), 1)
        launches = (_lib.lib().vdt_kernel_launches() - n0) // (steps + 1)
        out["this_path"] = {**rate(ms), "loss_last_step": loss,
                            "kernels_per_step": int(launches), "operands": net.operand_dtype,
                            "state": "parity-green composition over per-call kernel hooks, untuned (DESIGN.md section 7)"}
        del ts
    except Exception as e:                                              # noqa: BLE001 -- report, never break the bench line
        out["this_path"] = {"error": repr(e)[:400]}
    torch.cuda.empty_cache()
    try:
        if not reference_staged():
            out["reference_gpu_eager"] = {"unavailable": "oracle/_ref not staged"}
        else:
            model, rdiff = reference_objects(sd0, device)
            model.train()
            opt = torch.optim.AdamW(model.parameters(), lr=lr, weight_decay=wd)
            params = [p for p in model.parameters()]
            shadow = [p.detach().clone() for p in params]
            count = [0]

            def ref_step():
                t = torch.rand((batch,), dtype=torch.float64, device=device)                 # Trainer.loss, T = 0
                noise = torch.randn_like(x)
                loss = rdiff.train_loss(model, x_0=x, t=t, y=y.clone(), noise=noise).mean()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(params, max_norm=gn)
                opt.step()
                opt.zero_grad(set_to_none=True)
                count[0] += 1
                d = min(decay, (1 + count[0]) / (10 + count[0]))
                with torch.no_grad():
                    torch._foreach_lerp_(shadow, [p.detach() for p in params], 1 - d)      # EMA.update, utils.py:144-149
                return loss.detach()
            ref = {"note": "unmodified reference (oracle/_ref): train_loss + autograd + clip_grad_norm_ + AdamW + EMA, torch eager"}
            saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
            try:
                for mode, tf32 in (("stock_flags_tf32_convs", True), ("strict_fp32", False)):
                    torch.backends.cudnn.allow_tf32 = tf32
                    ms, loss = timed(ref_step, 1 if mode == "strict_fp32" else 2)
                    ref[mode] = {**rate(ms), "loss_last_step": loss}
            finally:
                torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
            out["reference_gpu_eager"] = ref
    except Exception as e:                                              # noqa: BLE001
        out["reference_gpu_eager"] = {"error": repr(e)[:400]}
    print("TRAIN_STEP " + json.dumps(out), flush=True)


def train_step_block(timeout_s=120):
    """Runs train_step_child in its own process (a fault there cannot touch this process's CUDA context or its bench line)."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--train-step-child"], capture_output=True, text=True,
                           timeout=timeout_s, cwd=ROOT)
        for ln in r.stdout.splitlines():
            if ln.startswith("TRAIN_STEP "):
                return json.loads(ln[len("TRAIN_STEP "):])
        return {"error": f"child rc={r.returncode}: " + (r.stderr or r.stdout)[-400:]}
    except Exception as e:                                              # noqa: BLE001
        return {"error": repr(e)[:400]}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, x):
    """--dump-outputs: the images the timed path left in x after its last step (what a caller of it receives), written
    as out_dir/samples.npy in float32 so that two builds can be compared on the same seeded inputs.  A batch above
    DUMP_MAX_BYTES is cut to a fixed, seeded subset of its images, kept in batch order."""
    import numpy as np
    import torch
    x = x.detach().float().cpu()
    per_image = x[0].numel() * 4
    if x.shape[0] * per_image > DUMP_MAX_BYTES:
        keep = torch.randperm(x.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_MAX_BYTES // per_image]
        x = x[keep.sort().values]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "samples.npy"), x.numpy())


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path on the host cores -- the unmodified
    reference staged under oracle/_ref (kind "reference"); the oracle port (kind "port") only if it is absent --
    same metric / config, each step a bounded sample (B = 2 images = 4 UNet rows) of the workload."""
    if rank != 0:
        return
    import torch
    torch.set_num_threads(os.cpu_count())
    net, _ = build_model("cpu", seed=0)
    B = 2
    g = torch.Generator().manual_seed(1234)
    x_t = torch.randn(B, 3, 32, 32, generator=g)
    label = torch.randint(10, (B,), generator=g) + 1
    kind, x_last, dt, n = cpu_reference_trajectory(net.state_dict(), x_t, label, args.warmup, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x_last)
    val = B / (dt * T_STEPS)
    line = {"metric": METRIC, "value": val, "unit": "images/s", "n_gpus": args.gpus, "steps": n,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "CIFAR-10 cond UNet (cifar10_cond.json), CFG w=1 as 2B rows, 100-step DDIM; "
                                   f"bounded sample B={B} images per step on the host CPU"},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": torch.get_num_threads(), "kind": kind,
                             "sample": f"B={B} images (4 UNet rows) per denoising step, {n} steps of the "
                                       + ("unmodified reference's p_sample_step (oracle/_ref)" if kind == "reference" else "oracle port")},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_b200(args, rank, world, local_rank):
    import ctypes as C
    import torch
    import torch.distributed as dist
    from v_diffusion_b200 import _lib

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        # keep stdout to the single JSON line: NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION/WARN,
        # so the communicator is brought up (init + first collective) with fd 1 pointed at stderr
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier(device_ids=[local_rank])
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    L = _lib.lib()
    wl = WORKLOADS[args.workload]
    res = 32 if wl is None else wl[3]
    use_cfg = wl is None or bool(wl[6])
    T, w_guide, use_ddim, in_ch = workload_params(args.workload)
    B, K, W = (args.batch if args.batch > 0 else (4096 if wl is None else wl[7])), args.steps, max(args.warmup, 3)
    net, diff = build_model(device, seed=0, workload=args.workload)
    net.max_rows = args.max_rows
    plan = net.plan_for(res, device)
    sc = diff.sampler_config(use_ddim=use_ddim, seed=1234 + rank)
    g = torch.Generator(device=device).manual_seed(1234 + rank)      # SURVEY §8d cfg 2: per-rank seeds 1234+rank
    noise = torch.randn(B, in_ch, res, res, device=device, generator=g)
    label = (torch.randint(10, (B,), device=device, generator=g) + 1) if use_cfg else None
    stream = torch.cuda.current_stream()

    def run_range(x, first, n):
        _lib.check(L.vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(label), None, B, first, n, None,
                                        C.c_void_p(stream.cuda_stream)))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    x = noise.clone()
    run_range(x, T - 1, W)                                      # warm-up (eager pass + graph capture)
    barrier()
    x = noise.clone()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = L.vdt_kernel_launches()
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record(stream)
        done, first = 0, T - 1
        while done < K:                                               # K may exceed one trajectory
            n = min(K - done, first + 1)
            run_range(x, first, n)
            done += n
            first = T - 1 if first - n < 0 else first - n
        ev1.record(stream)
        barrier()
    launches = L.vdt_kernel_launches() - n0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x)
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=device, dtype=torch.float64)
    per_rank = None
    if world > 1:
        # every rank's own device time and median SM clock, so that the spread behind the max is visible
        mine = torch.tensor([ms.item() / K, float(clocks.summary().get("sm_mhz") or 0.0)], device=device, dtype=torch.float64)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"ms_per_step": [round(t[0].item(), 3) for t in allr], "sm_mhz": [t[1].item() for t in allr]}
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = ms.item()
    ms_step = ms_total / K
    value = world * B / (ms_step * 1e-3 * T)

    # ---- per-kernel-family timing of the same step (CUDA events around every launch, on the launching stream)
    L.vdt_profile_enable(1)
    xs = noise.clone()
    run_range(xs, T - 1, 1)
    torch.cuda.synchronize()
    fam_ms, fam_n = (C.c_double * 4)(), (C.c_uint64 * 4)()
    L.vdt_profile_read(fam_ms, fam_n)
    L.vdt_profile_enable(0)
    fc, fa, fl = C.c_double(), C.c_double(), C.c_double()
    L.vdt_plan_flops(plan, C.byref(fc), C.byref(fa), C.byref(fl))
    rows = (2 if use_cfg else 1) * B
    flop_per_row = fc.value + fa.value + fl.value
    fexec = C.c_double()
    L.vdt_plan_conv_flops_executed(plan, 1 if use_cfg else 0, C.byref(fexec))
    conv_tflops = fc.value * rows / (fam_ms[0] * 1e-3) / 1e12 if fam_ms[0] > 0 else 0.0
    peaks = read_peaks()
    prof_total = sum(fam_ms)
    # DRAM bytes per conv launch: cannot be measured outside a profiler, so it comes from the committed ncu capture of
    # this same step (scripts/gpu_profile_round.sh + summarize_profiles.py write it with the commit it was taken on)
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_conv_dram_traffic.json")) as f:
            tr = json.load(f)
        if wl is None:
            traffic = tr["avg_dram_bytes_per_conv_launch_scaled_to_rows"] * min(rows, args.max_rows) / tr["rows"]
            traffic_src = f"profiles/r2_conv_dram_traffic.json (ncu capture at commit {tr.get('git_head')}, {tr.get('summarised_utc')})"
    except Exception:
        traffic = None
    roofline = {"bound": "tensor", "kernel": "conv_gemm_kernel (tcgen05 implicit GEMM, all conv/1x1 launches of a step)",
                "achieved": conv_tflops, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": conv_tflops / peaks["tflops"],
                "peak_source": peaks["source"] + " sustained bf16 cuBLAS", "traffic": traffic,
                "traffic_source": traffic_src,
                "traffic_note": "avg dram__bytes_read+write per conv launch (ncu, one chunk of chunk_rows UNet rows); "
                                "launches_per_step counts every chunk's launches",
                "algorithmic_flop_per_launch_avg": fc.value * rows / max(1, fam_n[0]),
                "executed_over_algorithmic_conv_flops": fexec.value / fc.value,
                "executed_note": "achieved / frac count the reference graph's FLOPs; the kernels execute fewer (sub-pixel "
                                 "upsampling convs, the CFG pair's shared label-independent prefix) -- multiply by this ratio for the tensor-pipe rate",
                "avg_launch_ms": fam_ms[0] / max(1, fam_n[0]), "launches_per_step": int(fam_n[0]),
                "step_share": {"conv": fam_ms[0] / prof_total, "groupnorm": fam_ms[1] / prof_total,
                               "attention": fam_ms[2] / prof_total, "other": fam_ms[3] / prof_total},
                "family_ms_per_step": {"conv": fam_ms[0], "groupnorm": fam_ms[1], "attention": fam_ms[2], "other": fam_ms[3]},
                "unet_tflops_whole_step": flop_per_row * rows / (ms_step * 1e-3) / 1e12,
                "unet_frac_of_peak_whole_step": flop_per_row * rows / (ms_step * 1e-3) / 1e12 / peaks["tflops"],
                "unet_frac_of_nominal_2250": flop_per_row * rows / (ms_step * 1e-3) / 1e12 / 2250.0}

    # ---- end to end through the public API: host noise/labels in (pinned), CPU images out, all 100 steps
    noise_h = noise.cpu().pin_memory()
    label_h = label.cpu().pin_memory() if label is not None else None
    barrier()
    t0 = time.perf_counter()
    imgs = diff.p_sample(net, (B, in_ch, res, res), noise=noise_h, label=label_h, device=device, seed=1234 + rank,
                         use_ddim=use_ddim)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        gathered = [torch.empty_like(noise) for _ in range(world)]   # the only collective: final image gather
        dist.all_gather(gathered, imgs.to(device))
    assert torch.isfinite(imgs).all()
    # outside every timed region: three images of the full-size run recomputed on their own (size-independent
    # property: a sample's trajectory does not depend on its batch or chunk; expected difference 0)
    pick = torch.tensor([0, B // 2, B - 1])
    if use_ddim:
        alone = diff.p_sample(net, (3, in_ch, res, res), noise=noise_h[pick], label=None if label_h is None else label_h[pick],
                              device=device, use_ddim=True)
        selfcheck = (alone - imgs[pick]).abs().max().item()
    else:
        selfcheck = None      # on-device ancestral noise is indexed by batch position: a sub-batch draws other noise
    e2e = {"value": world * B / e2e_s.item(), "unit": "images/s",
           "h2d_bytes_per_step": (noise_h.numel() * 4 + (label_h.numel() * 8 if label_h is not None else 0)) / T,
           "d2h_bytes_per_step": imgs.numel() * 4 / T,
           "note": f"one GaussianDiffusion.p_sample call = {T} denoising steps; bytes are per call / {T}",
           "seconds_per_call": e2e_s.item(), "selfcheck_max_abs_3_images_recomputed_alone": selfcheck}

    if rank == 0:
        metric = METRIC if wl is None else (f"ddim_images_per_sec_{args.workload}_100step" if use_ddim else
                                             f"ancestral_images_per_sec_{args.workload}_{T}step")
        wtext = ("CIFAR-10 class-conditional UNet (cifar10_cond.json), CFG w=1 batched cond/uncond (2B rows), 100-step DDIM"
                 if wl is None else wl[8])
        line = {"metric": metric, "value": value, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": net.operand_dtype, "data": "synthetic",
                "config": {"workload": f"{wtext}, batch {B} per GPU; step = one denoising step over the batch",
                           "batch_per_gpu": B, "rows_per_unet_call": rows, "chunk_rows": args.max_rows,
                           "steps_per_image": T, "l2": "inputs_exceed_l2", "parallelism": f"replicas x{world}",
                           "operands": net.operand_dtype + " tensor-core operands (same tcgen05 kind::f16 rate as bf16)",
                           "accumulate": "fp32", "residual_stream": "fp32"},
                "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline}
        if per_rank is not None:
            line["per_rank"] = per_rank
        if world == 1 and not args.no_cpu_baseline and wl is None:
            line["cpu_baseline"] = cpu_baseline(net, diff, noise_h[:2].clone(), label_h[:2].clone(), device)
            line["reference_gpu_eager"] = reference_gpu_eager(net, diff, noise, label, device)
            eager = line["reference_gpu_eager"].get("stock_flags_tf32_convs")
            if eager:
                line["reference_gpu_eager"]["speedup_e2e_over_stock_eager"] = e2e["value"] / eager["images_per_s"]
            if not args.no_train_step:
                line["train_step"] = train_step_block()      # BASELINE configs[4], outside every timed region, own process
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: 4096 for cifar10_cond, BASELINE configs[1])")
    ap.add_argument("--workload", default="cifar10_cond", choices=sorted(WORKLOADS))
    ap.add_argument("--max-rows", type=int, default=int(os.environ.get("VDT_MAX_ROWS", "1024")))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train-step", action="store_true", help="skip the BASELINE configs[4] training-step block of the N=1 line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the images of the last timed step (rank 0) to DIR/samples.npy, float32, at most 64 MB")
    ap.add_argument("--train-step-child", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.train_step_child:
        train_step_child()
        return
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run on this node
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        os.execv(sys.executable, cmd)
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
