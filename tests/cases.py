"""Shared definitions of the seeded parity cases.

Used by ``tests/golden/make_golden.py`` (which runs the unmodified reference on them in
the build container) and by the CPU / GPU tests (which run the oracle and the CUDA path
on the very same inputs).  Everything is regenerated from integer seeds with CPU
generators, so only outputs need to be stored under ``tests/golden/``.
"""
import zlib

import numpy as np
import torch


def golden_sample_index(numel, n, key):
    """Sorted flat positions of a fixed sample of n of an output's numel entries, seeded by ``key``: what a fixture keeps of
    an output too large to store in full."""
    g = torch.Generator().manual_seed(zlib.crc32(key.encode()) & 0x7fffffff)
    return torch.randperm(numel, generator=g)[:n].sort().values.numpy().astype(np.int32)


def _cfg(in_channels=3, hid=64, out_channels=3, mult=(1, 2), nrb=2, attn=(False, True),
         embedding_dim=None, head_dim=None, num_heads=1, num_classes=0, multitags=False):
    if head_dim is None and num_heads is None:
        num_heads = 1
    return dict(in_channels=in_channels, hid_channels=hid, out_channels=out_channels,
                ch_multipliers=list(mult), num_res_blocks=nrb, apply_attn=list(attn),
                embedding_dim=embedding_dim or 4 * hid, head_dim=head_dim, num_heads=num_heads,
                num_classes=num_classes, multitags=multitags)


# cifar10_{cond,uncond}.json + defaults.json -> UNet ctor integers (checked against
# tests/golden/merged_configs.json by test_config_merge)
CIFAR_COND = _cfg(hid=256, mult=(1, 1, 1), nrb=3, attn=(False, True, True), num_heads=1, num_classes=10)
CIFAR_UNCOND = _cfg(hid=256, mult=(1, 1, 1), nrb=3, attn=(False, True, True), num_heads=1, num_classes=0)
CELEBA = _cfg(hid=192, out_channels=6, mult=(1, 2, 3, 4), nrb=3, attn=(False, True, True, True),
              embedding_dim=768, head_dim=64, num_heads=1, num_classes=0)

UNET_CASES = {
    # small: two levels, concat widths 192/256/128 (6-channel groups straddling the concat seam)
    # trace_keep: the fixture stores each traced feature map at that many seeded positions (golden_sample_index)
    "small_cond": dict(cfg=_cfg(num_classes=10), seed=11, B=3, res=16, labels=[0, 3, 10], trace_keep=4096,
                       trace=["in_conv", "downsamples.level_0.0", "downsamples.level_0.2",
                              "downsamples.level_1.0", "middle", "upsamples.level_1.0",
                              "upsamples.level_1.3", "upsamples.level_0.2"]),
    # three levels with an attention-bearing resample block (N = 1024 / 256 / 64 tokens), head_dim 64
    "small_hd64": dict(cfg=_cfg(out_channels=6, mult=(1, 1, 2), nrb=1, attn=(False, True, True),
                                embedding_dim=192, head_dim=64, num_heads=1),
                       seed=12, B=2, res=32, labels=None, trace=[]),
    # the real CIFAR-10 conditional network (BASELINE configs[1]) at batch 2
    "cifar_cond": dict(cfg=CIFAR_COND, seed=13, B=2, res=32, labels=[7, 0], trace=["middle"]),
}

SAMPLE_CASES = {
    # BASELINE configs[1] in miniature: v-prediction, CFG w=1, DDIM
    "ddim_cfg_v": dict(unet="small_cond", seed=21, B=4, res=16, T=8, model_out_type="v", w_guide=1.0,
                       use_ddim=True, var_type="fixed_medium", intp_frac=0.3, labels=[1, 5, 10, 2]),
    # BASELINE configs[0] in miniature: x0-prediction, unconditional, DDIM
    "ddim_x0_uncond": dict(unet="small_hd64_x0", seed=22, B=3, res=32, T=6, model_out_type="x0",
                           w_guide=0.0, use_ddim=True, var_type="fixed_large", labels=None),
    # BASELINE configs[3] in miniature: ancestral, CFG w=3, injected per-step noise.  64 steps: a w=3 ancestral
    # trajectory of 10 coarse steps on a random-weight network is chaotic (round 1: unrelated kernel changes moved its
    # final-sample error between 1.9e-2 and 3.0e-2 while every per-step error stayed put), so it pinned nothing
    "ancestral_cfg_v": dict(unet="small_cond", seed=23, B=2, res=16, T=64, model_out_type="v", w_guide=3.0,
                            use_ddim=False, var_type="fixed_medium", intp_frac=0.3, labels=[4, 9]),
    # x0eps_coef=True (diffusion.py:137-140, 335-343): posterior mean written in (eps, x0), eps re-derived from the
    # clipped x0.  (v-prediction: an eps-prediction network at logsnr_min = -20 amplifies any rounding by e^10 before
    # the clip -- the reference under its own TF32 numerics moves by 0.5 on such a fixture.)
    "ancestral_x0eps": dict(unet="small_cond", seed=25, B=2, res=16, T=6, model_out_type="v", w_guide=0.5,
                            use_ddim=False, var_type="fixed_small", labels=[3, 8], x0eps_coef=True),
    # same under DDIM: the reference hands back LOG coefficients there (diffusion.py:180-182) -- reproduced as is
    "ddim_x0eps": dict(unet="small_cond", seed=26, B=2, res=16, T=5, model_out_type="v", w_guide=0.0,
                       use_ddim=True, var_type="fixed_small", labels=[1, 6], x0eps_coef=True),
    # CelebA-style "both" output (2C channels), ancestral fixed_large
    "ancestral_both": dict(unet="small_hd64", seed=24, B=2, res=32, T=5, model_out_type="both", w_guide=0.0,
                           use_ddim=False, var_type="fixed_large", labels=None),
}
# BASELINE configs[3] geometry: 1-channel 28x28 conditional UNet, 28 -> 14 -> 7, attention at 14x14 and 7x7 (N = 196 / 49)
# and in the attention-bearing upsampling block at 28x28 (N = 784)
UNET_CASES["mnist28"] = dict(cfg=_cfg(in_channels=1, out_channels=1, mult=(1, 2, 2), nrb=1, attn=(False, True, True),
                                      num_classes=10), seed=16, B=3, res=28, labels=[2, 0, 9], trace=[])
SAMPLE_CASES["ancestral_mnist28"] = dict(unet="mnist28", seed=27, B=2, res=28, T=64, model_out_type="v", w_guide=3.0,
                                         use_ddim=False, var_type="fixed_medium", intp_frac=0.3, labels=[5, 10])
# multitag (multi-hot) class conditioning as used by the reference's conditional CelebA checkpoints
UNET_CASES["small_multitag"] = dict(cfg=_cfg(mult=(1, 2), nrb=1, attn=(False, True), num_classes=40, multitags=True),
                                    seed=15, B=3, res=16, labels="multihot", trace=[])
SAMPLE_CASES["ddim_cfg_multitag"] = dict(unet="small_multitag", seed=25, B=3, res=16, T=6, model_out_type="v", w_guide=1.0,
                                         use_ddim=True, var_type="fixed_large", labels="multihot")
UNET_CASES["small_hd64_x0"] = dict(cfg=_cfg(out_channels=3, mult=(1, 1, 2), nrb=1, attn=(False, True, True),
                                            embedding_dim=192, head_dim=64, num_heads=1),
                                   seed=14, B=2, res=32, labels=None, trace=[])


def build_inputs(case):
    """x fp32 NCHW, t fp64 in (0,1], y int64 | None — seeded, CPU."""
    g = torch.Generator().manual_seed(case["seed"] + 1000)
    cfg = case["cfg"]
    x = torch.randn(case["B"], cfg["in_channels"], case["res"], case["res"], generator=g)
    t = torch.rand(case["B"], generator=g, dtype=torch.float64) * 0.98 + 0.01
    y = _labels(case, cfg, g)
    return x, t, y


def _labels(case, cfg, g):
    if case["labels"] is None:
        return None
    if case["labels"] == "multihot":        # ~5 of 40 attributes set per image; first row all zero (clamp(min=1) path)
        y = (torch.rand(case["B"], cfg["num_classes"], generator=g) < 0.12).float()
        y[0] = 0
        return y
    return torch.tensor(case["labels"], dtype=torch.int64)


def build_sample_inputs(case, cfg):
    """initial noise, labels, and the per-step draws the reference would take from
    ``torch.Generator('cpu').manual_seed(seed)``: one ``empty(shape).normal_()`` per step in loop
    order ti = T-1 .. 0 (diffusion.py:389, 410), stored at index ti."""
    g0 = torch.Generator().manual_seed(case["seed"] + 2000)
    shape = (case["B"], cfg["in_channels"], case["res"], case["res"])
    noise = torch.randn(shape, generator=g0)
    label = _labels(case, cfg, g0)
    g = torch.Generator().manual_seed(case["seed"])
    step_noise = torch.empty((case["T"],) + shape)
    for ti in reversed(range(case["T"])):
        step_noise[ti] = torch.empty(shape).normal_(generator=g)
    return noise, label, step_noise


# ---------------------------------------------------------------------------------------------------------------
# Full-length trajectories of the real CIFAR-10 networks (BASELINE configs[0] and configs[1]), SURVEY §8d recipe:
# the network is the reference's own random initialisation under torch.manual_seed(init_seed) -- this package's UNet
# constructor consumes the RNG exactly like the reference's (checked bit for bit in make_golden.py), so the GPU box can
# rebuild the weights without the reference -- with every all-zero matrix "de-zeroed" (oracle.dezero_, generator seed 7).
FULL_CASES = {
    # configs[0]: cifar10_uncond.json, x0-prediction, fixed_large, 10-step DDIM, batch 16
    "cifar10_uncond_ddim10": dict(cfg=CIFAR_UNCOND, init_seed=0, dezero_seed=7, B=16, T=10, model_out_type="x0",
                                  var_type="fixed_large", intp_frac=None, w_guide=0.0, use_ddim=True, noise_seed=1234,
                                  labelled=False, keep_rows=16, keep_entries=4096),
    # (per-step model outputs: the first keep_rows rows, stored at keep_entries seeded positions of a step, golden_sample_index)
    # configs[1] at B=8: cifar10_cond.json, v-prediction, CFG w=1 (16 UNet rows per step), 100-step DDIM
    "cifar10_cond_cfg_ddim100": dict(cfg=CIFAR_COND, init_seed=0, dezero_seed=7, B=8, T=100, model_out_type="v",
                                     var_type="fixed_medium", intp_frac=0.3, w_guide=1.0, use_ddim=True, noise_seed=1234,
                                     labelled=True, keep_rows=4, keep_entries=1024),
}


def build_full_inputs(case):
    """noise = randn(B, 3, 32, 32) from Generator().manual_seed(noise_seed); labels = randint(10) + 1 from the same
    generator afterwards (generate.py:134)."""
    g = torch.Generator().manual_seed(case["noise_seed"])
    noise = torch.randn(case["B"], 3, 32, 32, generator=g)
    label = (torch.randint(10, (case["B"],), generator=g) + 1) if case["labelled"] else None
    return noise, label


def full_state_dict(case, unet_cls):
    """State dict of ``unet_cls`` (the reference's UNet or this package's) initialised under manual_seed(init_seed)
    and de-zeroed.  Restores the global RNG state afterwards."""
    from oracle.unet_ref import dezero_
    cfg = case["cfg"]
    state = torch.get_rng_state()
    try:
        torch.manual_seed(case["init_seed"])
        net = unet_cls(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"],
                       cfg["num_res_blocks"], cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], drop_rate=0.2,
                       head_dim=cfg["head_dim"], num_heads=cfg["num_heads"], num_classes=cfg["num_classes"],
                       multitags=cfg["multitags"])
    finally:
        torch.set_rng_state(state)
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    return dezero_(sd, case["dezero_seed"]), net


# ---------------------------------------------------------------------------------------------------------------
# GaussianDiffusion.train_loss (diffusion.py:492-545; BASELINE configs[4]): x_0 ~ U[-1, 1], t ~ U[0, 1) fp64, eps ~ N(0, 1),
# labels 1..10.  The fixtures hold what the reference computes around the model call: x_t, the per-sample loss and the
# autograd gradient of loss.mean() with respect to the model output.
TRAIN_CASES = {
    # the config[4] objective: v-prediction, truncated-SNR reweighting (max of the x0 and eps errors)
    "v_snr_trunc": dict(unet="small_cond", seed=41, B=4, res=16, model_out_type="v", reweight_type="snr_trunc"),
    "eps_snr_trunc": dict(unet="small_cond", seed=42, B=3, res=16, model_out_type="eps", reweight_type="snr_trunc"),
    "x0_snr_trunc": dict(unet="small_cond", seed=43, B=3, res=16, model_out_type="x0", reweight_type="snr_trunc"),
    "both_snr_trunc": dict(unet="small_hd64", seed=44, B=2, res=32, model_out_type="both", reweight_type="snr_trunc"),
    # single-target reweightings compare the target with the RAW model output (diffusion.py:541), reproduced as is
    "x0_constant": dict(unet="small_cond", seed=45, B=3, res=16, model_out_type="x0", reweight_type="constant"),
    "eps_snr": dict(unet="small_cond", seed=46, B=3, res=16, model_out_type="eps", reweight_type="snr"),
    "v_snr_1plus": dict(unet="small_cond", seed=47, B=3, res=16, model_out_type="v", reweight_type="snr_1plus"),
}


def build_train_inputs(case, cfg):
    g = torch.Generator().manual_seed(case["seed"] + 3000)
    shape = (case["B"], cfg["in_channels"], case["res"], case["res"])
    x0 = torch.rand(shape, generator=g) * 2 - 1
    t = torch.rand(case["B"], generator=g, dtype=torch.float64)
    noise = torch.randn(shape, generator=g)
    y = (torch.randint(10, (case["B"],), generator=g) + 1) if cfg["num_classes"] else None
    return x0, t, noise, y


# ---- gradients of the training step, from the unmodified reference's autograd (tests/golden/make_train_grad_golden.py) ----
# every block type of the CIFAR network at a quarter of the width: 128 / 256-channel norms, 1x1 skips, an avg-pool and a
# nearest-upsample block, attention at 8x8 and (after the upsample) 16x16, class-conditional; objective of configs[4]
TRAIN_GRAD_CASE = dict(cfg=_cfg(hid=128, mult=(1, 1), nrb=1, attn=(False, True), num_classes=10), wseed=51, seed=52, B=4, res=16,
                       model_out_type="v", reweight_type="snr_trunc")


# BASELINE configs[4]'s own network (cifar10_cond.json) at batch 4, 32x32
TRAIN_GRAD_CASE_CIFAR = dict(cfg=CIFAR_COND, wseed=53, seed=54, B=4, res=32, model_out_type="v", reweight_type="snr_trunc")
TRAIN_GRAD_CASES = {"small": TRAIN_GRAD_CASE, "cifar": TRAIN_GRAD_CASE_CIFAR}


def build_train_grad_inputs(case=TRAIN_GRAD_CASE):
    cfg = case["cfg"]
    g = torch.Generator().manual_seed(case["seed"])
    shape = (case["B"], cfg["in_channels"], case["res"], case["res"])
    x0 = torch.rand(shape, generator=g) * 2 - 1
    t = torch.rand(case["B"], generator=g, dtype=torch.float64)
    noise = torch.randn(shape, generator=g)
    y = torch.randint(10, (case["B"],), generator=g) + 1
    y[1] = 0                                                    # one unconditional row
    return x0, t, noise, y


def grad_probe(name, shape):
    """Seeded N(0, 1) direction a gradient tensor is projected on (fixtures store |g| and <g, probe> per tensor)."""
    import zlib
    g = torch.Generator().manual_seed(zlib.crc32(name.encode()) & 0x7fffffff)
    return torch.randn(shape, generator=g, dtype=torch.float64)
