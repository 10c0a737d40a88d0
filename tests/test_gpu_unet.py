"""GPU parity of the whole path through the reference-shaped API: UNet.forward and
GaussianDiffusion.p_sample against (a) golden outputs of the unmodified reference and (b) the oracle run on
this box's CPU.  Tolerances are the north-star's production bars: per-step model output rel-L2 <= 1e-2,
final samples max-abs <= 2e-2 (default operand format: fp16 operands, fp32 accumulate / norm / softmax /
residual stream).  The bf16 operand format is measured next to it as calibration (looser bound)."""
import json
import os

import numpy as np
import pytest
import torch

from tests.cases import (UNET_CASES, SAMPLE_CASES, FULL_CASES, TRAIN_CASES, build_inputs, build_sample_inputs,
                         build_full_inputs, full_state_dict, build_train_inputs)
from tests.cases import _cfg as _cfg_case

pytestmark = pytest.mark.gpu
REL_L2 = 1e-2
SAMPLE_MAX_ABS = 2e-2
VALIDATION_MAX_ABS = 1e-3        # north-star: TF32/fp32 validation mode


def _model(cfg, seed, operand="fp16"):
    from oracle.unet_ref import make_state_dict
    from v_diffusion_b200 import UNet
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"],
               cfg["num_res_blocks"], cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], head_dim=cfg["head_dim"],
               num_heads=cfg["num_heads"], num_classes=cfg["num_classes"], multitags=cfg["multitags"])
    net.load_state_dict(make_state_dict(cfg, seed), strict=True)
    net.operand_dtype = operand
    return net.cuda().eval()


def _diffusion(case):
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), case["T"], case["model_out_type"],
                             case["var_type"], "snr_trunc", "mse", intp_frac=case.get("intp_frac"),
                             w_guide=case["w_guide"], x0eps_coef=case.get("x0eps_coef", False))


@pytest.mark.parametrize("name", sorted(UNET_CASES))
def test_unet_forward_vs_reference_golden(golden_dir, name):
    case = UNET_CASES[name]
    ref = torch.from_numpy(np.load(os.path.join(golden_dir, f"unet_{name}.npz"))["out"])
    net = _model(case["cfg"], case["seed"])
    x, t, y = build_inputs(case)
    out = net(x.cuda(), t.cuda(), None if y is None else y.cuda()).cpu()
    assert out.shape == ref.shape and torch.isfinite(out).all()
    rel = ((out - ref).norm() / ref.norm()).item()
    print(f"{name}: rel-L2 {rel:.3e} max-abs {(out - ref).abs().max().item():.3e}")
    assert rel <= REL_L2
    # second call replays the captured CUDA graph; third with a different batch builds a new exec
    out2 = net(x.cuda(), t.cuda(), None if y is None else y.cuda()).cpu()
    assert torch.equal(out, out2)
    out3 = net(x[:1].cuda(), t[:1].cuda(), None if y is None else y[:1].cuda()).cpu()
    assert ((out3 - ref[:1]).norm() / ref[:1].norm()).item() <= REL_L2


def test_unet_forward_vs_oracle_on_this_box():
    from oracle import unet_forward, make_state_dict
    case = UNET_CASES["small_cond"]
    cfg = case["cfg"]
    g = torch.Generator().manual_seed(99)
    B = 5                                     # odd batch, chunked by max_rows = 2 -> 2 + 2 + 1
    x = torch.randn(B, 3, 16, 16, generator=g)
    t = torch.rand(B, generator=g, dtype=torch.float64)
    y = torch.tensor([0, 1, 2, 9, 10])
    net = _model(cfg, 5)
    net.max_rows = 2
    out = net(x.cuda(), t.cuda(), y.cuda()).cpu()
    ref = unet_forward(make_state_dict(cfg, 5), cfg, x, t, y)
    assert ((out - ref).norm() / ref.norm()).item() <= REL_L2
    # y=None on a conditional model skips the class embedding entirely (unet.py:289)
    out_n = net(x.cuda(), t.cuda(), None).cpu()
    ref_n = unet_forward(make_state_dict(cfg, 5), cfg, x, t, None)
    assert ((out_n - ref_n).norm() / ref_n.norm()).item() <= REL_L2


def test_three_level_network_down_to_4x4_vs_oracle():
    """Three levels from 16x16 bottom out at 4x4 with attention over N = 64 and N = 16 tokens: 16 pixels per image is
    less than one 32-row statistics slab (two-pass GroupNorm there), eight images share one GEMM tile, and the
    attention key tile is ragged (16 of 64 keys).  Odd batch -> ragged GEMM tiles at every level."""
    from oracle import unet_forward, make_state_dict
    cfg = _cfg_case(mult=(1, 2, 2), nrb=1, attn=(False, True, True), num_classes=5)
    g = torch.Generator().manual_seed(123)
    B = 3
    x = torch.randn(B, 3, 16, 16, generator=g)
    t = torch.rand(B, generator=g, dtype=torch.float64)
    y = torch.tensor([0, 2, 5])
    net = _model(cfg, 31)
    out = net(x.cuda(), t.cuda(), y.cuda()).cpu()
    ref = unet_forward(make_state_dict(cfg, 31), cfg, x, t, y)
    rel = ((out - ref).norm() / ref.norm()).item()
    print(f"16 -> 8 -> 4 network: rel-L2 {rel:.3e}")
    assert rel <= REL_L2
    out1 = net(x[1:2].cuda(), t[1:2].cuda(), y[1:2].cuda()).cpu()      # a single image: M = 16 rows at the lowest level
    assert (out1 - out[1:2]).abs().max().item() <= 1e-5
    with pytest.raises(RuntimeError, match="feature-map size 2"):       # 8 -> 4 -> 2 is refused, loudly
        net(x[:, :, :8, :8].contiguous().cuda(), t.cuda(), y.cuda())


@pytest.mark.parametrize("name", sorted(SAMPLE_CASES))
def test_p_sample_vs_reference_golden(golden_dir, name):
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    g = np.load(os.path.join(golden_dir, f"sample_{name}.npz"))
    ref, ref_mo = torch.from_numpy(g["out"]), torch.from_numpy(g["model_out"])
    net = _model(ucase["cfg"], ucase["seed"])
    diff = _diffusion(case)
    noise, label, step_noise = build_sample_inputs(case, ucase["cfg"])
    # (1) fused path: whole loop inside the library, one CUDA graph per step
    out = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=case["use_ddim"],
                        step_noise=None if case["use_ddim"] else step_noise)
    assert out.device.type == "cpu" and out.shape == ref.shape
    err = (out - ref).abs().max().item()
    # flat north-star bar on every fixture; the reference's own deviation under TF32 convolutions (its default GPU
    # numerics, tests/golden/make_tf32_dev.py) is printed next to it as calibration only
    tf32 = json.load(open(os.path.join(golden_dir, "ref_tf32_deviation.json")))[name]["max_abs"]
    bar = SAMPLE_MAX_ABS
    print(f"{name}: fused max-abs {err:.3e} (bar {bar:.1e}; the reference under TF32 convs moves by {tf32:.3e})")
    assert err <= bar
    # (2) generic-callable path with a recorder: per-step model outputs along the trajectory
    rec = []

    def wrapped(x, t, y):
        o = net(x, t, y)
        rec.append(o.cpu())
        return o
    out2 = diff.p_sample(wrapped, tuple(noise.shape), noise=noise, label=label, device="cuda",
                         use_ddim=case["use_ddim"], step_noise=None if case["use_ddim"] else step_noise)
    assert (out2 - ref).abs().max().item() <= bar
    assert len(rec) == case["T"]
    worst = max(((o - ref_mo[i]).norm() / ref_mo[i].norm()).item() for i, o in enumerate(rec))
    print(f"{name}: worst per-step rel-L2 {worst:.3e}")
    assert worst <= REL_L2
    assert (out - out2).abs().max().item() <= 1e-5      # both drivers run the same kernels


def test_p_sample_chunking_and_roundtrip_properties():
    """Size-independent properties at a batch larger than one chunk: per-sample independence (a sample's
    trajectory does not depend on its neighbours or on the chunking) and determinism."""
    case = SAMPLE_CASES["ddim_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    net = _model(ucase["cfg"], ucase["seed"])
    diff = _diffusion(case)
    g = torch.Generator().manual_seed(5)
    B = 11
    noise = torch.randn(B, 3, 16, 16, generator=g)
    label = torch.randint(0, 11, (B,), generator=g)
    net.max_rows = 64
    a = diff.p_sample(net, (B, 3, 16, 16), noise=noise, label=label, device="cuda", use_ddim=True)
    net.max_rows = 6                                       # 3 images per chunk -> 3 + 3 + 3 + 2
    b = diff.p_sample(net, (B, 3, 16, 16), noise=noise, label=label, device="cuda", use_ddim=True)
    assert (a - b).abs().max().item() <= 1e-5
    perm = torch.randperm(B, generator=g)
    c = diff.p_sample(net, (B, 3, 16, 16), noise=noise[perm], label=label[perm], device="cuda", use_ddim=True)
    assert (c - b[perm]).abs().max().item() <= 1e-5


@pytest.mark.parametrize("name", ["ddim_cfg_v", "ancestral_cfg_v", "ddim_cfg_multitag", "ancestral_mnist28"])
def test_cfg_shared_prefix_is_bit_identical(name, monkeypatch):
    """Under CFG the cond / uncond rows of a sample share in_conv, norm1 and conv1 of block 0 (computed once per sample:
    they do not depend on the label).  Same arithmetic in the same order: the samples must be bit-identical to the
    row-by-row path (VDT_NO_CFG_SHARE=1), for one chunk and for several ragged chunks.  At 28x28 the shared residual
    takes the generic epilogue with the 7-tile pair order."""
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    diff = _diffusion(case)
    noise, label, step_noise = build_sample_inputs(case, ucase["cfg"])
    outs = []
    for off in (False, True):
        if off:
            monkeypatch.setenv("VDT_NO_CFG_SHARE", "1")
        for max_rows in (64, 6):
            net = _model(ucase["cfg"], ucase["seed"])            # a fresh plan: the switch is read when an exec is built
            net.max_rows = max_rows
            outs.append(diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=case["use_ddim"],
                                      step_noise=step_noise))
    assert torch.equal(outs[0], outs[2]) and torch.equal(outs[1], outs[3])
    assert torch.isfinite(outs[0]).all()


def test_p_sample_edge_batches():
    """Edge batches of the sampler: empty (nothing launched, empty tensor back), a single image and an odd batch under CFG
    (2B rows, ragged last tile) reproduce the same images as inside a larger batch; a noise tensor of the wrong shape and
    an unknown output type raise like the reference (ValueError / NotImplementedError, diffusion.py:253-257)."""
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    case = SAMPLE_CASES["ddim_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    net = _model(ucase["cfg"], ucase["seed"])
    diff = _diffusion(case)
    g = torch.Generator().manual_seed(9)
    noise = torch.randn(5, 3, 16, 16, generator=g)
    label = torch.randint(0, 11, (5,), generator=g)
    full = diff.p_sample(net, (5, 3, 16, 16), noise=noise, label=label, device="cuda", use_ddim=True)
    empty = diff.p_sample(net, (0, 3, 16, 16), noise=noise[:0], label=label[:0], device="cuda", use_ddim=True)
    assert tuple(empty.shape) == (0, 3, 16, 16) and empty.device.type == "cpu"
    one = diff.p_sample(net, (1, 3, 16, 16), noise=noise[2:3], label=label[2:3], device="cuda", use_ddim=True)
    three = diff.p_sample(net, (3, 3, 16, 16), noise=noise[1:4], label=label[1:4], device="cuda", use_ddim=True)
    assert (one - full[2:3]).abs().max().item() <= 1e-5 and (three - full[1:4]).abs().max().item() <= 1e-5
    with pytest.raises(ValueError):
        diff.p_sample(net, (5, 3, 16, 16), noise=noise[:4], label=label, device="cuda", use_ddim=True)
    with pytest.raises(NotImplementedError):
        GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 10, "velocity", "fixed_large", "constant", "mse")
    with pytest.raises(RuntimeError):                        # no CPU fallback
        diff.p_sample(net, (1, 3, 16, 16), noise=noise[:1], label=label[:1], device="cpu", use_ddim=True)


@pytest.mark.parametrize("name", ["cifar_cond", "small_cond"])
def test_bf16_operand_mode_forward(golden_dir, name):
    """bf16 operands (the north-star's nominal format): same kernels, 8-bit mantissa.  A single UNet call stays inside
    the 1e-2 per-call bar; it is several times looser than the fp16 default."""
    case = UNET_CASES[name]
    ref = torch.from_numpy(np.load(os.path.join(golden_dir, f"unet_{name}.npz"))["out"])
    x, t, y = build_inputs(case)
    outs = {}
    for mode in ("fp16", "bf16"):
        net = _model(case["cfg"], case["seed"], operand=mode)
        out = net(x.cuda(), t.cuda(), None if y is None else y.cuda()).cpu()
        outs[mode] = ((out - ref).norm() / ref.norm()).item()
    print(f"{name}: rel-L2 fp16 {outs['fp16']:.3e} bf16 {outs['bf16']:.3e}")
    assert outs["bf16"] <= REL_L2 and outs["fp16"] <= 0.5 * outs["bf16"]


@pytest.mark.parametrize("name", sorted(SAMPLE_CASES))
def test_bf16_operand_mode_sampler_status(golden_dir, name):
    """Honest status of the north-star's "bf16 production mode": with bf16 tensor-core operands the *samples* miss
    the 2e-2 bar on most fixtures (an 8-bit mantissa on every GEMM operand of a 27-block residual network, amplified
    by guidance), which is why fp16 -- same width, same tcgen05 rate, 10-bit mantissa, saturating conversions and a
    range monitor (vdt_plan_saturations) -- is the production format.  The test records the measured numbers and holds
    bf16 only to 'finite and within 0.25'; the xfail marks the fixtures over the contract bar instead of hiding them."""
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    ref = torch.from_numpy(np.load(os.path.join(golden_dir, f"sample_{name}.npz"))["out"])
    net = _model(ucase["cfg"], ucase["seed"], operand="bf16")
    diff = _diffusion(case)
    noise, label, step_noise = build_sample_inputs(case, ucase["cfg"])
    out = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=case["use_ddim"],
                        step_noise=None if case["use_ddim"] else step_noise)
    err = (out - ref).abs().max().item()
    print(f"{name} [bf16 operands]: max-abs {err:.3e}")
    assert torch.isfinite(out).all() and err <= 0.25
    if err > SAMPLE_MAX_ABS:
        pytest.xfail(f"bf16 operands: {err:.3e} > {SAMPLE_MAX_ABS:.0e} (documented: fp16 is the production format)")


def test_fp16_range_monitor_and_bf16_fallback():
    """fp16 operands saturate at +-65504 instead of overflowing.  A checkpoint whose residual stream leaves that range
    must be *noticed*: scale the stream far past 65504 (huge in_conv gain on a concat network), check that the plan's
    saturation counter fires and the output stays finite, that the same network in bf16 operands (fp32 exponent range)
    counts nothing, and that the in-range network counts nothing either."""
    import ctypes as C
    from oracle.unet_ref import make_state_dict
    from v_diffusion_b200 import UNet, _lib
    case = UNET_CASES["small_cond"]
    cfg = case["cfg"]
    x, t, y = build_inputs(case)

    def run(sd, operand):
        net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"],
                   cfg["num_res_blocks"], cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], head_dim=cfg["head_dim"],
                   num_heads=cfg["num_heads"], num_classes=cfg["num_classes"], multitags=cfg["multitags"])
        net.load_state_dict(sd, strict=True)
        net.operand_dtype = operand
        net = net.cuda().eval()
        out = net(x.cuda(), t.cuda(), y.cuda()).cpu()
        n = C.c_uint64()
        _lib.check(_lib.lib().vdt_plan_saturations(net.plan_for(case["res"], torch.device("cuda", 0)), C.byref(n), 1))
        return out, n.value

    sd = make_state_dict(cfg, case["seed"])
    out, n = run(sd, "fp16")
    assert n == 0 and torch.isfinite(out).all()
    big = {k: v.clone() for k, v in sd.items()}
    big["in_conv.weight"] *= 3.0e5                         # stream (and the raw concat copies of the up path) ~ 1e5..1e6
    big["in_conv.bias"] *= 3.0e5
    out16, n16 = run(big, "fp16")
    outb, nb = run(big, "bf16")
    print(f"fp16 saturation events {n16}, bf16 {nb}")
    assert n16 > 0, "the raw stream left the fp16 range but nothing was counted"
    assert nb == 0
    assert torch.isfinite(out16).all() and torch.isfinite(outb).all()
    # bf16 keeps tracking the fp32 oracle on that network; saturated fp16 does not have to
    from oracle import unet_forward
    ref = unet_forward(big, cfg, x, t, y)
    assert ((outb - ref).norm() / ref.norm()).item() <= 3e-2


def test_celeba_config_forward_vs_oracle():
    """BASELINE configs[2] architecture (celeba.json: hid 192, mult 1-2-3-4, E 768, one 64-wide head, 6 output
    channels) at 64x64: channel counts that are not powers of two (6..48 channels per group, concat seams inside
    a group -> two-pass GroupNorm fallback), 192-wide N tiles, attention over 4096 / 1024 / 256 / 64 tokens."""
    from oracle import unet_forward, make_state_dict
    from tests.cases import CELEBA
    cfg = CELEBA
    g = torch.Generator().manual_seed(3)
    B = 2
    x = torch.randn(B, 3, 64, 64, generator=g)
    t = torch.rand(B, generator=g, dtype=torch.float64)
    sd = make_state_dict(cfg, 21)
    net = _model(cfg, 21)
    out = net(x.cuda(), t.cuda(), None).cpu()
    ref = unet_forward(sd, cfg, x, t, None)
    rel = ((out - ref).norm() / ref.norm()).item()
    print(f"celeba: rel-L2 {rel:.3e} max-abs {(out - ref).abs().max().item():.3e}")
    assert out.shape == (B, 6, 64, 64) and rel <= REL_L2


def test_mnist_style_ancestral_cfg_vs_oracle():
    """BASELINE configs[3] in miniature: 1-channel conditional UNet (defaults model block), CFG w=3, ancestral
    sampling with injected per-step noise (the reference's own MNIST is resized to 32x32, datasets.py:97-106)."""
    from oracle import unet_forward, make_state_dict, p_sample
    from tests.cases import _cfg
    cfg = _cfg(in_channels=1, hid=64, out_channels=1, mult=(1, 2), nrb=1, attn=(False, True), num_classes=10)
    sd = make_state_dict(cfg, 31)
    net = _model(cfg, 31)
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    T, B = 64, 3                     # (a dozen coarse w = 3 steps on random weights is chaotic: it sat at 1.9e-2)
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, "v", "fixed_medium", "snr_trunc", "mse",
                             intp_frac=0.3, w_guide=3.0)
    g = torch.Generator().manual_seed(8)
    noise = torch.randn(B, 1, 32, 32, generator=g)
    label = torch.tensor([1, 7, 10])
    step_noise = torch.randn(T, B, 1, 32, 32, generator=g)
    out = diff.p_sample(net, (B, 1, 32, 32), noise=noise, label=label, device="cuda", use_ddim=False, step_noise=step_noise)
    ref = p_sample(lambda x, t, y: unet_forward(sd, cfg, x, t, y), (B, 1, 32, 32), noise, label, T=T, model_out_type="v",
                   w_guide=3.0, use_ddim=False, var_type="fixed_medium", intp_frac=0.3, step_noise=step_noise)
    err = (out - ref).abs().max().item()
    print(f"mnist-style ancestral w=3: max-abs {err:.3e}")
    assert err <= SAMPLE_MAX_ABS


def test_on_device_noise_stream():
    """Ancestral sampling without injected noise draws from the library's Philox stream: deterministic per seed,
    different across seeds, and statistically a unit normal (checked through one step with c1 = c2 = 0 removed:
    x_s - mean has the per-step std)."""
    case = SAMPLE_CASES["ancestral_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    net = _model(ucase["cfg"], ucase["seed"])
    diff = _diffusion(case)
    noise, label, _ = build_sample_inputs(case, ucase["cfg"])
    a = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", seed=5, use_ddim=False)
    b = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", seed=5, use_ddim=False)
    c = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", seed=6, use_ddim=False)
    assert torch.equal(a, b) and not torch.equal(a, c) and torch.isfinite(a).all()




@pytest.mark.parametrize("name", ["cifar_cond", "small_cond", "small_hd64"])
def test_validation_mode_forward(golden_dir, name):
    """operand_dtype="fp16x3": same tcgen05 kernels, every operand an fp16 hi/lo pair (three K segments per
    product), attention in fp32: agreement with the fp32 reference at the 1e-5 level."""
    case = UNET_CASES[name]
    ref = torch.from_numpy(np.load(os.path.join(golden_dir, f"unet_{name}.npz"))["out"])
    net = _model(case["cfg"], case["seed"], operand="fp16x3")
    x, t, y = build_inputs(case)
    out = net(x.cuda(), t.cuda(), None if y is None else y.cuda()).cpu()
    rel = ((out - ref).norm() / ref.norm()).item()
    err = (out - ref).abs().max().item()
    print(f"{name} [fp16x3]: rel-L2 {rel:.3e} max-abs {err:.3e}")
    assert rel <= 5e-5 and err <= 2e-4


@pytest.mark.parametrize("name", sorted(SAMPLE_CASES))
def test_validation_mode_sampler(golden_dir, name):
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    ref = torch.from_numpy(np.load(os.path.join(golden_dir, f"sample_{name}.npz"))["out"])
    net = _model(ucase["cfg"], ucase["seed"], operand="fp16x3")
    diff = _diffusion(case)
    noise, label, step_noise = build_sample_inputs(case, ucase["cfg"])
    out = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=case["use_ddim"],
                        step_noise=None if case["use_ddim"] else step_noise)
    err = (out - ref).abs().max().item()
    print(f"{name} [fp16x3]: max-abs {err:.3e}")
    assert err <= VALIDATION_MAX_ABS


@pytest.mark.parametrize("name", ["ddim_cfg_v", "ancestral_cfg_v"])
@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_p_sample_progressive_vs_reference_golden(golden_dir, name, operand):
    """diffusion.py:416-441 against the unmodified reference's own progressive loop, which carries an fp32 step
    tensor (:421): fp32 s / t quotients and an fp32 sinusoidal embedding.  x0 previews every pred_freq steps."""
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    g = np.load(os.path.join(golden_dir, f"progressive_{name}.npz"))
    ref, ref_preds, pred_freq = torch.from_numpy(g["out"]), torch.from_numpy(g["preds"]), int(g["pred_freq"])
    net = _model(ucase["cfg"], ucase["seed"], operand=operand)
    diff = _diffusion(case)
    noise, label, step_noise = build_sample_inputs(case, ucase["cfg"])
    x, preds = diff.p_sample_progressive(net, tuple(noise.shape), noise=noise, label=label, device="cuda",
                                         use_ddim=case["use_ddim"], pred_freq=pred_freq,
                                         step_noise=None if case["use_ddim"] else step_noise)
    assert preds.shape == ref_preds.shape
    bar = SAMPLE_MAX_ABS if operand == "fp16" else VALIDATION_MAX_ABS
    ex, ep = (x - ref).abs().max().item(), (preds - ref_preds).abs().max().item()
    print(f"progressive {name} [{operand}]: final {ex:.3e} previews {ep:.3e} (bar {bar:.0e})")
    assert ex <= bar
    # a guided preview is x0_c + w (x0_c - x0_u): the difference of two clipped predictions amplified by w on top
    assert ep <= bar * (1.0 + case["w_guide"])


def test_full_size_chunk_properties():
    """Size-independent properties on the real CIFAR-10 conditional network at a batch that spans full 1024-row
    chunks (BASELINE configs[1] geometry): a sample's trajectory does not depend on its batch neighbours, its
    chunk, or the chunk size, and the run is deterministic."""
    from tests.cases import CIFAR_COND
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    net = _model(CIFAR_COND, 13)
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 100, "v", "fixed_medium", "snr_trunc", "mse",
                             intp_frac=0.3, w_guide=1.0)
    g = torch.Generator().manual_seed(77)
    B = 520                                                # 512 images (one full 1024-row chunk) + 8
    noise = torch.randn(B, 3, 32, 32, generator=g)
    label = torch.randint(0, 11, (B,), generator=g)
    # only the first 2 of the 100 steps are run: the property is per step
    import ctypes as C
    from v_diffusion_b200 import _lib
    sc = diff.sampler_config(use_ddim=True)

    def run(n_idx, max_rows):
        net.max_rows = max_rows
        plan = net.plan_for(32, torch.device("cuda", 0))
        x = noise[n_idx].cuda().contiguous().clone()
        y = label[n_idx].cuda().contiguous()
        _lib.check(_lib.lib().vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(y), None, x.shape[0], 99, 2, None, None))
        torch.cuda.synchronize()
        return x.cpu()

    full = run(torch.arange(B), 1024)
    again = run(torch.arange(B), 1024)
    assert torch.equal(full, again)                        # deterministic (fixed-order statistics, no atomics)
    pick = torch.tensor([0, 255, 511, 512, 519])
    alone = run(pick, 1024)
    assert (alone - full[pick]).abs().max().item() <= 1e-5
    small_chunks = run(torch.arange(B), 128)
    assert (small_chunks - full).abs().max().item() <= 1e-5
    assert torch.isfinite(full).all() and (full - noise).abs().max().item() > 1e-3


def test_c_abi_host_entry_point_matches_python_api():
    """vdt_p_sample_host (host buffers in, host buffer out, copies inside the call) == GaussianDiffusion.p_sample."""
    import ctypes as C
    from v_diffusion_b200 import _lib
    case = SAMPLE_CASES["ancestral_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    net = _model(ucase["cfg"], ucase["seed"])
    diff = _diffusion(case)
    noise, label, step_noise = build_sample_inputs(case, ucase["cfg"])
    ref = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=False, step_noise=step_noise)
    plan = net.plan_for(noise.shape[2], torch.device("cuda", 0))
    sc = diff.sampler_config(use_ddim=False)
    out = torch.empty_like(noise)
    noise_h, label_h, sn_h = noise.contiguous(), label.contiguous(), step_noise.contiguous()
    rc = _lib.lib().vdt_p_sample_host(plan, C.byref(sc), _lib.ptr(noise_h), _lib.ptr(label_h), _lib.ptr(sn_h), _lib.ptr(out),
                                      noise.shape[0])
    assert rc == 0, _lib.lib().vdt_last_error()
    assert torch.equal(out, ref)
    # error path: a plan that is not finalized refuses to run and says why
    from v_diffusion_b200 import UNet
    cfg = ucase["cfg"]
    blank = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
                 cfg["apply_attn"], num_classes=cfg["num_classes"]).cuda().eval()
    handle = C.c_void_p()
    ucfg = _lib.UNetConfig()
    ucfg.in_channels, ucfg.hid_channels, ucfg.out_channels, ucfg.num_levels = 3, 64, 3, 2
    ucfg.ch_multipliers[0], ucfg.ch_multipliers[1] = 1, 2
    ucfg.apply_attn[1] = 1
    ucfg.num_res_blocks, ucfg.num_heads, ucfg.resolution, ucfg.max_rows = 1, 1, 16, 8
    assert _lib.lib().vdt_plan_create(C.byref(ucfg), C.byref(handle)) == 0
    assert _lib.lib().vdt_plan_finalize(handle) != 0 and b"missing key" in _lib.lib().vdt_last_error()
    rc = _lib.lib().vdt_p_sample_host(handle, C.byref(sc), _lib.ptr(noise_h), None, None, _lib.ptr(out), noise.shape[0])
    assert rc != 0 and b"not finalized" in _lib.lib().vdt_last_error()
    _lib.lib().vdt_plan_destroy(handle)
    del blank


# ---------------------------------------------------------------------------------------------------------------
# Full-length trajectories of the real CIFAR-10 networks against the unmodified reference (tests/golden/full_*.npz)
def _full_model(case, operand):
    from v_diffusion_b200 import UNet
    sd, net = full_state_dict(case, UNet)
    net.load_state_dict(sd, strict=True)
    net.operand_dtype = operand
    return net.cuda().eval()


def _full_diffusion(case):
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), case["T"], case["model_out_type"], case["var_type"],
                             "snr_trunc", "mse", intp_frac=case["intp_frac"], w_guide=case["w_guide"])


@pytest.mark.parametrize("name", sorted(FULL_CASES))
@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_full_trajectory_vs_reference_golden(golden_dir, name, operand):
    """BASELINE configs[0] (cifar10_uncond, 10-step DDIM, batch 16, exactly the SURVEY §8d recipe) and configs[1] at
    batch 8 (cifar10_cond, v-prediction, CFG w = 1, all 100 DDIM steps) on the real 60.8 M-parameter networks.
    Production mode (fp16 operands): final samples within 2e-2, every per-step model output within 1e-2 rel-L2;
    validation mode (fp16x3): final samples within 1e-3."""
    case = FULL_CASES[name]
    g = np.load(os.path.join(golden_dir, f"full_{name}.npz"))
    ref, ref_mo = torch.from_numpy(g["out"]), torch.from_numpy(g["model_out"])       # model_out: seeded sample of each step
    idx = torch.from_numpy(g["model_out_index"]).long()
    net = _full_model(case, operand)
    diff = _full_diffusion(case)
    noise, label = build_full_inputs(case)
    out = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=True)
    err = (out - ref).abs().max().item()
    bar = SAMPLE_MAX_ABS if operand == "fp16" else VALIDATION_MAX_ABS
    print(f"full {name} [{operand}]: final-sample max-abs {err:.3e} (bar {bar:.0e})")
    assert err <= bar
    # per-step model outputs along the trajectory (generic-callable path, same kernels), rows the fixture kept
    keep = case["keep_rows"]
    rec = []

    def wrapped(x, t, y):
        o = net(x, t, y)
        rec.append(o[:keep].cpu().reshape(-1)[idx])
        return o
    out2 = diff.p_sample(wrapped, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=True)
    assert (out2 - out).abs().max().item() <= 1e-5
    assert len(rec) == case["T"] == ref_mo.shape[0]
    rels = [((o - ref_mo[i]).norm() / ref_mo[i].norm()).item() for i, o in enumerate(rec)]
    print(f"full {name} [{operand}]: per-step rel-L2 worst {max(rels):.3e} median {sorted(rels)[len(rels) // 2]:.3e}")
    assert max(rels) <= (REL_L2 if operand == "fp16" else 1e-3)


def test_seed_none_draws_fresh_noise_and_seed_reproduces():
    """Ancestral sampling without injected noise: seed=None must not replay one noise trajectory (the reference draws
    from the global generator, diffusion.py:401-402); an explicit seed -- or torch.manual_seed -- reproduces a run."""
    case = SAMPLE_CASES["ancestral_x0eps"]
    ucase = UNET_CASES[case["unet"]]
    net = _model(ucase["cfg"], ucase["seed"])
    diff = _diffusion(case)
    noise, label, _ = build_sample_inputs(case, ucase["cfg"])
    kw = dict(noise=noise, label=label, device="cuda", use_ddim=False)
    a = diff.p_sample(net, tuple(noise.shape), **kw)
    b = diff.p_sample(net, tuple(noise.shape), **kw)
    assert not torch.equal(a, b)
    torch.manual_seed(123); c = diff.p_sample(net, tuple(noise.shape), **kw)
    torch.manual_seed(123); d = diff.p_sample(net, tuple(noise.shape), **kw)
    assert torch.equal(c, d)
    e = diff.p_sample(net, tuple(noise.shape), seed=9, **kw)
    f = diff.p_sample(net, tuple(noise.shape), seed=9, **kw)
    assert torch.equal(e, f) and not torch.equal(e, a)


def test_label_validation():
    """Out-of-range class ids and wrongly shaped multitag labels raise (F.one_hot raises in the reference,
    modules.py:191-196; unet.py:291 asserts y.ndim == 2) instead of indexing outside the embedding tables."""
    case = UNET_CASES["small_cond"]
    net = _model(case["cfg"], case["seed"])
    x, t, y = build_inputs(case)
    with pytest.raises(RuntimeError, match="class ids"):
        net(x.cuda(), t.cuda(), torch.tensor([0, 11, 3]).cuda())
    with pytest.raises(RuntimeError, match="class ids"):
        net(x.cuda(), t.cuda(), torch.tensor([0, -1, 3]).cuda())
    scase = SAMPLE_CASES["ddim_cfg_v"]
    diff = _diffusion(scase)
    noise, label, _ = build_sample_inputs(scase, case["cfg"])
    with pytest.raises(RuntimeError, match="class ids"):
        diff.p_sample(net, tuple(noise.shape), noise=noise, label=label + 10, device="cuda", use_ddim=True)
    with pytest.raises(ValueError, match="one class id per sample"):
        diff.p_sample(net, tuple(noise.shape), noise=noise, label=label[:2], device="cuda", use_ddim=True)
    mcase = UNET_CASES["small_multitag"]
    mnet = _model(mcase["cfg"], mcase["seed"])
    mdiff = _diffusion(SAMPLE_CASES["ddim_cfg_multitag"])
    mnoise, mlabel, _ = build_sample_inputs(SAMPLE_CASES["ddim_cfg_multitag"], mcase["cfg"])
    with pytest.raises(ValueError, match="multitag labels must have shape"):
        mdiff.p_sample(mnet, tuple(mnoise.shape), noise=mnoise, label=torch.ones(mnoise.shape[0]), device="cuda", use_ddim=True)
    # p_sample_progressive shares the label preparation: multi-hot float rows reach the C side as fp32
    a = mdiff.p_sample(mnet, tuple(mnoise.shape), noise=mnoise, label=mlabel, device="cuda", use_ddim=True)
    b, _ = mdiff.p_sample_progressive(mnet, tuple(mnoise.shape), noise=mnoise, label=mlabel, device="cuda", use_ddim=True, pred_freq=2)
    assert (a - b).abs().max().item() <= 5e-3              # same trajectory up to the fp32-t rounding of the progressive loop


def test_sampler_exec_cache_is_reused_across_noise_tensors_and_seeds():
    """Per-call values (injected-noise tensor, seed) live in device state: a new noise tensor or seed must not rebuild
    the workspace or re-capture the CUDA graph (round-1 advice), and the LRU cache keeps the other entries."""
    import time
    case = SAMPLE_CASES["ancestral_x0eps"]
    ucase = UNET_CASES[case["unet"]]
    net = _model(ucase["cfg"], ucase["seed"])
    diff = _diffusion(case)
    noise, label, step_noise = build_sample_inputs(case, ucase["cfg"])
    ref = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=False, step_noise=step_noise)
    diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=False, step_noise=step_noise)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(5):
        sn = step_noise.clone()                                # a fresh allocation every call
        out = diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=False, step_noise=sn)
        assert torch.equal(out, ref)
        diff.p_sample(net, tuple(noise.shape), noise=noise, label=label, device="cuda", use_ddim=False, seed=100 + k)
    per_call = (time.perf_counter() - t0) / 10
    print(f"cached sampler call: {per_call * 1e3:.1f} ms")
    assert per_call < 0.25          # a rebuild (workspace allocation + eager pass + capture) costs far more


def test_images_to_uint8_matches_generate_py():
    """generate.py:149 on the device: (x * 127.5 + 127.5).clamp(0, 255).to(uint8).permute(0, 2, 3, 1)."""
    from v_diffusion_b200.generate import images_to_uint8
    g = torch.Generator().manual_seed(4)
    for shape in [(5, 3, 32, 32), (3, 1, 28, 28), (2, 3, 64, 64)]:
        x = (torch.randn(shape, generator=g) * 0.8).cuda()
        x[0, 0, 0, :4] = torch.tensor([-1.0, 1.0, 1.7, -3.0])          # exact ends and out-of-range (guided samples exceed 1)
        want = (x * 127.5 + 127.5).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1)
        got = images_to_uint8(x)
        assert got.dtype == torch.uint8 and got.shape == want.shape
        assert torch.equal(got, want)


@pytest.mark.parametrize("world,schedule", [(1, "static"), (2, "static"), (1, "dynamic"), (2, "dynamic")])
def test_generate_driver_end_to_end(tmp_path, world, schedule):
    """`python -m v_diffusion_b200.generate` (the sharded batch loop of generate.py:100-150) as a user runs it: a
    reference-format checkpoint + config JSONs in, uint8 NHWC images out; on 2 GPUs under torchrun with the NCCL image
    gather.  The gathered images must equal what p_sample gives in-process for every rank's seeded noise / labels."""
    import subprocess
    import sys
    from oracle.unet_ref import make_state_dict
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    from v_diffusion_b200.generate import shard_bounds, images_to_uint8
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ucase = UNET_CASES["small_cond"]
    cfg = ucase["cfg"]
    sd = make_state_dict(cfg, ucase["seed"])
    torch.save({"model": {"module." + k: v for k, v in sd.items()}}, tmp_path / "ckpt.pt")     # DDP prefix, generate.py:40-42
    merged = json.load(open(os.path.join(root, "tests", "golden", "merged_configs.json")))["cifar10_cond"]
    model_block = dict(in_channels=3, hid_channels=64, ch_multipliers=[1, 2], num_res_blocks=2, apply_attn=[False, True],
                       drop_rate=0.2, num_heads=1)
    json.dump({"data": {"name": "cifar10"}, "model": model_block, "diffusion": merged["diffusion"],
               "conditional": merged["conditional"]}, open(tmp_path / "cfg.json", "w"))
    json.dump({}, open(tmp_path / "defaults.json", "w"))
    total, bs, T, seed = 22, 4, 6, 77
    args = ["--config-path", str(tmp_path / "cfg.json"), "--default-config-path", str(tmp_path / "defaults.json"),
            "--ckpt-path", str(tmp_path / "ckpt.pt"), "--sample-timesteps", str(T), "--w-guide", "1.0", "--batch-size", str(bs),
            "--total-size", str(total), "--save-path", str(tmp_path / "out.pt"), "--seed", str(seed), "--schedule", schedule]
    if world == 1:
        cmd = [sys.executable, "-m", "v_diffusion_b200.generate"] + args
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr",
               "127.0.0.1", "--master-port", "29533" if schedule == "static" else "29534", "-m", "v_diffusion_b200.generate"] + args
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run(cmd, cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = torch.load(tmp_path / "out.pt")
    assert got.dtype == torch.uint8 and tuple(got.shape) == (total, 32, 32, 3)
    # expected: every rank's slice, batch by batch, with the generator protocol of generate.sample_fn (ancestral sampling:
    # noise, labels and the per-batch noise seed all come from Generator(seed + rank))
    net = _model(cfg, ucase["seed"])
    d = merged["diffusion"]
    diff = GaussianDiffusion(get_logsnr_schedule(d["logsnr_schedule"], d["logsnr_min"], d["logsnr_max"]), T, d["model_out_type"],
                             d["model_var_type"], d["reweight_type"], d["loss_type"], intp_frac=d["intp_frac"], w_guide=1.0)
    want = []
    # static: rank r owns a contiguous slice and one generator (seed + r); dynamic: global batch k has its own
    # generator (seed + k) whichever rank claims it from the queue
    slices = [(shard_bounds(total, r, world), seed + r) for r in range(world)] if schedule == "static" else \
        [((b0, min(b0 + bs, total)), seed + b0 // bs) for b0 in range(0, total, bs)]
    for (s0, e0), gseed in slices:
        gen = torch.Generator(device="cuda").manual_seed(gseed)
        for b0 in range(s0, e0, bs):
            n = min(bs, e0 - b0)
            noise = torch.randn((n, 3, 32, 32), device="cuda", generator=gen)
            label = torch.randint(10, (n,), device="cuda", generator=gen) + 1
            call_seed = int(torch.randint(0, 2 ** 62, (1,), device="cuda", generator=gen).item())
            want.append(diff.p_sample(net, (n, 3, 32, 32), noise=noise, label=label, device="cuda", seed=call_seed, use_ddim=False))
    want = images_to_uint8(torch.cat(want).cuda()).cpu()
    diffpix = (got.int() - want.int()).abs()
    print(f"generate x{world} {schedule}: {int((diffpix > 0).sum())} of {diffpix.numel()} uint8 values differ, max {int(diffpix.max())}")
    assert int(diffpix.max()) == 0


# ---------------------------------------------------------------------------------------------------------------
# Training step, first slice (SURVEY §8 f2): GaussianDiffusion.train_loss around the model call
@pytest.mark.parametrize("name", sorted(TRAIN_CASES))
def test_train_loss_vs_reference_golden(golden_dir, name):
    """q_sample + from_model_out_to_pred + re-weighted MSE (diffusion.py:492-545) against the unmodified reference:
    (1) with the reference's own model output injected, x_t, the per-sample loss and d loss.mean() / d model_out (the
    reference's autograd) must agree to fp32 rounding; (2) with this package's UNet as denoise_fn the loss agrees within
    the operand format's accuracy.  The p_uncond label dropout acts on the caller's y after the model call only."""
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    case = TRAIN_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    g = np.load(os.path.join(golden_dir, f"train_{name}.npz"))
    x0, t, noise, y = build_train_inputs(case, cfg)
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 1000, case["model_out_type"], "fixed_large",
                             case["reweight_type"], "mse", p_uncond=0.1)
    ref_out = torch.from_numpy(g["model_out"]).cuda()
    seen = {}

    def injected(x_t, tt, yy):
        seen["x_t"] = x_t.clone()
        return ref_out
    torch.manual_seed(case["seed"])                        # the label-dropout mask comes from the global CPU generator
    yy = None if y is None else y.clone().cuda()
    loss, grad = diff.train_loss(injected, x0.cuda(), t, yy, noise=noise.cuda(), return_grad=True)
    assert (seen["x_t"].cpu() - torch.from_numpy(g["x_t"])).abs().max().item() <= 1e-6
    np.testing.assert_allclose(loss.cpu().numpy(), g["loss"], rtol=2e-6)
    ref_grad = torch.from_numpy(g["grad_out"])
    assert (grad.cpu() - ref_grad).abs().max().item() <= 2e-6 * max(1.0, ref_grad.abs().max().item())
    if y is not None:
        assert np.array_equal(yy.cpu().numpy(), g["y_after"])   # same mask, same in-place side effect, loss unaffected
    # (2) the CUDA UNet as the model (eval mode: the fixture's reference ran in eval mode too)
    for operand, tol in (("fp16", 1e-2), ("fp16x3", 1e-4)):
        net = _model(cfg, ucase["seed"], operand=operand)
        l2 = diff.train_loss(net, x0.cuda(), t.cuda(), None if y is None else y.clone().cuda(), noise=noise.cuda())
        rel = ((l2.cpu() - torch.from_numpy(g["loss"])).abs() / torch.from_numpy(g["loss"])).max().item()
        print(f"train_loss {name} [{operand}]: worst relative loss error {rel:.3e}")
        assert rel <= tol


def test_train_mode_forward_dropout():
    """UNet.forward in .train() mode (nn.Dropout(drop_rate, inplace=True) between act2 and conv2, unet.py:135, 146): with
    drop_rate = 0 it is bit-identical to .eval(); with drop_rate > 0 the masks follow the per-call seed drawn from torch's
    global generator (reproducible under manual_seed, fresh otherwise) and the output stays a perturbation of the eval one."""
    from oracle.unet_ref import make_state_dict
    from v_diffusion_b200 import UNet
    case = UNET_CASES["small_cond"]
    cfg = case["cfg"]
    x, t, y = build_inputs(case)

    def build(drop):
        net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
                   cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], drop_rate=drop, head_dim=cfg["head_dim"],
                   num_heads=cfg["num_heads"], num_classes=cfg["num_classes"])
        net.load_state_dict(make_state_dict(cfg, case["seed"]), strict=True)
        return net.cuda()
    ev = build(0.2).eval()(x.cuda(), t.cuda(), y.cuda())
    assert torch.equal(build(0.0).train()(x.cuda(), t.cuda(), y.cuda()), ev)
    net = build(0.2).train()
    torch.manual_seed(3); a = net(x.cuda(), t.cuda(), y.cuda())
    torch.manual_seed(3); b = net(x.cuda(), t.cuda(), y.cuda())
    c = net(x.cuda(), t.cuda(), y.cuda())
    assert torch.equal(a, b) and not torch.equal(a, c) and torch.isfinite(a).all()
    rel = ((a - ev).norm() / ev.norm()).item()
    print(f"train-mode forward, drop 0.2: rel-L2 distance to the eval output {rel:.3f}")
    assert 0.02 < rel < 1.5
    assert torch.equal(net.eval()(x.cuda(), t.cuda(), y.cuda()), ev)          # .eval() switches it off again


def test_optimizer_step_vs_torch_adamw_and_reference_ema():
    """clip_grad_norm_ -> AdamW.step -> EMA.update of the reference trainer (train_utils.py:159-166, train.py:158,
    utils.py:144-149; hyper-parameters of cifar10_cond.json) as two fused kernels per tensor: parameters, both Adam moments
    and the EMA shadow follow torch's own optimizer over several steps, with the clip active on some steps and not on others."""
    from v_diffusion_b200.optim import AdamWEMA
    g = torch.Generator(device="cuda").manual_seed(3)
    shapes = {"conv.weight": (256, 64, 3, 3), "conv.bias": (256,), "fc.weight": (70, 33), "odd": (7,)}
    mine = {k: torch.randn(s, device="cuda", generator=g) * 0.1 for k, s in shapes.items()}
    ref = {k: torch.nn.Parameter(v.clone()) for k, v in mine.items()}
    lr, betas, wd, max_norm, decay = 2e-4, (0.9, 0.999), 0.001, 1.0, 0.9999
    opt_ref = torch.optim.AdamW(list(ref.values()), lr=lr, betas=betas, weight_decay=wd)
    shadow_ref = {k: v.detach().clone() for k, v in ref.items()}
    opt = AdamWEMA(mine, lr=lr, betas=betas, weight_decay=wd, grad_norm=max_norm, ema_decay=decay)
    worst = 0.0
    for step, scale in enumerate([3.0, 1e-4, 0.5, 2.0], start=1):       # total norms above and below max_norm
        grads = {k: torch.randn(s, device="cuda", generator=g) * scale for k, s in shapes.items()}
        for k, p in ref.items():
            p.grad = grads[k].clone()
        total = torch.nn.utils.clip_grad_norm_(list(ref.values()), max_norm=max_norm)
        opt_ref.step()
        d = min(decay, (1 + step) / (10 + step))
        for k, p in ref.items():
            shadow_ref[k] += (1 - d) * (p.data - shadow_ref[k])
        sq = opt.step(grads)
        torch.cuda.synchronize()
        assert abs(sq.item() ** 0.5 - total.item()) <= 1e-5 * total.item()
        for k in shapes:
            stt = opt_ref.state[ref[k]]
            for a, b in ((mine[k], ref[k].data), (opt.exp_avg[k], stt["exp_avg"]), (opt.exp_avg_sq[k], stt["exp_avg_sq"]),
                         (opt.shadow[k], shadow_ref[k])):
                worst = max(worst, ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item())
    print(f"optimizer step: worst rel-L2 over params / moments / EMA shadow after 4 steps {worst:.2e}")
    assert worst <= 2e-6
    again = opt.step(grads).item()
    assert again == opt.step(grads).item()                              # fixed-order norm reduction


def test_bench_dump_outputs_is_the_timed_trajectory(tmp_path):
    """bench.py --dump-outputs writes what its timed loop computed: with --steps 100 the timed loop is exactly one 100-step DDIM
    trajectory from the bench's seeded noise, so the dump equals GaussianDiffusion.p_sample on the bench's model and inputs."""
    import subprocess
    import sys
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    B = 4
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--batch", str(B), "--steps", "100", "--warmup", "3",
                        "--no-cpu-baseline", "--no-train-step", "--dump-outputs", str(tmp_path)], cwd=root, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = torch.from_numpy(np.load(tmp_path / "samples.npy"))
    device = torch.device("cuda", 0)
    net, diff = bench.build_model(device, seed=0)
    g = torch.Generator(device=device).manual_seed(1234)                # bench.run_b200's draws for rank 0
    noise = torch.randn(B, 3, 32, 32, device=device, generator=g)
    label = torch.randint(10, (B,), device=device, generator=g) + 1
    want = diff.p_sample(net, (B, 3, 32, 32), noise=noise.cpu(), label=label.cpu(), device=device, use_ddim=True)
    err = (got - want.cpu()).abs().max().item()
    print(f"bench dump vs p_sample: max-abs {err:.3e}")
    assert got.dtype == torch.float32 and got.shape == want.shape and err <= 1e-3
