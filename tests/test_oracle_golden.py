"""CPU: the oracle restatement against fixtures produced by the unmodified reference
(tests/golden/make_golden.py).  This is what pins the oracle (SURVEY §8c)."""
import json
import math
import os

import numpy as np
import pytest
import torch

from oracle import unet_forward, make_state_dict, step_coefficients, p_sample, timestep_embedding
from oracle.unet_ref import unet_config_from_json
from tests.cases import (UNET_CASES, SAMPLE_CASES, FULL_CASES, TRAIN_CASES, CIFAR_COND, CIFAR_UNCOND, CELEBA, build_inputs,
                         build_sample_inputs, build_full_inputs, full_state_dict, build_train_inputs)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


@pytest.mark.parametrize("name", sorted(UNET_CASES))
def test_unet_forward_matches_reference(golden_dir, name):
    case = UNET_CASES[name]
    g = _load(golden_dir, f"unet_{name}.npz")
    sd = make_state_dict(case["cfg"], case["seed"])
    x, t, y = build_inputs(case)
    trace = {}
    out = unet_forward(sd, case["cfg"], x, t, y, trace=trace)
    ref = torch.from_numpy(g["out"])
    assert out.shape == ref.shape
    # same fp32 library kernels, different op grouping -> tiny reassociation differences only
    assert (out - ref).abs().max().item() <= 2e-4 * max(1.0, ref.abs().max().item())
    for key in g.files:
        if key.startswith("trace:"):
            mod = key[len("trace:"):]
            got = trace[mod] if mod in trace else trace[mod + ".1"] if mod + ".1" in trace else None
            if mod == "middle":
                got = trace["middle.2"]
            elif got is None:
                got = trace[mod + ".0"]
            if "trace_index:" + mod in g.files:                 # stored at a seeded sample of positions (cases.golden_sample_index)
                got = got.reshape(-1)[torch.from_numpy(g["trace_index:" + mod]).long()]
            r = torch.from_numpy(g[key])
            assert (got - r).abs().max().item() <= 2e-4 * max(1.0, r.abs().max().item()), mod


@pytest.mark.parametrize("name", sorted(SAMPLE_CASES))
def test_sampler_matches_reference(golden_dir, name):
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    g = _load(golden_dir, f"sample_{name}.npz")
    sd = make_state_dict(cfg, ucase["seed"])
    noise, label, step_noise = build_sample_inputs(case, cfg)
    rec = []
    out = p_sample(lambda x, t, y: unet_forward(sd, cfg, x, t, y), tuple(noise.shape), noise, label,
                   T=case["T"], model_out_type=case["model_out_type"], w_guide=case["w_guide"],
                   use_ddim=case["use_ddim"], var_type=case["var_type"], intp_frac=case.get("intp_frac"),
                   step_noise=step_noise, record=rec, x0eps_coef=case.get("x0eps_coef", False))
    ref = torch.from_numpy(g["out"])
    assert (out - ref).abs().max().item() <= 5e-4
    mo = torch.from_numpy(g["model_out"])
    assert len(rec) == mo.shape[0] == case["T"]
    for i, (ti, o) in enumerate(rec):
        assert ti == case["T"] - 1 - i
        rel = (o - mo[i]).norm() / mo[i].norm()
        assert rel.item() <= 1e-4


@pytest.mark.parametrize("name,pred_freq", [("ddim_cfg_v", 3), ("ancestral_cfg_v", 16)])
def test_progressive_matches_reference(golden_dir, name, pred_freq):
    """p_sample_progressive (diffusion.py:416-441) feeds an fp32 step tensor (:421): fp32 s / t, fp32 sinusoid."""
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    g = _load(golden_dir, f"progressive_{name}.npz")
    assert int(g["pred_freq"]) == pred_freq
    sd = make_state_dict(cfg, ucase["seed"])
    noise, label, step_noise = build_sample_inputs(case, cfg)
    rec = []
    out = p_sample(lambda x, t, y: unet_forward(sd, cfg, x, t, y), tuple(noise.shape), noise, label,
                   T=case["T"], model_out_type=case["model_out_type"], w_guide=case["w_guide"],
                   use_ddim=case["use_ddim"], var_type=case["var_type"], intp_frac=case.get("intp_frac"),
                   step_noise=step_noise, pred_record=rec, t_fp32=True)
    assert (out - torch.from_numpy(g["out"])).abs().max().item() <= 5e-4
    preds = torch.from_numpy(g["preds"])
    want = [p for ti, p in rec if (ti + 1) % pred_freq == 0]       # loop order: ti descending -> preds index descending
    assert len(want) == preds.shape[0] == case["T"] // pred_freq
    for k, p in enumerate(want):
        assert (p - preds[preds.shape[0] - 1 - k]).abs().max().item() <= 5e-4


def test_full_trajectory_configs0_matches_reference(golden_dir):
    """BASELINE configs[0] exactly as SURVEY §8d specifies it: cifar10_uncond.json network initialised under
    manual_seed(0) and de-zeroed (seed 7), x0 / fixed_large, 10-step DDIM, batch 16, noise from Generator(1234).
    Also proves that this package's UNet constructor reproduces the reference's initialisation bit for bit (the
    fixture was generated with the reference's own module)."""
    from v_diffusion_b200 import UNet
    case = FULL_CASES["cifar10_uncond_ddim10"]
    g = _load(golden_dir, "full_cifar10_uncond_ddim10.npz")
    sd, _ = full_state_dict(case, UNet)
    noise, label = build_full_inputs(case)
    rec = []
    out = p_sample(lambda x, t, y: unet_forward(sd, case["cfg"], x, t, y), tuple(noise.shape), noise, label,
                   T=case["T"], model_out_type=case["model_out_type"], w_guide=case["w_guide"], use_ddim=True,
                   var_type=case["var_type"], record=rec)
    assert (out - torch.from_numpy(g["out"])).abs().max().item() <= 5e-4
    mo, idx = torch.from_numpy(g["model_out"]), torch.from_numpy(g["model_out_index"]).long()   # seeded sample of each step
    assert len(rec) == mo.shape[0] == case["T"]
    for i, (ti, o) in enumerate(rec):
        o = o[:case["keep_rows"]].reshape(-1)[idx]
        assert ((o - mo[i]).norm() / mo[i].norm()).item() <= 1e-4


def test_full_trajectory_configs1_matches_reference(golden_dir):
    """BASELINE configs[1] at reduced batch: cifar10_cond.json network, v-prediction, CFG w = 1, all 100 DDIM steps.
    The fixture holds 8 images; trajectories are independent per sample, so the oracle replays the first two
    (4 UNet rows per step) to keep the CPU suite short."""
    from v_diffusion_b200 import UNet
    case = FULL_CASES["cifar10_cond_cfg_ddim100"]
    g = _load(golden_dir, "full_cifar10_cond_cfg_ddim100.npz")
    sd, _ = full_state_dict(case, UNet)
    noise, label = build_full_inputs(case)
    rec = []
    out = p_sample(lambda x, t, y: unet_forward(sd, case["cfg"], x, t, y), (2, 3, 32, 32), noise[:2], label[:2],
                   T=case["T"], model_out_type="v", w_guide=1.0, use_ddim=True, var_type="fixed_medium", intp_frac=0.3,
                   record=rec)
    assert (out - torch.from_numpy(g["out"])[:2]).abs().max().item() <= 1e-3
    mo = torch.from_numpy(g["model_out"])                       # (100, keep_entries): seeded sample of the rows of the first two images
    idx = torch.from_numpy(g["model_out_index"]).long()
    assert len(rec) == 100
    for i, (ti, o) in enumerate(rec):
        o = o.reshape(-1)[idx]
        assert ((o - mo[i]).norm() / mo[i].norm()).item() <= 2e-4, ti


@pytest.mark.parametrize("name", sorted(TRAIN_CASES))
def test_train_loss_matches_reference(golden_dir, name):
    """GaussianDiffusion.train_loss (diffusion.py:492-545) restated in the oracle, against the reference's own x_t,
    model output and per-sample loss (the fixture's model output is also what the oracle's UNet computes)."""
    from oracle import train_loss
    case = TRAIN_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    g = _load(golden_dir, f"train_{name}.npz")
    sd = make_state_dict(cfg, ucase["seed"])
    x0, t, noise, y = build_train_inputs(case, cfg)
    seen = {}

    def fn(x_t, tt, yy):
        seen["out"] = unet_forward(sd, cfg, x_t, tt, yy)
        return seen["out"]
    loss, x_t = train_loss(fn, x0, t, y, noise, model_out_type=case["model_out_type"], reweight_type=case["reweight_type"])
    assert (x_t - torch.from_numpy(g["x_t"])).abs().max().item() <= 1e-6
    mo = torch.from_numpy(g["model_out"])
    assert ((seen["out"] - mo).norm() / mo.norm()).item() <= 1e-4
    np.testing.assert_allclose(loss.numpy(), g["loss"], rtol=2e-4)


def test_step_coefficients_known_answers(golden_dir):
    g = _load(golden_dir, "coefs_T100.npz")
    dd = step_coefficients(100, use_ddim=True)
    np.testing.assert_array_equal(dd["logsnr_s"], g["logsnr_s"])
    np.testing.assert_array_equal(dd["logsnr_t"], g["logsnr_t"])
    np.testing.assert_allclose(dd["c1"], g["ddim_c1"], rtol=2e-7, atol=0)
    np.testing.assert_allclose(dd["c2"], g["ddim_c2"], rtol=2e-7, atol=1e-12)
    np.testing.assert_array_equal(dd["alpha_t"], g["alpha_t"])
    np.testing.assert_array_equal(dd["sigma_t"], g["sigma_t"])
    assert np.all(dd["std"] == 0)
    for vt in ("fixed_small", "fixed_large", "fixed_medium"):
        an = step_coefficients(100, use_ddim=False, var_type=vt, intp_frac=0.3)
        np.testing.assert_allclose(an["c1"], g[f"{vt}_c1"], rtol=2e-7, atol=1e-12)
        np.testing.assert_allclose(an["c2"], g[f"{vt}_c2"], rtol=2e-7, atol=1e-12)
        np.testing.assert_allclose(an["logvar"], g[f"{vt}_logvar"], rtol=2e-7, atol=1e-9)
    # x0eps_coef=True (diffusion.py:137-140); the DDIM pair is the un-exponentiated one the reference returns (180-182)
    xd = step_coefficients(100, use_ddim=True, x0eps_coef=True)
    np.testing.assert_allclose(xd["c1"], g["x0eps_ddim_c1"], rtol=2e-7, atol=1e-12)
    np.testing.assert_allclose(xd["c2"], g["x0eps_ddim_c2"], rtol=2e-7, atol=1e-12)
    assert np.all(xd["c1"] < 0) and np.all(xd["c2"] < 0)
    xa = step_coefficients(100, use_ddim=False, var_type="fixed_small", x0eps_coef=True)
    np.testing.assert_allclose(xa["c1"], g["x0eps_small_c1"], rtol=2e-7, atol=1e-12)
    np.testing.assert_allclose(xa["c2"], g["x0eps_small_c2"], rtol=2e-7, atol=1e-12)
    np.testing.assert_allclose(xa["logvar"], g["x0eps_small_logvar"], rtol=2e-7, atol=1e-9)
    # SURVEY §10.2 table (values printed by the reference)
    assert abs(dd["c1"][50] - 0.984656036) < 1e-7 and abs(dd["c2"][50] - 0.021871394) < 1e-7
    assert abs(dd["alpha_t"][1] - 0.999505162) < 1e-7 and abs(dd["sigma_t"][1] - 0.031454321) < 1e-7
    an = step_coefficients(100, use_ddim=False, var_type="fixed_medium", intp_frac=0.3)
    assert abs(an["c1"][50] - 0.954199851) < 1e-7 and abs(an["logvar"][1] - (-8.175132)) < 1e-5


def test_timestep_embedding_known_answers(golden_dir):
    g = _load(golden_dir, "coefs_T100.npz")
    t = torch.from_numpy(g["temb_t"])
    np.testing.assert_allclose(timestep_embedding(t, 256).numpy(), g["temb_256"], rtol=0, atol=1e-7)
    np.testing.assert_allclose(timestep_embedding(t, 64).numpy(), g["temb_64"], rtol=0, atol=1e-7)
    e = timestep_embedding(torch.tensor([0.37], dtype=torch.float64), 256)[0]
    assert abs(e[0].item() - (-0.650264919)) < 1e-6 and abs(e[128].item() - 0.759707510) < 1e-6


def test_config_merge_gives_case_configs(golden_dir):
    with open(os.path.join(golden_dir, "merged_configs.json")) as f:
        merged = json.load(f)
    assert unet_config_from_json(merged["cifar10_cond"]["model"], 3, 3, num_classes=10) == CIFAR_COND
    assert unet_config_from_json(merged["cifar10_uncond"]["model"], 3, 3) == CIFAR_UNCOND
    assert unet_config_from_json(merged["celeba"]["model"], 3, 6) == CELEBA


def test_all_schedules_known_answers(golden_dir):
    g = _load(golden_dir, "coefs_T100.npz")
    for sched in ("cosine", "linear", "sigmoid", "legacy"):
        an = step_coefficients(50, use_ddim=False, var_type="fixed_large", schedule=sched)
        np.testing.assert_allclose(an["logsnr_s"], g[f"{sched}_logsnr_s"], rtol=2e-6, atol=1e-6)
        np.testing.assert_allclose(an["logsnr_t"], g[f"{sched}_logsnr_t"], rtol=2e-6, atol=1e-6)
        np.testing.assert_allclose(an["c1"], g[f"{sched}_c1"], rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(an["c2"], g[f"{sched}_c2"], rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(an["logvar"], g[f"{sched}_logvar"], rtol=1e-5, atol=1e-6)


def test_tf32_calibration_covers_every_sampler_fixture(golden_dir):
    """tests/golden/make_tf32_dev.py: deviation of the unmodified reference under its own default GPU numerics (TF32
    convolutions) per sampler fixture.  Reported next to the CUDA path's error in the GPU tests; the bar itself is the
    flat north-star 2e-2 on every fixture, so every fixture must leave room under it."""
    with open(os.path.join(golden_dir, "ref_tf32_deviation.json")) as f:
        dev = json.load(f)
    assert set(dev) == set(SAMPLE_CASES)
    for name, d in dev.items():
        assert d["w_guide"] == SAMPLE_CASES[name]["w_guide"] and d["T"] == SAMPLE_CASES[name]["T"]
        assert d["max_abs"] <= 1.5e-2, name


@pytest.mark.parametrize("name", ["ddim_cfg_v", "ancestral_cfg_v"])
def test_numerics_model_of_the_cuda_path(golden_dir, name):
    """oracle.unet_forward(operand_round=...) rounds every tensor the CUDA path keeps in 16 bits.  With fp16 it must
    stay inside the production bar on the fixtures (this is what the GPU tests then measure for real); with bf16 it
    does not -- the reason fp16 is the shipped operand format (DESIGN.md §2)."""
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    ref = torch.from_numpy(_load(golden_dir, f"sample_{name}.npz")["out"])
    sd = make_state_dict(cfg, ucase["seed"])
    noise, label, step_noise = build_sample_inputs(case, cfg)
    err = {}
    for mode in ("fp16", "bf16"):
        out = p_sample(lambda x, t, y: unet_forward(sd, cfg, x, t, y, operand_round=mode), tuple(noise.shape), noise, label,
                       T=case["T"], model_out_type=case["model_out_type"], w_guide=case["w_guide"],
                       use_ddim=case["use_ddim"], var_type=case["var_type"], intp_frac=case.get("intp_frac"),
                       step_noise=step_noise)
        err[mode] = (out - ref).abs().max().item()
    print(name, err)
    assert err["fp16"] <= 2e-2 and err["bf16"] > err["fp16"]


@pytest.mark.parametrize("which", ["small", "cifar"])
def test_oracle_backward_matches_reference_gradients(golden_dir, which):
    """The training step's gradients: torch autograd through the oracle UNet + the oracle train_loss against the gradients
    the UNMODIFIED reference's own UNet / train_loss / autograd produced (tests/golden/make_train_grad_golden.py) -- loss,
    every parameter gradient's norm and probe projection, and the small tensors in full.  This pins the checker the GPU
    training tests compare the CUDA path with."""
    from oracle import train_loss
    from oracle.unet_ref import _unet_forward
    from tests.cases import TRAIN_GRAD_CASES, build_train_grad_inputs, grad_probe
    case = TRAIN_GRAD_CASES[which]                                      # "cifar": cifar10_cond.json's own network (configs[4])
    cfg = case["cfg"]
    g = _load(golden_dir, f"train_grads_{which}.npz")
    sd = {k: v.clone().requires_grad_(True) for k, v in make_state_dict(cfg, case["wseed"]).items()}
    x0, t, noise, y = build_train_grad_inputs(case)
    with torch.enable_grad():
        loss, _ = train_loss(lambda a, b, c: _unet_forward(sd, cfg, a, b, c, None), x0, t, y, noise,
                             model_out_type=case["model_out_type"], reweight_type=case["reweight_type"])
        loss.mean().backward()
    np.testing.assert_allclose(loss.detach().numpy(), g["loss"], rtol=1e-5)
    names = [str(n) for n in g["names"]]
    assert sorted(names) == sorted(sd)
    for k in names:
        gr = sd[k].grad.double()
        n_ref = float(g["norm/" + k])
        assert abs(gr.norm().item() - n_ref) <= 1e-4 * n_ref + 1e-9, k
        p_ref = float(g["proj/" + k])
        assert abs((gr * grad_probe(k, gr.shape)).sum().item() - p_ref) <= 1e-3 * n_ref + 1e-9, k
        if ("full/" + k) in g.files:
            full = torch.from_numpy(g["full/" + k]).double()
            assert (gr - full).norm().item() <= 1e-4 * n_ref + 1e-9, k
