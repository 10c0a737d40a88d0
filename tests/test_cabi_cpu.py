"""CPU: the C-ABI library loads, exports every symbol include/vdt_b200.h declares, and its host-side
schedule code agrees with the reference-generated known answers (no GPU work)."""
import ctypes as C
import os
import re

import numpy as np
import torch

from v_diffusion_b200 import _lib, GaussianDiffusion, get_logsnr_schedule, fill_with_defaults, UNet


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    hdr = open(_lib.INCLUDE).read()
    declared = set(re.findall(r"\b(vdt_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(L, name), name
    assert L.vdt_version() == 1


def test_struct_layout_matches_header():
    assert C.sizeof(_lib.UNetConfig) == 4 * (4 + 8 + 1 + 8 + 8)
    assert C.sizeof(_lib.SamplerConfig) == 8 * 4 + 4 * 8 + 8
    assert C.sizeof(_lib.ConvOp) == 12 * 8 + 10 * 4               # vdt_conv_op: 12 pointers, 10 int32


def test_step_coefficients_match_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "coefs_T100.npz"))
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 100, "v", "fixed_medium", "snr_trunc", "mse",
                          intp_frac=0.3, w_guide=1.0)
    dd = d.step_coefficients(use_ddim=True).numpy()
    np.testing.assert_allclose(dd[:, 10], g["logsnr_s"], rtol=1e-6)
    np.testing.assert_allclose(dd[:, 11], g["logsnr_t"], rtol=1e-6)
    np.testing.assert_allclose(dd[:, 0], g["alpha_t"], rtol=2e-6, atol=1e-9)
    np.testing.assert_allclose(dd[:, 1], g["sigma_t"], rtol=2e-6, atol=1e-9)
    np.testing.assert_allclose(dd[:, 6], g["ddim_c1"], rtol=2e-6)
    np.testing.assert_allclose(dd[:, 7], g["ddim_c2"], rtol=2e-6, atol=1e-10)
    assert np.all(dd[:, 8] == 0)
    for vt in ("fixed_small", "fixed_large", "fixed_medium"):
        d.model_var_type = vt
        an = d.step_coefficients(use_ddim=False).numpy()
        np.testing.assert_allclose(an[:, 6], g[f"{vt}_c1"], rtol=2e-6, atol=1e-10)
        np.testing.assert_allclose(an[:, 7], g[f"{vt}_c2"], rtol=2e-6, atol=1e-10)
        np.testing.assert_allclose(an[:, 9], g[f"{vt}_logvar"], rtol=2e-6, atol=1e-7)
        np.testing.assert_allclose(an[:, 8], np.exp(0.5 * g[f"{vt}_logvar"]), rtol=1e-5)
    # x0eps_coef=True: posterior mean in (eps, x0) (diffusion.py:137-140); the DDIM pair is returned by the reference
    # as logarithms (180-182 never reach the .exp_() of line 199) and is reproduced as such
    x = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 100, "eps", "fixed_small", "snr_trunc", "mse",
                          x0eps_coef=True)
    xd, xa = x.step_coefficients(use_ddim=True).numpy(), x.step_coefficients(use_ddim=False).numpy()
    np.testing.assert_allclose(xd[:, 6], g["x0eps_ddim_c1"], rtol=2e-6, atol=1e-10)
    np.testing.assert_allclose(xd[:, 7], g["x0eps_ddim_c2"], rtol=2e-6, atol=1e-10)
    np.testing.assert_allclose(xa[:, 6], g["x0eps_small_c1"], rtol=2e-6, atol=1e-10)
    np.testing.assert_allclose(xa[:, 7], g["x0eps_small_c2"], rtol=2e-6, atol=1e-10)
    np.testing.assert_allclose(xa[:, 9], g["x0eps_small_logvar"], rtol=2e-6, atol=1e-7)
    lt = g["logsnr_t"].astype(np.float64)
    np.testing.assert_allclose(xa[:, 12], np.sqrt(1.0 + np.exp(lt)), rtol=2e-6)      # rsqrt(sigmoid(-l_t))
    np.testing.assert_allclose(xa[:, 13], np.exp(0.5 * lt), rtol=2e-6)
    assert np.all(xa[:, 14] == 1) and np.all(dd[:, 14] == 0)


def test_error_behaviour_mirrors_reference():
    import pytest
    with pytest.raises(NotImplementedError):
        get_logsnr_schedule("quadratic")                         # diffusion.py:96
    with pytest.raises(NotImplementedError):
        GaussianDiffusion(get_logsnr_schedule("cosine"), 10, "w", "fixed_large", "snr", "mse")   # diffusion.py:253
    d = GaussianDiffusion(get_logsnr_schedule("cosine"), 10, "v", "learned", "snr", "mse")
    with pytest.raises(NotImplementedError):
        d.sampler_config(use_ddim=False)                         # diffusion.py:161
    net = UNet(3, 64, 3, (1, 2), 1, (False, True)).eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 3, 16, 16), torch.zeros(1, dtype=torch.float64))    # no CPU fallback
    with pytest.raises(RuntimeError, match="CUDA"):
        d.p_sample(net, (1, 3, 16, 16), device="cpu", use_ddim=True)


def test_reference_init_semantics():
    torch.manual_seed(0)
    net = UNet(3, 64, 3, (1, 2), 2, (False, True), num_classes=10)
    sd = net.state_dict()
    zero = [k for k, v in sd.items() if v.ndim >= 2 and not bool(v.any())]
    # conv2 of every res block, proj_out of every attention block, the last conv (SURVEY §9.1)
    assert all(k.endswith(("conv2.weight", "proj_out.weight", "out_conv.2.weight")) for k in zero) and len(zero) > 0
    assert sd["class_embed.1.weight"].shape == (256, 10)
    w = sd["in_conv.weight"]
    assert abs(w.std().item() * (27 ** 0.5) - 0.88) < 0.1       # truncated normal at 2 sigma: std ~0.88/sqrt(fan_in)


def test_fill_with_defaults_semantics():
    cfg = {"a": None, "b": {"c": 1, "d": None}}
    fill_with_defaults(cfg, {"a": 2, "b": {"c": 3, "d": 4, "e": 5}, "f": 6})
    assert cfg == {"a": 2, "b": {"c": 1, "d": 4, "e": 5}, "f": 6}     # utils.py:204-224 demo


def test_all_schedules_match_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "coefs_T100.npz"))
    for sched in ("cosine", "linear", "sigmoid", "legacy"):
        d = GaussianDiffusion(get_logsnr_schedule(sched, -20., 20.), 50, "eps", "fixed_large", "snr", "mse")
        an = d.step_coefficients(use_ddim=False).numpy()
        np.testing.assert_allclose(an[:, 10], g[f"{sched}_logsnr_s"], rtol=2e-6, atol=1e-6)
        np.testing.assert_allclose(an[:, 11], g[f"{sched}_logsnr_t"], rtol=2e-6, atol=1e-6)
        np.testing.assert_allclose(an[:, 6], g[f"{sched}_c1"], rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(an[:, 7], g[f"{sched}_c2"], rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(an[:, 9], g[f"{sched}_logvar"], rtol=1e-5, atol=1e-6)
        # the Python-side callable (API parity with get_logsnr_schedule's closure) agrees too
        fn = get_logsnr_schedule(sched, -20., 20.)
        tt = torch.arange(50, dtype=torch.float64) / 50
        np.testing.assert_allclose(fn(tt).to(torch.float32).numpy(), g[f"{sched}_logsnr_s"], rtol=2e-6, atol=1e-6)


def test_reference_checkpoint_interop(tmp_path, golden_dir):
    """A checkpoint written in the reference's format (train_utils.py:328-348: model / ema.shadow, optionally with
    DDP's "module." prefix) loads into the drop-in UNet built from the reference's merged config."""
    import json
    from oracle.unet_ref import make_state_dict
    from tests.cases import CIFAR_COND
    from v_diffusion_b200 import build_from_config
    from v_diffusion_b200.generate import load_reference_checkpoint
    sd = make_state_dict(CIFAR_COND, 3)
    ema = {k: v * 0.5 for k, v in sd.items()}
    path = tmp_path / "ckpt_last.pt"
    torch.save({"model": {"module." + k: v for k, v in sd.items()}, "ema": {"decay": 0.9999, "shadow": ema, "num_updates": 7},
                "optimizer": {}, "scheduler": {}, "epoch": 3}, path)
    with open(os.path.join(golden_dir, "merged_configs.json")) as f:
        merged = json.load(f)["cifar10_cond"]
    config = {"data": {"name": "cifar10"}, "model": merged["model"], "diffusion": merged["diffusion"]}
    for use_ema, want in ((False, sd), (True, ema)):
        state_dict, use_cfg = load_reference_checkpoint(str(path), use_ema)
        assert use_cfg                                                  # class_embed.* present (generate.py:44)
        diffusion, model, chw = build_from_config(config, use_cfg, w_guide=1.0, sample_timesteps=100)
        model.load_state_dict(state_dict)                               # strict: same 414 keys and shapes
        assert chw == (3, 32, 32) and diffusion.model_out_type == "v" and model.num_classes == 10
        got = model.state_dict()
        assert all(torch.equal(got[k], want[k]) for k in want) and len(got) == len(want) == 414
    import pytest
    bad = dict(sd); bad.pop("in_conv.bias")
    _, model, _ = build_from_config(config, True, 1.0, 100)
    with pytest.raises(RuntimeError, match="in_conv.bias"):
        model.load_state_dict(bad)


def test_statistics_slab_layout_follows_the_conv_tiling():
    """Host logic: GroupNorm statistics slabs per image = 4 per image-aligned M tile (include/vdt_b200.h)."""
    L = _lib.lib()
    want = {32: 32, 16: 8, 64: 128, 128: 512,      # whole 128-row tiles: HW / 32
            28: 28, 14: 8,                          # ragged tiles of 112 / 98 rows: 4 slabs per tile
            8: 2,                                   # two images per tile, 64 pixels each
            7: 0, 4: 0}                             # a slab would mix two images -> no layout, two-pass GroupNorm
    for r, n in want.items():
        assert L.vdt_stat_slabs_per_image(r, r) == n, r
