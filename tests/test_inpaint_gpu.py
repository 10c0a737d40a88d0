"""GPU: inpainting by replacement.  The fused update kernel against an fp64 step, the statistics of its own z' stream, whole
small networks against the reference loop (each in a child process, tests/inpaint_worker.py), the bit-identical properties
of the fused path, and the closed-form Gaussian case through the generic path.  Bars are the sampler's existing ones
(tests/test_gpu_unet.py)."""
import json
import os
import subprocess
import sys
import zlib

import pytest
import torch

from tests.test_dpm_solver_gpu import REL_L2, SAMPLE_MAX_ABS, VALIDATION_MAX_ABS, _step_fp64

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=1800):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "tests.inpaint_worker", *map(str, args)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=timeout)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:] + "\n" + r.stderr[-2500:])
    res = json.loads(lines[-1][len("RESULT "):])
    print(" ".join(map(str, args)), "->", json.dumps(res))
    return res


def _odd(t):
    """A device copy of ``t`` that starts 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, device="cuda")
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


def _op(L, _lib, mo, x, noise, xs, B, Cc, hw, cfg, out_type, ti, row, w, hist, known, mask, kn, seed, prev):
    _lib.check(L.vdt_op_sampler_step_known(_lib.ptr(mo), _lib.ptr(x), _lib.ptr(noise), _lib.ptr(xs), B, Cc, hw, int(cfg),
                                           _lib.OUT_TYPES[out_type], ti, _lib.ptr(row), w, _lib.ptr(hist), _lib.ptr(known),
                                           _lib.ptr(mask), _lib.ptr(kn), seed, _lib.ptr(prev), _lib.current_stream_ptr()))


@pytest.mark.parametrize("out_type", ["x0", "eps", "both", "v"])
@pytest.mark.parametrize("cfg", [False, True])
@pytest.mark.parametrize("hw,odd", [((16, 16), False), ((16, 16), True), ((5, 7), True)])   # 5 x 7: the VEC = 1 kernel
def test_sampler_step_known_kernel_vs_fp64(out_type, cfg, hw, odd):
    """A 2M row, an ancestral row with injected noise and the last step, with a soft mask and injected z'; known, mask and z'
    at 16-byte-aligned or odd offsets."""
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib
    L = _lib.lib()
    T, B, Cc, w = 20, 3, 3, 1.5
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, out_type, "fixed_large", "snr_trunc", "mse", w_guide=w)
    g = torch.Generator().manual_seed(zlib.crc32(f"{out_type}{cfg}{hw}{odd}".encode()))
    H, W = hw
    shape = (B, Cc, H, W)
    Cm = 2 * Cc if out_type == "both" else Cc
    x = torch.randn(shape, generator=g)
    mo = torch.randn((B * (2 if cfg else 1), Cm, H, W), generator=g) * 0.6
    prev = torch.rand(shape, generator=g) * 2 - 1
    known = torch.rand(shape, generator=g) * 2 - 1
    mask = torch.rand(shape, generator=g)
    mask[0, 0] = 0.0
    mask[1, 1] = 1.0
    z, zk = torch.randn(shape, generator=g), torch.randn(shape, generator=g)
    put = _odd if odd else (lambda t: t.cuda())
    mo_d, x_d, z_d, kd, md, zkd = mo.cuda(), x.cuda(), z.cuda(), put(known), put(mask), put(zk)
    for name, use_ddim, solver, ti in (("2m", True, "dpmpp_2m", 9), ("ancestral", False, None, 9), ("last", True, None, 0)):
        coefs = d.step_coefficients(use_ddim, solver)
        cf = coefs[ti].double()
        mean, pred = _step_fp64(_lib.OUT_TYPES[out_type], mo, x, coefs[ti], cfg, w, prev)
        if ti == 0:
            want = mask * known + (1 - mask) * pred
        else:
            if not use_ddim:
                mean = mean + cf[8] * z.double()
            k = coefs[ti - 1, 0].double() * known + coefs[ti - 1, 1].double() * zk
            want = mask * k + (1 - mask) * mean
        xs, hist = torch.empty(shape, device="cuda"), prev.cuda()
        _op(L, _lib, mo_d, x_d, None if use_ddim else z_d, xs, B, Cc, H * W, cfg, out_type, ti, coefs[ti].contiguous(), w,
            hist if solver else None, kd, md, zkd, 0, coefs[ti - 1].contiguous() if ti > 0 else None)
        rel = ((xs.cpu().double() - want).abs().max() / want.abs().max()).item()
        print(f"{out_type} cfg={cfg} {hw} odd={odd} {name}: x_s {rel:.2e}")
        assert rel <= 2e-6, name
        if solver:                                              # the history holds the model's guided x0, not replaced
            assert ((hist.cpu().double() - pred).abs().max() / pred.abs().max()).item() <= 1e-6
        ones, zeros = mask == 1, mask == 0
        if ti == 0:
            assert torch.equal(xs.cpu()[ones], known[ones])
        # mask 0 returns the plain step bit for bit
        plain = torch.empty_like(xs)
        _op(L, _lib, mo_d, x_d, None if use_ddim else z_d, plain, B, Cc, H * W, cfg, out_type, ti, coefs[ti].contiguous(), w,
            prev.cuda() if solver else None, None, None, None, 0, None)
        assert torch.equal(xs.cpu()[zeros], plain.cpu()[zeros])


def test_inpainting_noise_stream():
    """Mask 1 without injected z' returns alpha_s known + sigma_s z' from the library's stream: z' is standard normal, is
    uncorrelated with the ancestral draws of the same step and seed, and changes with the seed."""
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib
    L = _lib.lib()
    T, ti, B, Cc, H, W = 20, 9, 16, 4, 256, 256                             # 2^22 elements
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, "v", "fixed_large", "snr_trunc", "mse", w_guide=0.0)
    coefs = d.step_coefficients(False)
    row, prev_row = coefs[ti].contiguous(), coefs[ti - 1].contiguous()
    a, s, sd = coefs[ti - 1, 0].item(), coefs[ti - 1, 1].item(), coefs[ti, 8].item()
    shape = (B, Cc, H, W)
    g = torch.Generator(device="cuda").manual_seed(3)
    mo, x = torch.randn(shape, device="cuda", generator=g), torch.randn(shape, device="cuda", generator=g)
    known = torch.rand(shape, device="cuda", generator=g) * 2 - 1
    ones, zeros = torch.ones(shape, device="cuda"), torch.zeros(shape, device="cuda")
    hw = H * W

    def step(noise, mask, seed):
        out = torch.empty(shape, device="cuda")
        _op(L, _lib, mo, x, noise, out, B, Cc, hw, False, "v", ti, row, 0.0, None, known, mask, None, seed, prev_row)
        return out.double()
    zk = (step(None, ones, 77) - a * known.double()) / s
    z = (step(None, zeros, 77) - step(zeros, zeros, 77)) / sd               # the ancestral draws of the same step and seed
    zk2 = (step(None, ones, 78) - a * known.double()) / s
    corr = lambda u, v: (((u - u.mean()) * (v - v.mean())).mean() / (u.std() * v.std())).item()   # noqa: E731
    stats = dict(mean=zk.mean().item(), std=zk.std().item(), corr_ancestral=corr(zk, z), corr_seed=corr(zk, zk2),
                 z_std=z.std().item())
    print(stats)
    assert abs(stats["mean"]) <= 5e-3 and abs(stats["std"] - 1) <= 5e-3
    assert abs(stats["z_std"] - 1) <= 5e-3
    assert abs(stats["corr_ancestral"]) <= 5e-3 and abs(stats["corr_seed"]) <= 5e-3


@pytest.mark.parametrize("name,T,solver", [("ddim_cfg_v", 12, "none"), ("ddim_cfg_v", 12, "dpmpp_2m"),
                                           ("ancestral_x0", 10, "none"), ("ddim_cfg_multitag", 8, "dpmpp_2m")])
@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_unet_inpainting_vs_reference(name, T, solver, operand):
    """small_cond (CFG, DDIM and 2M), small_hd64_x0 (ancestral, injected step noise and z') and small_multitag: fused and
    generic inpainting against the reference loop over the oracle UNet, with a half-image box plus a random soft mask."""
    res = _run("parity", name, T, operand, solver)
    bar = SAMPLE_MAX_ABS if operand == "fp16" else VALIDATION_MAX_ABS
    assert res["finite"] and res["steps"] == T
    assert res["fused_max_abs"] <= bar and res["generic_max_abs"] <= bar, res
    assert res["worst_step_rel"] <= REL_L2, res
    assert res["fused_vs_generic"] <= 1e-5 and res["seeded_fused_vs_generic"] <= 1e-5, res
    assert res["ones_equal"], res
    assert res["differs_from_plain"] > 1e-2, res


@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_progressive_inpainting_vs_reference(operand):
    res = _run("progressive", "ddim_cfg_v", 20, operand)
    bar = SAMPLE_MAX_ABS if operand == "fp16" else VALIDATION_MAX_ABS
    for tag in ("ddim", "dpmpp_2m"):
        assert res[f"{tag}_previews"] == 6
        assert res[f"{tag}_final_max_abs"] <= bar, res
        assert res[f"{tag}_previews_max_abs"] <= bar * (1.0 + res["w_guide"]), res


def test_fused_inpainting_exactness_properties():
    res = _run("exactness")
    assert res["finite"]
    assert res["mask0_equal"], res                          # m = 0 is the plain call
    assert res["ones_equal"], res                           # m = 1 pixels are `known`
    assert res["same_seed_equal"] and res["other_seed_differs"] > 1e-3, res
    assert res["split_equal"], res                          # range calls carrying pred_x0 == one call
    assert res["repeat_fresh_equal"], res                   # a cached exec never keeps another call's known / mask
    # chunking: the existing sampler's bar (conv tiles depend on the chunk's image count); bit-identical whenever the
    # plain sampler is
    assert res["chunked_max_abs"] <= 1e-5, res
    assert res["chunked_equal"] or not res["ddim_chunked_equal"], res


def test_closed_form_case_through_the_generic_path():
    """The per-pixel Gaussian denoiser of tests/test_dpm_solver_cpu.py as a generic callable: the reference's inpainted
    trajectory to fp32 rounding, and under a binary mask the free pixels of the plain GPU run bit for bit."""
    from tests.inpaint_ref import p_sample as ref_p_sample
    from tests.test_dpm_solver_cpu import _posterior_mean
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    g = torch.Generator().manual_seed(0)
    shape, T = (2, 3, 8, 8), 20
    xT = 0.75 * torch.randn(shape, generator=g)
    known = torch.rand(shape, generator=g) * 2 - 1
    mask = (torch.rand(shape, generator=g) < 0.5).float()
    known_noise = torch.randn((T,) + shape, generator=g)
    fn = lambda x, t, y: _posterior_mean(x.cpu(), t.cpu()).cuda()           # noqa: E731
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, "x0", "fixed_large", "snr_trunc", "mse", w_guide=0.0)
    for solver in (None, "dpmpp_2m"):
        got = d.p_sample(fn, shape, noise=xT, device="cuda", use_ddim=True, solver=solver, known=known, mask=mask,
                         known_noise=known_noise)
        plain = d.p_sample(fn, shape, noise=xT, device="cuda", use_ddim=True, solver=solver)
        ref = ref_p_sample(_posterior_mean, shape, xT, None, T=T, model_out_type="x0", use_ddim=True, solver=solver, known=known,
                           mask=mask, known_noise=known_noise)
        err = (got - ref).abs().max().item()
        print(f"closed form {solver}: GPU generic path vs reference {err:.2e}")
        assert err <= 1e-5
        free = mask == 0
        assert torch.equal(got[free], plain[free]) and torch.equal(got[~free], known[~free])
