"""GPU: DDIM inversion and sampling from an intermediate step.  The fused inversion kernel against the fp64 step formula, the
closed-form Gaussian round trip through the generic path against the reference, whole small networks against the reference
inversion over the oracle UNet (each in a child process, tests/inversion_worker.py), and the bit-identical properties of the
fused paths.  Per-step model outputs hold the sampler's 1e-2 rel-L2 bar; the latent bars sit 2-5x above the worst values
measured on a B200 (profiles/r8_inversion_parity.txt)."""
import json
import os
import subprocess
import sys
import zlib

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REL_L2 = 1e-2
SAMPLE_MAX_ABS = 2e-2
VALIDATION_MAX_ABS = 1e-3
# latents relative to their max-abs value (they grow with t: c1' = sigma_t / sigma_s > 1)
LATENT_REL = {"fp16": 5e-3, "fp16x3": 5e-4}


def _run(*args, timeout=1800):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "tests.inversion_worker", *map(str, args)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=timeout)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:] + "\n" + r.stderr[-2500:])
    res = json.loads(lines[-1][len("RESULT "):])
    print(" ".join(map(str, args)), "->", json.dumps(res))
    return res


def _invert_fp64(out_type, model_out, x, coef, cfg, w, mag=False):
    """One guided inversion step in fp64 from the fp32 coefficient row: unclipped x0, x_t = c1' x + c2' x0.  mag=True: the
    same sum with every term's absolute value, the scale of the fp32 rounding error (c1' x and c2' x0 cancel to a large
    degree for v, eps and "both" at small t, where c1' >> 1)."""
    cf, x = coef.double(), x.double()
    f = torch.abs if mag else (lambda v: v)

    def x0(o):
        if out_type == 3:
            return f(x * cf[0]) - (-1 if mag else 1) * f(o * cf[1])
        if out_type == 0:
            return f(o)
        if out_type == 1:
            return f(x * cf[2]) - (-1 if mag else 1) * f(o * cf[3])
        xo, eo = o.chunk(2, dim=1)
        return f(xo * cf[5]) + (f(x * cf[2]) - (-1 if mag else 1) * f(eo * cf[3])) * cf[4]
    mo = model_out.double()
    if cfg:
        x0c, x0u = x0(mo[0::2]), x0(mo[1::2])
        pred = (1 + w) * x0c + w * x0u if mag else x0c + w * (x0c - x0u)
    else:
        pred = x0(mo)
    return f(cf[6] * x) + f(cf[7] * pred)


def _offset(t, off):
    """A copy of t whose storage starts `off` floats into a fresh buffer (off = 1: not 16-byte aligned)."""
    buf = torch.empty(t.numel() + off, device="cuda")
    v = buf[off:].view(t.shape)
    v.copy_(t)
    return v


@pytest.mark.parametrize("out_type", ["x0", "eps", "both", "v"])
@pytest.mark.parametrize("cfg", [False, True])
@pytest.mark.parametrize("hw,off", [((16, 16), 0), ((16, 16), 1), ((5, 7), 0)])   # odd offset / odd C*H*W: the scalar kernel
def test_invert_step_kernel_vs_fp64(out_type, cfg, hw, off):
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib
    L = _lib.lib()
    T, B, Cc = 20, 3, 3
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, out_type, "fixed_large", "snr_trunc", "mse", w_guide=1.5)
    coefs = d.invert_coefficients()
    g = torch.Generator().manual_seed(zlib.crc32(f"{out_type}{cfg}{hw}{off}".encode()))
    H, W = hw
    Cm = 2 * Cc if out_type == "both" else Cc
    for j in (0, 9, T - 1):                                          # t = 0 (l = 20), the middle, the last step
        x = torch.randn(B, Cc, H, W, generator=g)
        mo = torch.randn(B * (2 if cfg else 1), Cm, H, W, generator=g) * 1.5     # x0 beyond [-1, 1]: no clip may act
        want = _invert_fp64(_lib.OUT_TYPES[out_type], mo, x, coefs[j], cfg, 1.5)
        scale = _invert_fp64(_lib.OUT_TYPES[out_type], mo, x, coefs[j], cfg, 1.5, mag=True)
        mo_d, x_d = _offset(mo.cuda(), off), _offset(x.cuda(), off)
        xn = _offset(torch.zeros(B, Cc, H, W, device="cuda"), off)
        _lib.check(L.vdt_op_invert_step(_lib.ptr(mo_d), _lib.ptr(x_d), _lib.ptr(xn), B, Cc, H * W, int(cfg),
                                        _lib.OUT_TYPES[out_type], _lib.ptr(coefs[j].contiguous()), 1.5, _lib.current_stream_ptr()))
        rel = ((xn.cpu().double() - want).abs() / scale).max().item()      # error in units of the terms' magnitude
        print(f"{out_type} cfg={cfg} {hw} off={off} step {j}: {rel:.2e}")
        assert rel <= 1e-6, (j, rel)
        # in place (x_next = x)
        _lib.check(L.vdt_op_invert_step(_lib.ptr(mo_d), _lib.ptr(x_d), _lib.ptr(x_d), B, Cc, H * W, int(cfg),
                                        _lib.OUT_TYPES[out_type], _lib.ptr(coefs[j].contiguous()), 1.5, _lib.current_stream_ptr()))
        assert torch.equal(x_d, xn)


def test_closed_form_round_trip_through_the_generic_path():
    """The Gaussian closed-form denoiser of tests/test_dpm_solver_cpu.py as a generic callable on the GPU: inversion equals the
    reference inversion to fp32 rounding (amplified by c1' >> 1 in the first steps; 7e-5 measured at T = 20), and DDIM
    sampling from the latent (start_step = T, and from the halfway latent with start_step = T/2) returns the input with the
    reference's round-trip error."""
    from tests.dpm_solver_ref import p_sample as ref_p_sample
    from tests.inversion_ref import ddim_invert as ref_invert, p_sample_from as ref_sample_from
    from tests.test_dpm_solver_cpu import S, _posterior_mean
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    x0 = (S * torch.randn(2, 3, 8, 8, generator=torch.Generator().manual_seed(0))).clamp(-0.8, 0.8)
    den = lambda x, t, y: _posterior_mean(x.cpu(), t.cpu()).cuda()                     # noqa: E731
    for T in (20, 80):
        d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, "x0", "fixed_large", "snr_trunc", "mse", w_guide=0.0)
        lat = d.ddim_invert(den, x0)
        ref = ref_invert(_posterior_mean, x0, None, T=T, model_out_type="x0")
        err = ((lat - ref).abs().max() / ref.abs().max()).item()
        back = d.p_sample(den, tuple(x0.shape), noise=lat, device="cuda", use_ddim=True, start_step=T)
        ref_back = ref_p_sample(_posterior_mean, tuple(x0.shape), ref, None, T=T, model_out_type="x0", use_ddim=True)
        half = d.ddim_invert(den, x0, num_steps=T // 2)
        back_half = d.p_sample(den, tuple(x0.shape), noise=half, device="cuda", use_ddim=True, start_step=T // 2)
        ref_half = ref_sample_from(_posterior_mean, ref_invert(_posterior_mean, x0, None, T=T, model_out_type="x0",
                                                               num_steps=T // 2), None, T=T, start_step=T // 2, model_out_type="x0")
        rt, rt_ref = (back - x0).abs().max().item(), (ref_back - x0).abs().max().item()
        print(f"closed form T={T}: inversion vs reference {err:.2e} (rel), round trip {rt:.3e} (reference {rt_ref:.3e}), "
              f"halfway round trip {(back_half - x0).abs().max().item():.3e}")
        assert err <= 3e-4
        assert abs(rt - rt_ref) <= 5e-4 and (back - ref_back).abs().max().item() <= 5e-4
        assert (back_half - ref_half).abs().max().item() <= 5e-4


@pytest.mark.parametrize("name,T", [("ddim_cfg_v", 10), ("ddim_cfg_multitag", 8), ("ancestral_both", 8)])
@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_unet_inversion_vs_reference(name, T, operand):
    """small_cond (v, CFG w = 1), small_multitag (v, CFG w = 1, multi-hot labels) and small_hd64 ("both", unconditional):
    fused and generic inversion against the reference inversion over the oracle UNet, and DDIM sampling from the halfway
    latent (start_step = T/2) against the reference start-k loop."""
    res = _run("parity", name, T, operand)
    assert res["finite"] and res["steps"] == T and res["sample_steps"] == T // 2
    assert res["worst_step_rel"] <= REL_L2 and res["sample_worst_step_rel"] <= REL_L2, res
    assert res["fused_rel"] <= LATENT_REL[operand] and res["generic_rel"] <= LATENT_REL[operand], res
    assert res["fused_vs_generic"] <= 1e-5, res
    bar = SAMPLE_MAX_ABS if operand == "fp16" else VALIDATION_MAX_ABS
    assert res["sample_fused_max_abs"] <= bar and res["sample_generic_max_abs"] <= bar, res
    assert res["sample_fused_vs_generic"] <= 1e-5, res


def test_fused_exactness_properties():
    res = _run("exactness")
    assert res["finite"]
    assert res["split_equal"], res                          # [0, k) then [k, T) == [0, T)
    assert res["repeat_fresh_equal"], res                   # a cached exec reused after sampling == a fresh plan
    assert all(res["start_T_equal"]), res                   # p_sample(start_step=T) == p_sample()
    assert all(res["start_k_equal_range"]), res             # start_step=k == vdt_p_sample_range(k-1, k)
    assert res["m2_first_step_ddim_equal"], res             # under 2M the first step from k is DDIM's
    assert res["m2_differs_from_ddim"] > 1e-4, res
    # chunking: the existing sampler's chunking bar, relative to the latent's scale
    assert res["chunked_rel"] <= 1e-5 and res["chunked_sample_max_abs"] <= 1e-5, res
