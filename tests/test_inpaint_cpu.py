"""CPU: inpainting by replacement (p_sample(..., known=, mask=)).  The reference loop (tests/inpaint_ref.py) is pinned against
the plain samplers and the closed-form per-pixel Gaussian case, and every refusal of the Python and C layers is exercised
before any device work."""
import ctypes as C

import pytest
import torch

from tests import dpm_solver_ref
from tests.inpaint_ref import p_sample
from tests.test_dpm_solver_cpu import _posterior_mean
from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib

SHAPE = (2, 3, 8, 8)


def _inputs(T, seed=0):
    g = torch.Generator().manual_seed(seed)
    xT = torch.randn(SHAPE, generator=g)
    known = torch.rand(SHAPE, generator=g) * 2 - 1
    step_noise = torch.randn((T,) + SHAPE, generator=g)
    known_noise = torch.randn((T,) + SHAPE, generator=g)
    return xT, known, step_noise, known_noise


def _linear_denoiser(x, t, y=None):
    """A smooth v-prediction stand-in that mixes pixels (so the test does not rely on independence)."""
    return 0.5 * x + 0.25 * x.roll(1, dims=3) - 0.1 * t.reshape(-1, 1, 1, 1).float()


@pytest.mark.parametrize("use_ddim,solver", [(True, None), (True, "dpmpp_2m"), (False, None)])
def test_reference_mask_zero_and_one(use_ddim, solver):
    T = 12
    xT, known, step_noise, known_noise = _inputs(T)
    kw = dict(T=T, model_out_type="v", use_ddim=use_ddim, var_type="fixed_large", step_noise=step_noise, solver=solver)
    plain = dpm_solver_ref.p_sample(_linear_denoiser, SHAPE, xT, None, **kw)
    zero = p_sample(_linear_denoiser, SHAPE, xT, None, known=known, mask=torch.zeros(SHAPE), known_noise=known_noise, **kw)
    one = p_sample(_linear_denoiser, SHAPE, xT, None, known=known, mask=torch.ones(SHAPE[:1] + (1,) + SHAPE[2:]),
                   known_noise=known_noise, **kw)
    assert torch.equal(zero, plain)
    assert torch.equal(one, known)
    assert not torch.equal(plain, known)


@pytest.mark.parametrize("solver", [None, "dpmpp_2m"])
def test_closed_form_unknown_pixels_are_untouched(solver):
    """The exact per-pixel posterior mean of N(0, 0.3^2) data treats pixels independently, so under DDIM the pixels with
    mask 0 of an inpainted run are those of the plain run bit for bit, and the pixels with mask 1 are ``known``."""
    T = 20
    xT, known, _, known_noise = _inputs(T, 1)
    mask = (torch.rand(SHAPE, generator=torch.Generator().manual_seed(2)) < 0.5).float()
    kw = dict(T=T, model_out_type="x0", use_ddim=True, solver=solver)
    plain = dpm_solver_ref.p_sample(_posterior_mean, SHAPE, xT, None, **kw)
    inp = p_sample(_posterior_mean, SHAPE, xT, None, known=known, mask=mask, known_noise=known_noise, **kw)
    free = mask == 0
    assert torch.equal(inp[free], plain[free])
    assert torch.equal(inp[~free], known[~free])


def _diffusion(T=10):
    return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, "v", "fixed_large", "snr_trunc", "mse", w_guide=1.0)


def _p_sample_raises(match, progressive=False, **kw):
    d = _diffusion()
    fn = d.p_sample_progressive if progressive else d.p_sample
    with pytest.raises(ValueError, match=match):
        fn(lambda x, t, y: x, SHAPE, device="cuda", use_ddim=True, **kw)


@pytest.mark.parametrize("progressive", [False, True])
def test_python_refusals(progressive):
    known, mask = torch.zeros(SHAPE), torch.ones(SHAPE)
    kn = torch.zeros((10,) + SHAPE)
    r = lambda match, **kw: _p_sample_raises(match, progressive, **kw)         # noqa: E731
    r("both known and mask", known=known)
    r("both known and mask", mask=mask)
    r("known_noise needs known and mask", known_noise=kn)
    r("known has shape", known=torch.zeros(2, 3, 8, 7), mask=mask)
    r("mask has shape", known=known, mask=torch.ones(2, 2, 8, 8))
    r("mask has shape", known=known, mask=torch.ones(1, 1, 8, 8))
    r("known_noise has shape", known=known, mask=mask, known_noise=torch.zeros((9,) + SHAPE))
    bad = known.clone()
    bad[1, 2, 3, 4] = float("nan")
    r("known must be finite", known=bad, mask=mask)
    bad[1, 2, 3, 4] = float("inf")
    r("known must be finite", known=bad, mask=mask)
    for v in (1.5, -0.25, float("nan")):
        m = mask.clone()
        m[0, 0, 0, 0] = v
        r(r"mask values must lie in \[0, 1\]", known=known, mask=m)
    bad_kn = kn.clone()
    bad_kn[3, 0, 0, 0, 0] = float("-inf")
    r("known_noise must be finite", known=known, mask=mask, known_noise=bad_kn)


def test_python_accepts_soft_and_channel_broadcast_masks():
    d = _diffusion()
    known = torch.zeros(SHAPE)
    for m in (torch.rand(SHAPE), torch.rand(SHAPE[:1] + (1,) + SHAPE[2:]), torch.ones(SHAPE, dtype=torch.bool)):
        got = d._check_inpaint(SHAPE, known, m, None)
        assert got[1].dtype == torch.float32
        held, ip = d._inpaint_on(got, SHAPE, "cpu")
        assert held[1].shape == SHAPE and held[1].is_contiguous() and ip.known_noise is None


def _plan():
    L = _lib.lib()
    cfg = _lib.UNetConfig(in_channels=3, hid_channels=64, out_channels=3, num_levels=2, num_res_blocks=1, resolution=16,
                          max_rows=8, num_heads=1)
    cfg.ch_multipliers[0], cfg.ch_multipliers[1] = 1, 2
    plan = C.c_void_p()
    _lib.check(L.vdt_plan_create(C.byref(cfg), C.byref(plan)))
    return L, plan


def test_c_side_pair_refusals():
    """The library refuses known without mask, mask without known and known_noise without both through vdt_last_error,
    before any device work (the plan is not even finalized)."""
    L, plan = _plan()
    try:
        sc = _diffusion().sampler_config(True)
        x = torch.zeros(1, 3, 16, 16)
        rows = _diffusion().step_coefficients(True)
        row, prev = rows[5].contiguous(), rows[4].contiguous()
        bad = [(_lib.ptr(x), None, None, "both known and mask"), (None, _lib.ptr(x), None, "both known and mask"),
               (None, None, _lib.ptr(x), "known_noise needs known and mask")]
        for known, mask, kn, msg in bad:
            ip = _lib.Inpaint(known, mask, kn)
            assert L.vdt_p_sample_range_inpaint(plan, C.byref(sc), C.byref(ip), _lib.ptr(x), None, None, 1, 9, 1, None, None) != 0
            assert msg in L.vdt_last_error().decode()
            assert L.vdt_p_sample_inpaint(plan, C.byref(sc), C.byref(ip), _lib.ptr(x), None, None, _lib.ptr(x), 1, None) != 0
            assert msg in L.vdt_last_error().decode()
            assert L.vdt_op_sampler_step_known(_lib.ptr(x), _lib.ptr(x), None, _lib.ptr(x), 1, 3, 256, 0, 3, 5, _lib.ptr(row),
                                               1.0, None, known, mask, kn, 0, _lib.ptr(prev), None) != 0
            assert msg in L.vdt_last_error().decode()
        # a step after the first needs the previous coefficient row for alpha_s, sigma_s
        assert L.vdt_op_sampler_step_known(_lib.ptr(x), _lib.ptr(x), None, _lib.ptr(x), 1, 3, 256, 0, 3, 5, _lib.ptr(row), 1.0,
                                           None, _lib.ptr(x), _lib.ptr(x), None, 0, None, None) != 0
        assert "needs coefficient row 4" in L.vdt_last_error().decode()
        # no inpainting: the call goes on to the existing checks
        ip = _lib.Inpaint(None, None, None)
        assert L.vdt_p_sample_range_inpaint(plan, C.byref(sc), C.byref(ip), _lib.ptr(x), None, None, 1, 9, 1, None, None) != 0
        assert "not finalized" in L.vdt_last_error().decode()
    finally:
        L.vdt_plan_destroy(plan)

