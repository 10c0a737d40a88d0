"""CPU: DDIM inversion and sampling from an intermediate step.  The C library's inversion table against the fp64 formulas, the
reference inversion (tests/inversion_ref.py) pinned by a closed-form case, the reference start-k loop pinned to the oracle's
whole loop at k = T, and every refusal of the Python and C layers (no GPU work)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.diffusion_ref import logsnr_schedule
from tests.dpm_solver_ref import p_sample
from tests.inversion_ref import ddim_invert, invert_coefficients, p_sample_from
from tests.test_dpm_solver_cpu import S, _posterior_mean, _rho
from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib


def _diffusion(T=20, out="v", x0eps=False, schedule="cosine"):
    return GaussianDiffusion(get_logsnr_schedule(schedule, -20., 20.), T, out, "fixed_large", "snr_trunc", "mse", w_guide=1.0,
                             x0eps_coef=x0eps)


@pytest.mark.parametrize("T", [1, 2, 20, 100])
@pytest.mark.parametrize("schedule", ["cosine", "linear", "sigmoid", "legacy"])
def test_invert_table_matches_fp64_formulas(T, schedule):
    d = _diffusion(T, schedule=schedule)
    got = d.invert_coefficients().numpy()
    co = invert_coefficients(T, schedule)
    ddim = d.step_coefficients(True).numpy()
    # the same (s, t) pair as sampler step j, with the library's schedule evaluation (the oracle's numpy restatement differs
    # in the last bit near the linear schedule's end point)
    np.testing.assert_array_equal(got[:, 10:12], ddim[:, 10:12])
    np.testing.assert_allclose(got[:, 10], co["logsnr_s"], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(got[:, 11], co["logsnr_t"], rtol=1e-6, atol=1e-6)
    ls, lt = got[:, 10].astype(np.float64), got[:, 11].astype(np.float64)
    alpha = lambda l: np.sqrt(1.0 / (1.0 + np.exp(-l)))                       # noqa: E731
    sigma = lambda l: np.sqrt(1.0 / (1.0 + np.exp(l)))                        # noqa: E731
    c1 = sigma(lt) / sigma(ls)
    c2 = alpha(lt) - alpha(ls) * c1                                           # = -alpha_t expm1((l_s - l_t) / 2)
    np.testing.assert_allclose(got[:, 6], c1, rtol=1e-6)
    np.testing.assert_allclose(got[:, 7], c2, rtol=1e-5)
    np.testing.assert_allclose(got[:, 6], co["c1"], rtol=1e-6)
    np.testing.assert_allclose(got[:, 7], co["c2"], rtol=1e-5)
    assert np.all(got[:, 6] >= 1) and np.all(got[:, 7] <= 0)
    # the converters at l_s: row j-1 of the sampling table has them at its t = j/T, bit for bit
    conv = [0, 1, 2, 3, 4, 5, 12, 13]
    np.testing.assert_array_equal(got[1:, conv], ddim[:-1, conv])
    l0 = np.float32(logsnr_schedule(0.0, schedule))
    assert got[0, 10] == l0 and np.isclose(got[0, 0], alpha(float(l0)), rtol=1e-6)
    zero = [8, 9, 14, 15]
    assert np.all(got[:, zero] == 0)


def test_oracle_inversion_closed_form_convergence():
    """Gaussian data N(0, 0.3^2) (clamped to |x| <= 0.8 so that the sampler's clip never binds) with the exact posterior mean
    as denoiser, cosine schedule over [-20, 20].  The probability-flow ODE keeps x / rho(t) constant, so exact inversion
    from 0 to 1 is x rho(1) / rho(0) (max 2.67 here).  Measured max-abs errors of the reference inversion, and of inversion
    followed by T-step DDIM sampling against the input:

        T           10       20       40       80       160
        inversion   5.45e-1  2.84e-1  1.46e-1  7.36e-2  3.71e-2
        round trip  2.93e-1  1.61e-1  8.49e-2  4.36e-2  2.21e-2

    Both fall 1.8-2.0x per doubling of T: first order, like DDIM itself."""
    x0 = (S * torch.randn(2, 3, 8, 8, generator=torch.Generator().manual_seed(0))).clamp(-0.8, 0.8)
    exact = x0.double() * _rho(1.0) / _rho(0.0)
    Ts = (10, 20, 40, 80, 160)
    inv, rt = {}, {}
    for T in Ts:
        lat = ddim_invert(_posterior_mean, x0, None, T=T, model_out_type="x0")
        inv[T] = (lat.double() - exact).abs().max().item()
        back = p_sample(_posterior_mean, tuple(x0.shape), lat, None, T=T, model_out_type="x0", use_ddim=True)
        rt[T] = (back.double() - x0.double()).abs().max().item()
        print(f"T={T}: inversion {inv[T]:.3e}  round trip {rt[T]:.3e}")
    for a, b in zip(Ts, Ts[1:]):
        assert 1.7 < inv[a] / inv[b] < 2.2, (a, b, inv)
        assert 1.7 < rt[a] / rt[b] < 2.2, (a, b, rt)
    assert inv[160] < 0.04 and rt[160] < 0.025


def _toy(x, t, y):
    """A smooth stand-in network whose output depends on x, t and the label."""
    yv = 0. if y is None else y.double().reshape(-1, 1, 1, 1) * 0.05
    return torch.tanh(0.7 * x.double() + t.reshape(-1, 1, 1, 1) + yv).float()


@pytest.mark.parametrize("use_ddim,solver", [(True, None), (False, None), (True, "dpmpp_2m")])
def test_reference_start_step_T_is_the_whole_loop(use_ddim, solver):
    g = torch.Generator().manual_seed(3)
    x, T = torch.randn(4, 3, 8, 8, generator=g), 12
    label = torch.tensor([1, 0, 5, 2])
    sn = torch.randn((T,) + tuple(x.shape), generator=g)
    a = p_sample_from(_toy, x, label, T=T, start_step=T, model_out_type="v", w_guide=1.5, use_ddim=use_ddim, solver=solver,
                      step_noise=sn)
    b = p_sample(_toy, tuple(x.shape), x, label, T=T, model_out_type="v", w_guide=1.5, use_ddim=use_ddim, solver=solver,
                 step_noise=sn)
    assert torch.equal(a, b)


@pytest.mark.parametrize("T", [2, 10, 100])
def test_inversion_row_undoes_the_ddim_row_for_a_fixed_x0(T):
    """For a fixed x0, DDIM step j (x_t -> x_s = c1 x_t + c2 x0) and inversion step j (x_s -> c1' x_s + c2' x0) over the same
    (s, t) pair are exact inverses: c1' c1 = 1 and c1' c2 + c2' = 0, up to the fp32 rounding of each coefficient."""
    d = _diffusion(T)
    inv, ddim = d.invert_coefficients().double(), d.step_coefficients(True).double()
    assert torch.allclose(inv[:, 6] * ddim[:, 6], torch.ones(T, dtype=torch.float64), rtol=3e-7, atol=0)
    assert torch.allclose(inv[:, 6] * ddim[:, 7] + inv[:, 7], torch.zeros(T, dtype=torch.float64), rtol=0,
                          atol=1e-6 * float(inv[:, 7].abs().max()))


# ------------------------------------------------------------------ refusals
def _sc(d, **kw):
    sc = d.sampler_config(True)
    for k, v in kw.items():
        setattr(sc, k, v)
    return sc


def _c_table_refusal(sc):
    out = torch.empty((max(sc.sample_timesteps, 1), _lib.COEF_STRIDE), dtype=torch.float32)
    assert _lib.lib().vdt_invert_coefficients(C.byref(sc), _lib.ptr(out)) != 0
    return _lib.lib().vdt_last_error().decode()


def test_c_table_refusals():
    d = _diffusion(10)
    assert "use_ddim" in _c_table_refusal(_sc(d, use_ddim=0))
    assert "x0eps_coef" in _c_table_refusal(_sc(d, x0eps_coef=1))
    assert "solver" in _c_table_refusal(_sc(d, solver=1))
    assert "t_fp32" in _c_table_refusal(_sc(d, t_fp32=1))
    assert "sample_timesteps" in _c_table_refusal(_sc(d, sample_timesteps=0))
    assert _lib.lib().vdt_invert_coefficients(None, None) != 0


@pytest.fixture
def plan():
    L = _lib.lib()
    cfg = _lib.UNetConfig(in_channels=3, hid_channels=64, out_channels=3, num_levels=2, num_res_blocks=1, resolution=16,
                          max_rows=8, num_heads=1)
    cfg.ch_multipliers[0], cfg.ch_multipliers[1] = 1, 2
    p = C.c_void_p()
    _lib.check(L.vdt_plan_create(C.byref(cfg), C.byref(p)))
    yield p
    L.vdt_plan_destroy(p)


def test_c_invert_range_refusals(plan):
    """Every refusal comes before any CUDA call (the plan here is never finalized, and nothing touches a device)."""
    L = _lib.lib()
    d = _diffusion(10)
    x = torch.zeros(1, 3, 16, 16)

    def refused(sc, first, num, xp=_lib.ptr(x)):
        assert L.vdt_ddim_invert_range(plan, C.byref(sc), xp, None, 1, first, num, None) != 0
        return L.vdt_last_error().decode()
    assert "use_ddim" in refused(_sc(d, use_ddim=0), 0, 10)
    assert "x0eps_coef" in refused(_sc(d, x0eps_coef=1), 0, 10)
    assert "solver" in refused(_sc(d, solver=1), 0, 10)
    assert "t_fp32" in refused(_sc(d, t_fp32=1), 0, 10)
    for first, num in ((-1, 1), (10, 0), (0, 11), (9, 2), (3, -1)):
        assert "leave [0, 10)" in refused(_sc(d), first, num), (first, num)
    assert "null" in refused(_sc(d), 0, 1, None)
    assert "not finalized" in refused(_sc(d), 0, 10)                  # a valid range reaches the plan check


def test_c_sample_from_refusals(plan):
    L = _lib.lib()
    d = _diffusion(10)
    x = torch.zeros(1, 3, 16, 16)

    def refused(sc, first, inp=None):
        assert L.vdt_p_sample_from(plan, C.byref(sc), inp, _lib.ptr(x), None, None, 1, first, None) != 0
        return L.vdt_last_error().decode()
    for first in (-1, 10):
        assert "outside [0, 10)" in refused(_sc(d), first)
    assert "use_ddim" in refused(_sc(d, use_ddim=0, solver=1), 5)
    assert "unknown solver" in refused(_sc(d, solver=9), 5)
    assert "needs both known and mask" in refused(_sc(d), 5, C.byref(_lib.Inpaint(_lib.ptr(x), None, None)))
    assert "not finalized" in refused(_sc(d, solver=1), 5)           # 2M from an inner step needs no pred_x0


def test_c_op_invert_step_refusals():
    L = _lib.lib()
    x = torch.zeros(1, 3, 4, 4)
    row = torch.zeros(_lib.COEF_STRIDE)
    args = (_lib.ptr(x), _lib.ptr(x), _lib.ptr(x), 1, 3, 16, 0)
    assert L.vdt_op_invert_step(*args, 7, _lib.ptr(row), 0.0, None) != 0
    assert "unknown model_out_type 7" in L.vdt_last_error().decode()
    assert L.vdt_op_invert_step(*args, 3, None, 0.0, None) != 0
    assert "null" in L.vdt_last_error().decode()
    assert L.vdt_op_invert_step(_lib.ptr(x), _lib.ptr(x), _lib.ptr(x), 1, 0, 16, 0, 3, _lib.ptr(row), 0.0, None) != 0
    assert "bad image shape" in L.vdt_last_error().decode()


def test_python_refusals():
    d = _diffusion(10)
    f = lambda x, t, y: x                                                       # noqa: E731
    x = torch.zeros(1, 3, 16, 16)
    with pytest.raises(NotImplementedError, match="x0eps_coef"):
        _diffusion(10, x0eps=True).ddim_invert(f, x)
    with pytest.raises(NotImplementedError, match="x0eps_coef"):
        _diffusion(10, x0eps=True).invert_coefficients()
    for n in (-1, 11, 2.0, True):
        with pytest.raises(ValueError, match="num_steps"):
            d.ddim_invert(f, x, num_steps=n)
    with pytest.raises(RuntimeError, match="CUDA"):
        d.ddim_invert(f, x, device="cpu")
    for k in (0, 11, 5.0, False):
        with pytest.raises(ValueError, match="start_step"):
            d.p_sample(f, (1, 3, 16, 16), device="cuda", use_ddim=True, start_step=k)
    with pytest.raises(RuntimeError, match="CUDA"):
        d.p_sample(f, (1, 3, 16, 16), device="cpu", use_ddim=True, start_step=5)
