"""CPU: DPM-Solver++(2M) sampling (solver="dpmpp_2m").  The reference solver (tests/dpm_solver_ref.py) is pinned by a closed-form case; the C library's
coefficient slot 15 (c2k) is checked against the fp64 formula, and every refusal of the solver is exercised (no GPU work)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.diffusion_ref import logsnr_schedule
from tests.dpm_solver_ref import p_sample, step_coefficients
from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib

S = 0.3                                                  # data ~ N(0, S^2 I)


def _alpha_sigma(t):
    lam = torch.from_numpy(logsnr_schedule(t.double().numpy()))
    return torch.sigmoid(lam).sqrt(), torch.sigmoid(-lam).sqrt()


def _posterior_mean(x, t, y=None):
    """Exact E[x0 | x_t] for Gaussian data: alpha S^2 x / (alpha^2 S^2 + sigma^2)."""
    a, s = _alpha_sigma(t)
    a, s = a.reshape(-1, 1, 1, 1), s.reshape(-1, 1, 1, 1)
    return (a * S * S * x.double() / (a * a * S * S + s * s)).float()


def _rho(t):
    a, s = _alpha_sigma(torch.tensor([t], dtype=torch.float64))
    return float((a * a * S * S + s * s).sqrt())


def _closed_form_errors(T, xT):
    """Max-abs distance of the oracle's final DDIM and 2M samples from the exact one.  The probability-flow ODE keeps
    x / rho(t) constant (rho^2 = alpha^2 S^2 + sigma^2), so the exact x at t = 1/T is x_T rho(1/T) / rho(1), and the
    last step returns the posterior mean there."""
    x1 = xT.double() * _rho(1.0 / T) / _rho(1.0)
    exact = _posterior_mean(x1, torch.full((xT.shape[0],), 1.0 / T, dtype=torch.float64)).double()
    assert exact.abs().max().item() < 1.0                 # the clip never binds: the sampler sees the exact denoiser
    errs = []
    for solver in (None, "dpmpp_2m"):
        out = p_sample(_posterior_mean, tuple(xT.shape), xT, None, T=T, model_out_type="x0", use_ddim=True, solver=solver)
        errs.append((out.double() - exact).abs().max().item())
    return errs


def test_oracle_closed_form_convergence():
    """Gaussian data with the exact posterior mean as denoiser, cosine schedule over [-20, 20].  Measured max-abs errors
    (max |x_T| = 2.95; the sampler is linear in x_T here):

        T      10       20       40       80       160
        DDIM   7.82e-2  6.52e-2  4.07e-2  2.25e-2  1.18e-2
        2M     4.98e-3  1.58e-2  1.34e-2  5.97e-3  2.09e-3

    2M is 3-16x closer at every T.  Its error changes sign near T = 12 (the schedule's first and last steps are long in
    log-SNR), so the small-T ratios are pre-asymptotic; from T = 40 on, 2M falls by 2.2x then 2.9x per doubling (second
    order approaching 4x), DDIM by 1.8x then 1.9x (first order approaching 2x)."""
    xT = 0.75 * torch.randn(2, 3, 8, 8, generator=torch.Generator().manual_seed(0))     # linear ODE: any x_T
    Ts = (10, 20, 40, 80, 160)
    errs = {T: _closed_form_errors(T, xT) for T in Ts}
    for T in Ts:
        print(f"T={T}: DDIM {errs[T][0]:.3e}  2M {errs[T][1]:.3e}")
        assert errs[T][1] < 0.5 * errs[T][0]
    for a, b in ((40, 80), (80, 160)):
        ddim_ratio, m2_ratio = errs[a][0] / errs[b][0], errs[a][1] / errs[b][1]
        assert ddim_ratio < 2.0 and m2_ratio > 2.1 and m2_ratio > ddim_ratio + 0.3, (a, b, ddim_ratio, m2_ratio)


def _diffusion(T=20, out="v", x0eps=False):
    return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, out, "fixed_medium", "snr_trunc", "mse",
                             intp_frac=0.3, w_guide=1.0, x0eps_coef=x0eps)


@pytest.mark.parametrize("T", [1, 2, 3, 20, 100])
@pytest.mark.parametrize("t_fp32", [False, True])
def test_c2k_slot_matches_fp64_formula(T, t_fp32):
    d = _diffusion(T)
    def table(solver):
        sc = d.sampler_config(True, t_fp32=t_fp32, solver=solver)
        out = torch.empty((T, _lib.COEF_STRIDE), dtype=torch.float32)
        _lib.check(_lib.lib().vdt_step_coefficients(C.byref(sc), _lib.ptr(out)))
        return out.numpy()
    got, ddim = table("dpmpp_2m"), table(None)
    # every other slot is the DDIM row, bit for bit
    assert np.array_equal(got[:, :15], ddim[:, :15]) and np.all(ddim[:, 15] == 0)
    ls, lt = got[:, 10].astype(np.float64), got[:, 11].astype(np.float64)
    co = step_coefficients(T, True, t_fp32=t_fp32)
    np.testing.assert_array_equal(got[:, 10], co["logsnr_s"])
    h = 0.5 * (ls - lt)
    c2 = np.exp(np.log(-np.expm1(0.5 * (lt - ls))) + 0.5 * -np.logaddexp(0.0, -ls))     # alpha_s (1 - e^-h), fp64
    want = np.zeros(T)
    want[1:T - 1] = c2[1:T - 1] * h[1:T - 1] / (2.0 * h[2:T])
    np.testing.assert_allclose(got[:, 15], want, rtol=1e-6, atol=0)
    assert got[0, 15] == 0 and got[T - 1, 15] == 0                        # first step DDIM, last step returns x0
    if T >= 3:
        assert np.all(got[1:T - 1, 15] > 0)
    oracle = step_coefficients(T, True, t_fp32=t_fp32, solver="dpmpp_2m")["c2k"]
    np.testing.assert_allclose(got[:, 15], oracle, rtol=1e-6, atol=0)
    if not t_fp32:
        assert np.array_equal(d.step_coefficients(True, solver="dpmpp_2m").numpy(), got)


@pytest.mark.parametrize("var", ["fixed_small", "fixed_large", "fixed_medium"])
def test_slot15_is_zero_for_first_order_rows(var):
    for x0eps in (False, True):
        d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 50, "eps", var, "snr_trunc", "mse", intp_frac=0.3,
                              x0eps_coef=x0eps)
        for use_ddim in (True, False):
            assert np.all(d.step_coefficients(use_ddim).numpy()[:, 15] == 0)


def _c_refusal(sc):
    out = torch.empty((max(sc.sample_timesteps, 1), _lib.COEF_STRIDE), dtype=torch.float32)
    assert _lib.lib().vdt_step_coefficients(C.byref(sc), _lib.ptr(out)) != 0
    return _lib.lib().vdt_last_error().decode()


def test_c_side_refusals():
    d = _diffusion(10)
    sc = d.sampler_config(True)
    sc.solver = 1
    sc.use_ddim = 0
    assert "use_ddim" in _c_refusal(sc)
    sc = d.sampler_config(True)
    sc.solver, sc.x0eps_coef = 1, 1
    assert "x0eps_coef" in _c_refusal(sc)
    sc = d.sampler_config(True)
    sc.solver = 7
    assert "unknown solver 7" in _c_refusal(sc)


def test_python_refusals():
    d = _diffusion(10)
    with pytest.raises(NotImplementedError, match="use_ddim"):
        d.sampler_config(False, solver="dpmpp_2m")
    with pytest.raises(NotImplementedError, match="use_ddim"):
        d.p_sample(lambda x, t, y: x, (1, 3, 16, 16), device="cuda", use_ddim=False, solver="dpmpp_2m")
    with pytest.raises(NotImplementedError, match="use_ddim"):
        d.p_sample_progressive(lambda x, t, y: x, (1, 3, 16, 16), device="cuda", use_ddim=False, solver="dpmpp_2m")
    with pytest.raises(NotImplementedError, match="unknown solver"):
        d.step_coefficients(True, solver="dpmpp_3m")
    with pytest.raises(NotImplementedError, match="x0eps_coef"):
        _diffusion(10, x0eps=True).step_coefficients(True, solver="dpmpp_2m")
    with pytest.raises(NotImplementedError):
        step_coefficients(10, False, solver="dpmpp_2m")
    with pytest.raises(NotImplementedError):
        step_coefficients(10, True, solver="unipc")


def test_generate_driver_refuses_solver_without_ddim():
    import subprocess
    import sys
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "v_diffusion_b200.generate", "--config-path", "x.json", "--default-config-path",
                        "y.json", "--solver", "dpmpp_2m"], cwd=root, capture_output=True, text=True, timeout=300,
                       env=dict(os.environ, PYTHONPATH=root))
    assert r.returncode == 2 and "--solver dpmpp_2m needs --use-ddim" in r.stderr, r.stderr[-2000:]


def test_sub_range_without_history_is_refused():
    """A DPM-Solver++(2M) range that starts after the first step needs the previous step's guided x0 in pred_x0."""
    L = _lib.lib()
    cfg = _lib.UNetConfig(in_channels=3, hid_channels=64, out_channels=3, num_levels=2, num_res_blocks=1, resolution=16,
                          max_rows=8, num_heads=1)
    cfg.ch_multipliers[0], cfg.ch_multipliers[1] = 1, 2
    plan = C.c_void_p()
    _lib.check(L.vdt_plan_create(C.byref(cfg), C.byref(plan)))
    try:
        sc = _diffusion(10).sampler_config(True, solver="dpmpp_2m")
        x = torch.zeros(1, 3, 16, 16)
        rc = L.vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), None, None, 1, 5, 2, None, None)
        assert rc != 0 and "needs pred_x0" in L.vdt_last_error().decode()
        sc.use_ddim = 0
        assert L.vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), None, None, 1, 9, 1, None, None) != 0
        assert "use_ddim" in L.vdt_last_error().decode()
    finally:
        L.vdt_plan_destroy(plan)
