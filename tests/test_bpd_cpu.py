"""CPU: the likelihood bound in bits/dim.  The library's coefficient table against the fp64 formulas, every refusal in Python
and in C, the reference's decoder against an exact-CDF bin integral, and closed-form pins of the reference bound
(tests/bpd_ref.py) on Gaussian data (no GPU work)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
from scipy.stats import norm

from oracle.diffusion_ref import _logsigmoid, logsnr_schedule
from tests.bpd_ref import LN2, bpd_coefficients, calc_all_bpd, discretized_gaussian_loglik, prior_bpd
from tests.test_dpm_solver_cpu import S, _alpha_sigma
from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib

VAR_TYPES = ["fixed_small", "fixed_large", "fixed_medium"]


def _diffusion(T=20, out="v", var="fixed_large", schedule="cosine", x0eps=False, loss="mse"):
    return GaussianDiffusion(get_logsnr_schedule(schedule, -20., 20.), T, out, var, "snr_trunc", loss, intp_frac=0.3,
                             w_guide=1.0, x0eps_coef=x0eps)


@pytest.mark.parametrize("schedule", ["cosine", "linear", "sigmoid", "legacy"])
@pytest.mark.parametrize("var", VAR_TYPES)
def test_bpd_coefficients_match_fp64_formulas(schedule, var):
    T = 50
    d = _diffusion(T, var=var, schedule=schedule)
    got = d.bpd_coefficients().numpy()
    # slots 0-13 are the ancestral table's
    np.testing.assert_array_equal(got[:, :14], d.step_coefficients(False).numpy()[:, :14])
    co = bpd_coefficients(T, var, 0.3, schedule)
    np.testing.assert_allclose(got[:, 14], co["K"], rtol=1e-6, atol=0)
    np.testing.assert_allclose(got[:, 15], co["k"], rtol=1e-6, atol=0)
    if var == "fixed_small":
        assert np.all(got[:, 14] == 0)                     # the model's variance is the true posterior's: only the means differ
    else:
        assert np.all(got[1:, 14] > 0)                     # KL of two centred Gaussians with different variances
    assert np.all(got[:, 15] > 0) and np.all(np.isfinite(got))


def _c_table_error(sc):
    out = torch.empty((max(sc.sample_timesteps, 1), _lib.COEF_STRIDE), dtype=torch.float32)
    assert _lib.lib().vdt_bpd_coefficients(C.byref(sc), _lib.ptr(out)) != 0
    return _lib.lib().vdt_last_error().decode()


def test_c_side_refusals():
    L = _lib.lib()
    d = _diffusion(10)
    sc = d.sampler_config(False)
    sc.x0eps_coef = 1
    assert "x0eps_coef" in _c_table_error(sc)
    sc = d.sampler_config(False)
    sc.t_fp32 = 1
    assert "t_fp32" in _c_table_error(sc)
    sc = d.sampler_config(False)
    sc.model_var_type = 3
    assert "model_var_type" in _c_table_error(sc)
    # every argument is checked before the first CUDA call: these fail without a device (the plan pointer is never read)
    dummy = torch.zeros(64)
    fake = _lib.ptr(dummy)
    sc = d.sampler_config(False)
    for first, num in ((-1, 1), (10, 0), (3, 8), (0, -1)):
        assert L.vdt_calc_bpd_range(fake, C.byref(sc), fake, None, None, 1, 1, first, num, fake, fake, None) != 0
        assert "leave [0, 10)" in L.vdt_last_error().decode()
    assert L.vdt_calc_bpd_range(fake, C.byref(sc), fake, None, None, 1, -2, 0, 1, fake, fake, None) != 0
    assert "batch" in L.vdt_last_error().decode()
    assert L.vdt_calc_bpd_range(None, C.byref(sc), fake, None, None, 1, 1, 0, 1, fake, fake, None) != 0
    assert "null argument" in L.vdt_last_error().decode()
    sc.x0eps_coef = 1
    assert L.vdt_calc_bpd_range(fake, C.byref(sc), fake, None, None, 1, 1, 0, 1, fake, fake, None) != 0
    assert "x0eps_coef" in L.vdt_last_error().decode()
    assert L.vdt_bpd_prior(C.byref(sc), fake, 1, 3, fake, None) != 0
    assert "x0eps_coef" in L.vdt_last_error().decode()
    row = torch.zeros(_lib.COEF_STRIDE)
    for step, T, typ in ((10, 10, 3), (-1, 10, 3), (0, 10, 4)):
        assert L.vdt_op_bpd_term(fake, fake, fake, 1, 3, 4, typ, step, T, _lib.ptr(row), 1, fake, fake, None) != 0
    assert "unknown model_out_type 4" in L.vdt_last_error().decode()


def test_python_refusals():
    with pytest.raises(NotImplementedError, match="x0eps_coef"):
        _diffusion(10, x0eps=True).calc_all_bpd(lambda x, t, y: x, torch.zeros(1, 3, 4, 4))
    with pytest.raises(NotImplementedError, match="fixed model_var_type"):
        _diffusion(10, var="learned").calc_all_bpd(lambda x, t, y: x, torch.zeros(1, 3, 4, 4))
    with pytest.raises(NotImplementedError, match="x0eps_coef"):
        _diffusion(10, x0eps=True).bpd_coefficients()
    with pytest.raises(RuntimeError, match="CUDA"):
        _diffusion(10).calc_all_bpd(lambda x, t, y: x, torch.zeros(1, 3, 4, 4), device="cpu")
    # the continuous-time training loss of the bound stays refused
    with pytest.raises(NotImplementedError, match="kl"):
        _diffusion(10, loss="kl").train_loss(lambda x, t, y: x, torch.zeros(1, 3, 4, 4), torch.zeros(1), None)


def test_decoder_matches_exact_bin_integral():
    """The tanh CDF is within 3e-4 of the normal CDF, so each bin probability is within twice that of the exact integral of
    N(mean, scale^2) over the bin; the edge bins integrate to -inf and +inf."""
    k = torch.arange(256, dtype=torch.float64)
    x = (k / 255.0 - 0.5) / 0.5
    for mean, log_scale in ((0.1, math.log(0.05)), (-0.6, math.log(0.01)), (0.97, math.log(0.02)), (0.0, math.log(0.3))):
        got = discretized_gaussian_loglik(x, torch.full_like(x, mean), torch.tensor(log_scale, dtype=torch.float64)).exp()
        sc = math.exp(log_scale)
        hi = norm.cdf((x.numpy() + 1 / 255 - mean) / sc)
        lo = norm.cdf((x.numpy() - 1 / 255 - mean) / sc)
        want = hi - lo
        want[0], want[-1] = hi[0], 1.0 - lo[-1]               # open edge bins
        err = np.abs(got.numpy() - want)
        assert err.max() <= 6e-4 + 1e-12, (mean, log_scale, err.max())
        assert abs(got.sum().item() - 1.0) <= 1e-3           # the bins partition the real line
    # bins far from the mean are clamped at 1e-12
    far = discretized_gaussian_loglik(torch.tensor([0.0]), torch.tensor([0.9]), torch.tensor(math.log(1e-3)))
    assert far.item() == pytest.approx(math.log(1e-12))


def _gaussian_x0(B, seed):
    return (S * torch.randn(B, 3, 16, 16, generator=torch.Generator().manual_seed(seed))).clamp(-1, 1)


def test_cheating_denoiser_leaves_prior_and_decoder():
    """An x0 model that returns the true x0, under fixed_small: the posterior means coincide and the variances are equal, so every
    term with i > 0 is exactly 0 and the total is the prior plus the decoder term."""
    T, B = 12, 3
    x0 = _gaussian_x0(B, 1)
    noise = torch.randn((T,) + tuple(x0.shape), generator=torch.Generator().manual_seed(2))
    total, terms, prior, mse = calc_all_bpd(lambda x, t, y: x0, x0, None, noise, T=T, model_out_type="x0", var_type="fixed_small")
    assert torch.all(terms[:, 1:] == 0) and torch.all(mse == 0)
    assert torch.equal(total, terms[:, 0] + prior)
    # lv_p(row 0) is about -20 on the +-20 cosine schedule: the decoder is a near-delta, and an exact x0_hat puts all mass in the bin
    assert terms[:, 0].abs().max().item() < 1e-6


def test_posterior_mean_mse_matches_closed_form():
    """x0 ~ N(0, S^2) and the exact posterior mean as an x0 model (fp64, no clip): x0_hat - x0 ~ N(0, S^2 sigma^2 / (alpha^2 S^2 +
    sigma^2)), so the mean of mse_i over 16 x 768 draws has a relative standard error of sqrt(2 / 12288) = 1.3 %; the bar is 5 of
    those.  Measured worst relative deviation over the 20 steps: 1.3 %."""
    T, B = 20, 16
    g = torch.Generator().manual_seed(3)
    x0 = S * torch.randn(B, 3, 16, 16, generator=g, dtype=torch.float64)
    noise = torch.randn((T,) + tuple(x0.shape), generator=g)

    def posterior_mean(x, t, y=None):
        a, s = _alpha_sigma(t)
        a, s = a.reshape(-1, 1, 1, 1), s.reshape(-1, 1, 1, 1)
        return a * S * S * x.double() / (a * a * S * S + s * s)
    _, _, _, mse = calc_all_bpd(posterior_mean, x0.float(), None, noise, T=T, model_out_type="x0", var_type="fixed_large",
                                clip_denoised=False)
    t = torch.arange(1, T + 1, dtype=torch.float64) / T
    a, s = _alpha_sigma(t)
    want = S * S * s * s / (a * a * S * S + s * s)
    rel = (mse.mean(0) / want - 1).abs()
    print("worst relative deviation of mean mse from the closed form:", rel.max().item())
    assert rel.max().item() <= 5 * math.sqrt(2 / (B * 768))


def test_prior_matches_analytic_kl():
    """prior = KL(N(alpha_1 x0, sigma_1^2) || N(0, 1)) per dimension in bits, written here from alpha_1 and sigma_1."""
    x0 = _gaussian_x0(4, 5).double()
    l1 = float(np.float32(logsnr_schedule(1.0)))
    a1 = math.sqrt(1 / (1 + math.exp(-l1)))
    s1sq = 1 / (1 + math.exp(l1))
    kl = 0.5 * ((a1 * x0) ** 2 + s1sq - 1 - math.log(s1sq))
    want = kl.flatten(1).mean(1) / LN2
    torch.testing.assert_close(prior_bpd(x0), want, rtol=1e-12, atol=1e-15)
    assert float(_logsigmoid(-l1)) == pytest.approx(math.log(s1sq), rel=1e-12)
