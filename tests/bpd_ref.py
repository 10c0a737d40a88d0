"""Reference likelihood bound in bits/dim for the tests.  The reference's own likelihood lines are not in this repository, so
the standard definition (Ho et al., 2020, section 3.3; Nichol & Dhariwal, 2021, _vb_terms_bpd / calc_bpd_loop) is restated
here on this project's time grid and coefficient table, on top of the oracle's schedule, coefficients and prediction
converters (oracle/diffusion_ref.py), which it does not change.  include/vdt_b200.h (vdt_calc_bpd_range) states the same.

Step i = 0 ... T-1 (s = i/T, t = (i+1)/T): x_t = alpha_t x0 + sigma_t eps_i (fp32, two products and a sum), the model sees x_t
at fp64 time t, x0_hat comes from its output at the fp32 log-SNR l_t (clipped iff clip_denoised), mse_i = mean (x0_hat - x0)^2.
i > 0: term_i = K_i + k_i mse_i, the KL between the true posterior and the model's, in bits per dimension.  i = 0: the 8-bit
discretized-Gaussian decoder's negative log-likelihood with log-scale lv_p(row 0) / 2.  prior = KL(q(x_1 | x0) || N(0, I)).
Everything after the model call is fp64 here but the decoder, which is defined in fp32.  Where the decoder's bins are far in the
tails (x0_hat many scales from x0) its fp32 CDF differences cancel, and one ulp of tanh moves a per-element log-likelihood by
up to the 1e-12 clamp: there the library and this restatement agree only to about 1 %.
"""
import math
from typing import Callable, Optional

import numpy as np
import torch

from oracle.diffusion_ref import _log1mexp, _logsigmoid, _pred_x0, logsnr_schedule, step_coefficients

LN2 = math.log(2.0)


def bpd_coefficients(T: int, var_type: str, intp_frac=None, schedule: str = "cosine", logsnr_min: float = -20.,
                     logsnr_max: float = 20.):
    """The oracle's ancestral coefficients plus fp32 K and k (fp64 from the fp32 log-SNRs, rounded once) and fp64 lv_p."""
    co = step_coefficients(T, False, var_type, intp_frac, schedule, logsnr_min, logsnr_max)
    ls, lt = co["logsnr_s"].astype(np.float64), co["logsnr_t"].astype(np.float64)
    l1mr = _log1mexp(lt - ls)
    lo, hi = l1mr + _logsigmoid(-ls), l1mr + _logsigmoid(-lt)
    lv_p = {"fixed_small": lo, "fixed_large": hi}.get(var_type)
    if lv_p is None:
        lv_p = lo + intp_frac * (hi - lo)
    c2 = np.exp(l1mr + 0.5 * _logsigmoid(ls))
    dlv = lv_p - lo                                   # -1 + dlv + e^(-dlv), exactly 0 for dlv = 0
    co["K"] = (0.5 * (np.expm1(-dlv) + dlv) / LN2).astype(np.float32)
    co["k"] = (0.5 * c2 * c2 * np.exp(-lv_p) / LN2).astype(np.float32)
    co["lv_p"] = lv_p
    return co


def approx_std_normal_cdf(x):
    return 0.5 * (1.0 + torch.tanh(math.sqrt(2.0 / math.pi) * (x + 0.044715 * x.pow(3))))


def discretized_gaussian_loglik(x, means, log_scale):
    """log P(bin of x) under N(means, exp(log_scale)^2), 8-bit bins of half-width 1/255 on [-1, 1], open edge bins, logs
    clamped at 1e-12 (IDDPM's discretized_gaussian_log_likelihood)."""
    c = x - means
    inv_stdv = torch.exp(-log_scale)
    cdf_plus = approx_std_normal_cdf(inv_stdv * (c + 1.0 / 255.0))
    cdf_min = approx_std_normal_cdf(inv_stdv * (c - 1.0 / 255.0))
    log_cdf_plus = torch.log(cdf_plus.clamp(min=1e-12))
    log_one_minus_cdf_min = torch.log((1.0 - cdf_min).clamp(min=1e-12))
    log_delta = torch.log((cdf_plus - cdf_min).clamp(min=1e-12))
    return torch.where(x < -0.999, log_cdf_plus, torch.where(x > 0.999, log_one_minus_cdf_min, log_delta))


def flat_mean(x):
    return x.flatten(1).mean(1)


def q_sample(x0, eps, co, i):
    """fp32 alpha_t x0 + sigma_t eps, each product rounded (as vdt_q_sample)."""
    a, s = torch.tensor(co["alpha_t"][i]), torch.tensor(co["sigma_t"][i])
    return x0.float() * a + eps.float() * s


def step_terms(out, x_t, x0, i, co, model_out_type, clip_denoised=True):
    """(term_i, mse_i) per sample in fp64 from the model output at step i."""
    lt = torch.tensor(float(co["logsnr_t"][i]), dtype=torch.float64)
    x0_hat = _pred_x0(x_t.double(), out.double(), lt, model_out_type)
    if clip_denoised:
        x0_hat = x0_hat.clamp(-1., 1.)
    x0 = x0.double()
    mse = flat_mean((x0_hat - x0) ** 2)
    if i == 0:                                        # the decoder is defined in fp32, like the reference's tensors
        ll = discretized_gaussian_loglik(x0.float(), x0_hat.float(), torch.tensor(0.5 * float(co["logvar"][0])))
        return -flat_mean(ll.double()) / LN2, mse
    return float(co["K"][i]) + float(co["k"][i]) * mse, mse


def prior_bpd(x0, schedule: str = "cosine", logsnr_min: float = -20., logsnr_max: float = 20.):
    l1 = float(np.float32(logsnr_schedule(1.0, schedule, logsnr_min, logsnr_max)))
    a2, lv1 = math.exp(float(_logsigmoid(l1))), float(_logsigmoid(-l1))
    return flat_mean(0.5 * (-1.0 - lv1 + math.exp(lv1) + a2 * x0.double() ** 2)) / LN2


@torch.no_grad()
def calc_all_bpd(denoise_fn: Callable, x0: torch.Tensor, y: Optional[torch.Tensor], noise: torch.Tensor, *, T: int,
                 model_out_type: str, var_type: str, intp_frac=None, clip_denoised: bool = True, schedule: str = "cosine",
                 logsnr_min: float = -20., logsnr_max: float = 20., record: Optional[list] = None):
    """(total [B], terms [B, T], prior [B], mse [B, T]) in fp64, eps_i = noise[i].  ``record`` collects (i, model_out)."""
    co = bpd_coefficients(T, var_type, intp_frac, schedule, logsnr_min, logsnr_max)
    B = x0.shape[0]
    terms = torch.zeros((B, T), dtype=torch.float64)
    mse = torch.zeros((B, T), dtype=torch.float64)
    for i in reversed(range(T)):
        x_t = q_sample(x0, noise[i], co, i)
        t = torch.full((B,), float(co["t_model"][i]), dtype=torch.float64)
        out = denoise_fn(x_t, t, y)
        if record is not None:
            record.append((i, out.clone()))
        terms[:, i], mse[:, i] = step_terms(out, x_t, x0, i, co, model_out_type, clip_denoised)
    prior = prior_bpd(x0, schedule, logsnr_min, logsnr_max)
    return terms.sum(1) + prior, terms, prior, mse
