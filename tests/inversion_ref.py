"""Reference DDIM inversion and sampling from an intermediate step, for the tests.  Neither is in the reference repository, so
both are restated here on top of the oracle's schedule and prediction converters (oracle/diffusion_ref.py) and the
DPM-Solver reference (tests/dpm_solver_ref.py), which they do not change.

Inversion step j (0 <= j < T) maps x at s = j/T to x at t = (j+1)/T: the model sees x at fp64 time s, x0 comes from its raw
output at the fp32 log-SNR l_s without the clip (under CFG the guided x0c + w (x0c - x0u)), and
x_t = c1' x_s + c2' x0 with c1' = sigma_t / sigma_s, c2' = alpha_t - alpha_s c1' (fp64 from the fp32 log-SNRs, rounded once).

Sampling from step k runs steps k-1 ... 0 of the T-step loop on the given x (at t = k/T) as a fresh trajectory: under
DPM-Solver++(2M) step k-1 is first-order.
"""
from typing import Callable, Optional

import numpy as np
import torch

from oracle.diffusion_ref import _logsigmoid, _pred_x0, logsnr_schedule
from tests.dpm_solver_ref import step_coefficients


def invert_coefficients(T: int, schedule: str = "cosine", logsnr_min: float = -20., logsnr_max: float = 20.):
    """fp32 arrays of length T: logsnr_s, logsnr_t, c1 (= c1'), c2 (= c2'), and fp64 t_model = j/T (the model's time)."""
    i = np.arange(T, dtype=np.float64)
    s, t = i / T, (i + 1) / T
    ls32 = logsnr_schedule(s, schedule, logsnr_min, logsnr_max).astype(np.float32)
    lt32 = logsnr_schedule(t, schedule, logsnr_min, logsnr_max).astype(np.float32)
    ls, lt = ls32.astype(np.float64), lt32.astype(np.float64)
    c1 = np.exp(0.5 * (_logsigmoid(-lt) - _logsigmoid(-ls)))
    c2 = -np.exp(0.5 * _logsigmoid(lt)) * np.expm1(0.5 * (ls - lt))
    return dict(logsnr_s=ls32, logsnr_t=lt32, c1=c1.astype(np.float32), c2=c2.astype(np.float32), t_model=s)


def _cfg_inputs(x, t, label, use_cfg):
    if not use_cfg:
        return x, t, label
    yin = label.repeat_interleave(2, dim=0).clone()               # rows 2i cond, 2i+1 uncond (diffusion.py:368-372)
    yin[1::2] = 0
    return x.repeat_interleave(2, dim=0), t.repeat_interleave(2), yin


@torch.no_grad()
def ddim_invert(denoise_fn: Callable, x0: torch.Tensor, label: Optional[torch.Tensor], *, T: int, model_out_type: str,
                w_guide: float = 0., num_steps: Optional[int] = None, schedule: str = "cosine", logsnr_min: float = -20.,
                logsnr_max: float = 20., record: Optional[list] = None) -> torch.Tensor:
    """x at t = num_steps / T (None: T) from the image x0.  ``record`` collects (j, model_out)."""
    n = T if num_steps is None else num_steps
    co = invert_coefficients(T, schedule, logsnr_min, logsnr_max)
    B = x0.shape[0]
    x = x0.clone().float()
    use_cfg = (w_guide > 0) and (label is not None)
    for j in range(n):
        ls = torch.tensor(co["logsnr_s"][j])
        t = torch.full((B,), float(co["t_model"][j]), dtype=torch.float64)
        xin, tin, yin = _cfg_inputs(x, t, label, use_cfg)
        out = denoise_fn(xin, tin, yin)
        if record is not None:
            record.append((j, out.clone()))
        x0p = _pred_x0(xin, out, ls, model_out_type)               # not clipped
        if use_cfg:
            x0p = x0p[0::2] + w_guide * (x0p[0::2] - x0p[1::2])
        x = torch.tensor(co["c1"][j]) * x + torch.tensor(co["c2"][j]) * x0p
    return x


@torch.no_grad()
def p_sample_from(denoise_fn: Callable, x_k: torch.Tensor, label: Optional[torch.Tensor], *, T: int, start_step: int,
                  model_out_type: str, w_guide: float = 0., use_ddim: bool = True, solver: Optional[str] = None,
                  var_type: str = "fixed_large", intp_frac=None, step_noise: Optional[torch.Tensor] = None,
                  schedule: str = "cosine", logsnr_min: float = -20., logsnr_max: float = 20.,
                  record: Optional[list] = None) -> torch.Tensor:
    """Steps start_step-1 ... 0 of the T-step loop on x_k (x at t = start_step / T); start_step = T is the oracle's p_sample.
    ``step_noise`` (T, B, ...) indexed by step, as in the oracle."""
    co = step_coefficients(T, use_ddim, var_type, intp_frac, schedule, logsnr_min, logsnr_max, solver=solver)
    c2k = co["c2k"].copy() if solver is not None else np.zeros(T, dtype=np.float32)
    c2k[start_step - 1] = 0                                         # a fresh trajectory: no previous guided x0
    B = x_k.shape[0]
    x_t = x_k.clone().float()
    use_cfg = (w_guide > 0) and (label is not None)
    pred_prev = None
    for ti in reversed(range(start_step)):
        lt = torch.tensor(co["logsnr_t"][ti])
        t = torch.full((B,), float(co["t_model"][ti]), dtype=torch.float64)
        xin, tin, yin = _cfg_inputs(x_t, t, label, use_cfg)
        out = denoise_fn(xin, tin, yin)
        if record is not None:
            record.append((ti, out.clone()))
        x0 = _pred_x0(xin, out, lt, model_out_type).clamp(-1., 1.)
        mean = x0 if ti == 0 else torch.tensor(float(co["c1"][ti])) * xin + torch.tensor(float(co["c2"][ti])) * x0
        pred = x0
        if use_cfg:
            mc, mu = mean[0::2], mean[1::2]
            mean = mc + w_guide * (mc - mu)
            pred = x0[0::2] + w_guide * (x0[0::2] - x0[1::2])
        if c2k[ti] != 0:
            mean = mean + torch.tensor(c2k[ti]) * (pred - pred_prev)
        pred_prev = pred
        if ti > 0 and not use_ddim:
            assert step_noise is not None, "ancestral sampling needs injected step noise"
            mean = mean + torch.tensor(co["std"][ti]) * step_noise[ti]
        x_t = mean
    return x_t
