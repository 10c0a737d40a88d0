"""Reference DPM-Solver++(2M) (Lu et al., 2022) for the tests: the solver is not in the reference repository, so it is restated
here on top of the oracle's schedule, coefficients and prediction converters (oracle/diffusion_ref.py), which it does not change.

The solver runs on the DDIM time grid t = i/T.  With lambda = l/2 and h_i = (l_s - l_t)/2 of step i (fp32-rounded log-SNRs):
  * the first step (i = T-1) is DDIM;
  * 0 < i < T-1: x_s = [guided DDIM mean] + c2k_i (pred_i - pred_{i+1}), c2k_i = c2_i h_i / (2 h_{i+1}) in fp64, rounded once;
  * the last step (i = 0) returns the guided x0, like DDIM.
pred is the guided, clipped x0 prediction: x0c + w (x0c - x0u) under CFG.
"""
from typing import Callable, Optional

import numpy as np
import torch

from oracle.diffusion_ref import _log1mexp, _logsigmoid, _pred_x0
from oracle.diffusion_ref import p_sample as _p_sample_first_order
from oracle.diffusion_ref import step_coefficients as _step_coefficients_first_order

SOLVERS = (None, "dpmpp_2m")


def _check(solver, use_ddim, x0eps_coef):
    if solver not in SOLVERS:
        raise NotImplementedError(solver)
    if solver is not None and (not use_ddim or x0eps_coef):
        raise NotImplementedError("dpmpp_2m is defined for DDIM with x0eps_coef=False only")


def step_coefficients(T: int, use_ddim: bool, var_type: str = "fixed_large", intp_frac=None, schedule: str = "cosine",
                      logsnr_min: float = -20., logsnr_max: float = 20., x0eps_coef: bool = False, t_fp32: bool = False,
                      solver: Optional[str] = None):
    """oracle.diffusion_ref.step_coefficients, plus a ``c2k`` column (fp32, 0 in rows 0 and T-1) for solver="dpmpp_2m"."""
    _check(solver, use_ddim, x0eps_coef)
    co = _step_coefficients_first_order(T, use_ddim, var_type, intp_frac, schedule, logsnr_min, logsnr_max, x0eps_coef, t_fp32)
    if solver == "dpmpp_2m":
        ls, lt = co["logsnr_s"].astype(np.float64), co["logsnr_t"].astype(np.float64)
        c2 = np.exp(_log1mexp(0.5 * (lt - ls)) + 0.5 * _logsigmoid(ls))          # alpha_s (1 - e^-h), fp64
        h = 0.5 * (ls - lt)
        c2k = np.zeros(T, dtype=np.float64)
        c2k[1:T - 1] = c2[1:T - 1] * (h[1:T - 1] / (2.0 * h[2:T]))
        co["c2k"] = c2k.astype(np.float32)
    return co


@torch.no_grad()
def p_sample(denoise_fn: Callable, shape, noise: torch.Tensor, label: Optional[torch.Tensor], *, T: int, model_out_type: str,
             w_guide: float = 0., use_ddim: bool = True, schedule: str = "cosine", logsnr_min: float = -20.,
             logsnr_max: float = 20., record: Optional[list] = None, pred_record: Optional[list] = None,
             x0eps_coef: bool = False, t_fp32: bool = False, solver: Optional[str] = None, **first_order) -> torch.Tensor:
    """oracle.diffusion_ref.p_sample for solver=None; the 2M loop above for solver="dpmpp_2m" (same record / pred_record /
    t_fp32 conventions)."""
    _check(solver, use_ddim, x0eps_coef)
    if solver is None:
        return _p_sample_first_order(denoise_fn, shape, noise, label, T=T, model_out_type=model_out_type, w_guide=w_guide,
                                     use_ddim=use_ddim, schedule=schedule, logsnr_min=logsnr_min, logsnr_max=logsnr_max,
                                     record=record, pred_record=pred_record, x0eps_coef=x0eps_coef, t_fp32=t_fp32,
                                     **first_order)
    B = shape[0]
    co = step_coefficients(T, True, schedule=schedule, logsnr_min=logsnr_min, logsnr_max=logsnr_max, t_fp32=t_fp32,
                           solver=solver)
    x_t = noise.clone().float()
    use_cfg = (w_guide > 0) and (label is not None)
    pred_prev = None
    for ti in reversed(range(T)):
        lt = torch.tensor(co["logsnr_t"][ti])
        c1, c2 = float(co["c1"][ti]), float(co["c2"][ti])
        t = torch.full((B,), float(co["t_model"][ti]), dtype=torch.float32 if t_fp32 else torch.float64)
        if use_cfg:                                   # rows 2i cond, 2i+1 uncond (diffusion.py:368-372)
            xin, tin = x_t.repeat_interleave(2, dim=0), t.repeat_interleave(2)
            yin = label.repeat_interleave(2, dim=0).clone()
            yin[1::2] = 0
        else:
            xin, tin, yin = x_t, t, label
        out = denoise_fn(xin, tin, yin)
        if record is not None:
            record.append((ti, out.clone()))
        x0 = _pred_x0(xin, out, lt, model_out_type).clamp(-1., 1.)
        mean = x0 if ti == 0 else torch.tensor(c1) * xin + torch.tensor(c2) * x0
        pred = x0
        if use_cfg:
            mc, mu = mean[0::2], mean[1::2]
            mean = mc + w_guide * (mc - mu)
            pred = x0[0::2] + w_guide * (x0[0::2] - x0[1::2])
        if pred_record is not None:
            pred_record.append((ti, pred.clone()))
        if co["c2k"][ti] != 0:
            mean = mean + torch.tensor(co["c2k"][ti]) * (pred - pred_prev)
        pred_prev = pred
        x_t = mean
    return x_t
