"""Reference inpainting loop for the tests: replacement (Song et al., 2021, App. I; RePaint without resampling) is not in the
reference repository, so the reverse loop is restated here on top of tests/dpm_solver_ref.py's coefficients and the oracle's
prediction converter (oracle/diffusion_ref.py), neither of which it changes.

After step i has produced x_s (first order or DPM-Solver++(2M), DDIM or ancestral, with CFG):
  * i > 0: x_s = m k_s + (1 - m) x_s, k_s = alpha_s known + sigma_s z'_i, alpha_s / sigma_s = alpha_t / sigma_t of row i - 1;
  * i = 0: x_0 = m known + (1 - m) x_0.
pred (the guided x0, and the 2M history) is never replaced.  z' must be injected (known_noise, indexed by step like
step_noise).  mask = None runs the plain loop.
"""
from typing import Callable, Optional

import numpy as np
import torch

from oracle.diffusion_ref import _pred_x0
from tests.dpm_solver_ref import step_coefficients


@torch.no_grad()
def p_sample(denoise_fn: Callable, shape, noise: torch.Tensor, label: Optional[torch.Tensor], *, T: int, model_out_type: str,
             known: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None,
             known_noise: Optional[torch.Tensor] = None, w_guide: float = 0., use_ddim: bool = True,
             var_type: str = "fixed_large", intp_frac=None, step_noise: Optional[torch.Tensor] = None,
             schedule: str = "cosine", logsnr_min: float = -20., logsnr_max: float = 20., record: Optional[list] = None,
             pred_record: Optional[list] = None, x0eps_coef: bool = False, t_fp32: bool = False,
             solver: Optional[str] = None) -> torch.Tensor:
    B = shape[0]
    co = step_coefficients(T, use_ddim, var_type, intp_frac, schedule, logsnr_min, logsnr_max, x0eps_coef, t_fp32, solver)
    c2k = co.get("c2k", np.zeros(T, dtype=np.float32))
    if mask is not None:
        known = known.float()
        mask = mask.float().expand(tuple(shape))
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
        xt_or_eps = xin
        if x0eps_coef:                                # eps re-derived from the clipped x0 (diffusion.py:335-343, 222-223)
            xt_or_eps = xin * torch.sigmoid(-lt).rsqrt() - x0 * (lt * 0.5).exp()
        mean = x0 if ti == 0 else torch.tensor(c1) * xt_or_eps + torch.tensor(c2) * x0
        pred = x0
        if use_cfg:
            mc, mu = mean[0::2], mean[1::2]
            mean = mc + w_guide * (mc - mu)
            pred = x0[0::2] + w_guide * (x0[0::2] - x0[1::2])
        if pred_record is not None:
            pred_record.append((ti, pred.clone()))
        if ti > 0 and not use_ddim:
            mean = mean + torch.tensor(co["std"][ti]) * step_noise[ti]
        if c2k[ti] != 0:
            mean = mean + torch.tensor(c2k[ti]) * (pred - pred_prev)
        pred_prev = pred
        if mask is not None:
            if ti > 0:
                k = torch.tensor(co["alpha_t"][ti - 1]) * known + torch.tensor(co["sigma_t"][ti - 1]) * known_noise[ti]
            else:
                k = known
            mean = mask * k + (1 - mask) * mean
        x_t = mean
    return x_t
