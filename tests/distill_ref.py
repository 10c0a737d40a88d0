"""Reference progressive distillation (Salimans & Ho, 2022, Algorithm 2) in fp64, for the tests.  The reference repository has
no distillation, so this restates the paper literally on top of the oracle's schedule and prediction converters
(oracle/diffusion_ref.py), which it does not change.

Student grid N, step index i: t = (i+1)/N, t' = (2i+1)/(2N), t'' = i/N.  The teacher takes two DDIM steps t -> t' -> t'' from z_t
with its (guided, clipped) x0 predictions x1 at t and x2 at t'; the target is the x0 with which one student DDIM step from z_t
lands on z_t'': x~ = (z_t'' - (sigma_t''/sigma_t) z_t) / (alpha_t'' - (sigma_t''/sigma_t) alpha_t).  The library computes the same
x~ as c_a x1 + c_b x2 (include/vdt_b200.h); ``closed_form`` gives those coefficients in fp64.
"""
import numpy as np
import torch

from oracle.diffusion_ref import _logsigmoid, _pred_x0, logsnr_schedule


def times(N, i):
    """fp64 (t, t', t'') of student step i: the sampler's grid at N and at 2N."""
    return (i + 1) / N, (2 * i + 1) / (2 * N), i / N


def logsnrs(N, i, schedule="cosine", logsnr_min=-20., logsnr_max=20.):
    """The fp32-rounded log-SNRs at (t, t', t''), as fp64 numbers."""
    return tuple(float(np.float32(logsnr_schedule(s, schedule, logsnr_min, logsnr_max))) for s in times(N, i))


def alpha_sigma(l):
    return float(np.exp(0.5 * _logsigmoid(l))), float(np.exp(0.5 * _logsigmoid(-l)))


def ddim_step(z, x0, l_from, l_to):
    """DDIM (eta = 0) from l_from to l_to with the prediction x0: alpha_to x0 + sigma_to (z - alpha_from x0) / sigma_from."""
    a0, s0 = alpha_sigma(l_from)
    a1, s1 = alpha_sigma(l_to)
    return a1 * x0 + s1 * (z - a0 * x0) / s0


def algorithm2_target(z_t, z_tpp, l_t, l_tpp):
    """The paper's target x~ = (z_t'' - (sigma_t''/sigma_t) z_t) / (alpha_t'' - (sigma_t''/sigma_t) alpha_t)."""
    a, s = alpha_sigma(l_t)
    a2, s2 = alpha_sigma(l_tpp)
    r = s2 / s
    return (z_tpp - r * z_t) / (a2 - r * a)


def two_teacher_steps(z_t, x1, x2_fn, l_t, l_tp, l_tpp):
    """z_t' = DDIM(t -> t') with x1, x2 = x2_fn(z_t'), z_t'' = DDIM(t' -> t'') with x2.  Returns (z_t', x2, z_t'')."""
    z_tp = ddim_step(z_t, x1, l_t, l_tp)
    x2 = x2_fn(z_tp)
    return z_tp, x2, ddim_step(z_tp, x2, l_tp, l_tpp)


def closed_form(l_t, l_tp, l_tpp):
    """(c_a, c_b) of x~ = c_a x1 + c_b x2, fp64 from the given log-SNRs (no t'' = 0 special case)."""
    den = np.expm1(0.5 * (l_t - l_tpp))
    return float(np.exp(0.5 * (l_tp - l_tpp)) * np.expm1(0.5 * (l_t - l_tp)) / den), float(np.expm1(0.5 * (l_tp - l_tpp)) / den)


def ddim_c1_c2(l_from, l_to):
    """fp64 c1, c2 of the DDIM step from l_from to l_to (diffusion.py:178-187 with s = the target time)."""
    c1 = np.exp(0.5 * (_logsigmoid(-l_to) - _logsigmoid(-l_from)))
    c2 = -np.exp(0.5 * _logsigmoid(l_to)) * np.expm1(0.5 * (l_from - l_to))
    return float(c1), float(c2)


def guided_x0(x, out, l, model_out_type, w, cfg):
    """The teacher's prediction in fp64: per branch from the raw output, clipped to [-1, 1], then x0c + w (x0c - x0u) under CFG
    (rows 2b conditional, 2b+1 unconditional).  ``l``: the fp32-rounded log-SNR, a scalar tensor or one per sample (B, 1, 1, 1)."""
    x, out, l = x.double(), out.double(), torch.as_tensor(l).double()
    if not cfg:
        return _pred_x0(x, out, l, model_out_type).clamp(-1., 1.)
    xc = _pred_x0(x, out[0::2], l, model_out_type).clamp(-1., 1.)
    xu = _pred_x0(x, out[1::2], l, model_out_type).clamp(-1., 1.)
    return xc + w * (xc - xu)


def distill_targets(teacher_fn, z_t, steps, y, *, N, model_out_type, w_guide=0., schedule="cosine"):
    """x~ and eps~ per sample, fp64, for the student steps ``steps`` (B,) from the literal Algorithm 2: the teacher's two DDIM
    steps from z_t, then the target formula.  At t'' = 0 the teacher's last step returns x2, and so does the target (the
    student's last step returns its x0).  Returns (x~, eps~, intermediates)."""
    B = z_t.shape[0]
    use_cfg = w_guide > 0 and y is not None
    z = z_t.double()
    steps = [int(i) for i in steps]
    trow = torch.tensor([times(N, i) for i in steps], dtype=torch.float64)
    lrow = torch.tensor([logsnrs(N, i, schedule) for i in steps], dtype=torch.float64)

    def call(x, col):
        t = trow[:, col]
        if use_cfg:
            yin = y.repeat_interleave(2, dim=0).clone()
            yin[1::2] = 0
            return teacher_fn(x.float().repeat_interleave(2, dim=0), t.repeat_interleave(2), yin)
        return teacher_fn(x.float(), t, y)
    shp = (B, 1, 1, 1)
    lt, ltp, ltpp = (lrow[:, k].reshape(shp) for k in range(3))
    a_t, s_t = torch.sigmoid(lt).sqrt(), torch.sigmoid(-lt).sqrt()
    a_tp, s_tp = torch.sigmoid(ltp).sqrt(), torch.sigmoid(-ltp).sqrt()
    a_tpp, s_tpp = torch.sigmoid(ltpp).sqrt(), torch.sigmoid(-ltpp).sqrt()
    x1 = guided_x0(z, call(z, 0), lt, model_out_type, w_guide, use_cfg)
    z_tp = a_tp * x1 + s_tp * (z - a_t * x1) / s_t
    x2 = guided_x0(z_tp, call(z_tp, 1), ltp, model_out_type, w_guide, use_cfg)
    last = torch.tensor(steps).reshape(shp) == 0
    z_tpp = torch.where(last, x2, a_tpp * x2 + s_tpp * (z_tp - a_tp * x2) / s_tp)
    r = s_tpp / s_t
    x_tgt = torch.where(last, x2, (z_tpp - r * z) / (a_tpp - r * a_t))
    eps_tgt = (z - a_t * x_tgt) / s_t
    return x_tgt, eps_tgt, dict(x1=x1, z_tp=z_tp, x2=x2, z_tpp=z_tpp, t=trow, l=lrow)
